"""Host-side ARZ records and closures of the drop-in API.

Only what callers of the reference touch lives here: the per-cell record ``ARZ.FullQ`` /
``ARZ.Q`` and the scalar closures u_eq, u, y (reference: model/macro/_arz.py:1-149).  They
accept Python floats or tensors (any shape, any device) and are differentiated by autograd
with the TRUE derivative, as the reference's 0-dim tensor arithmetic is.  The Riemann solver
and its Jacobians (_arz.py:155-332, darz.py) are NOT here: they run inside the CUDA kernels
(diff-hybrid-traffic-sim_b200/csrc/dhts_arz_lean.cuh).
"""
import math

import torch

GAMMA = 0.5
EPSILON = 1e-5


def _is_t(x):
    return isinstance(x, torch.Tensor)


def _floor_at(x, lo):
    """max(x, lo) the way Python's max treats a tensor: pass x (and its gradient) when x > lo."""
    if _is_t(x):
        return torch.clamp(x, min=lo)
    return x if x > lo else lo


def _pow(x, e):
    if _is_t(x):
        return torch.sqrt(x) if e == 0.5 else torch.pow(x, e)
    return math.sqrt(x) if e == 0.5 else math.pow(x, e)


class ARZ:
    class Q:
        """(density r, relative flow y) of a cell."""

        def __init__(self, r=0, y=0):
            self.r = r
            self.y = y

        @staticmethod
        def from_r_y(r, y):
            return ARZ.Q(r, y)

        @staticmethod
        def from_r_u(r, u, u_max):
            return ARZ.Q(r, ARZ.compute_y(r, u, u_max))

        def __mul__(self, c):
            return ARZ.Q(self.r * c, self.y * c)

        def __add__(self, o):
            return ARZ.Q(self.r + o.r, self.y + o.y)

        def __sub__(self, o):
            return ARZ.Q(self.r - o.r, self.y - o.y)

        def clear(self):
            self.r, self.y = 0, 0

    class FullQ:
        """Q plus the speed u and equilibrium speed u_eq STORED on the cell (the step reads the stored
        values, it does not re-derive them: SURVEY.md App. B.3)."""

        def __init__(self, u_max):
            self.q = ARZ.Q()
            self.u_max = u_max
            self.u = u_max
            self.u_eq = u_max

        @staticmethod
        def from_q(q, u_max):
            s = ARZ.FullQ(u_max)
            s.q = q
            s.u = ARZ.compute_u(q.r, q.y, u_max)
            s.u_eq = ARZ.compute_u_eq(q.r, u_max)
            return s

        @staticmethod
        def from_r_u(r, u, u_max):
            s = ARZ.FullQ(u_max)
            s.set_r_u(r, u, u_max)
            return s

        def set_r_u(self, r, u, u_max):
            self.u_max = u_max
            self.u_eq = ARZ.compute_u_eq(r, u_max)
            self.q = ARZ.Q(r, r * (u - self.u_eq))
            self.u = u

        def set_r_y(self, r, y, u_max):
            self.u_max = u_max
            self.q = ARZ.Q(r, y)
            self.u = ARZ.compute_u(r, y, u_max)
            self.u_eq = ARZ.compute_u_eq(r, u_max)

        def flux_r(self):
            return self.q.r * self.u

        def flux_y(self):
            return self.q.y * self.u

        def flux(self):
            return ARZ.Q(self.flux_r(), self.flux_y())

        def lambda_0(self):
            return self.u + self.q.r * ARZ.compute_u_eq_prime(self.q.r, self.u_max)

        def lambda_1(self):
            return self.u

        def __sub__(self, o):
            return ARZ.FullQ.from_q(self.q - o.q, self.u_max)

        def clear(self):
            self.q.clear()
            self.u = self.u_max
            self.u_eq = self.u_max

    @staticmethod
    def compute_u_eq(r, u_max, gamma=GAMMA):
        return u_max * (1.0 - _pow(_floor_at(r, 0.0) + EPSILON, gamma))

    @staticmethod
    def compute_u_eq_prime(r, u_max, gamma=GAMMA):
        return -u_max * gamma * _pow(_floor_at(r, EPSILON), gamma - 1)

    @staticmethod
    def compute_y(r, u, u_max):
        return r * (u - ARZ.compute_u_eq(r, u_max))

    @staticmethod
    def compute_u(r, y, u_max):
        rc = _floor_at(r, EPSILON)
        return y / rc + ARZ.compute_u_eq(rc, u_max)

    @staticmethod
    def compute_r_from_u_eq(u_eq, u_max, gamma=GAMMA):
        return _pow(1.0 - u_eq / _floor_at(u_max, EPSILON), 1.0 / _floor_at(gamma, EPSILON))

    @staticmethod
    def riemann_solve(*_a, **_k):
        raise NotImplementedError("the Riemann solver of this build runs inside the CUDA step "
                                  "(dhts_arz_step_fwd_*; pass want_case=True for the outcome per interface)")
