"""ctypes binding of libdhts_b200.so (the C ABI declared in include/dhts.h).

There is NO fallback: if the shared library is missing or a symbol does not
resolve, importing / calling fails loudly.  Every call passes raw device
pointers of torch tensors plus torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libdhts_b200.so")

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA = 0, 1, 2, 3
FLAG_CFL, FLAG_NAN_GRAD, FLAG_COLLISION, FLAG_ROUTE, FLAG_VEH_OVERFLOW = 1, 2, 4, 8, 16
_ERR = {ERR_INVALID: "invalid argument", ERR_UNSUPPORTED: "unsupported shape for the fused kernel",
        ERR_CUDA: "CUDA launch failed"}

# every exported symbol of include/dhts.h; tests/test_cabi.py checks this list against the header
SYMBOLS = [
    "dhts_version", "dhts_fp64_probe", "dhts_csr_expand", "dhts_idm_rollout_max_lane", "dhts_idm_rollout_max_ckpt_every", "dhts_hyb_aux_size",
] + [f"dhts_{op}_{suf}" for suf in ("f64", "f32") for op in (
    "arz_step_fwd", "arz_step_bwd", "arz_rollout_fwd", "arz_rollout_scratch_elems", "arz_rollout_ckpt_elems", "arz_rollout_bwd",
    "idm_step_fwd", "idm_step_bwd", "idm_step_bwd_params", "idm_rollout_fwd", "idm_rollout_bwd", "idm_rollout_bwd_params",
    "m2c_fwd", "m2c_bwd", "c2m_fwd", "c2m_bwd", "net_rollout_fwd", "net_rollout_bwd", "hyb_rollout_fwd", "hyb_rollout_bwd")]

_lib = None


class UnsupportedShape(RuntimeError):
    """The fused kernel cannot take this shape; callers step with the per-step kernels instead."""


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for the simulation step)")
        lib = ctypes.CDLL(SO_PATH)
        for name in SYMBOLS:
            fn = getattr(lib, name)      # AttributeError if the ABI is incomplete
            fn.restype = ctypes.c_longlong if ("_elems" in name or name == "dhts_fp64_probe") else ctypes.c_int
        _lib = lib
    return _lib


def suffix(dtype: torch.dtype) -> str:
    if dtype == torch.float64:
        return "f64"
    if dtype == torch.float32:
        return "f32"
    raise TypeError(f"dhts kernels are built for float64 / float32, got {dtype}")


def creal(dtype: torch.dtype, x: float):
    return ctypes.c_double(x) if dtype == torch.float64 else ctypes.c_float(x)


def ptr(t):
    if t is None:
        return ctypes.c_void_p(0)
    assert t.is_cuda and t.is_contiguous(), "dhts kernels take contiguous CUDA tensors"
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def check(rc: int, what: str):
    if rc == OK:
        return
    if rc == ERR_UNSUPPORTED:
        raise UnsupportedShape(f"{what}: {_ERR[rc]}")
    raise RuntimeError(f"{what}: {_ERR.get(rc, 'error %d' % rc)}")


def require_cuda(*tensors):
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("the dhts simulation step runs on CUDA only (no CPU fallback); got a CPU tensor")
        dev = dev or t.device
        if t.device != dev:
            raise RuntimeError("all tensors of one call must live on the same CUDA device")
    return dev


class Flags:
    """Device-side condition flags of a rollout, mapped to the reference's error conventions."""

    def __init__(self, device):
        self.t = torch.zeros(4, dtype=torch.int32, device=device)

    def reset(self):
        self.t.zero_()

    def read(self):
        v = self.t.cpu().tolist()
        return v[0], v[1]

    def check(self, quiet_collisions: bool = False):
        bits, ncol = self.read()
        # road/lane/_macro_lane.py:141-146
        assert not (bits & FLAG_CFL), "Time step size does not meet CFL condition. Please try smaller delta_time."
        # road/lane/dmacro_lane.py:308
        assert not (bits & FLAG_NAN_GRAD), ""
        if bits & FLAG_VEH_OVERFLOW:
            raise RuntimeError("hybrid network rollout: a vehicle ring, spawn-route list or deposit log overflowed "
                               "(raise veh_cap / max_spawn)")
        if bits & FLAG_ROUTE:
            # road/network/road_network.py:332-339: self.lane[-1] when the step's MacroRoute selects no neighbour
            raise KeyError(-1)
        if (bits & FLAG_COLLISION) and not quiet_collisions:
            # road/lane/_micro_lane.py:155-160 prints and continues
            print("Collision detected (%d vehicle-steps)" % ncol)
            print("Set deltas to 0, but please check traffic flow for unrealistic behavior...")
        return bits, ncol
