"""Populate the git-ignored ``baseline/_ref/`` with the UNMODIFIED reference (SURVEY sec. 7 step 0).

``baseline/_ref`` is the reference install of the bench contract: it is never committed (``.gitignore``), but it
travels to the GPU box with the ``gpurun`` snapshot, which is what makes "the reference CPU path timed in the same
run" (north star) and "the unchanged example drivers on the GPU path" possible there.  Nothing is edited:

  * ``model/ road/ dmath/ example/`` are copied file by file from ``/root/reference`` (``example/_result`` --
    53 MB of published curves -- and byte-code caches are left out);
  * ``example/**/__init__.py`` are ADDED as empty files: site-packages ships an ``example.py`` that shadows the
    reference's namespace package (SURVEY 8c [probe]);
  * ``_stubs/cma.py`` and ``_stubs/matplotlib/pyplot.py`` are import stand-ins for the two packages
    ``example/inverse/_inverse.py:4,10`` imports at module top and ``solve_gd`` never touches.

    DHTS_REFERENCE=<checkout of the original project> python baseline/install_ref.py
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "_ref")
STUBS = os.path.join(REF, "_stubs")
SRC = os.environ.get("DHTS_REFERENCE", "")         # a checkout of the original project
PACKAGES = ("model", "road", "dmath", "example")


def available() -> bool:
    return os.path.isdir(os.path.join(REF, "road")) and os.path.isdir(os.path.join(REF, "example", "inverse"))


def install(force: bool = False) -> str | None:
    """Copy the reference into baseline/_ref (no-op when it is already there or the source is absent)."""
    if available() and not force:
        return REF
    if not (SRC and os.path.isdir(os.path.join(SRC, "road"))):
        return None
    os.makedirs(REF, exist_ok=True)
    for pkg in PACKAGES:
        if os.path.isdir(os.path.join(REF, pkg)):
            shutil.rmtree(os.path.join(REF, pkg))
    ignore = shutil.ignore_patterns("_result", "__pycache__", "*.pyc")
    # the contract's way first: pip-install the reference's own setup.py (from a copy under /tmp, the checkout is
    # read-only and setuptools writes build/ next to setup.py) with --target baseline/_ref ...
    tmp = tempfile.mkdtemp(prefix="dhts_ref_")
    try:
        for pkg in PACKAGES:
            shutil.copytree(os.path.join(SRC, pkg), os.path.join(tmp, pkg), ignore=ignore)
        shutil.copy(os.path.join(SRC, "setup.py"), tmp)
        r = subprocess.run([sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
                            "--find-links", "/opt/wheelhouse", "--target", REF, "--upgrade", tmp],
                           capture_output=True, text=True, cwd=tmp)
        how = "pip install --target" if r.returncode == 0 else "file copy (pip failed: %s)" % r.stderr.strip()[-200:]
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    # ... then (or instead, when pip is unavailable) a plain copy of whatever setup.py's package list left out
    # (example/sanity, example/__init__): same files, nothing edited
    for pkg in PACKAGES:
        shutil.copytree(os.path.join(SRC, pkg), os.path.join(REF, pkg), ignore=ignore, dirs_exist_ok=True)
    with open(os.path.join(REF, "INSTALL.txt"), "w") as f:
        f.write("unmodified copy of %s (%s); added: empty example/**/__init__.py, _stubs/\n" % (SRC, how))
    for root, _dirs, _files in os.walk(os.path.join(REF, "example")):
        init = os.path.join(root, "__init__.py")
        if not os.path.exists(init):
            open(init, "w").close()
    os.makedirs(os.path.join(STUBS, "matplotlib"), exist_ok=True)
    with open(os.path.join(STUBS, "cma.py"), "w") as f:
        f.write('"""Import stand-in (baseline/install_ref.py): the gradient-descent driver never calls cma."""\n')
    with open(os.path.join(STUBS, "matplotlib", "__init__.py"), "w") as f:
        f.write('"""Import stand-in (baseline/install_ref.py)."""\n')
    with open(os.path.join(STUBS, "matplotlib", "pyplot.py"), "w") as f:
        f.write('"""Import stand-in (baseline/install_ref.py): solve_gd never plots."""\n')
    return REF


def add_to_path(with_core: bool = True) -> None:
    """Put the reference install on sys.path, ahead of site-packages (whose ``example.py`` would shadow the
    reference's ``example`` package).  with_core=False is for running the reference's DRIVERS on top of the
    drop-in packages: the install then goes right BEHIND the first path entry (the drop-in directory placed there
    by ``dhts_b200.dropin.install()``), so ``road/ model/ dmath/`` keep resolving to the drop-in and only
    ``example`` and the stubs come from here."""
    assert available(), "baseline/_ref is missing: run `python baseline/install_ref.py` in the build container"
    try:
        import cma  # noqa: F401
        import matplotlib.pyplot  # noqa: F401
    except Exception:
        if STUBS not in sys.path:
            sys.path.append(STUBS)
    if REF in sys.path:
        sys.path.remove(REF)
    sys.path.insert(0 if with_core else 1, REF)


if __name__ == "__main__":
    print(install(force="--force" in sys.argv))
