"""TEST INFRASTRUCTURE ONLY -- builds oracle/philox_sampler.c with gcc and stages the reference for the CPU arm.

``build()``      the CPU replay of the Philox sampler stream -> ``oracle/_build/liboracle.so``.
``build_ref()``  the reference is pure Python, so "building" it means staging the UNMODIFIED hot-path modules
                 (pmgt/pmgt/{datasets,models,modeling_pmgt,configuration_pmgt,utils}.py, pmgt/optimizers.py and the
                 two package __init__ files) from the upstream checkout ``ref_shim`` finds (``PMGT_REFERENCE_ROOT``, or
                 an importable ``pmgt`` package) into the git-ignored ``oracle/_ref/``.  That directory is build output:
                 it never enters the history, but a copy of the tree that carries it lets ``bench.py --impl reference``
                 and the ``cpu_baseline`` leg time the reference's OWN sampler and model code on the host cores
                 (``kind: "reference"``) instead of the oracle port.  Without a checkout an existing staged copy is used
                 as is.
"""
import ctypes
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "philox_sampler.c")
OUT_DIR = os.path.join(HERE, "_build")
OUT = os.path.join(OUT_DIR, "liboracle.so")


def build(force: bool = False) -> str:
    os.makedirs(OUT_DIR, exist_ok=True)
    if force or not os.path.exists(OUT) or os.path.getmtime(OUT) < os.path.getmtime(SRC):
        subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-std=c99", "-o", OUT, SRC])
    return OUT


REF_OUT = os.path.join(HERE, "_ref")
REF_FILES = ["pmgt/__init__.py", "pmgt/optimizers.py", "pmgt/pmgt/__init__.py", "pmgt/pmgt/datasets.py",
             "pmgt/pmgt/models.py", "pmgt/pmgt/modeling_pmgt.py", "pmgt/pmgt/configuration_pmgt.py", "pmgt/pmgt/utils.py"]


def build_ref(force: bool = False) -> str:
    """Stage the reference's hot-path modules into ``oracle/_ref/`` (byte-for-byte copies); returns the directory, or
    "" when neither the reference tree nor a staged copy is available."""
    import shutil

    from oracle.ref_shim import REFERENCE_ROOT as REF_ROOT

    if REF_ROOT and os.path.isdir(os.path.join(REF_ROOT, "pmgt", "pmgt")):
        for rel in REF_FILES:
            src, dst = os.path.join(REF_ROOT, rel), os.path.join(REF_OUT, rel)
            os.makedirs(os.path.dirname(dst), exist_ok=True)
            if force or not os.path.exists(dst) or os.path.getmtime(dst) < os.path.getmtime(src):
                shutil.copyfile(src, dst)
    return REF_OUT if os.path.isdir(os.path.join(REF_OUT, "pmgt", "pmgt")) else ""


_lib = None


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(OUT):
            build()
        _lib = ctypes.CDLL(OUT)
    return _lib


if __name__ == "__main__":
    print(build(force=True))
    print(build_ref(force=True) or "(reference tree not present: oracle/_ref not staged)")
