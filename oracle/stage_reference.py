"""Byte-compile the original FactorVAE project's Python files into oracle/_ref/ (git-ignored): module.pyc, main.pyc,
train_model.pyc, dataset.pyc, utils.pyc.  Python imports a sourceless .pyc found on sys.path, so these serve two checkers
without any of the original sources entering the tree: `bench.py --impl reference` and bench.py's CPU / eager baselines (kind
"reference": the unmodified module.py) and tests/test_dropin_reference_drivers_gpu.py (the unmodified drivers on dropin/).

__graft_entry__.build() calls stage() where the original project is present: FVAE_REFERENCE_DIR, else /root/reference (where
the golden-vector generators under oracle/ read it too).  Elsewhere it does nothing, and the checkers fall back or skip.
The .pyc files are tied to the Python minor version that compiled them; run build() with the interpreter that will load them.

    python oracle/stage_reference.py [original project directory]
"""
import os
import py_compile
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
REF_FILES = ("module.py", "train_model.py", "main.py", "dataset.py", "utils.py")


def reference_dir() -> str:
    return os.environ.get("FVAE_REFERENCE_DIR", "/root/reference")


def stage(src_dir=None) -> bool:
    """Compile every file of REF_FILES found in src_dir into OUT; returns False (and leaves OUT alone) when src_dir does not
    hold the original project's module.py or cannot be read."""
    src_dir = src_dir or reference_dir()
    if not os.access(os.path.join(src_dir, "module.py"), os.R_OK):
        return False
    os.makedirs(OUT, exist_ok=True)
    for f in REF_FILES:
        src = os.path.join(src_dir, f)
        if os.path.exists(src):
            py_compile.compile(src, cfile=os.path.join(OUT, f[:-3] + ".pyc"), dfile=f, doraise=True)
    return True


if __name__ == "__main__":
    ok = stage(sys.argv[1] if len(sys.argv) > 1 else None)
    print(OUT if ok else "no original project found; nothing staged")
