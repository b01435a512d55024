"""Compiles the original HR-VITON modules into oracle/_ref/ (git-ignored): every .py of a checkout of sangyun884/HR-VITON is
byte-compiled to a sourceless .pyc at the same relative path, which Python imports like the module itself.  The reference's own
training scripts (tests/test_reference_scripts_gpu.py) and bench.py's reference arms run from there on machines that have the built
tree but no checkout.  __graft_entry__.build() calls build(); without a checkout it leaves oracle/_ref/ as it is.

    python oracle/build_reference.py [checkout]      (default: $HRV_REFERENCE_DIR, else /root/reference)
"""
import os
import py_compile
import shutil
import sys

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def default_checkout():
    return os.environ.get("HRV_REFERENCE_DIR") or "/root/reference"


def build(src=None):
    """Returns OUT when it holds the compiled modules, None when there is neither a checkout nor an earlier build."""
    src = src or default_checkout()
    if not os.path.isfile(os.path.join(src, "train_generator.py")):
        return OUT if os.path.isfile(os.path.join(OUT, "train_generator.pyc")) else None
    tmp = OUT + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    for dirpath, dirnames, filenames in os.walk(src):
        dirnames[:] = sorted(d for d in dirnames if not d.startswith(".") and d not in ("__pycache__", "figures", "data"))
        rel = os.path.relpath(dirpath, src)
        for f in sorted(filenames):
            if f.endswith(".py"):
                py_compile.compile(os.path.join(dirpath, f), cfile=os.path.join(tmp, rel, f + "c"),
                                   dfile=os.path.normpath(os.path.join("HR-VITON", rel, f)), doraise=True)
    shutil.rmtree(OUT, ignore_errors=True)
    os.replace(tmp, OUT)
    return OUT


if __name__ == "__main__":
    print(build(sys.argv[1] if len(sys.argv) > 1 else None))
