"""Stage the original OpenRec's tf2_examples scripts into oracle/_ref/tf2_examples/ (git-ignored).

The original project's sources are not part of this repository.  `tests/test_reference_examples_cpu.py` and
`tests/test_gpu_reference_examples.py` run its UNMODIFIED example scripts against openrec_b200, and read them from
oracle/_ref/, so that no test reaches outside the tree.  `__graft_entry__.build()` calls this; where the original
checkout is not readable nothing is staged and those tests skip.  The checkout is found at $OPENREC_REFERENCE, by
default /root/reference.
    python -m oracle.build_ref"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(os.environ.get("OPENREC_REFERENCE", "/root/reference"), "tf2_examples")
DST = os.path.join(HERE, "_ref", "tf2_examples")
FILES = ("bpr_citeulike.py", "dlrm_criteo.py", "dataloader.py")


def stage():
    """-> the staged directory, or None when the original checkout is not readable."""
    if not all(os.access(os.path.join(SRC, f), os.R_OK) for f in FILES):
        return None
    os.makedirs(DST, exist_ok=True)
    for f in FILES:
        shutil.copyfile(os.path.join(SRC, f), os.path.join(DST, f))
    return DST


if __name__ == "__main__":
    d = stage()
    print(d if d else f"{SRC} not readable: nothing staged")
    sys.exit(0)
