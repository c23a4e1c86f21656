"""GPU: the reference's tf2_examples/bpr_citeulike.py and dlrm_criteo.py run UNMODIFIED against liborx.so -- the real
kernels behind the reference's own class surface and step protocol (north_star: "tf2_examples/*.py run unmodified").
The scripts are not part of this repo: build() stages them into the git-ignored oracle/_ref/ (oracle/build_ref.py)
where the original checkout is readable, and these tests skip where it staged nothing."""
import subprocess
import sys

import pytest

from _examples_common import (REF_EXAMPLES, check_bpr_line, check_dlrm_line, make_citeulike, make_criteo,
                              needs_ref_examples, run_until, runner_code)

pytestmark = [pytest.mark.gpu, needs_ref_examples]


def test_bpr_citeulike_runs_unmodified_on_gpu(tmp_path):
    work = make_citeulike(tmp_path)
    out, ok = run_until([sys.executable, "-c", runner_code(REF_EXAMPLES, "bpr_citeulike.py", False)], str(work),
                        [b"Iter: 0, Loss:", b"3 iter training."], 600)
    assert ok, out[-3000:]
    check_bpr_line(out)


def test_dlrm_criteo_runs_unmodified_on_gpu(tmp_path):
    work = make_criteo(tmp_path)
    r = subprocess.run([sys.executable, "-c", runner_code(REF_EXAMPLES, "dlrm_criteo.py", False)], cwd=str(work),
                       capture_output=True, text=True, timeout=900)
    out = (r.stdout + r.stderr).replace("\r", "\n")
    assert r.returncode == 0, out[-3000:]
    check_dlrm_line(out)
