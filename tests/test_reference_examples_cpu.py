"""CPU: the reference's tf2_examples/bpr_citeulike.py and dlrm_criteo.py run UNMODIFIED against
openrec_b200's `openrec.tf2` + `tensorflow` surfaces (compat/).  The scripts are read from oracle/_ref/ (staged there by
build(), see oracle/build_ref.py), fed synthetic files under ../dataset/, and the liborx engine is replaced by the
oracle-backed stand-in of tests/fake_engine.py (no GPU here).  What this pins is the host side: import paths,
constructor/kwarg surface, sampler workers, the GradientTape -> apply_gradients step protocol, evaluation generator,
metrics, printing.  Skipped where build() staged nothing; the same scripts on the real kernels:
tests/test_gpu_reference_examples.py."""
import subprocess
import sys

from _examples_common import (REF_EXAMPLES, check_bpr_line, check_dlrm_line, make_citeulike, make_criteo,
                              needs_ref_examples, run_until, runner_code)

pytestmark = needs_ref_examples


def test_bpr_citeulike_runs_unmodified(tmp_path):
    work = make_citeulike(tmp_path)
    out, ok = run_until([sys.executable, "-c", runner_code(REF_EXAMPLES, "bpr_citeulike.py", True)], str(work),
                        [b"Iter: 0, Loss:", b"3 iter training."], 600)
    assert ok, out[-3000:]
    check_bpr_line(out)


def test_dlrm_criteo_runs_unmodified(tmp_path):
    """tf2_examples/dlrm_criteo.py: tf.data pipeline -> DLRM under GradientTape -> Adam -> keras AUC.
    The script makes one pass over its (here: small synthetic) training slice and exits by itself."""
    work = make_criteo(tmp_path)
    r = subprocess.run([sys.executable, "-c", runner_code(REF_EXAMPLES, "dlrm_criteo.py", True)], cwd=str(work),
                       capture_output=True, text=True, timeout=900)
    out = (r.stdout + r.stderr).replace("\r", "\n")
    assert r.returncode == 0, out[-3000:]
    check_dlrm_line(out)
