"""Shared by the CPU and GPU runs of the reference's unmodified tf2_examples scripts: synthetic ../dataset/ files of the
shapes tf2_examples/dataloader.py expects, and a runner that stops the (endless) BPR script once it has printed what
the test looks for."""
import os
import signal
import subprocess
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# staged by __graft_entry__.build() (oracle/build_ref.py) where the original checkout was readable
REF_EXAMPLES = os.path.join(ROOT, "oracle", "_ref", "tf2_examples")
needs_ref_examples = pytest.mark.skipif(not os.path.exists(os.path.join(REF_EXAMPLES, "bpr_citeulike.py")),
                                        reason="original tf2_examples not staged under oracle/_ref/ by build()")

RUNNER = r"""
import sys, runpy
sys.path[:0] = [{compat!r}, {root!r}, {tests!r}, {ref!r}]
{prolog}
runpy.run_path({script!r}, run_name="__main__")
"""


def runner_code(ref_dir, script, fake_engine):
    prolog = "import fake_engine\nfake_engine.install()" if fake_engine else ""
    return RUNNER.format(compat=os.path.join(ROOT, "compat"), root=ROOT, tests=os.path.join(ROOT, "tests"), ref=ref_dir,
                         script=os.path.join(ref_dir, script), prolog=prolog)


def make_citeulike(tmp_path, n_pairs=30000):
    rng = np.random.default_rng(0)
    U, I = 5551, 16980                                    # tf2_examples/dataloader.py:22-23
    d = tmp_path / "dataset" / "citeulike"
    d.mkdir(parents=True)
    pairs = np.unique(np.stack([rng.integers(0, U, n_pairs), rng.integers(0, I, n_pairs)], 1), axis=0)
    rng.shuffle(pairs)
    raw = np.empty(len(pairs), dtype=[("user_id", np.int32), ("item_id", np.int32)])
    raw["user_id"], raw["item_id"] = pairs[:, 0], pairs[:, 1]
    np.save(d / "user_data_train.npy", raw[200:])
    np.save(d / "user_data_val.npy", raw[:120])
    np.save(d / "user_data_test.npy", raw[120:200])
    work = tmp_path / "work"
    work.mkdir()
    return work


def make_criteo(tmp_path, n=24000):
    rng = np.random.default_rng(1)
    counts = rng.integers(3, 400, 26)
    d = tmp_path / "dataset" / "criteo"
    d.mkdir(parents=True)
    np.savez(d / "kaggle_processed.npz", X_int=rng.integers(0, 100, (n, 13)), y=(rng.random(n) < 0.25).astype(np.int64),
             X_cat=np.stack([rng.integers(0, c, n) for c in counts], 1), counts=counts)   # dataloader.py:50-55
    work = tmp_path / "work"
    work.mkdir()
    return work


def run_until(cmd, cwd, needles, timeout):
    p = subprocess.Popen(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, start_new_session=True)
    os.set_blocking(p.stdout.fileno(), False)
    buf, t0 = b"", time.time()
    try:
        while time.time() - t0 < timeout:
            chunk = p.stdout.read()
            if chunk:
                buf += chunk
            if all(n in buf for n in needles):
                return buf.decode(errors="replace"), True
            if p.poll() is not None:
                break
            time.sleep(0.2)
        return buf.decode(errors="replace"), False
    finally:
        try:
            os.killpg(p.pid, signal.SIGTERM)     # the script loops forever (total_iter is unused): stop our own group
        except ProcessLookupError:
            pass
        p.wait(timeout=30)


def check_bpr_line(out):
    line = [l for l in out.replace("\r", "\n").splitlines() if l.startswith("Iter: 0")][0]
    loss = float(line.split("Loss:")[1].split(",")[0])
    auc = float(line.split("AUC:")[1].split(",")[0])
    # fresh U(-0.05,0.05) tables: BPR loss ~ log 2 = 0.69, l2 ~ 0.5*3000*50*(0.05^2/3) = 62.5; the script prints the
    # mean of the two numbers (SURVEY Q4) => ~31.6
    assert 29.0 < loss < 34.0 and 0.3 < auc < 0.7, line


def check_dlrm_line(out):
    line = [l for l in out.splitlines() if l.startswith("Iter: 0")][0]
    loss = float(line.split("Loss:")[1].split(",")[0])
    auc = float(line.split("AUC:")[1])
    # MSE of a ~0.5 sigmoid output against 25% positives; the reference's interaction is identically zero (Q1)
    assert 0.15 < loss < 0.35 and 0.3 < auc < 0.7, line
