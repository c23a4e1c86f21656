#!/usr/bin/env python
"""bench.py -- the openrec.tf2 training step on B200: BPR (headline), UCML, DLRM; roofline + CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload bpr|ucml|dlrm] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (BASELINE.json configs): bpr = configs[1] (N = 1) / configs[4] shape (N > 1), ucml = configs[2],
dlrm = configs[3].  A "step" = one pass of the hot path over one batch of synthetic input:
  bpr / ucml : gather -> score -> loss -> sparse gradient -> dedup -> Adagrad over 65 536 triplets against 1M x 128 user /
               item tables (ucml: + censor_vec, the three LatentFactor.censor calls of its training loop);
  dlrm       : 26 embedding gathers -> bottom MLP -> pairwise interaction -> top MLP -> MSE -> backward -> Adagrad (sparse
               for the 26 x 1M x 128 tables, dense for the MLPs), batch 32 768.

 value : whole-job units/s, inputs already resident in HBM, liborx called as directly as the path allows.
 e2e   : the same metric through the public API a user calls (openrec.tf2 model + GradientTape + optimizer.apply_gradients),
         inputs copied from pinned HOST memory and the loss read back to the host every step, inside the timed region.
 roofline : the dominant kernel timed live with CUDA events on its launch stream (a dedicated instrumented loop of the
         same step right after the timed region, so that the event records do not sit inside it).
 cpu_baseline / --impl reference : the CPU restatement of the reference step on the box's host cores
         (oracle/: C+OpenMP port for the pairwise steps, numpy/BLAS oracle for DLRM; TensorFlow is not installable here).
At N = 1 the default (bpr) line also carries the ucml and dlrm lines, same schema, under "secondary".
Prints exactly ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

U = I = 1_000_000
D = 128
B = 65_536
N_BATCHES = 16
LR = 0.05
# SURVEY 8(d): bytes/triplet = 12 + 4*(3D+2)*(2+2S); Adagrad S=1, D=128 -> 6188
ALG_BYTES_PER_TRIPLET = 12 + 4 * (3 * D + 2) * (2 + 2 * 1)
METRICS = {"bpr": ("bpr_triplets_per_sec", "triplets/s"), "ucml": ("ucml_triplets_per_sec", "triplets/s"),
           "dlrm": ("dlrm_samples_per_sec", "samples/s")}
# DLRM (configs[3]); the MLP widths are this repo's choice (MLPerf-DLRM-like), BASELINE.json leaves them open
DLRM_T, DLRM_VOCAB, DLRM_B, DLRM_DENSE = 26, 1_000_000, 32_768, 13
DLRM_BOT, DLRM_TOP = [512, 256, D], [1024, 1024, 512, 256, 1]
DLRM_LR = 0.01
# --dump-outputs: rows sampled from each 1M-row table, so that the three workloads together stay under DUMP_LIMIT
# (BPR and UCML 2 MB per table, DLRM 26 x 0.5 MB of tables + 9 MB of MLP weights)
DUMP_ROWS, DLRM_DUMP_ROWS = 4096, 1024
DUMP_LIMIT = 64 << 20


def dlrm_layers():
    P = (DLRM_T + 1) * DLRM_T // 2
    dims = [(DLRM_DENSE, DLRM_BOT[0])] + list(zip(DLRM_BOT[:-1], DLRM_BOT[1:]))
    dims += [(D + P, DLRM_TOP[0])] + list(zip(DLRM_TOP[:-1], DLRM_TOP[1:]))
    return dims


def dlrm_flops_per_sample():
    """fwd + dgrad + wgrad of the Dense layers, and the interaction's batched Z Z^T (fwd) + its two backward products."""
    mlp = 3 * 2 * sum(i * o for i, o in dlrm_layers())
    return mlp + 3 * 2 * (DLRM_T + 1) ** 2 * D


def workload_name(wl, n_gpus):
    if wl == "dlrm":
        return (f"DLRM {DLRM_T} sparse features x {DLRM_VOCAB} vocab x dim {D}, {DLRM_DENSE} dense, batch {DLRM_B}, bottom MLP "
                f"{DLRM_DENSE}-{'-'.join(map(str, DLRM_BOT))}, top MLP {D + (DLRM_T + 1) * DLRM_T // 2}-{'-'.join(map(str, DLRM_TOP))}, "
                f"MSE, Adagrad lr {DLRM_LR}, interaction_mode=dlrm (strictly-lower triangle; the reference's own interaction "
                "is identically zero, SURVEY Q1), ids uniform i.i.d., 4 rotating batches")
    items = I if n_gpus == 1 else 12_500_000 * n_gpus          # BASELINE configs[1] / configs[4] (100M items on 8 GPUs)
    name = "BPR" if wl == "bpr" else "UCML (margin 0.5, + censor_vec)"
    s = (f"{name} {U} users x {items} items, dim {D}, batch {B} per GPU, Adagrad lr {LR} (acc init 0.1), "
         f"ids uniform i.i.d. int32, {N_BATCHES} rotating id batches")
    if n_gpus > 1:
        mode = os.environ.get("ORX_SHARDED", "home")
        how = {"home": "home-routed: a triplet is computed on the rank owning its user row; item rows and item gradient rows "
                       "travel as peer stores into IPC-mapped mailboxes over NVLink (no collective in the step)"}.get(
                           mode, "NCCL all-to-all exchange of counts / ids / rows / gradient rows")
        s += f", user and item tables row-sharded over {n_gpus} GPUs (row r on rank r % N, 12.5M item rows per GPU); {how}"
    return s


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1500.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------
# clocks: a separate process polls NVML so the timed Python loop keeps the GIL.  It is started before torch is imported
# and the bench waits for its first sample, so that even a 2 ms timed region has samples around it.
# ---------------------------------------------------------------------------------------
_CLOCK_SRC = r"""
import sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
out = open(sys.argv[2], "w")
mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
while True:
    try:
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
    except Exception:
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
    out.write("%f %d %d %d\n" % (time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), mx, r))
    out.flush()
    time.sleep(0.002)
"""
_REASONS = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
            0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
            0x100: "display_clock_setting"}


class ClockSampler:
    def __init__(self, index):
        self.path = tempfile.mktemp(prefix="orx_clocks_")
        try:
            self.p = subprocess.Popen([sys.executable, "-c", _CLOCK_SRC, str(index), self.path],
                                      stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        self.windows = []

    def wait_ready(self, timeout=20.0):
        t0 = time.time()
        while self.p is not None and time.time() - t0 < timeout:
            try:
                if os.path.getsize(self.path) > 0:
                    return True
            except OSError:
                pass
            if self.p.poll() is not None:
                return False
            time.sleep(0.01)
        return False

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def _rows(self):
        rows = []
        try:
            for line in open(self.path):
                f = line.split()
                if len(f) == 4:
                    rows.append((float(f[0]), int(f[1]), int(f[2]), int(f[3])))
        except Exception:
            pass
        return rows

    def report(self, final=False):
        """Clocks over the windows registered so far (under load: samples inside them, widened by one poll period)."""
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML sampler unavailable"}
        time.sleep(0.01)
        rows = self._rows()
        if final:
            self.p.terminate()
            try:
                os.unlink(self.path)
            except OSError:
                pass
        inside = [r for r in rows if any(a - 0.003 <= r[0] <= b + 0.003 for a, b in self.windows)]
        note = "samples inside the timed / instrumented regions"
        if not inside:
            lo = min((a for a, _ in self.windows), default=0.0)
            inside, note = [r for r in rows if r[0] >= lo - 0.5], "no sample fell inside the regions; samples from 0.5 s before on"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "no samples"}
        bits = 0
        for r in inside:
            bits |= r[3]
        return {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": float(inside[0][2]),
                "reasons": sorted(v for k, v in _REASONS.items() if bits & k), "samples": len(inside), "note": note}


# ---------------------------------------------------------------------------------------
# CPU arm: the restated reference step on the host cores
# ---------------------------------------------------------------------------------------
def _visible_cpus():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_arm_pairwise(kind, steps, warmup, budget_s, batch=B):
    """Times `steps` steps of `batch` triplets (bounded by budget_s) of the C/OpenMP port.  -> (units/s, ms, steps, info)."""
    from oracle import c_port
    from oracle import openrec_oracle as O
    rng = np.random.default_rng(0)

    def tab(rows, cols):
        return rng.random((rows, cols), dtype=np.float32) * np.float32(0.1) - np.float32(0.05)

    user, item, bias = tab(U, D), tab(I, D), tab(I, 1)
    acc = [np.full_like(a, 0.1) for a in (user, item, bias)]
    ids = [tuple(rng.integers(0, n, batch, dtype=np.int32) for n in (U, I, I)) for _ in range(4)]
    state = {"threads": c_port.num_threads()}

    def step(i):
        u, p, n = ids[i % len(ids)]
        out = c_port.pairwise_step(kind, user, acc[0], item, acc[1], bias, acc[2], u, p, n, 1, LR, nthreads=state["threads"])
        if kind == "ucml":
            O.ucml_censor_vec(user, item, u, p, n)
        return out

    # "all the host threads it can use": the port is memory-bound and SMT siblings slow it down (r1a: 0.17 M/s on 128
    # threads vs 0.80 M/s on 64), so each of all / half / quarter of the visible CPUs is timed best-of-3
    visible = _visible_cpus()
    cands = sorted({max(1, visible), max(1, visible // 2), max(1, visible // 4)}, reverse=True)
    best = None
    t_pick = time.perf_counter()
    for cand in cands:
        state["threads"] = cand
        step(0)                                   # first touch / warm
        ts = []
        for r in range(3):
            t = time.perf_counter()
            step(1 + r)
            ts.append(time.perf_counter() - t)
            if time.perf_counter() - t_pick > budget_s * 0.5:
                break
        if best is None or min(ts) < best[0]:
            best = (min(ts), cand)
    state["threads"] = best[1]
    t0 = time.perf_counter()
    for i in range(max(1, warmup)):
        step(i)
        if time.perf_counter() - t0 > budget_s * 0.15:
            break
    done, t0 = 0, time.perf_counter()
    while done < steps:
        step(done)
        done += 1
        if time.perf_counter() - t0 > budget_s * 0.5:
            break
    dt = time.perf_counter() - t0
    info = {"cores": best[1], "kind": "port",
            "sample": f"{done} steps x {batch} triplets of the same workload (same table sizes, Adagrad"
                      f"{', + numpy censor_vec' if kind == 'ucml' else ''}), C/OpenMP port of the oracle (oracle/c/orx_oracle.c), "
                      f"{best[1]} threads (fastest of {cands} of the {visible} visible CPUs, best of 3 steps each), {dt:.1f} s"}
    return done * batch / dt, dt / done * 1e3, done, info


def cpu_arm_dlrm(steps, warmup, budget_s):
    """numpy / BLAS restatement of the DLRM step (oracle/openrec_oracle.py) on a bounded sample: the full MLPs and feature
    count, batch 4096, vocab 100k per table (13 GB of host tables at the full vocab would take minutes to initialise)."""
    from oracle import openrec_oracle as O
    rng = np.random.default_rng(0)
    batch, vocab = 4096, 100_000
    f32 = np.float32
    tabs = [(rng.random((vocab, D), dtype=f32) * f32(0.1) - f32(0.05)) for _ in range(DLRM_T)]
    accs = [np.full_like(t, 0.1) for t in tabs]
    dims = dlrm_layers()
    nb = len(DLRM_BOT)
    ws = [(rng.random(d, dtype=f32) * 2 - 1) * f32(np.sqrt(6.0 / (d[0] + d[1]))) for d in dims]
    bs = [np.zeros(d[1], dtype=f32) for d in dims]
    wacc, bacc = [np.full_like(w, 0.1) for w in ws], [np.full_like(b, 0.1) for b in bs]
    dense = np.log1p(rng.integers(0, 100, (batch, DLRM_DENSE))).astype(f32)
    sparse = rng.integers(0, vocab, (batch, DLRM_T)).astype(np.int32)
    label = (rng.random(batch) < 0.25).astype(f32)

    def step():
        cache = O.dlrm_forward(tabs, ws[:nb], bs[:nb], ws[nb:], bs[nb:], dense, sparse, interaction_mode="dlrm")
        _, dpred = O.dlrm_loss(cache["pred"], label, "mse")
        g = O.dlrm_backward(cache, tabs, ws[:nb], ws[nb:], dense, sparse, dpred, interaction_mode="dlrm")
        for k in range(DLRM_T):
            O.adagrad_sparse(tabs[k], accs[k], sparse[:, k], g["emb"][k], DLRM_LR)
        for l, (dw, db) in enumerate(zip(list(g["bot_w"]) + list(g["top_w"]), list(g["bot_b"]) + list(g["top_b"]))):
            O.adagrad_dense(ws[l], wacc[l], dw, DLRM_LR)
            O.adagrad_dense(bs[l], bacc[l], db.reshape(bs[l].shape), DLRM_LR)

    t0 = time.perf_counter()
    for _ in range(max(1, warmup)):
        step()
        if time.perf_counter() - t0 > budget_s * 0.3:
            break
    done, t0 = 0, time.perf_counter()
    while done < steps:
        step()
        done += 1
        if time.perf_counter() - t0 > budget_s * 0.7:
            break
    dt = time.perf_counter() - t0
    info = {"cores": _visible_cpus(), "kind": "port",
            "sample": f"{done} steps x {batch} samples, {DLRM_T} tables x {vocab} x {D} (vocab reduced from {DLRM_VOCAB}), "
                      f"the full MLP stack, numpy/BLAS oracle (oracle/openrec_oracle.py dlrm_*), {dt:.1f} s"}
    return done * batch / dt, dt / done * 1e3, done, info


def cpu_arm(wl, steps, warmup, budget_s):
    if wl == "dlrm":
        return cpu_arm_dlrm(steps, warmup, budget_s)
    return cpu_arm_pairwise(wl, steps, warmup, budget_s)


def run_reference(args, rank, world):
    if rank != 0:
        return
    wl = args.workload
    budget = float(os.environ.get("ORX_CPU_BUDGET_S", "60"))
    v, ms, done, info = cpu_arm(wl, args.steps, args.warmup, budget)
    metric, unit = METRICS[wl]
    line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": done,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(wl, 1), "note": "CPU restatement of openrec.tf2 (TensorFlow not "
                       "installable): oracle/, all host threads; ALWAYS the single-GPU workload -- the reference has no "
                       "multi-device path and the 100M-item tables of the N > 1 runs need ~100 GB of host memory, so at "
                       "--gpus > 1 this arm and the GPU arm run different table sizes"},
            "cpu_baseline": {"value": v, "unit": unit, **info},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------
def _timed(fn_step, K, barrier, torch, clocks):
    """EXACTLY K steps between two events, barrier + synchronize on both sides.  -> seconds"""
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for i in range(K):
        fn_step(i)
    e1.record()
    barrier()
    if clocks:
        clocks.window(t0, time.time())
    return e0.elapsed_time(e1) * 1e-3


def _sample_rows(t, n):
    """n rows of a device tensor, picked by a fixed seed and kept in row order (all rows if it has no more), as float32."""
    import torch
    if t.shape[0] <= n:
        return t.float().cpu().numpy()
    idx = np.sort(np.random.default_rng(0).choice(t.shape[0], n, replace=False))
    return t.index_select(0, torch.from_numpy(idx).to(t.device)).float().cpu().numpy()


def write_dumps(out_dir, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {DUMP_LIMIT}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bench_pairwise(wl, args, eng, dev, barrier, clocks, with_extra=True):
    import torch
    from openrec_b200 import native as N
    kind = N.ORX_PAIR_BPR if wl == "bpr" else N.ORX_PAIR_UCML
    K, W = args.steps, max(3, args.warmup)
    tu, ti = torch.empty(U, D, device=dev), torch.empty(I, D, device=dev)
    tb = torch.empty(I, 1, device=dev)
    for k, t in enumerate((tu, ti, tb)):
        eng.fill_uniform(t, -0.05, 0.05, 1000 + k)
    acc = [torch.full_like(t, 0.1) for t in (tu, ti, tb)]
    tabs = (N.table(tu, acc[0]), N.table(ti, acc[1]), N.table(tb, acc[2]))
    g = torch.Generator(device="cpu").manual_seed(1)
    host_ids = [tuple(torch.randint(0, n, (B,), generator=g, dtype=torch.int32).pin_memory() for n in (U, I, I))
                for _ in range(N_BATCHES)]
    dev_ids = [tuple(x.to(dev) for x in b) for b in host_ids]
    out4 = torch.zeros(4, device=dev)
    opt = N.opt(N.ORX_OPT_ADAGRAD, LR)
    torch.cuda.synchronize()                       # the id batches are complete: ids_ready below is honest

    def step(i, kind=kind, o=opt, pipeline=True):
        u, p, n = dev_ids[i % N_BATCHES]
        eng.pairwise_step(kind, *tabs, u, p, n, o, out4)
        if kind == N.ORX_PAIR_UCML:                # UCML's training loop: censor the rows just touched (ucml.py:44-48)
            eng.censor(tu, u), eng.censor(ti, p), eng.censor(ti, n)
        if pipeline:                               # index of the next batch: side stream, beside the next step's predecessor
            eng.pairwise_prefetch(tabs[0], tabs[1], *dev_ids[(i + 1) % N_BATCHES], o.kind, ids_ready=True)

    eng.pairwise_prefetch(tabs[0], tabs[1], *dev_ids[0], opt.kind, ids_ready=True)
    for i in range(W):
        step(i - W)
    seconds = _timed(step, K, barrier, torch, clocks)
    dump = {}
    if args.dump_outputs:      # the last timed step's results, before the loops below train the same tables further
        dump = {f"{wl}_loss_l2": out4[:2].cpu().numpy(), f"{wl}_user_rows": _sample_rows(tu, DUMP_ROWS),
                f"{wl}_item_rows": _sample_rows(ti, DUMP_ROWS), f"{wl}_item_bias_rows": _sample_rows(tb, DUMP_ROWS)}
    loss_check = out4.cpu().numpy().tolist()
    # ---- roofline: the same loop, instrumented (events around the phases of every 8th step), >= 64 samples
    n_inst = 8 * 64 + 8
    eng.profile_enable(True)
    t0 = time.time()
    for i in range(n_inst):
        step(K + i)
    torch.cuda.synchronize()
    clocks and clocks.window(t0, time.time())
    phase_ms, n_prof = eng.profile_read()
    eng.profile_enable(False)

    extra = {"last_loss_value_path": loss_check[:2]}
    if with_extra:   # same tables, short loops: the un-pipelined step and the SGD variant
        def short(n=200, **kw):
            for i in range(5):
                step(i, **kw)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                step(i, **kw)
            e1.record()
            torch.cuda.synchronize()
            return n * B / (e0.elapsed_time(e1) * 1e-3)
        extra[f"{wl}_without_index_prefetch_triplets_per_sec"] = short(pipeline=False)
        if wl == "bpr":
            extra["bpr_sgd_triplets_per_sec"] = short(o=N.opt(N.ORX_OPT_SGD, LR))
            # SURVEY 8d: a Zipf(1.05) id distribution exposes duplicate contention (most lookups hit rows that other
            # triplets of the batch also hit: they go through the staging buffer and the tail instead of the in-register
            # update).  Ranks are shuffled over the row space so that hot rows are not neighbours.
            zr = np.random.default_rng(5)
            pk = np.arange(1, U + 1, dtype=np.float64) ** -1.05
            pk /= pk.sum()
            relabel = [zr.permutation(n).astype(np.int32) for n in (U, I)]
            saved = list(dev_ids)
            for k in range(N_BATCHES):
                draws = [zr.choice(U, size=B, p=pk) for _ in range(3)]
                dev_ids[k] = tuple(torch.from_numpy(relabel[min(j, 1)][d]).to(dev) for j, d in enumerate(draws))
            torch.cuda.synchronize()
            extra["bpr_zipf1.05_triplets_per_sec"] = short(pipeline=False)
            u0 = dev_ids[0][0]
            extra["bpr_zipf1.05_unique_user_rows_per_batch"] = int(torch.unique(u0).numel())
            dev_ids[:] = saved

    # ---- e2e: public API (openrec.tf2 model + GradientTape + Adagrad), host ids in, loss out, every step
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    import tensorflow as tf
    from openrec.tf2.recommenders import BPR, UCML
    del tu, ti, tb, acc, tabs
    torch.cuda.empty_cache()
    model = (BPR if wl == "bpr" else UCML)(dim_user_embed=D, dim_item_embed=D, total_users=U, total_items=I)
    optimizer = tf.keras.optimizers.Adagrad(learning_rate=LR)

    def train_step(user_id, p_item_id, n_item_id):
        with tf.GradientTape() as tape:
            loss_value = model(user_id, p_item_id, n_item_id)
        gradients = tape.gradient(loss_value, model.trainable_variables)
        optimizer.apply_gradients(zip(gradients, model.trainable_variables))
        if wl == "ucml":
            model.censor_vec(user_id, p_item_id, n_item_id)
        return loss_value

    state = {"prev": None, "last": 0.0}

    def e2e_step(i):
        loss_value = train_step(*host_ids[i % N_BATCHES])     # pinned host ids -> device inside the call
        if state["prev"] is not None:
            state["last"] = float(state["prev"][0])            # every step's loss is read on the host, one step
        state["prev"] = loss_value                             # behind so the copy overlaps the next launch

    for i in range(W):
        e2e_step(i)
    e2e_seconds = _timed(e2e_step, K, barrier, torch, clocks)
    state["last"] = float(state["prev"][0])
    extra["last_loss_e2e"] = state["last"]

    peak, _, peak_src = measured_peaks()
    step_ms = phase_ms[1] / max(n_prof, 1)
    achieved = ALG_BYTES_PER_TRIPLET * B / (step_ms * 1e-3) / 1e9 if step_ms > 0 else 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "k_pair_step_traffic.json")) as f:
            traffic = json.load(f)["dram_bytes_per_launch"]
    except Exception:
        pass
    kname = "k_pair_step<%s,ADAGRAD,D=128,CH=8,4 CTAs/SM>" % ("BPR" if wl == "bpr" else "UCML")
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic if wl == "bpr" else None, "peak_source": peak_src + " hbm_gbs, burst copy",
                "algorithmic_bytes_per_launch": ALG_BYTES_PER_TRIPLET * B, "kernel_ms": step_ms,
                "phase_ms_per_step": {"wait_for_prefetched_index": phase_ms[0] / max(n_prof, 1), "pair_step": step_ms,
                                      "tail": phase_ms[2] / max(n_prof, 1)},
                "step_level_frac": ALG_BYTES_PER_TRIPLET * B / (seconds / K) / 1e9 / peak,
                "timing": f"CUDA events on the launch stream around the phases of every 8th step of a {n_inst}-step "
                          f"instrumented loop of the same step right after the timed region ({n_prof} samples); the batch "
                          "index of step t+1 runs on the side stream during step t, so pair_step includes that contention"}
    launches = (3 + (3 if wl == "ucml" else 0)) * K
    return {"seconds": seconds, "e2e_seconds": e2e_seconds, "launches": launches, "units_per_step": B, "roofline": roofline,
            "h2d": 3 * 4 * B, "d2h": 16,
            "e2e_api": f"openrec.tf2.recommenders.{'BPR' if wl == 'bpr' else 'UCML'} + tf.GradientTape + "
                       "tf.keras.optimizers.Adagrad (shim); pinned host ids in, loss read to host each step",
            "extra": extra, "dump": dump}


def bench_dlrm(args, eng, dev, barrier, clocks):
    import torch
    K, W = args.steps, max(3, args.warmup)
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    import tensorflow as tf
    from openrec.tf2.recommenders import DLRM
    from openrec_b200.tf2 import mlp_ops
    rng = np.random.default_rng(0)
    model = DLRM(m_spa=D, ln_emb=[DLRM_VOCAB] * DLRM_T, ln_bot=DLRM_BOT, ln_top=DLRM_TOP, interaction_mode="dlrm")
    optimizer = tf.keras.optimizers.Adagrad(learning_rate=DLRM_LR)
    host = [(np.log1p(rng.integers(0, 100, (DLRM_B, DLRM_DENSE))).astype(np.float32),
             rng.integers(0, DLRM_VOCAB, (DLRM_B, DLRM_T)).astype(np.int32),
             (rng.random(DLRM_B) < 0.25).astype(np.float32)) for _ in range(4)]
    pinned = [tuple(torch.from_numpy(a).pin_memory() for a in b) for b in host]
    devb = [tuple(tf.constant(a) for a in b) for b in host]

    def train_step(d, s, y):
        with tf.GradientTape() as tape:
            loss = model(d, s, y)
        g = tape.gradient(loss, model.trainable_variables)
        optimizer.apply_gradients(zip(g, model.trainable_variables))
        return loss

    state = {"prev": None, "last": 0.0}

    def step(i):
        state["prev"] = train_step(*devb[i % 4])

    def e2e_step(i):
        loss = train_step(*pinned[i % 4])                     # pinned host arrays -> device inside the call
        if state["prev"] is not None:
            state["last"] = float(state["prev"])
        state["prev"] = loss

    for i in range(W):
        step(i)
    seconds = _timed(step, K, barrier, torch, clocks)
    loss_value = float(state["prev"])
    dump = {}
    if args.dump_outputs:      # the last timed step's results, before the loops below train the same model further
        dump["dlrm_loss"] = np.array([loss_value], dtype=np.float32)
        for k, v in enumerate(model.trainable_variables):     # 26 embedding tables, then the MLP kernels and biases
            dump[f"dlrm_var{k:02d}"] = _sample_rows(v.t, DLRM_DUMP_ROWS)
    # ---- roofline: the Dense-layer GEMMs (dominant kernels), timed with events around every GEMM call of a few steps
    prof = mlp_ops.GemmProfile()
    t0 = time.time()
    with prof:
        for i in range(4):
            step(K + i)
        torch.cuda.synchronize()
    clocks and clocks.window(t0, time.time())
    gemm_ms, gemm_flops, n_gemm = prof.totals()
    tc_ms, tc_flops, n_tc = prof.totals(pure_only=True)        # the forward layers: one k_gemm_tma launch each
    state["prev"] = None
    for i in range(W):
        e2e_step(i)
    e2e_seconds = _timed(e2e_step, K, barrier, torch, clocks)
    state["last"] = float(state["prev"])
    _, tf_peak, peak_src = measured_peaks()
    # 3xTF32 on kind::tf32 tensor cores: TF32 dense peak = half the bf16 peak, three MMAs per fp32-equivalent product
    peak = tf_peak / 2.0 / 3.0
    achieved = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    step_flops = dlrm_flops_per_sample() * DLRM_B
    roofline = {"bound": "tensor", "kernel": mlp_ops.GEMM_KERNEL_NAME, "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                "peak_source": peak_src + " bf16_tflops_sustained / 2 (TF32) / 3 (3xTF32 error-compensated fp32)",
                "algorithmic_flops_per_launch": tc_flops / max(n_tc, 1), "kernel_ms": tc_ms / max(n_tc, 1),
                "launches_timed": n_tc,
                "algorithmic_flops_per_step": step_flops, "dense_layer_flops_per_step": gemm_flops / 4,
                "dense_layer_ms_per_step": gemm_ms / 4, "dense_layer_calls_per_step": n_gemm // 4,
                "dense_layer_share_of_step": (gemm_ms / 4) / (seconds / K * 1e3),
                "dense_layer_tflops_all_calls": gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0,
                "step_level_tflops": step_flops / (seconds / K) / 1e12,
                "timing": "CUDA events on the launch stream around every Dense-layer call of 4 instrumented steps right after "
                          "the timed region.  achieved / kernel_ms: the forward layers on the tensor-core path, each exactly "
                          "one k_gemm_tma launch (bias + activation in its epilogue), flops = 2*M*N*K; dense_layer_*: all "
                          "calls, where a backward call = dgrad + wgrad GEMMs + activation-gradient and bias-sum kernels"}
    return {"seconds": seconds, "e2e_seconds": e2e_seconds, "launches": model._launches_per_step() * K,
            "units_per_step": DLRM_B, "roofline": roofline,
            "h2d": DLRM_B * (DLRM_DENSE * 4 + DLRM_T * 4 + 4), "d2h": 4,
            "e2e_api": "openrec.tf2.recommenders.DLRM + tf.GradientTape + tf.keras.optimizers.Adagrad (shim); pinned host "
                       "dense / sparse / label in, loss read to host each step",
            "extra": {"last_loss_value_path": loss_value, "last_loss_e2e": state["last"]}, "dump": dump}


def make_line(wl, args, world, result, clocks_report, cpu=None):
    metric, unit = METRICS[wl]
    K = args.steps
    units = K * result["units_per_step"] * world
    line = {"metric": metric, "value": units / result["seconds"], "unit": unit, "n_gpus": world, "steps": K,
            "warmup": max(3, args.warmup), "ms_per_step": result["seconds"] / K * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(wl, world), "optimizer": "Adagrad (Keras sparse semantics)",
                       "l2_flush": ("none needed: tables + accumulators >= 2 GB per GPU and >= 0.4 GB of random rows touched per "
                                    "step >> 126 MB L2; id batches rotate"),
                       "parallelism": "single GPU" if world == 1 else f"row-sharded tables x{world}"},
            "clocks": clocks_report,
            "e2e": {"value": units / result["e2e_seconds"], "unit": unit,
                    "h2d_bytes_per_step": result["h2d"] * world, "d2h_bytes_per_step": result["d2h"] * world,
                    "api": result["e2e_api"]},
            "gpu_launches": result["launches"], "roofline": result["roofline"]}
    if world > 1:
        line["config"]["reference_arm"] = ("bench.py --impl reference always runs the single-GPU workload (1M x 1M tables): "
                                           "same step, different table sizes")
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if result.get("extra"):
        line["extra"] = result["extra"]
    return line


def run_b200(args, rank, world, local_rank):
    clocks = ClockSampler(local_rank) if rank == 0 else None    # started before torch: ready when the timing starts
    import torch
    import torch.distributed as dist
    from openrec_b200 import native as N

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    real_stdout = None
    if world > 1:
        # The contract is ONE JSON line on stdout, and NCCL prints its version banner (and, with NCCL_DEBUG=INFO, its log)
        # there.  The driver's NCCL_DEBUG setting is left alone: file descriptor 1 points at stderr while the job runs and
        # the JSON line goes out through a saved copy of the real stdout.
        sys.stdout.flush()
        real_stdout = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    eng = N.engine(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if clocks:
        clocks.wait_ready()
    wl = args.workload
    if world > 1:
        if wl != "bpr":
            raise SystemExit("the multi-GPU bench is the row-sharded BPR step (BASELINE configs[4])")
        from openrec_b200 import sharded
        result = sharded.bench(args, rank, world, eng, barrier, clocks)
        t = torch.tensor([result["seconds"], result["e2e_seconds"]], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)   # max over ranks
        result["seconds"], result["e2e_seconds"] = t[0].item(), t[1].item()
        if rank == 0:
            real_stdout.write(json.dumps(make_line(wl, args, world, result, clocks.report(final=True))) + "\n")
            real_stdout.flush()
        dist.destroy_process_group()
        return
    run = {"bpr": lambda: bench_pairwise("bpr", args, eng, dev, barrier, clocks),
           "ucml": lambda: bench_pairwise("ucml", args, eng, dev, barrier, clocks, with_extra=False),
           "dlrm": lambda: bench_dlrm(args, eng, dev, barrier, clocks)}
    result = run[wl]()
    clocks_main = clocks.report()
    cpu_budget = float(os.environ.get("ORX_CPU_BUDGET_S", "24"))

    def cpu_of(w, budget):
        if args.no_cpu:
            return None
        v, ms, done, info = cpu_arm(w, 50, 2, budget)
        return {"value": v, "unit": METRICS[w][1], **info}

    line = make_line(wl, args, 1, result, clocks_main, cpu_of(wl, cpu_budget))
    dumps = dict(result["dump"])
    if wl == "bpr" and not args.no_secondary:
        line["secondary"] = []
        for w in ("ucml", "dlrm"):
            torch.cuda.empty_cache()
            clocks.windows = []
            try:
                r = run[w]()
                line["secondary"].append(make_line(w, args, 1, r, clocks.report(), cpu_of(w, cpu_budget / 2)))
                dumps.update(r["dump"])
            except Exception as e:                                 # a secondary workload must never cost the headline line
                line["secondary"].append({"metric": METRICS[w][0], "error": f"{type(e).__name__}: {e}"})
    clocks.report(final=True)
    if args.dump_outputs:
        write_dumps(args.dump_outputs, dumps)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="bpr", choices=["bpr", "ucml", "dlrm"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs (profiling runs)")
    ap.add_argument("--no-secondary", action="store_true", help="bpr only: do not append the ucml / dlrm lines")
    ap.add_argument("--check", action="store_true",
                    help="--gpus N > 1: after the timed loops run ONE more step on a fresh batch and verify it on rank 0 against "
                         "the oracle over the rows the global batch touches (tests/shard_check.py); the verdict goes to extra.check")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--gpus 1: write what the last timed step of each workload run computed to DIR/<name>.npy "
                         "(float32): the loss, and the trained tables and weights, each table a fixed sample of "
                         f"{DUMP_ROWS} (DLRM: {DLRM_DUMP_ROWS}) rows; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl b200 and --gpus 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and not (world == 1 and args.gpus == 1):
        if rank == 0:
            sys.stderr.write(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run\n")
        sys.exit(2)
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
