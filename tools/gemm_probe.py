"""Dense-layer GEMM alone at the DLRM shapes (forward, dgrad, wgrad): CUDA-event time and fp32-equivalent TFLOP/s;
also the ncu target for the tcgen05 kernel.   python tools/gemm_probe.py [reps]"""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from openrec_b200 import native as N
eng = N.engine()
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
B = 32768
for (K, Nn) in [(1024, 1024), (479, 1024), (1024, 512), (512, 256), (256, 128), (512, 256)]:
    Kp = (K + 3) // 4 * 4                      # row stride a multiple of 16 bytes, as DLRMGraph allocates (TMA)
    x = torch.randn(B, Kp, device='cuda')[:, :K]; w = torch.randn(K, Nn, device='cuda') * 0.03; b = torch.zeros(Nn, device='cuda')
    y = torch.empty(B, Nn, device='cuda'); dy = torch.randn(B, Nn, device='cuda'); dx = torch.empty(B, Kp, device='cuda')[:, :K]
    dw = torch.empty_like(w); db = torch.empty_like(b)
    def t(fn):
        for _ in range(3): fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps): fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    f = t(lambda: eng.mlp_fwd(x, w, b, 1, y))
    bw = t(lambda: eng.mlp_bwd(x, y, w, 1, dy, dx, dw, db))
    fl = 2.0 * B * K * Nn
    print(f"M={B} K={K} N={Nn}: fwd {f*1e3:.0f} us = {fl/f/1e9:.1f} TF/s   bwd(dgrad+wgrad+act+colsum) {bw*1e3:.0f} us = {2*fl/bw/1e9:.1f} TF/s")
