"""python scripts/gemm_pair_bench.py: CTA-pair GEMM vs the single-CTA kernel (pinned tile_n=256) at the step's big shapes, warm clocks."""
import os, sys, time
import torch
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from importlib import import_module
import fo1_b200  # noqa
ops = import_module("vlm-fo1_b200.ops")
shapes = [(131072, 3840, 1280, False), (131072, 1280, 1280, False), (131072, 6848, 1280, True), (131072, 1280, 3456, False),
          (38240, 2560, 2048, False), (38240, 22016, 2048, True), (38240, 2048, 11008, False), (73728, 1024, 4096, False), (294912, 768, 256, False)]
wa = torch.randn(8192, 8192, device="cuda", dtype=torch.bfloat16)
t0 = time.time()
while time.time() - t0 < 2.0:
    for _ in range(20): wa @ wa
    torch.cuda.synchronize()
for M, N, K, gated in shapes:
    a = (torch.randn(M, K, device="cuda") * 0.5).bfloat16(); w = (torch.randn(N, K, device="cuda") * 0.05).bfloat16()
    out = torch.empty(M, N // 2 if gated else N, device="cuda", dtype=torch.bfloat16)
    res = {}
    for rep in range(2):
        for tag in ("pair", "single"):
            tn = 256 if tag == "single" else 0
            for _ in range(3): ops.gemm(a, w, gated=gated, act="silu" if gated else None, out=out, tile_n=tn)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10): ops.gemm(a, w, gated=gated, act="silu" if gated else None, out=out, tile_n=tn)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            res[tag] = min(res.get(tag, 1e9), ms)
    fl = 2.0 * M * N * K
    print(f"{M}x{N}x{K}{' gated' if gated else ''}: pair {res['pair']:.3f} ms {fl / res['pair'] / 1e9:.0f} TFLOP/s | single {res['single']:.3f} ms {fl / res['single'] / 1e9:.0f} TFLOP/s", flush=True)
