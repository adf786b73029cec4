"""Kernel micro-benchmarks on one B200 (CUDA-event timing, L2 flushed between iterations).
Writes gpurun_out/microbench_<tag>.json.  Not the contract bench (bench.py)."""
import json
import os
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from importlib import import_module

import fo1_b200  # noqa: E402

ops = import_module("vlm-fo1_b200.ops")
H = import_module("vlm-fo1_b200.hfre")

PEAKS = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(REPO, "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
_flush = None


def flush_l2():
    global _flush
    if _flush is None:
        _flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    _flush.zero_()


def timeit(fn, iters=10, warm=3, flush=True):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush:
            flush_l2()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def bench_gemm(results):
    shapes = [(32768, 1280, 1280), (32768, 3840, 1280), (32768, 6912, 1280), (32768, 1280, 3456), (8192, 8192, 8192),
              (38240, 2048, 2048), (38240, 22016, 2048), (38240, 2048, 11008), (4096, 1280, 1280), (32, 2048, 2048)]
    for M, N, K in shapes:
        a = (torch.randn(M, K, device="cuda") * 0.5).to(torch.bfloat16)
        w = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        med, best = timeit(lambda: ops.gemm(a, w, out=out))
        tmed, tbest = timeit(lambda: torch.matmul(a, w.t(), out=out))
        fl = 2.0 * M * N * K
        r = {"kind": "gemm", "M": M, "N": N, "K": K, "ms": med, "tflops": fl / med / 1e9, "tflops_best": fl / best / 1e9,
             "cublas_ms": tmed, "cublas_tflops": fl / tmed / 1e9,
             "frac_of_measured_sustained": fl / med / 1e9 / PEAKS["bf16_tflops_sustained"]}
        print(json.dumps(r), flush=True)
        results.append(r)
        del a, w, out


def make_hfre_inputs(B, S, N, seed=0):
    g = torch.Generator().manual_seed(seed)
    chans = (256, 512, 1024, 2048)
    gh = S // 14
    aux_all, pyr_all, ba, bv, grids = [], [], [], [], []
    for b in range(B):
        aux = [torch.randn(S // (4 << i), S // (4 << i), c, device="cuda").to(torch.bfloat16) for i, c in enumerate(chans)]
        pyr = [torch.randn(int(gh * f), int(gh * f), 512, device="cuda").to(torch.bfloat16) for f in (4, 2, 1, 0.5)]
        gb = torch.Generator().manual_seed(2000 + b)
        w = torch.rand(N, generator=gb) * (S / 2 - 32) + 32; h = torch.rand(N, generator=gb) * (S / 2 - 32) + 32
        x1 = torch.rand(N, generator=gb) * (S - w); y1 = torch.rand(N, generator=gb) * (S - h)
        boxes = torch.stack([x1, y1, x1 + w, y1 + h], 1)
        aux_all.append(aux); pyr_all.append(pyr); ba.append(boxes.cuda()); bv.append((boxes * (gh * 14 / S)).cuda()); grids.append((gh, gh))
    return aux_all, pyr_all, ba, bv, grids


def bench_hfre(results, B=8, S=896, N=100, algo=0):
    aux_all, pyr_all, ba, bv, grids = make_hfre_inputs(B, S, N)
    cfg = H.HfreConfig(region_dim=5888, vt_mode="fpn", algo=algo)
    tot_unique = tot_gather = 0
    for b in range(B):
        shapes = [tuple(a.shape) for a in aux_all[b]] + [tuple(p.shape) for p in pyr_all[b]]
        H0 = aux_all[b][0].shape[0]
        boxes_l = [ba[b].cpu().numpy()] * 4 + [bv[b].cpu().numpy()] * 4
        scales = [0.25] * 4 + [1 / s for s in H.FPN_STRIDES]
        ups = [H0 // a.shape[0] for a in aux_all[b]] + [1] * 4
        ab = H.algorithmic_bytes(shapes, boxes_l, scales, ups, N, 5888)
        tot_unique += ab["unique_bytes"]; tot_gather += ab["gather_bytes"]
    med, best = timeit(lambda: H.hfre_forward(aux_all, pyr_all, ba, bv, cfg, grids), iters=10)
    # one profiled pass: CUDA-event time of each tagged kernel (the sweep / gather is the roofline kernel)
    import ctypes as C
    L = import_module("vlm-fo1_b200._lib").lib()
    L.fo1_profile_enable(1)
    for _ in range(3):
        flush_l2()
        H.hfre_forward(aux_all, pyr_all, ba, bv, cfg, grids)
    torch.cuda.synchronize()
    buf = C.create_string_buffer(1 << 20)
    L.fo1_profile_collect(buf, 1 << 20)
    L.fo1_profile_enable(0)
    prof = json.loads(buf.value.decode())
    kern = {k: round(v["ms"] / v["launches"], 4) for k, v in prof.items()}
    main = kern.get("hfre_sweep_mma") or kern.get("hfre_gather")
    r = {"kind": "hfre", "algo": algo, "B": B, "S": S, "N": N, "ms": med, "kernel_ms": kern,
         "kernel_unique_GBs": tot_unique / main / 1e6, "kernel_frac_of_measured_hbm": tot_unique / main / 1e6 / PEAKS["hbm_gbs"], "ms_best": best, "unique_MB": tot_unique / 1e6, "gather_MB": tot_gather / 1e6,
         "unique_GBs": tot_unique / med / 1e6, "gather_GBs": tot_gather / med / 1e6,
         "frac_of_measured_hbm": tot_unique / med / 1e6 / PEAKS["hbm_gbs"]}
    print(json.dumps(r), flush=True)
    results.append(r)


def bench_decode_gemms(results, M=32):
    """the four per-layer decode GEMMs + lm_head at batch M: weight-streaming, HBM-bound"""
    shapes = [("qkv", 2560, 2048, False), ("o", 2048, 2048, False), ("gateup", 22016, 2048, True), ("down", 2048, 11008, False),
              ("lm_head", 151936, 2048, False)]
    for name, N, K, gated in shapes:
        a = (torch.randn(M, K, device="cuda") * 0.5).to(torch.bfloat16)
        w = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
        fn = (lambda: ops.gemm(a, w, act="silu", gated=True)) if gated else (lambda: ops.gemm(a, w))
        med, best = timeit(fn, iters=20)
        byt = 2.0 * (N * K + M * K + M * N)
        r = {"kind": "decode_gemm", "name": name, "M": M, "N": N, "K": K, "us": med * 1e3, "GBs": byt / med / 1e6,
             "frac_of_measured_hbm": byt / med / 1e6 / PEAKS["hbm_gbs"]}
        print(json.dumps(r), flush=True)
        results.append(r)


if __name__ == "__main__":
    tag = sys.argv[1] if len(sys.argv) > 1 else "r1"
    which = sys.argv[2:] or ["gemm", "hfre"]
    res = []
    print("device", torch.cuda.get_device_name(0), "cpus", os.cpu_count(), flush=True)
    if "hfre" in which:
        for algo in (1, 3):
            bench_hfre(res, algo=algo)
        for algo in (1, 3):
            bench_hfre(res, B=8, S=896, N=32, algo=algo)     # COCO-like box count (mean 31.5)
    if "gemm" in which:
        bench_gemm(res)
    if "decode" in which:
        bench_decode_gemms(res)
    os.makedirs(os.path.join(REPO, "gpurun_out"), exist_ok=True)
    json.dump(res, open(os.path.join(REPO, "gpurun_out", f"microbench_{tag}.json"), "w"), indent=1)
