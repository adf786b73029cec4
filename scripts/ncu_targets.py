"""Tiny driver for `ncu --set full` captures: a representative big GEMM, the HFRE kernels at the C2 shape,
and one decode-shaped skinny GEMM.  Launch counts are kept minimal (ncu replays each kernel ~40x)."""
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "scripts"))
from importlib import import_module

import fo1_b200  # noqa

ops = import_module("vlm-fo1_b200.ops"); H = import_module("vlm-fo1_b200.hfre")
import microbench as MB  # noqa

which = sys.argv[1:] or ["gemm", "hfre", "skinny"]
if "gemm" in which:
    a = (torch.randn(32768, 1280, device="cuda") * 0.5).to(torch.bfloat16)
    w = (torch.randn(3840, 1280, device="cuda") * 0.05).to(torch.bfloat16)
    for _ in range(3):
        ops.gemm(a, w)
if "skinny" in which:
    a = (torch.randn(32, 2048, device="cuda") * 0.5).to(torch.bfloat16)
    w = (torch.randn(22016, 2048, device="cuda") * 0.05).to(torch.bfloat16)
    for _ in range(3):
        ops.gemm(a, w, act="silu", gated=True)
if "hfre" in which:
    aux_all, pyr_all, ba, bv, grids = MB.make_hfre_inputs(8, 896, 100)
    for algo in [int(a) for a in os.environ.get("NCU_HFRE_ALGOS", "1,3").split(",")]:
        cfg = H.HfreConfig(region_dim=5888, vt_mode="fpn", algo=algo)
        for _ in range(2):
            H.hfre_forward(aux_all, pyr_all, ba, bv, cfg, grids)
torch.cuda.synchronize()
