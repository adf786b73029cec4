"""Decode-loop probe: per-step decode time at B=32, L=1195 (prefill-only vs 64-token run); under ncu (PROBE_NCU=1, few steps)
it yields the exact per-kernel durations of one decode step."""
import json
import os
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from importlib import import_module

import fo1_b200  # noqa

E = import_module("vlm-fo1_b200.engine"); CK = import_module("vlm-fo1_b200.checkpoint")

B = int(os.environ.get("PROBE_B", 32)); L = int(os.environ.get("PROBE_L", 1195)); T = int(os.environ.get("PROBE_T", 64))
cfg = E.EngineConfig(); cfg.use_vit = cfg.use_davit = False; cfg.proj_aux_layers = 0
sds = CK.random_state_dicts(cfg, "cuda", 0)
eng = CK.load_engine(cfg, sds); del sds
emb = (torch.randn(B * L, 2048, device="cuda") * 0.02).to(torch.bfloat16)
pos = torch.arange(L, dtype=torch.int32, device="cuda").repeat(B).view(1, -1).expand(3, -1).contiguous()


def run(tokens):
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    out = eng.generate(emb, pos, [L] * B, [0] * B, tokens, stop_ids=[], pad_id=0, early_exit_interval=0)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1)


if os.environ.get("PROBE_PROF"):   # CUDA-event time of every tagged kernel of a short run (events break PDL / the graph)
    import ctypes as C
    lib_ = import_module("vlm-fo1_b200._lib").lib()
    run(4)
    lib_.fo1_profile_enable(1)
    run(T)
    buf = C.create_string_buffer(1 << 20)
    lib_.fo1_profile_collect(buf, 1 << 20)
    lib_.fo1_profile_enable(0)
    prof = json.loads(buf.value.decode())
    print(json.dumps({k: {"launches": v["launches"], "avg_us": round(1e3 * v["ms"] / v["launches"], 2)} for k, v in prof.items() if "skinny" in k or "decode" in k}))
elif os.environ.get("PROBE_NCU"):
    run(T)
else:
    run(4); run(4)
    p = min(run(1) for _ in range(3)); f = min(run(T) for _ in range(3))
    print(json.dumps({"B": B, "L": L, "T": T, "prefill_ms": p, "full_ms": f,
                      "decode_ms_per_step": (f - p) / (T - 1)}))
