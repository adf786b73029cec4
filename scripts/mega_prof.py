"""FO1_MEGA_PROF=1 python scripts/mega_prof.py [B] [L]: one generate() of the LLM alone at the 3B widths, prints the per-phase profile
of the persistent decode kernel (stderr) and the decode step time with / without it."""
import os, sys, time
import torch
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from importlib import import_module
import fo1_b200  # noqa
E = import_module("vlm-fo1_b200.engine"); CK = import_module("vlm-fo1_b200.checkpoint"); W = import_module("vlm-fo1_b200.weights")
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
L = int(sys.argv[2]) if len(sys.argv) > 2 else 1195
cfg = E.EngineConfig(); cfg.use_vit = cfg.use_davit = False; cfg.proj_aux_layers = 0
sd = CK.random_llm(cfg.llm, torch.Generator(device="cuda").manual_seed(5), "cuda")
eng = E.Engine(cfg); eng.set_weights(W.prepare_llm(sd, cfg.llm, eng.device)); eng.finalize(); del sd
emb = (torch.randn(B * L, 2048, device="cuda") * 0.05).to(torch.bfloat16)
pos = torch.arange(L, dtype=torch.int32).view(1, -1).expand(3, -1).repeat(1, B).contiguous()
def run(T):
    torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); eng.generate(emb, pos, [L] * B, [0] * B, T, stop_ids=[], pad_id=0, early_exit_interval=0); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1)
# clocks ramp up from idle over hundreds of milliseconds: warm the GPU first, then alternate the two paths and keep the best of each
wa = torch.randn(8192, 8192, device="cuda", dtype=torch.bfloat16)
t0 = time.time()
while time.time() - t0 < 3.0:
    for _ in range(20): wa @ wa
    torch.cuda.synchronize()
best = {"mega": 1e9, "per-kernel": 1e9}
prof = os.environ.pop("FO1_MEGA_PROF", None)
for rep in range(3):
    for tag in ("mega", "per-kernel"):
        if tag == "per-kernel": os.environ["FO1_NO_MEGA"] = "1"
        else: os.environ.pop("FO1_NO_MEGA", None)
        run(4); a = run(2); b = run(34)
        best[tag] = min(best[tag], (b - a) / 32)
for tag, v in best.items(): print(tag, "decode ms/step %.3f" % v, flush=True)
if prof:
    os.environ.pop("FO1_NO_MEGA", None); os.environ["FO1_MEGA_PROF"] = prof
    run(4)
