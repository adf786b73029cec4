#!/usr/bin/env python
"""bench.py -- contract benchmark of the FO1 hot path on N B200s (one rank per GPU).

Workload (BASELINE.json configs[2], the configuration the headline metric is quoted on): per GPU a batch of 32
synthetic 896x896 images, 64 boxes each, random-init 3B FO1 weights: dual vision towers (ViT + DaViT) -> SimpleFPN ->
HFRE region tokens -> projector -> splice -> Qwen2.5-3B prefill -> 64-token greedy decode; weak scaling (per-GPU batch
fixed), one NCCL all-gather of the decoded ids per step.  A "step" is one pass of that pipeline over one batch.

  value : images/sec, inputs already resident in HBM, CUDA-event timed, max over ranks.
  e2e   : the same through the public pipeline API from pinned HOST buffers: H2D of the raw uint8 images and the boxes,
          device-side pre-processing (bicubic smart-resize, normalise, patchify for both towers) and D2H of the token ids,
          all inside the timed region.
  roofline     : the dominant kernel (tcgen05 GEMM) -- algorithmic FLOPs / CUDA-event launch time (one extra
                 instrumented step after the timed region) vs the measured cuBLAS bf16 sustained peak.
  roofline_hfre: HFRE gather -- SURVEY 8d algorithmic bytes / launch time vs the measured HBM copy bandwidth.
  roofline_decode: one decode step -- bytes it must stream (bf16 weights + the live K/V) / its device time vs HBM.
  cpu_baseline : the reference's OWN modules (oracle/reference_path.py over the copy in baseline/_ref/, ``kind: "reference"``)
                 timed on the host cores on ONE full-depth image with a shortened decode (stated in ``sample``); the oracle
                 port (``kind: "port"``) only if that copy is absent.
``--impl reference`` times that CPU arm alone: one full-depth image per step, all decode tokens, every host thread.
``--dump-outputs DIR`` writes what the last timed step (of rank 0) returned as DIR/<name>.npy (dump_outputs); weights and inputs are
seeded, so two builds run with the same arguments can be compared output for output.

Workloads (``--workload``): c3 (default, the headline configuration), c4 (COCO shape: 640 px -> 46x46 grid, 100 boxes,
16 images / GPU), c5 (counting: 1344 px, 300 boxes, 128 tokens, 8 images / GPU), c2 (HFRE-only: towers + region tokens of
8 x 896 px x 100 boxes; value = GB/s of the HFRE operator).  ``--global-batch G`` fixes the TOTAL batch and splits it over
the ranks (strong scaling) instead of the per-GPU batch (weak scaling)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "images/sec (prefill+64-tok decode) 3B FO1"
UNIT = "images/s"
WORKLOADS = {   # BASELINE.json configs[1..4] (SURVEY.md section 8d "Config -> concrete workload"); batch = images per GPU
    "c3": dict(batch=32, size=896, boxes=64, tokens=64, name="configs[2] full prefill + 64-token decode"),
    "c4": dict(batch=16, size=640, boxes=100, tokens=64, name="configs[3] COCO-shape detection template (640 -> 644 px, grid 46x46)"),
    "c5": dict(batch=8, size=1344, boxes=300, tokens=128, name="configs[4] counting template (1344 px, 300 boxes, 128-token decode)"),
    "c2": dict(batch=8, size=896, boxes=100, tokens=0, name="configs[1] HFRE-only: dual-ViT forward + region-token extraction"),
}


def load_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.proc = None
        self.lines = []
        self.index = index

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx = max(mx, float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def reference_arm(args, cfg, steps, decode_tokens, warm=0):
    """The CPU arm: ONE image per step through the reference's own modules (oracle/reference_path.py; the oracle port if
    baseline/_ref is absent), fp32, FULL depth, on the host cores this process owns (affinity + cgroup quota: with every logical CPU of
    the box the OpenMP pool of a quota-limited container thrashes -- 455 s per image instead of ~45 s).  ``decode_tokens`` < args.tokens
    shortens the greedy loop; the remaining steps are then added at the measured per-token cost (the note says so).  --cpu-sample swaps the
    full depth for a bounded depth sample (8 of 32 ViT blocks, 4 of 36 decoder layers, DaViT stage 3 at 3 of 9) scaled to full depth.
    Returns (images/s, kind, cores, note, stage seconds of the last step)."""
    from importlib import import_module
    SY = import_module("vlm-fo1_b200.synthetic")
    from oracle import reference_path as RP
    cores = RP.usable_cores()
    torch.set_num_threads(cores)
    s = SY.synthetic_batch(0, 1, args.size, args.boxes)[0]
    T = max(args.tokens, 1)
    dt = max(1, min(decode_tokens, T))
    times, detail = [], None
    sample = dict(vit_blocks=8, llm_layers=4, davit_stage3=3) if getattr(args, "cpu_sample", False) else None
    depth_note = "FULL depth"
    if RP.available():
        kind = "reference"
        rp = RP.ReferencePath(cfg.vit, "davit-large", cfg.llm, region_dim=cfg.region_dim, davit_depths=cfg.davit["depths"], sample=sample)
        sc = rp.scale
        if any(v != 1.0 for v in sc.values()):
            depth_note = (f"DEPTH SAMPLE scaled to full depth: ViT {int(round(cfg.vit['depth'] / sc['vit']))} of {cfg.vit['depth']} blocks (x{sc['vit']:g}), "
                          f"DaViT stage 3 at {int(round(cfg.davit['depths'][2] / sc['davit3']))} of {cfg.davit['depths'][2]} (its measured time x{sc['davit3']:g}), "
                          f"LLM {int(round(cfg.llm['num_hidden_layers'] / sc['llm']))} of {cfg.llm['num_hidden_layers']} layers (x{sc['llm']:g}); "
                          "embeddings / merger / FPN / HFRE / projector / LM head in full")
        for i in range(warm + steps):
            out = rp.run(input_ids=s.input_ids, pixel_values=s.pixel_values, grid_hw=s.grid_hw, image_aux=s.image_aux, boxes=s.boxes,
                         max_new_tokens=dt)
            if i < warm:
                continue
            t = dict(out["timings"])
            per_tok = t["llm_decode_s"] / max(dt - 1, 1)
            total = t["total_s"] + (T - dt) * per_tok
            t["llm_decode_s_per_token"] = per_tok
            times.append(total); detail = t
        what = ("the reference's own modules (baseline/_ref copy of vlm_fo1: Qwen2_5_VisionTransformerPretrainedModel + custom_forward + "
                f"GATHER, DaViT, HFREModule incl. SimpleFP, mm_projector_aux, Qwen2_5_VLDecoderLayer; "
                f"attention '{rp.attn}'), model loop / splice / greedy loop restated")
    else:
        kind = "port"
        CK = import_module("vlm-fo1_b200.checkpoint")
        from oracle import pipeline as OP
        sds = CK.random_state_dicts(cfg, "cpu", 0)
        sds = {k: {n: v.float() for n, v in d.items()} for k, d in sds.items()}
        for _ in range(steps):
            with torch.no_grad():
                out = OP.run_sample(sds, cfg.vit, cfg.davit, cfg.llm, input_ids=s.input_ids, pixel_values=s.pixel_values, grid_hw=s.grid_hw,
                                    image_aux=s.image_aux, boxes=s.boxes, region_dim=cfg.region_dim, max_new_tokens=dt)
            t = {k: v for k, v in out["timings"].items() if isinstance(v, float)}
            per_tok = t.get("llm_decode_s_per_token", 0.0)
            total = t["vit_s"] + t["davit_s"] + t["fpn_s"] + t["hfre_s"] + t["proj_s"] + t["llm_prefill_s"] + (T - 1) * per_tok
            times.append(total); detail = t
        what = "oracle/pipeline.py (the CPU restatement of the reference; baseline/_ref is absent on this machine)"
    note = (f"1 image per step, {args.size}x{args.size}, {args.boxes} boxes, {depth_note} (ViT {cfg.vit['depth']} blocks, DaViT "
            f"{cfg.davit['depths']}, LLM {cfg.llm['num_hidden_layers']} layers), fp32, {cores} host threads, through {what}; "
            + (f"all {T} decode tokens executed" if dt >= T else
               f"{dt} of {T} decode tokens executed, the remaining {T - dt} added at the measured per-token time (extrapolated term: "
               f"{(T - dt) * detail.get('llm_decode_s_per_token', 0.0):.1f} s of {statistics.mean(times):.1f} s)"))
    return 1.0 / statistics.mean(times), kind, cores, note, detail


def hfre_algorithmic_bytes(HF, cfg, host, size):
    """SURVEY.md section 8d unique bytes of the HFRE stage for these samples (host-side rasterisation of the boxes)."""
    tot = 0
    for s in host:
        H0 = s.image_aux.shape[-1] // 4
        gh, gw = s.grid_hw
        Sa = s.image_aux.shape[-1]
        shapes = [(Sa // (4 << i), Sa // (4 << i), c) for i, c in enumerate(cfg.davit["dim_embed"])] + \
                 [(int(gh * f), int(gw * f), cfg.fpn_out) for f in (4, 2, 1, 0.5)]
        sc = gh * 14 / Sa
        bl = [s.boxes.numpy()] * 4 + [s.boxes.numpy() * sc] * 4
        scales = [0.25] * 4 + [1 / x for x in HF.FPN_STRIDES]
        ups = [H0 // sh[0] for sh in shapes[:4]] + [1] * 4
        tot += HF.algorithmic_bytes(shapes, bl, scales, ups, s.boxes.shape[0], cfg.region_dim)["unique_bytes"]
    return tot


DUMP_BYTES = 64_000_000


def dump_outputs(res: dict, out_dir: str) -> None:
    """Write the arrays one step returned as <out_dir>/<name>.npy: integers (token ids, lengths) as float64, which holds them
    exactly, floating-point values as float32.  An array larger than its share of DUMP_BYTES keeps a seeded sample of its rows,
    the same rows on every run, whose indices go to <name>_rows.npy."""
    arrays = {}
    for k, v in res.items():
        if v is None:
            continue
        if torch.is_tensor(v):
            v = v.detach().cpu()
            v = v.float() if v.is_floating_point() else v
        a = np.asarray(v)
        arrays[k] = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // max(len(arrays), 1) - 1024          # room for the .npy headers
    for k, a in arrays.items():
        if a.nbytes > share:
            row_bytes = a.nbytes // a.shape[0]
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], share // (row_bytes + 8), replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, f"{k}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def load_traffic(workload: str, per_gpu_batch: int):
    """DRAM bytes per launch of the roofline kernels from the committed ncu capture of this round (profiles/): the bench
    cannot run under ncu, so `traffic` is read from the capture of the same command -- one C3 step at 32 images per GPU
    (profiles/r02_ncu_dram_step.csv).  Any other workload / batch launches other shapes: no figure (null) rather than a wrong one."""
    p = os.path.join(REPO, "profiles", "r02_traffic.json")
    if workload != "c3" or per_gpu_batch != 32 or not os.path.exists(p):
        return {}
    return json.load(open(p))


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fo1", choices=["fo1", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="images per GPU (default: the workload's)")
    ap.add_argument("--global-batch", type=int, default=None, help="TOTAL images, split over the ranks (strong scaling)")
    ap.add_argument("--size", type=int, default=None)
    ap.add_argument("--boxes", type=int, default=None)
    ap.add_argument("--tokens", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", action="store_true", help="CPU legs run a bounded depth sample scaled to full depth instead of every block (~45 s per image)")
    ap.add_argument("--cpu-tokens", type=int, default=64, help="decode steps the in-run cpu_baseline executes (rest at the measured per-token time)")
    ap.add_argument("--profile-run", action="store_true", help="warm-up exactly as given, one timed pass, nothing else (for ncu)")
    ap.add_argument("--small", action="store_true", help="tiny architecture (plumbing check only; NOT a valid bench number)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path (--impl fo1)")
    wl = WORKLOADS[args.workload]
    for k in ("batch", "size", "boxes", "tokens"):
        if getattr(args, k) is None:
            setattr(args, k, wl[k])

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from importlib import import_module
    import fo1_b200  # noqa: F401
    E = import_module("vlm-fo1_b200.engine"); CK = import_module("vlm-fo1_b200.checkpoint"); DP = import_module("vlm-fo1_b200.dp")
    P = import_module("vlm-fo1_b200.pipeline"); SY = import_module("vlm-fo1_b200.synthetic"); HF = import_module("vlm-fo1_b200.hfre")
    cfg = E.EngineConfig()
    if args.small:
        cfg.vit = dict(cfg.vit, depth=4, fullatt_block_indexes=[1, 3])
        cfg.davit = dict(cfg.davit, depths=[1, 1, 1, 1])
        cfg.llm = dict(cfg.llm, num_hidden_layers=2)
    strong = args.global_batch is not None
    G = args.global_batch if strong else args.batch * world
    lo, hi = DP.shard_range(G, rank, world)                      # this rank's contiguous slice of the sample list
    B, T = hi - lo, args.tokens
    per_rank_max = max(DP.shard_range(G, r, world)[1] - DP.shard_range(G, r, world)[0] for r in range(world))
    hfre_only = args.workload == "c2"
    config = {"workload": f"{wl['name']}: {'global batch ' + str(G) if strong else 'batch ' + str(args.batch) + '/GPU'}, {args.size}x{args.size}, "
                          f"{args.boxes} boxes/img, {T}-token greedy decode, random-init 3B FO1 (variant B: SimpleFPN, D=5888, mlp2x_gelu projector)",
              "workload_id": args.workload, "global_batch": G, "per_gpu_batch": per_rank_max, "image_size": args.size,
              "boxes_per_image": args.boxes, "decode_tokens": T, "parallelism": f"dp{world}",
              "l2_policy": "working set (8.3 GB weights + GBs of activations per step) >> 126 MB L2; no flush needed",
              "small_arch": bool(args.small)}
    metric, unit = (METRIC, UNIT) if not hfre_only else ("HFRE GB/s (SURVEY 8d unique bytes / fo1_hfre_forward time), dual-ViT forward + region tokens", "GB/s")

    # ------------------------------------------------------------------ reference (CPU) arm
    if args.impl == "reference":
        if rank != 0:
            return
        # a step is ONE full-depth image (~45 s on 16 host cores); the untimed warm-up is bounded to one step (if any was asked for)
        steps = args.steps
        ips, kind, cores, note, detail = reference_arm(args, cfg, steps, min(args.cpu_tokens, max(T, 1)), warm=min(args.warmup, 1))
        value = ips
        if hfre_only:                                # the HFRE stage alone, same unit as the GPU arm
            host1 = SY.synthetic_batch(0, 1, args.size, args.boxes)
            sec = detail.get("fpn_hfre_s", detail.get("hfre_s", 0.0) + detail.get("fpn_s", 0.0))
            value = hfre_algorithmic_bytes(HF, cfg, host1, args.size) / max(sec, 1e-9) / 1e9
            note += "; value = unique HFRE bytes of that image / the reference's SimpleFP + HFREModule time"
        line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1),
                "ms_per_step": 1000.0 / ips, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": kind, "sample": note, "stage_seconds": detail},
                "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), file=out, flush=True)
        return

    # ------------------------------------------------------------------ fo1 arm
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    sds = CK.random_state_dicts(cfg, dev, 0)
    eng = CK.load_engine(cfg, sds, dev)
    keep_cpu = (rank == 0 and world == 1 and not args.no_cpu_baseline)
    del sds
    torch.cuda.empty_cache()
    pipe = P.Fo1Pipeline(eng)
    host = SY.synthetic_batch(lo, B, args.size, args.boxes)
    # end-to-end arm: the raw uint8 images in pinned host memory; resize / normalise / patchify run on the device (fo1_preprocess_*)
    host_u8 = [SY.synthetic_sample_u8(lo + k, args.size, args.boxes) for k in range(B)]
    for s in host_u8:
        s.image_u8 = s.image_u8.pin_memory(); s.boxes = s.boxes.pin_memory()
    resident = [P.SampleInputs(s.input_ids, s.pixel_values.to(dev), s.grid_hw, s.image_aux.to(dev), s.boxes.to(dev)) for s in host]
    Tc = max(T, 1)
    host_tokens = torch.empty((B, Tc), dtype=torch.int32).pin_memory()
    host_regions = torch.empty((B * args.boxes, cfg.llm["hidden_size"]), dtype=torch.bfloat16).pin_memory() if hfre_only else None

    def step(samples):
        if hfre_only:                                 # C2: towers + region tokens, no language model
            feats, img_off, region_tokens, region_f32 = pipe.encode(samples)
            return {"region_tokens": torch.cat(region_tokens, 0)}
        res = pipe.generate(samples, T, stop_ids=[], early_exit_interval=0)
        # the path's only collective: every rank's decoded ids (ragged shards padded to the largest) over NVLink
        res["all_tokens"], res["all_lens"] = DP.gather_ids(res["tokens"], res["lens"], world, per_rank_max)
        return res

    def step_e2e():
        moved = [P.SampleInputs(s.input_ids, None, None, None, s.boxes.to(dev, non_blocking=True), image_u8=s.image_u8.to(dev, non_blocking=True))
                 for s in host_u8]
        res = step(moved)
        if hfre_only:
            host_regions.copy_(res["region_tokens"], non_blocking=True)
        else:
            host_tokens.copy_(res["tokens"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return res

    def timed(fn, steps):
        """-> (ms of the steps, what the last step returned)"""
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), res

    L = fo1_b200.lib()
    if args.profile_run:
        for _ in range(args.warmup):
            step(resident)
        ms, res = timed(lambda: step(resident), args.steps)
        if rank == 0:
            if args.dump_outputs:
                dump_outputs(res, args.dump_outputs)
            print(json.dumps({"profile_run": True, "ms_per_step": ms / args.steps, "launches": int(L.fo1_launch_count())}), file=out, flush=True)
        return
    for _ in range(max(args.warmup, 3)):
        step(resident)
    torch.cuda.synchronize()
    L.fo1_launch_count_reset()
    with ClockSampler(local) as cs:
        ms, res = timed(lambda: step(resident), args.steps)
    launches = int(L.fo1_launch_count())
    clocks = cs.summary()
    ips = G * args.steps / (ms / 1000.0)
    if rank == 0 and args.dump_outputs:
        dump_outputs(res, args.dump_outputs)
    del res
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    ips_e2e = G * args.steps / (ms_e2e / 1000.0)
    h2d = sum(s.image_u8.numel() + s.boxes.numel() * 4 for s in host_u8)
    d2h = host_regions.numel() * 2 if hfre_only else B * Tc * 4

    line = {"metric": metric, "value": ips, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": ips_e2e, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "images_per_s": ips, "images_per_s_e2e": ips_e2e}

    if rank == 0:
        # ---- extra instrumented steps (rank 0 only, no collective: the other ranks are already at the final barrier) ----
        peaks = load_peaks()
        traffic = load_traffic(args.workload, B)
        if hfre_only:
            local_step = lambda: pipe.encode(resident)
        else:
            local_step = lambda: pipe.generate(resident, T, stop_ids=[], early_exit_interval=0)
        pipe.profile_stages = True
        local_step()
        line["stage_ms"] = pipe.stage_ms()          # un-instrumented kernels, CUDA events between the stages
        pipe.profile_stages = False
        L.fo1_profile_enable(1)
        local_step()
        buf = (__import__("ctypes").c_char * (1 << 20))()
        L.fo1_profile_collect(buf, 1 << 20)
        L.fo1_profile_enable(0)
        raw = json.loads(buf.value.decode())
        prof, shapes = {}, []
        for k, v in raw.items():
            base = k.split(":")[0]
            if base != k:
                shapes.append({"shape": k, **v, "tflops": (v["flops"] / v["ms"] / 1e9) if v["ms"] > 0 else 0.0,
                               "GBs": (v["bytes"] / v["ms"] / 1e6) if v["ms"] > 0 else 0.0})
            a = prof.setdefault(base, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0, "max_ms": 0.0})
            a["launches"] += v["launches"]; a["ms"] += v["ms"]; a["flops"] += v["flops"]; a["bytes"] += v["bytes"]
            a["max_ms"] = max(a["max_ms"], v["max_ms"])
        for v in prof.values():
            if v["flops"] > 0 and v["ms"] > 0:
                v["tflops"] = v["flops"] / v["ms"] / 1e9
        line["kernel_profile"] = prof
        line["gemm_shapes_top"] = sorted(shapes, key=lambda r: -r["ms"])[:14]
        step_ms = ms / args.steps
        g = prof.get("gemm")
        roof_gemm = None
        if g and g["ms"] > 0:
            ach = g["flops"] / g["ms"] / 1e9
            roof_gemm = {"kernel": "gemm_bf16_tcgen05_pair_kernel (CTA pairs, tcgen05.mma.cta_group::2; the few sub-wave problems: gemm_bf16_tcgen05_kernel), M > 128 launches of one step", "bound": "tensor", "achieved": ach,
                         "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"], "traffic": traffic.get("gemm_bytes_per_launch"),
                         "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']})",
                         "launches": g["launches"], "ms_per_launch": g["ms"] / g["launches"], "share_of_step": g["ms"] / step_ms,
                         "algorithmic_bytes_per_launch": g["bytes"] / g["launches"]}
        for tag in ("attn", "attn_causal"):
            a = prof.get(tag)
            if a and a["ms"] > 0 and a["flops"] > 0:
                ach = a["flops"] / a["ms"] / 1e9
                line["roofline_" + tag] = {"kernel": "attn_tc_kernel (tcgen05 flash attention" + (", causal GQA prefill)" if tag == "attn_causal" else ", ViT / DaViT)"),
                                           "bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"],
                                           "traffic": traffic.get(tag + "_bytes_per_launch"), "launches": a["launches"], "share_of_step": a["ms"] / step_ms}
        h = prof.get("hfre_sweep_mma") or prof.get("hfre_sweep") or prof.get("hfre_gather")
        roof_hfre = None
        if h and h["ms"] > 0:
            tot = hfre_algorithmic_bytes(HF, cfg, host, args.size)
            ach = tot / h["ms"] / 1e6
            hname = "hfre_sweep_mma_kernel" if "hfre_sweep_mma" in prof else ("hfre_sweep_kernel" if "hfre_sweep" in prof else "hfre_gather_kernel")
            stage = line["stage_ms"].get("hfre")
            roof_hfre = {"kernel": hname, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                         "traffic": traffic.get("hfre_bytes_per_launch"), "algorithmic_bytes": tot, "launches": h["launches"],
                         "algorithmic_bytes_per_launch": tot / h["launches"], "ms": h["ms"],
                         "operator_ms": stage, "operator_GBs": (tot / stage / 1e6) if stage else None,
                         "operator_frac": (tot / stage / 1e6 / peaks["hbm_gbs"]) if stage else None,
                         "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks['source']})"}
            line["roofline_hfre"] = roof_hfre
        if hfre_only and roof_hfre:
            # C2's metric IS the HFRE rate: value = whole operator (all its kernels), roofline = its sweep kernel
            line["value"] = roof_hfre["operator_GBs"]
            line["e2e"]["value"] = roof_hfre["operator_GBs"]; line["e2e"]["note"] = "images_per_s_e2e carries the host-buffer images/s of the C2 step"
            line["roofline"] = roof_hfre
        elif roof_gemm:
            line["roofline"] = roof_gemm
        if not hfre_only and T > 2:
            # one decode step: what it must stream (bf16 weights of every layer + head, K/V of the live prefixes) over its time
            lc = cfg.llm
            hd = lc["hidden_size"] // lc["num_attention_heads"]
            per_layer = lc["hidden_size"] * (lc["num_attention_heads"] + 2 * lc["num_key_value_heads"]) * hd + lc["hidden_size"] ** 2 + \
                3 * lc["hidden_size"] * lc["intermediate_size"]
            wbytes = 2 * (lc["num_hidden_layers"] * per_layer + lc["vocab_size"] * lc["hidden_size"])
            prompt = sum(len(s.input_ids) - 1 + s.grid_hw[0] * s.grid_hw[1] // 4 for s in host)
            kv = 2 * 2 * lc["num_hidden_layers"] * lc["num_key_value_heads"] * hd * (prompt + B * T / 2)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e2 = torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(); pipe.generate(resident, 2, stop_ids=[], early_exit_interval=0); e1.record()
            pipe.generate(resident, T, stop_ids=[], early_exit_interval=0); e2.record()
            torch.cuda.synchronize()
            dms = (e1.elapsed_time(e2) - e0.elapsed_time(e1)) / (T - 2)
            ach = (wbytes + kv) / dms / 1e6
            path = pipe.eng.last_decode_path()
            kname = ("decode_mega_kernel (persistent cooperative kernel: the whole greedy loop in one launch), per decode step" if path == 1
                     else "one greedy decode step (CUDA graph of the per-layer kernels)")
            line["roofline_decode"] = {"kernel": kname, "bound": "hbm", "achieved": ach,
                                       "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None,
                                       "algorithmic_bytes": wbytes + kv, "weight_bytes": wbytes, "kv_bytes": kv, "ms_per_step": dms,
                                       "share_of_step": dms * (T - 1) / step_ms}
        # ---- CPU baseline (rank 0, N = 1 only): the reference's own modules on the host cores ----
        if keep_cpu:
            try:
                cips, kind, cores, note, detail = reference_arm(args, cfg, 1, args.cpu_tokens)
                cval = cips
                if hfre_only:
                    sec = detail.get("fpn_hfre_s", detail.get("hfre_s", 0.0) + detail.get("fpn_s", 0.0))
                    cval = hfre_algorithmic_bytes(HF, cfg, host[:1], args.size) / max(sec, 1e-9) / 1e9
                line["cpu_baseline"] = {"value": cval, "unit": unit, "cores": cores, "kind": kind, "sample": note, "stage_seconds": detail}
            except Exception as exc:  # the baseline is a report, never a reason to lose the GPU number
                line["cpu_baseline"] = {"value": None, "unit": unit, "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {exc!r}"}
        print(json.dumps(line), file=out, flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def _claim_stdout():
    """stdout carries exactly ONE JSON line: libraries that print from C (NCCL's version banner) go to stderr instead.
    Returns a text handle on the original stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(os.dup(2), "w", buffering=1)
    return os.fdopen(real, "w", buffering=1)


if __name__ == "__main__":
    main()
