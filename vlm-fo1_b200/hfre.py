"""Host side of the HFRE operator: mirrors ``HFREModule.__call__``
(hybrid_finegrained_region_encoder.py:275-468) as called from ``encode_regions``
(omchat_qwen2_5_vl.py:75-128), over ``fo1_hfre_forward``.

Feature maps are channels-last bf16 ``[H, W, C]`` device tensors at NATIVE resolution (what the
towers of this engine emit); nothing is up-sampled or concatenated."""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import HfreImage, HfreLevel, HfreParams, check, lib

FPN_STRIDES = (3.5, 7.0, 14.0, 28.0)   # hybrid_finegrained_region_encoder.py:245
AUX_SCALE = 0.25                        # omchat_arch.py:29
VT_SCALE = 1.0 / 14.0                   # omchat_arch.py:27


@dataclass
class HfreConfig:
    """The ``mm_*`` flags that select the HFRE variant (omchat_arch.py:17-31)."""
    region_dim: int                       # mm_region_hidden_size
    vt_mode: str = "fpn"                  # 'fpn' (mm_use_simpleFPN_for_vt) | 'concat'
    roi_size: int = 7                     # mm_roi_output_size
    apply_pos_embed: bool = True          # mm_apply_position_embedding (bbox_based)
    algo: int = 0                         # fo1_hfre_params.algo: 0 auto, 1 per-box gather, 3 map sweep


class HfreWorkspace:
    """Grow-only device scratch for the per-box weight vectors (no allocation on the hot path once warm)."""

    def __init__(self) -> None:
        self.buf: Optional[torch.Tensor] = None

    def get(self, nbytes: int, device) -> torch.Tensor:
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        return self.buf


_default_ws = HfreWorkspace()


def _level_table(aux_shapes, vt_shapes, cfg: HfreConfig):
    """``(up_H, up_W, spatial_scale, box_set, out_offset)`` of every level, aux levels first, from the levels' native
    ``(H, W, C)`` shapes."""
    H0 = max(s[0] for s in aux_shapes)
    W0 = max(s[1] for s in aux_shapes)
    if cfg.vt_mode == "fpn":
        vt_scales = [1.0 / FPN_STRIDES[i] for i in range(len(vt_shapes))]
    elif cfg.vt_mode == "concat":
        vt_scales = [VT_SCALE] * len(vt_shapes)
    else:
        raise ValueError(f"unknown vt_mode {cfg.vt_mode!r}")
    rows = []
    off = 0
    for s in aux_shapes:  # aux levels are up-sampled to level 0's grid by the reference (:338-350)
        rows.append((H0, W0, AUX_SCALE, 0, off))
        off += s[2]
    for s, sc in zip(vt_shapes, vt_scales):
        rows.append((s[0], s[1], sc, 1, off))
        off += s[2]
    if off > cfg.region_dim:
        raise ValueError(f"levels provide {off} channels > region_dim {cfg.region_dim}")
    if len(rows) > _lib.FO1_HFRE_MAX_LEVELS:
        raise ValueError("too many feature levels")
    return rows


def _launch(imgs, n_images: int, cfg: HfreConfig, dev, workspace: Optional[HfreWorkspace]) -> None:
    p = HfreParams(cfg.region_dim, cfg.roi_size, 1 if cfg.apply_pos_embed else 0, cfg.algo)
    L = lib()
    need = L.fo1_hfre_workspace_bytes(imgs, n_images, C.byref(p))
    ws = (workspace or _default_ws).get(need, dev)
    check(L.fo1_hfre_forward(imgs, n_images, C.byref(p), C.c_void_p(ws.data_ptr()), ws.numel(),
                             C.c_void_p(torch.cuda.current_stream().cuda_stream)), "fo1_hfre_forward")


def _fill_image(img: HfreImage, aux_feats, vt_feats, boxes_aux, boxes_vt, out, out_bf16, cfg, vt_grid_hw):
    rows = _level_table([f.shape for f in aux_feats], [f.shape for f in vt_feats], cfg)
    for i, (f, (uh, uw, sc, bs, o)) in enumerate(zip(list(aux_feats) + list(vt_feats), rows)):
        if f.dtype != torch.bfloat16 or not f.is_contiguous() or f.dim() != 3 or not f.is_cuda:
            raise _lib.Fo1Error("HFRE levels must be contiguous channels-last bf16 CUDA tensors [H, W, C]")
        L = img.levels[i]
        L.data = f.data_ptr(); L.H, L.W, L.C = f.shape
        L.up_H, L.up_W = uh, uw
        L.spatial_scale = sc; L.box_set = bs; L.out_offset = o
    img.n_levels = len(rows)
    img.n_boxes = boxes_aux.shape[0]
    img.boxes_aux = boxes_aux.data_ptr(); img.boxes_vt = boxes_vt.data_ptr()
    img.out = out.data_ptr()
    img.out_bf16 = out_bf16.data_ptr() if out_bf16 is not None else None
    gh, gw = vt_grid_hw
    img.pos_img_w = gw / VT_SCALE   # :447-448 (python float, rounded to fp32 at the division like the reference)
    img.pos_img_h = gh / VT_SCALE
    img.pos_box_set = 1


def hfre_forward(aux_feats: Sequence[Sequence[torch.Tensor]], vt_feats: Sequence[Sequence[torch.Tensor]],
                 boxes_aux: Sequence[torch.Tensor], boxes_vt: Sequence[torch.Tensor], cfg: HfreConfig,
                 vt_grid_hw: Sequence[Sequence[int]], want_bf16: bool = False,
                 workspace: Optional[HfreWorkspace] = None):
    """Region features for a batch of images.  Per image ``b``: ``aux_feats[b]`` = 4 DaViT stage maps,
    ``vt_feats[b]`` = 4 SimpleFPN levels ('fpn') or the 4 ViT tap maps ('concat'), all [H, W, C] bf16;
    ``boxes_*[b]`` fp32 [N_b, 4] xyxy.  Returns a list of fp32 [N_b, D] (and bf16 copies if asked)."""
    B = len(aux_feats)
    imgs = (HfreImage * B)()
    outs, outs16 = [], []
    keep = []
    for b in range(B):
        ba = boxes_aux[b].to(torch.float32).contiguous()
        bv = boxes_vt[b].to(torch.float32).contiguous()
        keep += [ba, bv]
        n = ba.shape[0]
        o = torch.empty((n, cfg.region_dim), dtype=torch.float32, device=ba.device)
        o16 = torch.empty((n, cfg.region_dim), dtype=torch.bfloat16, device=ba.device) if want_bf16 else None
        outs.append(o); outs16.append(o16)
        _fill_image(imgs[b], aux_feats[b], vt_feats[b], ba, bv, o, o16, cfg, vt_grid_hw[b])
    _launch(imgs, B, cfg, outs[0].device if outs else torch.device("cuda"), workspace)
    return (outs, outs16) if want_bf16 else outs


_IMG_DTYPE = np.dtype(HfreImage)


def hfre_forward_packed(aux_levels: Sequence[torch.Tensor], vt_levels: Sequence[torch.Tensor], boxes_aux: torch.Tensor,
                        boxes_vt: torch.Tensor, counts: Sequence[int], cfg: HfreConfig, vt_grid_hw: Sequence[int],
                        want_bf16: bool = False, workspace: Optional[HfreWorkspace] = None):
    """hfre_forward for a batch whose images share their shapes (the serving case): ``aux_levels[l]`` / ``vt_levels[l]`` are the
    batch-contiguous maps bf16 [B, H_l, W_l, C_l] the towers emit, ``boxes_*`` fp32 [sum N_b, 4] packed in image order, ``counts[b]``
    = N_b.  Same operator, same descriptors -- they are filled with array arithmetic instead of a Python loop over images x levels,
    and the outputs are one packed fp32 [sum N_b, D] tensor (+ its bf16 copy), image b at rows sum(counts[:b]) .. ."""
    B = len(counts)
    dev = boxes_aux.device
    for f in list(aux_levels) + list(vt_levels):
        if f.dtype != torch.bfloat16 or not f.is_contiguous() or f.dim() != 4 or not f.is_cuda or f.shape[0] != B:
            raise _lib.Fo1Error("HFRE packed levels must be contiguous channels-last bf16 CUDA tensors [B, H, W, C]")
    if boxes_aux.dtype != torch.float32 or boxes_vt.dtype != torch.float32 or not boxes_aux.is_contiguous() or not boxes_vt.is_contiguous():
        raise _lib.Fo1Error("HFRE packed boxes must be contiguous fp32 [sum N, 4]")
    total = int(sum(counts))
    if boxes_aux.shape != (total, 4) or boxes_vt.shape != (total, 4):
        raise _lib.Fo1Error("HFRE packed boxes do not match counts")
    rows = _level_table([f.shape[1:] for f in aux_levels], [f.shape[1:] for f in vt_levels], cfg)
    out = torch.empty((total, cfg.region_dim), dtype=torch.float32, device=dev)
    out16 = torch.empty((total, cfg.region_dim), dtype=torch.bfloat16, device=dev) if want_bf16 else None
    imgs = (HfreImage * B)()
    a = np.frombuffer(imgs, dtype=_IMG_DTYPE)
    idx = np.arange(B, dtype=np.uint64)
    lv = a["levels"]
    for i, (f, (uh, uw, sc, bs, o)) in enumerate(zip(list(aux_levels) + list(vt_levels), rows)):
        lv["data"][:, i] = np.uint64(f.data_ptr()) + idx * np.uint64(f.stride(0) * 2)
        lv["H"][:, i], lv["W"][:, i], lv["C"][:, i] = f.shape[1], f.shape[2], f.shape[3]
        lv["up_H"][:, i], lv["up_W"][:, i] = uh, uw
        lv["spatial_scale"][:, i] = sc; lv["box_set"][:, i] = bs; lv["out_offset"][:, i] = o
    cnt = np.asarray(counts, dtype=np.uint64)
    row0 = np.concatenate([[0], np.cumsum(cnt)[:-1]]).astype(np.uint64)
    a["n_levels"] = len(rows)
    a["n_boxes"] = cnt.astype(np.int32)
    a["boxes_aux"] = np.uint64(boxes_aux.data_ptr()) + row0 * np.uint64(16)
    a["boxes_vt"] = np.uint64(boxes_vt.data_ptr()) + row0 * np.uint64(16)
    a["out"] = np.uint64(out.data_ptr()) + row0 * np.uint64(cfg.region_dim * 4)
    a["out_bf16"] = (np.uint64(out16.data_ptr()) + row0 * np.uint64(cfg.region_dim * 2)) if want_bf16 else np.uint64(0)
    gh, gw = vt_grid_hw
    a["pos_img_w"] = gw / VT_SCALE      # :447-448 (python float, rounded to fp32 at the division like the reference)
    a["pos_img_h"] = gh / VT_SCALE
    a["pos_box_set"] = 1
    _launch(imgs, B, cfg, dev, workspace)
    return (out, out16) if want_bf16 else out


def algorithmic_bytes(level_shapes, level_boxes, level_scales, level_up, n_boxes: int, out_dim: int) -> dict:
    """SURVEY.md section 8d accounting for one image: unique native-resolution bf16 cells inside the
    union of the boxes' sample windows x C x 2 B + fp32 output + the two box arrays; and the no-reuse
    figure (every box's window counted separately).  ``level_shapes[l] = (H, W, C)`` native,
    ``level_scales[l]`` the ROIAlign scale on the up-sampled grid, ``level_up[l]`` = up/native factor."""
    unique = 0
    gather = 0
    for (H, W, Cn), boxes, sc, up in zip(level_shapes, level_boxes, level_scales, level_up):
        mask = np.zeros((H, W), dtype=bool)
        Hu, Wu = H * up, W * up
        for x1, y1, x2, y2 in np.asarray(boxes, dtype=np.float64):
            ys, xs = y1 * sc, x1 * sc
            ye, xe = max(y2 * sc, ys + 1.0), max(x2 * sc, xs + 1.0)
            r0 = min(max(int(math.floor(ys)), 0), Hu - 1); r1 = min(max(int(math.floor(ye)) + 1, 0), Hu - 1)
            c0 = min(max(int(math.floor(xs)), 0), Wu - 1); c1 = min(max(int(math.floor(xe)) + 1, 0), Wu - 1)
            if up > 1:
                r0 = max(int(math.floor((r0 + 0.5) / up - 0.5)), 0); r1 = min(int(math.floor((r1 + 0.5) / up - 0.5)) + 1, H - 1)
                c0 = max(int(math.floor((c0 + 0.5) / up - 0.5)), 0); c1 = min(int(math.floor((c1 + 0.5) / up - 0.5)) + 1, W - 1)
            mask[r0:r1 + 1, c0:c1 + 1] = True
            gather += (r1 - r0 + 1) * (c1 - c0 + 1) * Cn * 2
        unique += int(mask.sum()) * Cn * 2
    io = n_boxes * out_dim * 4 + n_boxes * 16 * 2
    return {"unique_bytes": unique + io, "gather_bytes": gather + io, "io_bytes": io}
