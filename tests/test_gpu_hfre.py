"""-m gpu: the CUDA HFRE (through the C ABI) vs the oracle and vs the reference-module goldens."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _hwc(a):  # [C,H,W] numpy -> channels-last bf16 CUDA
    return torch.from_numpy(np.ascontiguousarray(a.transpose(1, 2, 0))).to("cuda", torch.bfloat16).contiguous()


def _nerr(got, ref):
    return float((got - ref).abs().max() / ref.abs().max())


@pytest.mark.parametrize("algo", [1, 3])
@pytest.mark.parametrize("tag", ["small", "rect"])
def test_hfre_matches_reference_goldens(golden_dir, tag, algo):
    import fo1_b200  # noqa: F401
    from importlib import import_module
    H = import_module("vlm-fo1_b200.hfre")
    z = np.load(os.path.join(golden_dir, f"hfre_{tag}.npz"))
    aux = [_hwc(z[f"aux{i}"]) for i in range(4)]
    taps = [_hwc(z[f"tap{i}"]) for i in range(4)]
    pyr = [_hwc(z[f"pyr{i}"]) for i in range(4)]
    boxes = torch.from_numpy(z["boxes"]).cuda(); vtb = torch.from_numpy(z["vt_boxes"]).cuda()
    grid = tuple(int(v) for v in z["grid_hw"])
    D = z["out_fpn"].shape[1]
    out_b = H.hfre_forward([aux], [pyr], [boxes], [vtb], H.HfreConfig(region_dim=D, vt_mode="fpn", algo=algo), [grid])[0]
    out_a = H.hfre_forward([aux], [taps], [boxes], [vtb], H.HfreConfig(region_dim=D, vt_mode="concat", algo=algo), [grid])[0]
    torch.cuda.synchronize()
    # tolerance: 1e-3 relative (north_star); measured against the golden's max magnitude per tensor
    assert _nerr(out_b.cpu(), torch.from_numpy(z["out_fpn"])) < 1e-3
    assert _nerr(out_a.cpu(), torch.from_numpy(z["out_concat"])) < 1e-3
    np.testing.assert_allclose(out_b.cpu().numpy(), z["out_fpn"], rtol=1e-3, atol=2e-4)
    np.testing.assert_allclose(out_a.cpu().numpy(), z["out_concat"], rtol=1e-3, atol=2e-4)


@pytest.mark.parametrize("algo", [1, 3])
@pytest.mark.parametrize("S,N", [(448, 37), (896, 100)])
def test_hfre_matches_oracle_full_shapes(S, N, algo):
    """DaViT-large / SimpleFPN shaped maps at real resolution, batch of 2 images, ragged box counts."""
    from importlib import import_module
    from oracle import hfre as O
    H = import_module("vlm-fo1_b200.hfre")
    g = torch.Generator().manual_seed(7)
    chans = (256, 512, 1024, 2048)
    B = 2
    aux_all, pyr_all, boxes_all, grid_all, n_all = [], [], [], [], [N, max(N // 3, 1)]
    gh = S // 14
    for b in range(B):
        aux = [torch.randn(S // (4 << i), S // (4 << i), c, generator=g).to(torch.bfloat16) for i, c in enumerate(chans)]
        pyr = [torch.randn(int(gh * f), int(gh * f), 512, generator=g).to(torch.bfloat16) for f in (4, 2, 1, 0.5)]
        n = n_all[b]
        w = torch.rand(n, generator=g) * (S / 2 - 32) + 32; h = torch.rand(n, generator=g) * (S / 2 - 32) + 32
        x1 = torch.rand(n, generator=g) * (S - w); y1 = torch.rand(n, generator=g) * (S - h)
        boxes = torch.stack([x1, y1, x1 + w, y1 + h], 1)
        aux_all.append(aux); pyr_all.append(pyr); boxes_all.append(boxes); grid_all.append((gh, gh))
    sc = gh * 14 / S
    cfg = H.HfreConfig(region_dim=5888, vt_mode="fpn", algo=algo)
    outs = H.hfre_forward([[a.cuda() for a in aux] for aux in aux_all], [[p.cuda() for p in pyr] for pyr in pyr_all],
                          [b.cuda() for b in boxes_all], [(b * sc).cuda() for b in boxes_all], cfg, grid_all)
    torch.cuda.synchronize()
    for b in range(B):
        nb = min(n_all[b], 12)  # the oracle materialises the up-sampled map: keep the CPU side to seconds
        ref = O.hfre_forward([a.float().permute(2, 0, 1) for a in aux_all[b]], boxes_all[b][:nb],
                             [p.float().permute(2, 0, 1) for p in pyr_all[b]], boxes_all[b][:nb] * sc,
                             vt_mode="fpn", region_dim=5888, vt_grid_hw=grid_all[b])
        assert _nerr(outs[b][:nb].cpu(), ref) < 1e-3


def test_hfre_empty_and_errors():
    from importlib import import_module
    H = import_module("vlm-fo1_b200.hfre")
    L = import_module("vlm-fo1_b200._lib")
    aux = [torch.zeros(8 >> i, 8 >> i, 8, dtype=torch.bfloat16, device="cuda") for i in range(4)]
    pyr = [torch.zeros(4, 4, 8, dtype=torch.bfloat16, device="cuda") for _ in range(4)]
    empty = torch.zeros(0, 4, device="cuda")
    out = H.hfre_forward([aux], [pyr], [empty], [empty], H.HfreConfig(region_dim=64), [(2, 2)])[0]
    assert out.shape == (0, 64)
    with pytest.raises(ValueError):   # region_dim smaller than the channels provided -> rejected on the host side
        H.hfre_forward([aux], [pyr], [empty], [empty], H.HfreConfig(region_dim=16), [(2, 2)])
    bad = [torch.zeros(8, 8, 12, dtype=torch.bfloat16, device="cuda")] + aux[1:]  # C % 8 != 0
    one = torch.tensor([[0.0, 0.0, 4.0, 4.0]], device="cuda")
    with pytest.raises(L.Fo1Error):
        H.hfre_forward([bad], [pyr], [one], [one], H.HfreConfig(region_dim=128), [(2, 2)])
    with pytest.raises(L.Fo1Error):   # algo: 0 auto, 1 gather, 3 sweep
        H.hfre_forward([aux], [pyr], [one], [one], H.HfreConfig(region_dim=128, algo=2), [(2, 2)])


def test_hfre_packed_batch_is_the_same_operator():
    """hfre_forward_packed (batch-contiguous maps, packed boxes, descriptors filled with array arithmetic) must give bit-identical
    rows to the per-image list form, ragged box counts included."""
    import fo1_b200  # noqa: F401
    from importlib import import_module
    H = import_module("vlm-fo1_b200.hfre")
    g = torch.Generator().manual_seed(11)
    B, S, D = 3, 224, 5888
    aux_b = [torch.randn(B, S // (4 << i), S // (4 << i), c, generator=g).to(torch.bfloat16).cuda() for i, c in enumerate((256, 512, 1024, 2048))]
    vt_b = [torch.randn(B, int(16 * f), int(16 * f), 512, generator=g).to(torch.bfloat16).cuda() for f in (4, 2, 1, 0.5)]
    counts = [5, 1, 9]
    boxes = []
    for n in counts:
        xy = torch.rand(n, 2, generator=g) * (S - 40)
        wh = torch.rand(n, 2, generator=g) * 120 + 2
        boxes.append(torch.cat([xy, torch.minimum(xy + wh, torch.tensor(float(S)))], 1).cuda())
    cfg = H.HfreConfig(region_dim=D, vt_mode="fpn")
    aux = [[aux_b[l][b] for l in range(4)] for b in range(B)]
    vt = [[vt_b[l][b] for l in range(4)] for b in range(B)]
    ref32, ref16 = H.hfre_forward(aux, vt, boxes, boxes, cfg, [(16, 16)] * B, want_bf16=True)
    ba = torch.cat(boxes, 0).contiguous()
    out32, out16 = H.hfre_forward_packed(aux_b, vt_b, ba, ba.clone(), counts, cfg, (16, 16), want_bf16=True)
    torch.cuda.synchronize()
    assert torch.equal(out32, torch.cat(ref32, 0)) and torch.equal(out16, torch.cat(ref16, 0))
    with pytest.raises(Exception):
        H.hfre_forward_packed(aux_b, vt_b, ba, ba, [5, 1, 8], cfg, (16, 16))
