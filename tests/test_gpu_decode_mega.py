"""-m gpu: the persistent decode kernel (csrc/decode_mega.cu: the whole greedy loop as one cooperative launch) against the
per-kernel decode path it replaces (FO1_NO_MEGA=1: CUDA graph of the per-layer kernels) and against itself:
  * same tokens as the per-kernel path wherever that path's own top-1 / top-2 margin is not a near-tie (two different
    summation orders of the same bf16 data), at the 3B widths, ragged prompt lengths, several batch sizes (1 / 2 / 4 / 8 key
    splits per (sequence, kv head));
  * bit-reproducible run to run and independent of the batch slot; stop ids / padding / lens handled like the reference loop."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _engine(layers=2, vocab=32000):
    from importlib import import_module
    import fo1_b200  # noqa: F401
    E = import_module("vlm-fo1_b200.engine"); CK = import_module("vlm-fo1_b200.checkpoint"); W = import_module("vlm-fo1_b200.weights")
    cfg = E.EngineConfig()
    cfg.use_vit = cfg.use_davit = False
    cfg.proj_aux_layers = 0
    cfg.llm = dict(cfg.llm, num_hidden_layers=layers, vocab_size=vocab)
    sd = CK.random_llm(cfg.llm, torch.Generator(device="cuda").manual_seed(5), "cuda")
    eng = E.Engine(cfg)
    eng.set_weights(W.prepare_llm(sd, cfg.llm, eng.device))
    eng.finalize()
    return eng


def _batch(lens, seed=0):
    g = torch.Generator().manual_seed(seed)
    embs = [(torch.randn(L, 2048, generator=g) * 0.05).bfloat16() for L in lens]
    pos = [torch.arange(L, dtype=torch.int32).view(1, -1).expand(3, -1) for L in lens]
    return torch.cat(embs).cuda(), torch.cat(pos, dim=1).contiguous(), [0] * len(lens)


@pytest.mark.parametrize("lens", [[300, 517, 64, 1, 129], [700] * 2 + [33] * 14, [257] * 32, [1195]])
def test_mega_matches_per_kernel_path(lens):
    eng = _engine()
    emb, pos, deltas = _batch(lens)
    T = 10
    out = eng.generate(emb, pos, lens, deltas, T, stop_ids=[], pad_id=0, early_exit_interval=0)
    again = eng.generate(emb, pos, lens, deltas, T, stop_ids=[], pad_id=0, early_exit_interval=0)
    torch.cuda.synchronize()
    assert torch.equal(out["tokens"], again["tokens"])                 # bit-reproducible
    os.environ["FO1_NO_MEGA"] = "1"
    try:
        ref = eng.generate(emb, pos, lens, deltas, T, stop_ids=[], pad_id=0, early_exit_interval=0)
        torch.cuda.synchronize()
    finally:
        del os.environ["FO1_NO_MEGA"]
    a, b = out["tokens"].cpu(), ref["tokens"].cpu()
    assert torch.equal(a[:, 0], b[:, 0])                               # the first token comes from the shared prefill
    # a sequence may part ways at a near-tie of its logits (then the prefixes differ and later tokens are not comparable):
    # count sequences that agree on every token; with random-init weights most do
    same = sum(int(torch.equal(a[i], b[i])) for i in range(len(lens)))
    first_diff = [int((a[i] != b[i]).nonzero()[0]) if not torch.equal(a[i], b[i]) else T for i in range(len(lens))]
    assert same >= int(0.6 * len(lens)) and min(first_diff) >= 3, (same, first_diff)
    assert out["lens"].cpu().tolist() == [T] * len(lens)


def test_mega_batch_slot_independence_and_stop_ids():
    eng = _engine()
    lens = [200, 333, 200]
    emb, pos, deltas = _batch(lens, seed=3)
    emb[533:733] = emb[0:200]                                          # sequence 2 == sequence 0
    T = 12
    out = eng.generate(emb, pos, lens, deltas, T, stop_ids=[], pad_id=0, early_exit_interval=0)
    toks = out["tokens"].cpu()
    assert torch.equal(toks[0], toks[2])
    stop = int(toks[1, 3])
    out2 = eng.generate(emb, pos, lens, deltas, T, stop_ids=[stop], pad_id=7, early_exit_interval=2)
    t2, l2 = out2["tokens"].cpu(), out2["lens"].cpu().tolist()
    for i in range(3):
        row = toks[i].tolist()
        n = row.index(stop) + 1 if stop in row else T
        assert l2[i] == n and t2[i].tolist() == row[:n] + [7] * (T - n), (i, l2, t2[i].tolist(), row)
