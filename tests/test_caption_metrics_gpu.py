"""coco-caption validation metrics on the device (sc_bleu_stats, sc_rouge_l, sc_cider_score, sc_caption_metrics_reduce via
metrics.CaptionMetrics) against the oracle, the CIDEr-D reward it shares its kernel with, and eval_on_split(metrics=...)."""
import os

import numpy as np
import pytest
import torch

from oracle import caption_metrics_oracle as M
from tests import golden_io

pytestmark = pytest.mark.gpu
DEV = "cuda"
EOS, PAD = 3, 0


def _random_split(seed, n_img, L=64):
    """Captions of lengths 0..64 over a small vocabulary (repeated n-grams), pads inside and garbage after <eos>, 1..7
    references per image, some longer than 64 tokens, a few ids near 65535."""
    rng = np.random.RandomState(seed)
    word = lambda: int(rng.randint(4, 12)) if rng.rand() < 0.97 else int(rng.randint(60000, 65536))
    refs, hyps = [], []
    rows = np.full((n_img, L), 7, dtype=np.int32)
    for i in range(n_img):
        refs.append([[word() for _ in range(rng.randint(1, 14) if rng.rand() < 0.85 else rng.randint(60, 100))]
                     for _ in range(rng.randint(1, 8))])
        n = int(rng.choice([0, 64, rng.randint(1, 20), rng.randint(1, 64)], p=[0.05, 0.05, 0.6, 0.3]))
        h = [word() for _ in range(n)]
        if i % 3 == 0 and n:                       # sometimes a copy of a reference's prefix
            src = refs[-1][0][:n]
            h = src + h[len(src):]
        hyps.append(h)
        pos = 0
        for j, w in enumerate(h):
            if pos + (n - j) < L and rng.rand() < 0.05:   # pads inside the caption are dropped
                rows[i, pos] = PAD
                pos += 1
            rows[i, pos] = w
            pos += 1
        if pos < L:
            rows[i, pos] = EOS
        hyps[-1] = [int(t) for t in rows[i, :pos] if t != PAD]
    return refs, hyps, torch.from_numpy(rows)


def _metrics(refs):
    from sparse_caption_b200.metrics import CaptionMetrics
    m = CaptionMetrics(eos_id=EOS, pad_id=PAD, device=DEV)
    m.set_refs(refs)
    return m


def test_device_metrics_match_the_oracle():
    refs, hyps, rows = _random_split(11, 300)
    m = _metrics(refs)
    perm = torch.from_numpy(np.random.RandomState(2).permutation(len(refs)))
    for part in (perm[:170], perm[170:]):       # two batches, images in shuffled order
        m.add(rows[part].to(DEV), part.to(DEV))
    scores, per = m.compute()
    want, want_per = M.evaluate(hyps, refs)
    for k in M.METRICS:
        assert scores[k] == pytest.approx(want[k], rel=1e-12, abs=1e-15), k
    assert per.dtype == torch.float64 and tuple(per.shape) == (len(refs), 6)
    np.testing.assert_allclose(per.numpy(), want_per, rtol=1e-12, atol=1e-15)
    # BLEU's sufficient statistics are exact integers
    stats = m._stats.cpu().numpy()
    for i, (h, rs) in enumerate(zip(hyps, refs)):
        c = M.bleu_cook_test(h, M.bleu_cook_refs(rs))
        assert stats[i].tolist() == c["correct"] + c["guess"] + [c["testlen"], c["reflen"]], i
    # one fixed reduction order: bitwise equal on a second run
    scores2, per2 = m.compute()
    assert scores2 == scores and torch.equal(per2, per)
    # reset() forgets the hypotheses, not the references
    m.reset()
    m.add(rows.to(DEV), torch.arange(len(refs), device=DEV))
    scores3, per3 = m.compute()
    assert scores3 == scores and torch.equal(per3, per)


def test_ciderd_reward_unchanged_on_the_golden():
    from sparse_caption_b200.cider import CiderD
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ciderd.npz"))
    unpad = lambda a: [[int(x) for x in r if x >= 0] for r in a]
    refs_flat, hyps = unpad(z["refs"]), unpad(z["hyps"])
    refs, o = [], 0
    for c in z["ref_count"]:
        refs.append(refs_flat[o: o + int(c)])
        o += int(c)
    ns = len(hyps) // len(refs)
    tok = torch.zeros(len(hyps), 16, dtype=torch.int32)
    for i, h in enumerate(hyps):
        tok[i, : len(h)] = torch.tensor(h, dtype=torch.int32)
        if len(h) < 16:
            tok[i, len(h)] = EOS
    table = {tuple(int(x) for x in k if x >= 0): float(c) for k, c in zip(z["df_ngrams"], z["df_counts"])}
    sc = CiderD(table, float(z["df_docs"]), device=DEV)
    sc.set_refs(refs)
    img = torch.arange(len(refs)).repeat_interleave(ns).to(DEV)
    got = sc.score(tok.to(DEV), img)
    np.testing.assert_allclose(got.cpu().numpy(), z["cached_scores"], rtol=1e-12, atol=1e-13)
    assert torch.equal(sc.score(tok.to(DEV), img), got)


def test_add_does_not_synchronise():
    refs, hyps, rows = _random_split(5, 64)
    m = _metrics(refs)
    seq, idx = rows.to(DEV).long(), torch.arange(len(refs), device=DEV)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        m.add(seq[:40], idx[:40])
        m.add(seq[40:], idx[40:])
    finally:
        torch.cuda.set_sync_debug_mode(0)
    scores, _ = m.compute()
    assert scores["CIDEr"] == pytest.approx(M.evaluate(hyps, refs)[0]["CIDEr"], rel=1e-12)


def test_every_image_needs_exactly_one_hypothesis():
    refs, hyps, rows = _random_split(3, 20)
    m = _metrics(refs)
    seq = rows.to(DEV)
    m.add(seq[:19], torch.arange(19, device=DEV))
    with pytest.raises(ValueError, match="1 of 20 images have none"):
        m.compute()
    m.add(seq[:2], torch.tensor([19, 4], device=DEV))
    with pytest.raises(ValueError, match="1 more than one"):
        m.compute()
    m.reset()
    m.add(seq, torch.arange(20, device=DEV))
    m.add(seq[:1], torch.tensor([20], device=DEV))
    with pytest.raises(ValueError, match="1 hypotheses have an image index outside"):
        m.compute()
    m.reset()
    m.add(seq, torch.arange(20, device=DEV))
    assert m.compute()[0]["CIDEr"] == pytest.approx(M.evaluate(hyps, refs)[0]["CIDEr"], rel=1e-12)


def _refs_for(rng, n_img, lo, hi):
    return [[[int(w) for w in rng.randint(lo, hi, rng.randint(2, 9))] for _ in range(rng.randint(1, 6))] for _ in range(n_img)]


def test_eval_on_split_scores_the_returned_captions():
    import sparse_caption_b200.relation_transformer as R
    from sparse_caption_b200 import evaluate as E
    z = golden_io.load("ort_tiny")
    w = dict(z["w"])
    bias = w["model.generator.proj.bias"].clone()
    bias[EOS] -= 4.0                             # the fixture's captions are all empty (<eos> first); this gives 8-word ones
    w["model.generator.proj.bias"] = bias
    m = R.get_model("relation_transformer")(z["cfg_dict"])
    m.load_state_dict(w, strict=True)
    m = m.to(DEV).eval()
    m.precision = "fp32"
    att, boxes = z["att_feats"].to(DEV), z["boxes"].to(DEV)
    refs = _refs_for(np.random.RandomState(4), att.shape[0], 20, 36)   # the words these captions use: n-grams match
    met = _metrics(refs)
    batches = [{"att_feats": att[1:], "boxes": boxes[1:], "image_ids": [102, 103], "image_idx": torch.tensor([1, 2], device=DEV)},
               {"att_feats": att[:1], "boxes": boxes[:1], "image_ids": [101], "image_idx": [0]}]
    preds, speed, _ = E.eval_on_split(m, batches, {"beam_size": 3}, decode_words=lambda ids: " ".join(map(str, ids)), metrics=met)
    hyps = [[int(w) for w in p.split()] for p in preds]
    hyps = [hyps[2], hyps[0], hyps[1]]          # split order
    scores, per = met.compute()
    want, want_per = M.evaluate(hyps, refs)
    for k in M.METRICS:
        assert scores[k] == pytest.approx(want[k], rel=1e-12, abs=1e-15), k
    np.testing.assert_allclose(per.numpy(), want_per, rtol=1e-12, atol=1e-15)
    assert all(len(h) for h in hyps) and scores["Bleu_1"] > 0 and scores["CIDEr"] > 0


def test_eval_on_split_radix_model():
    """ACORT-style radix model: digits -> word ids on the device, ids beyond vocab_len -> <unk> (which matches no reference)."""
    import sparse_caption_b200.relation_transformer as R
    from sparse_caption_b200 import evaluate as E
    z = golden_io.load("acort_tiny")
    m = R.get_model("relation_transformer")(z["cfg_dict"])
    m.load_state_dict(z["w"], strict=True)
    m = m.to(DEV).eval()
    m.precision = "fp32"
    base, tpw, vocab_len = 8, 2, 40
    refs = _refs_for(np.random.RandomState(6), 2, 4, 68)
    met = _metrics(refs)
    batches = [{"att_feats": z["att_feats"].to(DEV), "boxes": z["boxes"].to(DEV), "image_ids": [7, 9], "image_idx": [0, 1]}]
    preds, _, _ = E.eval_on_split(m, batches, {"beam_size": 3}, decode_words=lambda ids: " ".join(map(str, ids)), radix=(base, tpw),
                                  vocab_len=vocab_len, eos_id=base + 2, metrics=met)
    hyps = [[int(w) for w in p.split()] for p in preds]
    assert all(w < vocab_len for h in hyps for w in h)
    scores, per = met.compute()
    want, want_per = M.evaluate(hyps, refs)
    for k in M.METRICS:
        assert scores[k] == pytest.approx(want[k], rel=1e-12, abs=1e-15), k
    np.testing.assert_allclose(per.numpy(), want_per, rtol=1e-12, atol=1e-15)
