"""CPU tier: diverse beam search (group_size > 1, caption_model.py:30-226) - the restatement in tests/diverse_oracle.py
pinned to the reference goldens, a hand-worked case with scripted log-probs, and the option checks."""
import pytest
import torch

from oracle import ort_oracle as O
from tests import diverse_oracle as D
from tests import golden_io


@pytest.mark.parametrize("name", ["ort_tiny", "ort_tiny_masks", "acort_tiny"])
def test_lambda_zero_reproduces_reference_goldens_group_by_group(name):
    """With diversity_lambda = 0 the groups are independent width-bdash searches: each group's beams equal the reference's
    own beam-bdash search (golden fixtures of the imported reference)."""
    z = golden_io.load(name)
    am = z.get("att_masks")
    memory, src_mask = O.encode(z["w"], z["cfg"], z["att_feats"], z["boxes"], am)
    for key, opt in (("beam3", {"beam_size": 6, "group_size": 2}), ("beam2", {"beam_size": 6, "group_size": 3}),
                     ("beam3c", {"beam_size": 6, "group_size": 2, "decoding_constraint": 1, "length_penalty": "wu_0.5"})):
        opt = dict(opt, diversity_lambda=0.0)
        seq, lp, p = D.diverse_beam_search(z["w"], z["cfg"], memory, src_mask, opt)
        G, bdash, _ = D.diverse_groups(opt)
        assert tuple(seq.shape) == (z[key + "_seq"].shape[0], 6, z["cfg"].max_seq_length)
        for g in range(G):
            assert torch.equal(seq[:, g * bdash:(g + 1) * bdash], z[key + "_seq"]), (name, key, g)
            torch.testing.assert_close(lp[:, g * bdash:(g + 1) * bdash], z[key + "_lp"], rtol=1e-5, atol=2e-6)


V, L, EOS = 8, 4, 3
# scripted log-probs: the row a beam gets depends on the token it was just fed (and, for token 4, on its group)
_ROWS = {"bos": {4: -1.0, 5: -1.25, 6: -2.0, 7: -4.0, 3: -5.0},
         (0, 4): {6: -3.0, 7: -3.5, 3: -4.0}, (1, 4): {6: -0.1, 7: -3.5, 3: -4.0},
         5: {6: -0.25, 7: -0.5, 3: -2.0}, 6: {3: -0.5, 7: -0.75, 4: -2.0}, 7: {3: -1.0, 4: -1.5}, 3: {3: -0.5, 4: -1.0}}


def _row(key):
    r = torch.full((V,), -10.0)
    for c, v in _ROWS.get(key, {}).items():
        r[c] = v
    return r


def _scripted(opt):
    def advance(g, state_ix, it, tau):
        return torch.stack([_row((g, 4) if int(i) == 4 else int(i)) for i in it])
    return D.diverse_beam_core(_row("bos").unsqueeze(0), advance, 1, V, L, EOS, 0, opt)


def test_hand_worked_case():
    """beam 4, G = 2 (bdash 2), lambda 0.5, L = 4, EOS = 3.  Worked by hand:
      t=0  g0 tau0: [4] -1, [5] -1.25
      t=1  g0 tau1: both children of [5]: [5,6] -1.5, [5,7] -1.75  -> g0's CURRENT tokens at position 0 are {5, 5}
           g1 tau0: 5 penalised twice (-1.0): [4] -1, [6] -2      (lockstep, i.e. g0's tau-0 choices {4, 5}: [4] -1.5, [5] -1.75)
      t=2  g0 tau2: [5,6,3] -2.0 finishes (sum -> -1002), [5,6,7] -2.25      -> position 1 now {6, 6}
           g1 tau1: [4,6] -1 + (-0.1 - 1.0) = -2.1, [6,3] -2.5 finishes
      t=3  g0 tau3 (forced finish): [5,6,7,3] -3.25, [5,6,7,4] -3.75       -> position 2 now {7, 7}
           g1 tau2: [4,6,3] -2.6 finishes, [4,6,7] -2.1 + (-0.75 - 1.0) = -3.85
      t=4  g1 tau3 (forced finish; g0's final position 3 is {3, 4}): [4,6,7,3] -5.35, [4,6,7,4] -5.85
    Per group: finished beams sorted by the AUGMENTED p, two kept; groups concatenated.  [6,3] (p -2.5) ranks before
    [4,6,3] (p -2.6) although its unaugmented sum is lower (-2.5 vs -1.6)."""
    seq, lp, p, done = _scripted({"beam_size": 4, "group_size": 2, "diversity_lambda": 0.5})
    want_seq = [[5, 6, 3, 0], [5, 6, 7, 3], [6, 3, 0, 0], [4, 6, 3, 0]]
    want_lp = [[-1.25, -0.25, -0.5, 0.0], [-1.25, -0.25, -0.75, -1.0], [-2.0, -0.5, 0.0, 0.0], [-1.0, -0.1, -0.5, 0.0]]
    want_p = [-2.0, -3.25, -2.5, -2.6]
    assert seq[0].tolist() == want_seq
    torch.testing.assert_close(lp[0], torch.tensor(want_lp))
    torch.testing.assert_close(p[0], torch.tensor(want_p))
    assert [round(d["unaug_p"], 4) for d in done[0]] == [-2.0, -3.25, -2.5, -1.6]
    assert [d["seq"].tolist() for d in done[0]] == [[5, 6, 3], [5, 6, 7, 3], [6, 3], [4, 6, 3]]
    # group 0 is never penalised; without the penalty group 1 keeps [4] at local step 0 and its own best continuations
    seq0, _, p0, _ = _scripted({"beam_size": 4, "group_size": 2, "diversity_lambda": 0.0})
    assert seq0[0, :2].tolist() == want_seq[:2] and seq0[0, 2:].tolist() == [[4, 6, 3, 0], [4, 6, 7, 3]]
    assert p0[0].tolist() == pytest.approx([-2.0, -3.25, -1.6, -2.85])


def test_add_diversity_counts_duplicates_and_repeats_rows():
    table = [torch.tensor([[[5, 1], [5, 2]]]), torch.tensor([[[6, 1], [5, 1]]])]   # B=1, bdash=2, 2 positions
    lp = torch.zeros(2, 8)
    aug, unaug = D.add_diversity(table, lp, 0, 2, 0.5, 2)
    assert torch.equal(unaug, lp)
    assert aug[:, 5].tolist() == [-1.5, -1.5] and aug[:, 6].tolist() == [-0.5, -0.5] and float(aug[:, [0, 1, 7]].abs().sum()) == 0
    aug, _ = D.add_diversity(table, lp[:1], 0, 1, 0.5, 2)  # local step 0: one row per image
    assert aug[0, 5] == -1.0 and aug.shape == (1, 8)


def test_group_options_are_checked():
    from sparse_caption_b200.engine import diverse_groups
    assert diverse_groups({"beam_size": 6, "group_size": 3}) == (3, 2, 0.5)
    assert diverse_groups({"beam_size": 7, "group_size": 2, "diversity_lambda": 2.0}) == (2, 3, 2.0)
    for opt in ({"beam_size": 2, "group_size": 3}, {"beam_size": 18, "group_size": 2}, {"beam_size": 3, "group_size": 0}):
        with pytest.raises(ValueError, match="group_size"):
            diverse_groups(opt)
