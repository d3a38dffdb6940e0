"""SCST step, CPU tier: the option checks of scst_step, and the numpy restatement of sc_scst_targets (the teacher-forcing layout,
RewardCriterion's shifted mask, the mean-of-others baseline, the token count) pinned against the module recipe's own formula
(utils/training.py:239-255, utils/losses.py:10-29) on hand-made rollouts.  The GPU tier checks the kernel against the restatement."""
import numpy as np
import pytest
import torch

BOS, PAD, EOS = 2, 0, 3


def scst_targets_np(seq, score, base, S, cider_weight, bos=BOS, pad=PAD):
    """seq int [R, L], score float64 [R], base float64 [R // S] or None -> (tokens, targets, tok_w, key_valid) [R, L], mask sum,
    inv_norm, mean reward: what sc_scst_targets writes."""
    seq = np.asarray(seq)
    R, L = seq.shape
    score = np.asarray(score, dtype=np.float64)
    if base is None:
        tot = score.reshape(-1, S).sum(1)
        b = (np.repeat(tot, S) - score) / (S - 1)
    else:
        b = np.repeat(np.asarray(base, dtype=np.float64), S)
    reward = cider_weight * (score - b)
    tokens = np.concatenate([np.full((R, 1), bos), seq[:, :-1]], 1)
    mask = np.concatenate([np.ones((R, 1)), (seq[:, :-1] != pad)], 1).astype(np.float32)
    tok_w = reward.astype(np.float32)[:, None] * mask
    n = float(mask.sum())
    return tokens, seq.copy(), tok_w, (tokens != pad).astype(np.float32), n, np.float32(1.0) / np.float32(n), reward.mean()


def hand_rows(L=6):
    """Two images x three samples: EOS at position 0, EOS at L-1, no EOS, an all-pad row, and ordinary captions."""
    return np.array([[EOS, 0, 0, 0, 0, 0],
                     [5, 6, 7, 8, 9, EOS],
                     [5, 6, 7, 8, 9, 10],
                     [0, 0, 0, 0, 0, 0],
                     [11, 12, EOS, 0, 0, 0],
                     [13, EOS, 0, 0, 0, 0]], dtype=np.int32)[:, :L]


@pytest.mark.parametrize("baseline", ["greedy", "sample"])
def test_targets_restatement_matches_module_recipe(baseline):
    seq = hand_rows()
    R, L = seq.shape
    S = 3
    score = np.array([0.0, 1.25, 0.5, 0.0, 2.0, 0.75])
    base = np.array([0.4, 1.1]) if baseline == "greedy" else None
    tokens, targets, tok_w, key_valid, n, inv_norm, mean_r = scst_targets_np(seq, score, base, S, cider_weight=1.0)
    # the module recipe (tests/test_cider.py:112-119) on random log-probs
    lp = torch.randn(R, L, dtype=torch.float64)
    if base is None:  # CiderD.scst_reward's mean-of-others baseline
        sc = torch.tensor(score)
        b = (sc.view(-1, S).sum(-1).repeat_interleave(S) - sc) / (S - 1)
    else:
        b = torch.tensor(base).repeat_interleave(S)
    reward = (torch.tensor(score) - b).float()
    m = (torch.from_numpy(seq) != PAD).float()
    m = torch.cat([m.new_ones(R, 1), m[:, :-1]], 1)
    want = float((-lp.float() * reward[:, None] * m).sum() / m.sum())
    got = float(-(lp.float() * torch.from_numpy(tok_w)).sum() * float(inv_norm))
    assert abs(got - want) < 1e-5 * max(1.0, abs(want))
    assert n == float(m.sum())
    # layout of the teacher-forcing inputs: [BOS, s_0 .. s_{L-2}] -> [s_0 .. s_{L-1}]
    assert (tokens[:, 0] == BOS).all() and (tokens[:, 1:] == seq[:, :-1]).all() and (targets == seq).all()
    assert (key_valid == (tokens != PAD)).all()
    # edge rows: EOS at 0 -> positions 0 and 1 are weighted (the shifted mask keeps the step after the EOS, as the reference
    # does); no EOS / EOS at L-1 -> every position; all-pad -> position 0 only
    rw = reward.numpy()
    assert (tok_w[0, 2:] == 0).all() and (tok_w[0, :2] == rw[0]).all() and rw[0] != 0
    assert (tok_w[1] == rw[1]).all() and (tok_w[2] == rw[2]).all() and rw[1] != 0 and rw[2] != 0
    assert (tok_w[3, 1:] == 0).all() and tok_w[3, 0] == rw[3]
    assert abs(mean_r - float(reward.double().mean())) < 1e-7


def test_option_validation():
    from sparse_caption_b200.trainer import scst_samples
    assert scst_samples({"beam_size": 5}, "greedy") == 5
    assert scst_samples({"beam_size": 5}, "sample") == 5
    assert scst_samples({"num_random_sample": 5, "beam_size": 0}, "greedy") == 5
    assert scst_samples({"beam_size": 6, "group_size": 3}, "greedy") == 6
    assert scst_samples({"beam_size": 7, "group_size": 3}, "greedy") == 6
    with pytest.raises(ValueError, match="bleu"):
        scst_samples({"beam_size": 5}, "greedy", bleu_weight=0.5)
    with pytest.raises(ValueError, match="temperature"):
        scst_samples({"beam_size": 5, "temperature": 0.5}, "greedy")
    with pytest.raises(ValueError, match="beam_size == 1"):
        scst_samples({"beam_size": 1}, "greedy")
    with pytest.raises(ValueError, match="at least 2"):
        scst_samples({"num_random_sample": 1, "beam_size": 0}, "sample")
    with pytest.raises(ValueError, match="baseline"):
        scst_samples({"beam_size": 5}, "mean")
    with pytest.raises(AssertionError, match="Beam size must be < 1"):
        scst_samples({"num_random_sample": 5, "beam_size": 3}, "greedy")


def test_scst_step_rejects_options_before_any_device_work():
    """Both trainers validate the options first: the checks above surface from scst_step on a CPU-only machine too."""
    from sparse_caption_b200.trainer import ModuleTrainer, OrtTrainer
    for cls in (OrtTrainer, ModuleTrainer):
        tr = cls.__new__(cls)
        with pytest.raises(ValueError, match="bleu"):
            tr.scst_step(torch.zeros(1, 2, 4), torch.zeros(1, 2, 4), scorer=None, opt={"beam_size": 5}, bleu_weight=1.0, lr=1e-3)
        with pytest.raises(ValueError, match="at least 2"):
            tr.scst_step(torch.zeros(1, 2, 4), torch.zeros(1, 2, 4), scorer=None, opt={"num_random_sample": 1, "beam_size": 0},
                         baseline="sample", lr=1e-3)


def test_rollout_engine_rejects_unsupported_engine_options():
    from sparse_caption_b200.trainer import OrtTrainer
    tr = OrtTrainer.__new__(OrtTrainer)
    for kw in ({"ln_fold": True}, {"sparse_backend": "sell"}, {"sparse_backend": "auto"}):
        with pytest.raises(ValueError, match="dense operands"):
            tr._bound_engine(eval_masks=False, **kw)
