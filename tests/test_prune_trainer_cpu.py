"""CPU tier of the trainer's magnitude / SNIP mask updates: the option checks against PruningMixin's, the shared gradual schedule,
the trainer's mask order against the module's, and the selection contract - prune the first k in (criterion, position) order,
-0.0 as +0.0, NaN above every number - restated in numpy (the GPU tests hold sc_prune_select to this restatement)."""
import numpy as np
import pytest
import torch

from tests.test_host_cpu import _cfg


def restate_select(crit, groups, ks):
    """0/1 mask of float32 criteria ``crit`` [n]: in each group (index array in position order) the first k elements of a stable
    sort by criterion are pruned.  numpy's sort places NaN last and compares -0.0 equal to +0.0; stability orders ties by position."""
    mask = np.ones(crit.shape[0], dtype=np.float32)
    for idx, k in zip(groups, ks):
        order = np.argsort(crit[idx].astype(np.float32), kind="stable")
        mask[idx[order[:k]]] = 0.0
    return mask


def order_keys(crit, pos):
    """The kernel's 64-bit keys: order-preserving uint32 of the criterion (<< 32) | position."""
    c = np.where(crit == 0, np.float32(0.0), crit).astype(np.float32)
    u = c.view(np.uint32).astype(np.uint64)
    k = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    k = np.where(np.isnan(c), np.uint64(0xFFC00000), k)
    return (k.astype(np.uint64) << np.uint64(32)) | pos.astype(np.uint64)


def _trainer(mask_type, **kw):
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200.trainer import OrtTrainer
    from oracle import ort_oracle as O
    cfg = _cfg(prune_type=mask_type)
    ocfg = O.Cfg(**{k: cfg[k] for k in ("d_model", "dim_feedforward", "num_layers", "num_heads", "max_seq_length", "att_feat_size",
                                        "vocab_size")})
    sd = O.random_state_dict(ocfg, seed=3)
    return OrtTrainer(sd, ModelCfg(cfg), mask_type=mask_type, precision="fp32", device="cpu", **kw)


def _host(mask_type, **kw):
    import sparse_caption_b200.relation_transformer as R
    return R.get_model("relation_transformer_prune")(_cfg(prune_type=mask_type, **kw))


def _raises(fn):
    try:
        fn()
    except Exception as e:   # noqa: BLE001 - the type is what is compared
        return type(e)
    return None


@pytest.mark.parametrize("mask_type", ["supermask", "mask_freeze", "lottery_mask_freeze", "mag_blind", "snip"])
def test_update_masks_once_rejects_like_the_host(mask_type):
    """supermask / mask_freeze: AssertionError; lottery_mask_freeze: ValueError (no criterion); snip without saliency: the
    reference's ``m.grad is not None`` assert; a bad sparsity target: AssertionError."""
    tr, m = _trainer(mask_type), _host(mask_type)
    want = _raises(lambda: m.update_masks_once(0.5))
    if mask_type == "mag_blind":
        assert want is None
        want = _raises(lambda: m.update_masks_once(1.0))
        assert want is AssertionError and _raises(lambda: tr.update_masks_once(1.0)) is want
        assert _raises(lambda: tr.update_masks_once(0)) is AssertionError   # (an int, like the host's isinstance check)
        return
    assert want is not None and _raises(lambda: tr.update_masks_once(0.5)) is want
    assert want is (ValueError if mask_type == "lottery_mask_freeze" else AssertionError)


@pytest.mark.parametrize("mask_type", ["mag_blind", "mag_uniform", "mag_dist", "snip", "supermask"])
def test_update_masks_gradual_rejects_like_the_host(mask_type):
    tr, m = _trainer(mask_type), _host(mask_type)
    want = _raises(lambda: m.update_masks_gradual(0.9, 0, 0, 2))
    assert want is AssertionError and _raises(lambda: tr.update_masks_gradual(0.9, 0, 0, 2)) is want


def test_gradual_schedule_shared_with_the_host(monkeypatch):
    """PruningMixin.update_masks_gradual and OrtTrainer.update_masks_gradual prune to the same targets at the same steps,
    the ones prune.gradual_sparsity gives; bad frequencies / step counts assert in both."""
    from sparse_caption_b200 import prune as P
    tr, m = _trainer("mag_grad_blind"), _host("mag_grad_blind")
    seen = {"host": [], "trainer": []}
    monkeypatch.setattr(m, "update_masks_once", lambda sparsity_target: seen["host"].append(sparsity_target))
    monkeypatch.setattr(tr, "update_masks_once", lambda sparsity_target: seen["trainer"].append(sparsity_target))
    args = dict(start_step=1000, prune_steps=4, initial_sparsity=0.1, prune_frequency=500)
    want = []
    for step in range(0, 4001, 250):
        assert m.update_masks_gradual(0.9, step, **args) is False
        assert tr.update_masks_gradual(0.9, step, **args) is False
        s = P.gradual_sparsity(0.9, step, **args)
        if s is not None:
            want.append(s)
    assert seen["host"] == seen["trainer"] == want
    assert len(want) == 5 and abs(want[0] - 0.1) < 1e-12 and abs(want[-1] - 0.9) < 1e-12 and want == sorted(want)
    for bad in (dict(prune_frequency=0), dict(prune_steps=0)):
        a = dict(args, **bad)
        assert _raises(lambda: m.update_masks_gradual(0.9, 1000, **a)) is AssertionError
        assert _raises(lambda: tr.update_masks_gradual(0.9, 1000, **a)) is AssertionError


def test_trainer_mask_order_is_the_module_order():
    """Tie positions count along the concatenation of active_pruning_masks(): the trainer's masked tensors are in that order,
    and mask_freeze_scope selects the same active set."""
    m = _host("mag_blind")
    tr = _trainer("mag_blind")
    assert tr.masked == [n[: -len("_pruning_mask")] for n, _ in m.all_pruning_masks()]
    scope = "model.decoder.layers.1,att_embed"
    m = _host("mag_blind", prune_mask_freeze_scope=scope)
    tr = _trainer("mag_blind", mask_freeze_scope=m.mask_freeze_scope)
    want = [n[: -len("_pruning_mask")] for n, _ in m.active_pruning_masks()]
    assert tr.active_masked() == want and _trainer("mag_blind", mask_freeze_scope=scope).active_masked() == want
    assert len(want) < len(tr.masked) and not any(k.startswith("att_embed") for k in want)
    assert _trainer("mag_blind").active_masked() == tr.masked


def test_selection_contract_restatement():
    """The keys order exactly like the stable (criterion, position) sort, with -0.0 == +0.0 and NaN last; on tie-free criteria
    the restatement is torch.topk's mask (PruningMixin.compute_mask)."""
    from sparse_caption_b200.prune import PruningMixin
    g = np.random.default_rng(0)
    c = g.integers(-4, 5, 4000).astype(np.float32) * np.float32(0.25)
    c[g.integers(0, 4000, 50)] = -0.0
    c[g.integers(0, 4000, 20)] = np.nan
    c[g.integers(0, 4000, 10)] = np.inf
    c[g.integers(0, 4000, 10)] = -np.inf
    pos = np.arange(c.shape[0])
    by_key = np.argsort(order_keys(c, pos), kind="stable")
    assert np.array_equal(by_key, np.argsort(c, kind="stable"))
    n_nan = int(np.isnan(c).sum())
    assert n_nan > 0 and np.all(np.isnan(c[by_key[-n_nan:]])) and c[by_key[-n_nan - 1]] == np.inf
    for k in (0, 1, 1234, 3999):
        m = restate_select(c, [pos], [k])
        assert int((m == 0).sum()) == k and np.array_equal(np.sort(np.flatnonzero(m == 0)), np.sort(by_key[:k]))
    w = torch.randn(5000, generator=torch.Generator().manual_seed(1))
    for s in (0.0, 0.3, 0.999):
        want = PruningMixin.compute_mask(w.abs(), s).numpy()
        n = int(s * 5000)
        assert np.array_equal(restate_select(w.abs().numpy(), [np.arange(5000)], [n]), want)
