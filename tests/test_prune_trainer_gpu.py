"""Magnitude / SNIP mask updates on the trainer's own buffers: sc_prune_select against the numpy restatement (bit-exact), the
trainer's masks against PruningMixin on the same weights, what an update keeps (optimizer state, step counters, graphs, operand
pointers), training across a prune event against the module-tree recipe, the SNIP saliency against autograd, the rollout engine
after an update, and bitwise reproducibility (the data-parallel premise)."""
import numpy as np
import pytest
import torch

from tests import golden_io
from tests.test_prune_trainer_cpu import restate_select

pytestmark = pytest.mark.gpu
DEV = "cuda"
SUFFIX = "_pruning_mask"


# ---- sc_prune_select against the restatement ----------------------------------------------------------------------------------
def _select(src, sizes, groups, ks, criterion, sums=False):
    """Segments of `sizes` laid end to end in `src`, written to a separate mask buffer; `groups[i]` the group of segment i."""
    from sparse_caption_b200 import kernels as K
    segs, offs, pos = [], np.cumsum([0] + sizes), {}
    for i, (n, g) in enumerate(zip(sizes, groups)):
        segs.append((int(offs[i]), int(offs[i]), n, g, pos.get(g, 0)))
        pos[g] = pos.get(g, 0) + n
    desc, blocks = K.prune_descriptors(segs, DEV)
    x = torch.from_numpy(src).to(DEV)
    out = torch.full_like(x, 7.0)
    st = K.prune_stats(desc, blocks, x, centered=criterion == K.PRUNE_DIST) if sums else None
    K.prune_select(desc, blocks, torch.tensor(ks, dtype=torch.int64, device=DEV), criterion, x, out, sums=st)
    return out.cpu().numpy(), (None if st is None else st.cpu().numpy()), offs


def _group_idx(offs, groups, g):
    return np.concatenate([np.arange(offs[i], offs[i + 1]) for i in range(len(groups)) if groups[i] == g])


def test_select_kernel_matches_restatement():
    from sparse_caption_b200 import kernels as K
    rng = np.random.default_rng(0)
    sizes = [1, 64, 5_120_000, 777, 64, 3001]
    n = sum(sizes)
    # 1. random criteria, one global group: |w|
    w = rng.standard_normal(n).astype(np.float32)
    for frac in (0.0, 0.37, 0.9):
        k = int(frac * n)
        got, _, offs = _select(w, sizes, [0] * 6, [k], K.PRUNE_ABS)
        assert np.array_equal(got, restate_select(np.abs(w), [np.arange(n)], [k])), frac
    # 2. global and per-tensor groups in one launch, ties forced to straddle every threshold, -0.0 / +0.0, NaN, k = 0 and n - 1
    w = (rng.integers(-3, 4, n).astype(np.float32) * np.float32(0.5))
    w[rng.integers(0, n, 1000)] = -0.0
    w[rng.integers(0, n, 300)] = np.nan
    w[offs[3]: offs[3] + 5] = np.nan
    groups = [0, 1, 0, 2, 3, 0]
    sz = {g: sum(s for s, gg in zip(sizes, groups) if gg == g) for g in set(groups)}
    ks = [int(0.61 * sz[0]), 0, sz[2] - 1, 17]
    got, _, offs = _select(w, sizes, groups, ks, K.PRUNE_ABS)
    want = restate_select(np.abs(w), [_group_idx(offs, groups, g) for g in range(4)], ks)
    assert np.array_equal(got, want)
    assert got[offs[1]] == 1.0 and (got[offs[3]: offs[4]] == 1).sum() == 1 and np.isnan(w[offs[3]: offs[4]][got[offs[3]: offs[4]] == 1])
    # 3. SNIP: sal / (group sum); integer-valued saliency keeps the sums exact; a negative sum flips the order; signed zeros
    for sign in (1.0, -1.0):
        sal = rng.integers(-20, 25, n).astype(np.float32) * np.float32(sign)
        sal[rng.integers(0, n, 500)] = -0.0
        for g in range(4):
            idx = _group_idx(offs, groups, g)
            sal[idx[0]] += np.float32(sign * 3.0)    # every group sum is non-zero
        ks = [int(0.45 * sz[0]), int(0.3 * sz[1]), int(0.8 * sz[2]), 1]
        got, _, _ = _select(sal, sizes, groups, ks, K.PRUNE_SNIP, sums=True)
        gidx = [_group_idx(offs, groups, g) for g in range(4)]
        crit = sal.copy()
        for idx in gidx:
            crit[idx] = sal[idx] / np.float32(sal[idx].astype(np.float64).sum())
        assert all(sal[idx].astype(np.float64).sum() * sign > 0 for idx in gidx[:1])
        assert np.array_equal(got, restate_select(crit, gidx, ks)), sign
    # 4. DIST: |(w - mean) / std| with the segment statistics (two-pass double sums, fixed order); a constant segment whose value
    #    is not a dyadic fraction still has variance exactly 0, so its criterion is NaN and it sorts above every number
    w = rng.standard_normal(n).astype(np.float32) * np.float32(0.02) + np.float32(0.01)
    w[offs[4]: offs[5]] = np.float32(0.1)
    ks = [int(0.5 * n)]
    got, st, _ = _select(w, sizes, [0] * 6, ks, K.PRUNE_DIST, sums=True)
    crit = np.empty_like(w)
    for i in range(6):
        seg = w[offs[i]: offs[i + 1]]
        ref = seg.astype(np.float64)
        np.testing.assert_allclose(st[i], [ref.sum(), ((ref - ref.mean()) ** 2).sum()], rtol=1e-12, atol=1e-12)
        mean = st[i, 0] / seg.size
        std = np.float32(np.sqrt(st[i, 1] / seg.size))
        with np.errstate(divide="ignore", invalid="ignore"):
            crit[offs[i]: offs[i + 1]] = np.abs((seg - np.float32(mean)) / std)
    assert np.array_equal(got, restate_select(crit, [np.arange(n)], ks))
    assert st[4, 1] == 0.0 and np.all(np.isnan(crit[offs[4]: offs[5]])) and np.all(got[offs[4]: offs[5]] == 1.0)


# ---- the trainer against PruningMixin -------------------------------------------------------------------------------------------
def _tiny_sd(mask_type, seed=3):
    z = golden_io.load("ort_prune_tiny")
    sd = {k: v.clone() for k, v in z["w"].items()}
    g = torch.Generator().manual_seed(seed)
    for k in z["u"]:
        sd[k] = sd[k] + 0.01 * torch.randn(sd[k].shape, generator=g)   # continuous weights: no ties
        sd[k + SUFFIX] = torch.ones_like(sd[k])
    return z, sd


def _trainer(mask_type, sd, z, **kw):
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200.trainer import OrtTrainer
    kw.setdefault("precision", "fp32")
    return OrtTrainer(sd, ModelCfg(z["cfg_dict"]), mask_type=mask_type, dropout=0.0, drop_prob_src=0.0, **kw)


def _module(mask_type, z, tr, scope="", device="cpu"):
    import sparse_caption_b200.relation_transformer as R
    m = R.get_model("relation_transformer_prune")(dict(z["cfg_dict"], prune_type=mask_type, prune_mask_freeze_scope=scope))
    m.load_state_dict({k: v.cpu() for k, v in tr.state_dict().items()}, strict=False)
    return m.to(device)


def _host_criterion(m, mask_type):
    """PruningMixin's own criterion tensors (prune.py:268-279) per active mask, for the near-threshold exemption."""
    ws = m.active_pruned_weights(named=False)
    if mask_type == "snip":
        sal = torch.cat([p.grad.reshape(-1) for p in m.active_pruning_masks(named=False)])
        return sal / sal.sum()
    return torch.cat([torch.abs((w - w.mean()) / torch.std(w.reshape(-1), dim=0, unbiased=False)).reshape(-1) for w in ws])


def _compare(tr, m, mask_type, sparsity):
    got = torch.cat([tr.s[n[: -len(SUFFIX)]].reshape(-1).cpu() for n, _ in m.active_pruning_masks()])
    want = torch.cat([p.detach().reshape(-1).cpu() for p in m.active_pruning_masks(named=False)])
    if mask_type in ("mag_blind", "mag_grad_blind", "mag_uniform", "mag_grad_uniform", "lottery_mag_blind"):
        assert torch.equal(got, want)
        return 0
    k = int(sparsity * want.numel())
    assert int((got == 0).sum()) == int((want == 0).sum()) == k
    crit = _host_criterion(m, mask_type).cpu()
    kth = crit.sort().values[k - 1]
    near = (crit - kth).abs() <= 1e-5 * kth.abs()
    diff = got != want
    assert bool((~diff | near).all()), int((diff & ~near).sum())
    print(f"{mask_type}: {int(diff.sum())} mask differences, all within 1e-5 of the k-th value ({int(near.sum())} such elements)")
    return int(near.sum())


@pytest.mark.parametrize("mask_type", ["mag_blind", "mag_uniform", "mag_dist", "mag_grad_uniform", "lottery_mag_blind"])
def test_update_masks_once_matches_pruning_mixin(mask_type):
    z, sd = _tiny_sd(mask_type)
    tr = _trainer(mask_type, sd, z)
    for sparsity in (0.3, 0.8, 0.5):      # later events may bring pruned weights back, as in the reference
        tr.update_masks_once(sparsity)
        m = _module(mask_type, z, tr)
        for p in m.active_pruning_masks(named=False):
            p.data.fill_(1.0)
        m.update_masks_once(sparsity)
        _compare(tr, m, mask_type, sparsity)
    # mask_sparsities == all_mask_sparsities
    sp, nnz, per, names = tr.mask_sparsities()
    hsp, hnnz, hper, hnames = m.all_mask_sparsities
    assert names == hnames and nnz == float(hnnz) and abs(sp - float(hsp)) < 1e-6
    assert np.allclose(per, [float(x) for x in hper], atol=1e-6)


def test_mask_freeze_scope():
    z, sd = _tiny_sd("mag_blind")
    scope = "model.decoder.layers.1,att_embed"
    sd["att_embed.0.weight" + SUFFIX] = (torch.rand(sd["att_embed.0.weight"].shape, generator=torch.Generator().manual_seed(1)) < 0.5).float()
    tr = _trainer("mag_blind", sd, z, mask_freeze_scope=scope)
    frozen = {k: tr.s[k].clone() for k in tr.masked if k not in tr.active_masked()}
    assert "att_embed.0.weight" in frozen and "model.decoder.layers.1.feed_forward.w_1.weight" in frozen
    tr.update_masks_once(0.7)
    m = _module("mag_blind", z, tr, scope=scope)
    for p in m.active_pruning_masks(named=False):
        p.data.fill_(1.0)
    m.update_masks_once(0.7)
    _compare(tr, m, "mag_blind", 0.7)   # (frozen tensors are not in the global group: the pruned count is of the active ones)
    for k, v in frozen.items():
        assert torch.equal(tr.s[k], v), k
    # through the model: trainer() passes the model's scope
    m2 = _module("mag_blind", z, tr, scope=scope, device=DEV)
    assert m2.trainer().active_masked() == tr.active_masked()


def _batch(z):
    return z["att_feats"].to(DEV), z["boxes"].to(DEV), z["seqs"], z["masks"]


def test_snip_saliency_matches_autograd_and_accumulates():
    """fp32, dropout off: the saliency is mask.grad of the module tree; two calls accumulate; two half-batch shards with the
    global token count sum to the full batch; an all_reduce is applied to the gradient buffer; the masks match PruningMixin
    fed the same saliency."""
    z, sd = _tiny_sd("snip")
    att, boxes, seqs, masks = _batch(z)
    tr = _trainer("snip", sd, z)
    tr.snip_saliency(att, boxes, seqs, masks, seq_per_img=2)
    m = _module("snip", z, tr, device=DEV)
    m.precision = "fp32"
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    out = m(att_feats=att, boxes=boxes, seqs=seqs.to(DEV))
    T = out.shape[1]
    w = masks.to(DEV)[:, 1: T + 1]
    (-(out.gather(2, seqs.to(DEV)[:, 1: T + 1].unsqueeze(2)).squeeze(2) * w).sum() / w.sum()).backward()
    sal = {k: tr._saliency[tr._offs_s[k]: tr._offs_s[k] + tr.s[k].numel()].view(tr.s[k].shape).clone() for k in tr.masked}
    for n, p in m.all_pruning_masks():
        g = p.grad
        e = float((sal[n[: -len(SUFFIX)]] - g).abs().max() / g.abs().max().clamp_min(1e-6))
        assert e < 1e-3, (n, e)
    full = tr._saliency.clone()
    tr.snip_saliency(att, boxes, seqs, masks, seq_per_img=2)
    assert float((tr._saliency - 2 * full).abs().max()) <= 1e-5 * float(full.abs().max())
    # shards
    tr2 = _trainer("snip", sd, z)
    total = masks[:, 1:].sum().reshape(1).to(DEV)
    tr2.snip_saliency(att[:1], boxes[:1], seqs[:2], masks[:2], seq_per_img=2, global_tokens=total)
    tr2.snip_saliency(att[1:], boxes[1:], seqs[2:], masks[2:], seq_per_img=2, global_tokens=total)
    assert float((tr2._saliency - full).abs().max()) <= 1e-4 * float(full.abs().max())
    tr3 = _trainer("snip", sd, z)
    def all_reduce(t):   # a second rank holding the same batch
        t.mul_(2.0)

    tr3.snip_saliency(att, boxes, seqs, masks, seq_per_img=2, all_reduce=all_reduce)
    assert float((tr3._saliency - 2 * full).abs().max()) <= 1e-5 * float(full.abs().max())
    # the update consumes the saliency; with the host fed the trainer's saliency the masks agree
    for n, p in m.all_pruning_masks():
        k = n[: -len(SUFFIX)]
        p.grad = tr._saliency[tr._offs_s[k]: tr._offs_s[k] + tr.s[k].numel()].view(tr.s[k].shape).clone()
    m_cpu = m.cpu()
    tr.update_masks_once(0.6)
    m_cpu.update_masks_once(0.6)
    print("snip near-threshold elements:", _compare(tr, m_cpu, "snip", 0.6))
    assert not tr._has_saliency and float(tr._saliency.abs().max()) == 0.0
    with pytest.raises(AssertionError):
        tr.update_masks_once(0.6)
    # graph mode: the first call runs and captures the "fwdbwd" graph, the second replays it; both accumulate
    trg = _trainer("snip", sd, z, use_graph=True)
    for _ in range(2):
        trg.snip_saliency(att, boxes, seqs, masks, seq_per_img=2)
    graphs = next(iter(trg._ws.values())).graphs
    assert [key[0] for key in graphs] == ["fwdbwd"]
    assert float((trg._saliency - 2 * full).abs().max()) <= 1e-4 * float(full.abs().max())


@pytest.mark.parametrize("mask_type", ["mag_blind", "mag_uniform", "mag_dist", "snip", "mag_grad_uniform"])
def test_update_does_not_synchronise_the_host(mask_type):
    """update_masks_once / update_masks_gradual (first call included: descriptor tables, k values) enqueue work only."""
    z, sd = _tiny_sd(mask_type)
    att, boxes, seqs, masks = _batch(z)
    tr = _trainer(mask_type, sd, z, precision="bf16", use_graph=True)
    if mask_type == "snip":
        tr.snip_saliency(att, boxes, seqs, masks, seq_per_img=2)
    else:
        tr.train_step(att, boxes, seqs, masks, seq_per_img=2, lr=1e-3)
    torch.cuda.set_sync_debug_mode("error")
    try:
        if mask_type == "mag_grad_uniform":
            tr.update_masks_gradual(0.8, 1000, start_step=0, prune_steps=2, prune_frequency=1000)
        else:
            tr.update_masks_once(0.7)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert float((tr.flat_s[~tr._s_pad_mask] == 0).float().mean()) > 0.5


def test_update_keeps_premask_operand_pointers_bf16():
    """bf16 graph mode: the pre-masked operands (_wm, _wmT) and the premask descriptor table keep their memory across an update,
    and the next replayed step's operands carry the new masks."""
    z, sd = _tiny_sd("mag_blind")
    att, boxes, seqs, masks = _batch(z)
    tr = _trainer("mag_blind", sd, z, precision="bf16", use_graph=True)
    for _ in range(2):
        tr.train_step(att, boxes, seqs, masks, seq_per_img=2, lr=1e-3)
    ptrs = {key: (tr._wm[key].data_ptr(), tr._wmT[key].data_ptr()) for key in tr._premask_keys()}
    desc = tr._premask_desc[0].data_ptr()
    tr.update_masks_once(0.8)
    tr.train_step(att, boxes, seqs, masks, seq_per_img=2, lr=0.0)   # (lr 0: the weights the operands were built from stay put)
    torch.cuda.synchronize()
    assert {key: (tr._wm[key].data_ptr(), tr._wmT[key].data_ptr()) for key in tr._premask_keys()} == ptrs
    assert tr._premask_desc[0].data_ptr() == desc
    gen = "model.generator.proj.weight"
    V = tr.cfg.vocab_size
    assert torch.equal(tr._wm[(gen, 1)][:V], (tr.p[gen] * tr.s[gen]).bfloat16())


def test_update_keeps_state_and_graph_step_equals_eager():
    """mag_grad_uniform, graph mode: after an update mid-run the Adam moments, opt_step, step_id, graphs and operand pointers are
    the same objects / values; the next replayed step equals the next eager step."""
    z, sd = _tiny_sd("mag_grad_uniform")
    att, boxes, seqs, masks = _batch(z)
    res = {}
    for graph in (False, True):
        tr = _trainer("mag_grad_uniform", sd, z, use_graph=graph)
        losses = [float(tr.train_step(att, boxes, seqs, masks, seq_per_img=2, lr=1e-3)) for _ in range(3)]
        ws = next(iter(tr._ws.values()))
        before = dict(m_w=tr.m_w, v_w=tr.v_w, flat_w=tr.flat_w, flat_s=tr.flat_s, opt=tr.opt_step, step=tr.step_id,
                      graphs=dict(ws.__dict__.get("graphs", {})), m_w_val=tr.m_w.clone(), w_val=tr.flat_w.clone())
        tr.update_masks_gradual(0.6, 2000, start_step=0, prune_steps=4, prune_frequency=1000)
        torch.cuda.synchronize()
        assert tr.m_w is before["m_w"] and tr.v_w is before["v_w"] and tr.flat_s is before["flat_s"] and tr.flat_w is before["flat_w"]
        assert torch.equal(tr.m_w, before["m_w_val"]) and torch.equal(tr.flat_w, before["w_val"])
        assert tr.opt_step == before["opt"] == 3 and tr.step_id == before["step"] == 3
        assert float((tr.flat_s[~tr._s_pad_mask] == 0).float().mean()) > 0.4
        losses += [float(tr.train_step(att, boxes, seqs, masks, seq_per_img=2, lr=1e-3)) for _ in range(2)]
        if graph:
            now = ws.__dict__.get("graphs", {})
            assert before["graphs"] and all(now[k] is v for k, v in before["graphs"].items()) and len(now) == len(before["graphs"])
        res[graph] = (losses, tr.flat_w.clone(), tr.flat_s.clone())
    assert int((res[True][2] != res[False][2]).sum()) <= 8   # (same masks up to near-ties of the atomically summed weights)
    for a, b in zip(res[True][0], res[False][0]):
        assert abs(a - b) < 2e-3 * abs(b), (res[True][0], res[False][0])
    assert float((res[True][1] - res[False][1]).abs().mean() / res[False][1].abs().mean()) < 2e-3


def test_training_across_a_prune_event_matches_module_recipe():
    """fp32 mag_grad_uniform: two steps, a gradual update, two steps - against the module tree + PruningMixin.update_masks_gradual
    + torch Adam (clip_grad_value_ 0.1, betas (0.9, 0.98), eps 1e-9)."""
    z, sd = _tiny_sd("mag_grad_uniform")
    att, boxes, seqs, masks = _batch(z)
    tr = _trainer("mag_grad_uniform", sd, z)
    m = _module("mag_grad_uniform", z, tr, device=DEV)
    m.precision = "fp32"
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    m.train()
    params = [p for n, p in m.named_parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=1e-3, betas=(0.9, 0.98), eps=1e-9)
    sched = dict(start_step=1, prune_steps=2, prune_frequency=1)   # step 2: 0.7 * (1 - 0.5^3) = 0.6125
    for step in range(4):
        if step == 2:
            tr.update_masks_gradual(0.7, step, **sched)
            m.update_masks_gradual(0.7, step, **sched)
            got = torch.cat([tr.s[n[: -len(SUFFIX)]].reshape(-1) for n, _ in m.all_pruning_masks()])
            want = torch.cat([p.detach().reshape(-1) for p in m.all_pruning_masks(named=False)])
            assert int((got == 0).sum()) == int((want == 0).sum()) > 0
            assert int((got != want).sum()) <= 4, int((got != want).sum())   # (Adam's sign-like first steps: near-ties only)
        loss = float(tr.train_step(att, boxes, seqs, masks, seq_per_img=2, lr=1e-3))
        opt.zero_grad()
        out = m(att_feats=att, boxes=boxes, seqs=seqs.to(DEV))
        T = out.shape[1]
        w = masks.to(DEV)[:, 1: T + 1]
        ref = -(out.gather(2, seqs.to(DEV)[:, 1: T + 1].unsqueeze(2)).squeeze(2) * w).sum() / w.sum()
        ref.backward()
        torch.nn.utils.clip_grad_value_(params, 0.1)
        opt.step()
        ref = float(ref.detach())
        assert abs(loss - ref) < 1e-4 * abs(ref), (step, loss, ref)
    sdm = dict(m.named_parameters())
    got = torch.cat([tr.p[k].reshape(-1) for k in tr.names])
    want = torch.cat([sdm[k].detach().reshape(-1) for k in tr.names])
    err = float((got - want).abs().mean() / want.abs().mean())
    assert err < 2e-3, err   # (Adam's sign-like steps on near-zero gradients are the only differences, as in test_trainer_gpu)


def test_rollout_engine_after_update_equals_fresh_engine():
    from sparse_caption_b200.engine import OrtEngine
    from tests.test_scst_gpu import _folded, _operand_ptrs, _refs
    from sparse_caption_b200.cider import CiderD
    z, sd = _tiny_sd("mag_blind")
    att, boxes = z["att_feats"].to(DEV), z["boxes"].to(DEV)
    scorer = CiderD.from_corpus(_refs(z, att.shape[0]), device=DEV)
    for precision in ("fp32", "bf16"):
        tr = _trainer("mag_blind", sd, z, precision=precision, use_graph=True)
        opt = {"beam_size": 3}
        tr.scst_step(att, boxes, scorer=scorer, opt=opt, lr=1e-3)
        eng = tr.rollout_engine()
        ptrs = _operand_ptrs(eng)
        tr.update_masks_once(0.8)
        tr.scst_step(att, boxes, scorer=scorer, opt=opt, lr=1e-3)
        assert tr.rollout_engine() is eng and _operand_ptrs(eng) == ptrs
        tr._scst_masks(eng)
        seq, lp = eng.decode(eng.encode(att, boxes), opt)
        seq, lp = seq.clone(), lp.clone()
        fresh = OrtEngine(_folded(tr), tr.cfg, precision=precision, use_graphs=False)
        fseq, flp = fresh.decode(fresh.encode(att, boxes), opt)
        assert torch.equal(seq, fseq), precision
        torch.testing.assert_close(lp, flp, rtol=1e-5, atol=1e-5)
        assert abs(tr.mask_sparsities()[0] - 0.8) < 1e-3


@pytest.mark.parametrize("mask_type", ["mag_blind", "mag_dist", "mag_uniform", "snip"])
def test_two_trainers_produce_identical_masks(mask_type):
    z, sd = _tiny_sd(mask_type)
    att, boxes, seqs, masks = _batch(z)
    sal = None
    out = []
    for _ in range(2):
        tr = _trainer(mask_type, sd, z, precision="bf16")
        if mask_type == "snip":
            tr.snip_saliency(att, boxes, seqs, masks, seq_per_img=2)
            if sal is None:
                sal = tr._saliency.clone()
            tr._saliency.copy_(sal)   # the all-reduced saliency: the same on every rank
        tr.update_masks_once(0.75)
        out.append(tr.flat_s.clone())
    assert torch.equal(out[0], out[1])
