"""SCST step on the device: sc_scst_targets against its restatement, the trainer-bound rollout engine against an engine built
from scratch, the fused step's gradients against autograd through the oracle, graph mode against eager, shard additivity at full
size, the ACORT module path and the model surface."""
import numpy as np
import pytest
import torch

from oracle import ort_oracle as O
from tests import golden_io
from tests.test_scst_cpu import hand_rows, scst_targets_np

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _refs(z, B):
    return [[[int(t) for t in row[1:] if t not in (0, 3)] for row in z["seqs"][i * 2: (i + 1) * 2]] for i in range(B)]


def _tiny(mask_type, precision, use_graph=False, inject=True):
    from sparse_caption_b200.cider import CiderD
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200.trainer import OrtTrainer
    z = golden_io.load("ort_prune_tiny")
    sd = dict(z["w"])
    if mask_type == "mask_freeze":   # fixed 0/1 masks
        g = torch.Generator().manual_seed(5)
        for k in z["u"]:
            sd[k + "_pruning_mask"] = (torch.rand(sd[k].shape, generator=g) < 0.7).float()
    tr = OrtTrainer(sd, ModelCfg(z["cfg_dict"]), mask_type=mask_type, precision=precision, dropout=0.0, drop_prob_src=0.0,
                    uniforms=z["u"] if (inject and mask_type == "supermask") else None, use_graph=use_graph)
    B = z["att_feats"].shape[0]
    return z, tr, CiderD.from_corpus(_refs(z, B), device=DEV)


def _folded(tr):
    """The trainer's weights folded with the step's mask sample (injected uniforms / fixed masks), dense-class names."""
    from sparse_caption_b200 import kernels as K
    sd = {k: tr.p[k].clone() for k in tr.names}
    for k in tr.masked:
        sd[k] = K.apply_mask(tr.p[k].contiguous(), tr.s[k].contiguous(), tr.mask_mode(),
                             uniforms=None if tr.flat_u is None else tr._u(k).contiguous()[: tr.p[k].shape[0]].contiguous())
    sd["model.tgt_embed.1.pe"] = tr.pe[None]
    return sd


@pytest.mark.parametrize("baseline", ["greedy", "sample"])
def test_scst_targets_kernel_matches_restatement(baseline):
    from sparse_caption_b200 import kernels as K
    g = torch.Generator().manual_seed(1)
    S, L = 3, 6
    rows = [hand_rows(L)]
    for _ in range(40):   # random captions with EOS anywhere (or none) and pads after it
        r = torch.randint(4, 30, (S * 2, L), generator=g).numpy()
        for i in range(r.shape[0]):
            e = int(torch.randint(0, L + 1, (1,), generator=g))
            if e < L:
                r[i, e], r[i, e + 1:] = 3, 0
        rows.append(r)
    seq = np.concatenate(rows).astype(np.int32)
    R = seq.shape[0]
    score = torch.rand(R, generator=g, dtype=torch.float64) * 3
    base = torch.rand(R // S, generator=g, dtype=torch.float64) * 3 if baseline == "greedy" else None
    out = dict(tokens=torch.empty(R * L, dtype=torch.int32, device=DEV), targets=torch.empty(R * L, dtype=torch.int32, device=DEV),
               tok_w=torch.empty(R * L, device=DEV), key_valid=torch.empty(R * L, device=DEV), inv_norm=torch.empty(1, device=DEV),
               mask_sum=torch.empty(1, device=DEV), mean_reward=torch.empty(1, device=DEV))
    K.scst_targets(torch.from_numpy(seq).to(DEV), score.to(DEV), None if base is None else base.to(DEV), S=S, cider_weight=0.75,
                   bos=2, pad=0, **out)
    tokens, targets, tok_w, key_valid, n, inv_norm, mean_r = scst_targets_np(seq, score.numpy(), None if base is None else base.numpy(),
                                                                           S, 0.75)
    assert np.array_equal(out["tokens"].view(R, L).cpu().numpy(), tokens)
    assert np.array_equal(out["targets"].view(R, L).cpu().numpy(), targets)
    assert np.array_equal(out["key_valid"].view(R, L).cpu().numpy(), key_valid)
    np.testing.assert_allclose(out["tok_w"].view(R, L).cpu().numpy(), tok_w, rtol=1e-6, atol=1e-7)
    assert float(out["mask_sum"]) == n
    np.testing.assert_allclose(float(out["inv_norm"]), inv_norm, rtol=1e-7)
    np.testing.assert_allclose(float(out["mean_reward"]), mean_r, rtol=1e-6, atol=1e-7)
    # data parallel: an outside token count replaces the local one
    glob = torch.tensor([4.0 * n], device=DEV)
    K.scst_targets(torch.from_numpy(seq).to(DEV), score.to(DEV), None if base is None else base.to(DEV), S=S, cider_weight=0.75,
                   bos=2, pad=0, norm_in=glob, **{k: v for k, v in out.items() if k != "mask_sum"})
    np.testing.assert_allclose(float(out["inv_norm"]), 1.0 / (4.0 * n), rtol=1e-7)


def _operand_ptrs(eng):
    lins = [eng.att_embed, eng.generator] + [e[k] for e in eng.enc.values() for k in ("qkv", "o", "ff1", "ff2")]
    lins += [e[k] for e in eng.dec.values() for k in ("qkv", "o", "cq", "ckv", "co", "ff1", "ff2")]
    return [x.w.data_ptr() for x in lins] + [eng.table.data_ptr(), eng.wg_w_all.data_ptr()]


@pytest.mark.parametrize("mask_type", ["supermask", "mask_freeze"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_bound_engine_equals_fresh_engine(precision, mask_type):
    from sparse_caption_b200.engine import OrtEngine
    z, tr, scorer = _tiny(mask_type, precision, use_graph=True)
    att, boxes = z["att_feats"].to(DEV), z["boxes"].to(DEV)
    opt = {"beam_size": 3}
    graphs, ptrs = None, None
    for it in range(4):
        if it:
            tr.scst_step(att, boxes, scorer=scorer, opt=opt, lr=3e-3, mask_lr=5.0)
        eng = tr.rollout_engine()
        tr._scst_masks(eng)
        seq, lp = eng.decode(eng.encode(att, boxes), opt)
        seq, lp = seq.clone(), lp.clone()
        fresh = OrtEngine(_folded(tr), tr.cfg, precision=precision, use_graphs=False)
        fseq, flp = fresh.decode(fresh.encode(att, boxes), opt)
        assert torch.equal(seq, fseq), it
        torch.testing.assert_close(lp, flp, rtol=1e-5, atol=1e-5)
        now = {k: ws.graph for k, ws in eng._dec_ws.items()}, {k: ws.graph for k, ws in eng._enc_ws.items()}
        if graphs is None:
            graphs, ptrs = now, _operand_ptrs(eng)
        else:   # same graph objects (no capture after the first step), same operand memory
            assert all(now[0][k] is v for k, v in graphs[0].items()) and all(now[1][k] is v for k, v in graphs[1].items())
            assert _operand_ptrs(eng) == ptrs
    assert tr.opt_step == 3


def _oracle_grads(z, tr, sample, reward):
    """RewardCriterion on oracle.forward_tf with the trainer's (pre-step) weights and mask sample: (loss, dW, dS)."""
    cfg, full = z["cfg"], z["w"]
    W = {k: tr.p[k].detach().cpu().clone().requires_grad_(True) for k in tr.names}
    S = {k: tr.s[k].detach().cpu().clone().requires_grad_(True) for k in tr.masked}
    eff = dict(W)
    for k in tr.masked:
        p = torch.sigmoid(S[k])
        m = (z["u"][k] < p).float()
        eff[k] = (p + (m - p).detach()) * W[k]
    eff["model.tgt_embed.1.pe"] = full["model.tgt_embed.1.pe"]
    R, L = sample.shape
    seqs = torch.cat([torch.full((R, 1), 2, dtype=torch.long), sample.long()], 1)
    lp = O.forward_tf(eff, cfg, z["att_feats"], z["boxes"], seqs, None)
    lp = lp[:, :L].gather(2, sample.long().unsqueeze(2)).squeeze(2)
    mask = (sample != 0).float()
    mask = torch.cat([mask.new_ones(R, 1), mask[:, :-1]], 1)
    loss = (-lp * reward[:, None] * mask).sum() / mask.sum()
    loss.backward()
    return float(loss), {k: W[k].grad for k in W}, {k: S[k].grad for k in S}


@pytest.mark.parametrize("opt,baseline", [({"beam_size": 3}, "greedy"), ({"beam_size": 3}, "sample"),
                                          ({"num_random_sample": 3, "beam_size": 0}, "greedy"),
                                          ({"num_random_sample": 3, "beam_size": 0}, "sample")])
def test_gradients_match_oracle(opt, baseline):
    def err(a, b):
        a, b = a.double().cpu(), b.double()
        return float((a - b).abs().max() / b.abs().max().clamp_min(1e-5))

    for precision in ("fp32", "bf16"):
        z, tr, scorer = _tiny("supermask", precision)
        B = z["att_feats"].shape[0]
        # lr = 0: the step's gradients stay inspectable against the unchanged weights
        loss, mean_r, sample = tr.scst_step(z["att_feats"].to(DEV), z["boxes"].to(DEV), scorer=scorer, opt=opt, baseline=baseline,
                                            lr=0.0, mask_lr=0.0)
        L = tr.cfg.max_seq_length
        R = sample.shape[0] * sample.shape[1]
        ws = tr._get_ws(B, z["att_feats"].shape[1], sample.shape[1], L, False)
        reward = ws.tok_w.view(R, L)[:, 0].cpu()           # tok_w[r, 0] = reward[r] (mask[r, 0] = 1)
        assert float(reward.abs().max()) > 0 and abs(float(mean_r) - float(reward.double().mean())) < 1e-5
        tr.materialize_grads()
        o_loss, gW, gS = _oracle_grads(z, tr, sample.view(R, L).cpu(), reward)
        assert abs(float(loss) - o_loss) < (1e-4 if precision == "fp32" else 3e-2) * max(1.0, abs(o_loss))
        if precision == "fp32":
            for k in tr.names:
                assert err(tr.g[k], gW[k]) < 1e-3, k
            for k in tr.masked:
                assert err(tr.gs[k], gS[k]) < 1e-3, k + "_pruning_mask"
        else:
            errs = sorted(err(tr.g[k], gW[k]) for k in tr.names)
            assert errs[len(errs) // 2] < 3e-2, errs[len(errs) // 2]


@pytest.mark.parametrize("mask_type", ["supermask", "mask_freeze"])
def test_graph_mode_matches_eager(mask_type):
    res = {}
    for graph in (False, True):
        z, tr, scorer = _tiny(mask_type, "fp32", use_graph=graph)
        s0 = tr.flat_s.clone()
        losses = []
        for step in range(2):
            loss, _, _ = tr.scst_step(z["att_feats"].to(DEV), z["boxes"].to(DEV), scorer=scorer, opt={"beam_size": 3}, lr=1e-3 * (step + 1))
            losses.append(float(loss))
            if mask_type == "mask_freeze":
                assert torch.equal(tr.flat_s, s0)    # fixed masks are never updated
        res[graph] = losses, tr.flat_w.clone(), tr.flat_s.clone()
    for a, b in zip(res[True][0], res[False][0]):
        assert abs(a - b) < 2e-3 * max(abs(b), 1e-3), (res[True][0], res[False][0])
    assert float((res[True][1] - res[False][1]).abs().mean() / res[False][1].abs().mean()) < 2e-3


def test_full_size_gradient_is_additive_over_image_shards():
    """configs[1] (ORT 6x512, V = 10000), 50 images x beam 5, bf16, fixed 0/1 masks at 95 %: the gradient of the whole batch equals
    the sum over two image shards that normalise by the global token count (the all_reduce of scst_step)."""
    import bench
    from sparse_caption_b200 import synthetic
    from sparse_caption_b200.cider import CiderD
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200.trainer import OrtTrainer
    cfg = ModelCfg(dict(bench.CFG))
    sd = synthetic.random_state_dict(cfg, seed=1234, device=DEV)
    g = torch.Generator(device="cpu").manual_seed(2)
    for k in [k for k, v in sd.items() if k.endswith(".weight") and v.dim() == 2]:
        sd[k + "_pruning_mask"] = (torch.rand(sd[k].shape, generator=g) >= 0.95).float().to(DEV)
    B, S, L = 50, 5, cfg.max_seq_length
    att, boxes = synthetic.synthetic_inputs(B, 36, 2048, seed=3)
    att, boxes = att.to(DEV), boxes.to(DEV)
    tr = OrtTrainer(sd, cfg, mask_type="mask_freeze", precision="bf16", device=DEV, seed=9, dropout=0.0, drop_prob_src=0.0)
    # references: each image's own greedy caption and a random one, so that the beams' CIDEr-D differ
    eng = tr.rollout_engine()
    tr._scst_masks(eng)
    greedy, _ = eng.decode(eng.encode(att, boxes), {"beam_size": 1})
    refs = [[[int(t) for t in greedy[i, 0].tolist() if t not in (0, 3)] or [5],
             torch.randint(4, 10000, (8,), generator=g).tolist()] for i in range(B)]
    scorer = CiderD.from_corpus(refs, device=DEV)
    opt = {"beam_size": 5}

    def step(lo, hi, total=None):
        tr.step_id = 0
        def ar(t):   # data parallel stand-in: the token count of the whole batch; the gradient buckets stay local
            if t.numel() == 1:
                t.fill_(total)
        loss, _, seq = tr.scst_step(att[lo:hi], boxes[lo:hi], scorer=scorer, image_ids=torch.arange(lo, hi, device=DEV), opt=opt,
                                    lr=0.0, all_reduce=None if total is None else ar)
        ws = tr._get_ws(hi - lo, 36, S, L, False)
        torch.cuda.synchronize()
        return float(loss), tr.flat_gw.clone(), seq.clone(), float(ws.mask_sum)

    l_all, g_all, s_all, total = step(0, B)
    l_a, g_a, s_a, _ = step(0, 20, total)
    l_b, g_b, s_b, _ = step(20, B, total)
    assert torch.equal(torch.cat([s_a, s_b]), s_all)
    assert float(g_all.abs().max()) > 0 and torch.isfinite(g_all).all()
    assert abs(l_all - (l_a + l_b)) < 1e-3 * max(abs(l_all), 1e-6)
    d = (g_a + g_b - g_all).abs().max() / g_all.abs().max()
    assert float(d) < 2e-3, float(d)


def _acort_model():
    import sparse_caption_b200.relation_transformer as RT
    z = golden_io.load("acort_tiny")
    m = RT.get_model("relation_transformer")(z["cfg_dict"])   # (the fixture holds the dense ACORT weights)
    m.load_state_dict(z["w"], strict=True)
    m = m.cuda()
    m.precision = "fp32"
    return z, m


def test_module_trainer_scst_step_acort():
    from sparse_caption_b200.cider import CiderD
    from sparse_caption_b200.trainer import ModuleTrainer
    z, m = _acort_model()
    att, boxes = z["att_feats"].cuda(), z["boxes"].cuda()
    B = att.shape[0]
    scorer = CiderD.from_corpus(_refs(z, B), device=DEV)
    tr = m.trainer()
    assert isinstance(tr, ModuleTrainer)
    before = {k: v.detach().clone() for k, v in m.named_parameters()}
    loss, mean_r, seq = tr.scst_step(att, boxes, scorer=scorer, opt={"num_random_sample": 3, "beam_size": 0}, baseline="sample", lr=1e-3)
    assert torch.isfinite(loss) and tuple(seq.shape) == (B, 3, m.cfg.max_seq_length) and torch.isfinite(mean_r).all()
    assert all(p.grad is None or torch.isfinite(p.grad).all() for p in m.parameters())
    assert any(not torch.equal(before[k], v) for k, v in m.named_parameters())

    # a fixed (deterministic) rollout: beam search, no dropout -> the explicit recipe of test_cider.py
    z, m = _acort_model()
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    tr = m.trainer()
    loss, _, seq = tr.scst_step(att, boxes, scorer=scorer, opt={"beam_size": 3}, lr=0.0, mask_lr=0.0)
    got = {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    for p in m.parameters():
        p.grad = None
    m.eval()
    greedy, _ = m(att_feats=att, boxes=boxes, opt={"beam_size": 1}, mode="sample")
    m.train()
    sc_s, sc_b = scorer.scst_reward(seq, greedy)
    reward = (sc_s - sc_b).float()
    L = seq.shape[-1]
    sample = seq.reshape(B * 3, L).long()
    seqs = torch.cat([torch.full((B * 3, 1), m.bos_idx, device=DEV), sample], 1)
    logp = m(att_feats=att, boxes=boxes, seqs=torch.cat([seqs, torch.zeros(B * 3, 1, dtype=torch.long, device=DEV)], 1))
    lp = logp[:, :L].gather(2, sample.view(B * 3, L, 1)).squeeze(2)
    mask = (sample != m.pad_idx).float()
    mask = torch.cat([mask.new_ones(B * 3, 1), mask[:, :-1]], 1)
    want = (-lp * reward[:, None] * mask).sum() / mask.sum()
    want.backward()
    assert abs(float(loss) - float(want)) < 1e-5 * max(1.0, abs(float(want)))
    for n, p in m.named_parameters():
        if p.grad is not None and n in got:
            assert float((got[n] - p.grad).abs().max()) <= 1e-4 * max(float(p.grad.abs().max()), 1e-6), n


@pytest.mark.parametrize("name", ["relation_transformer", "relation_transformer_prune"])
def test_model_surface(name):
    import sparse_caption_b200.relation_transformer as RT
    from sparse_caption_b200.cider import CiderD
    z = golden_io.load("ort_prune_tiny")
    cfg = dict(z["cfg_dict"])
    m = RT.get_model(name)(cfg)
    w = z["w"] if name.endswith("prune") else {k: v for k, v in z["w"].items() if not k.endswith("_pruning_mask")}
    m.load_state_dict(w, strict=True)
    m = m.cuda()
    att, boxes = z["att_feats"].cuda(), z["boxes"].cuda()
    B, L = att.shape[0], cfg["max_seq_length"]
    scorer = CiderD.from_corpus(_refs(z, B), device=DEV)
    tr = m.trainer()
    for opt, S in (({"beam_size": 3}, 3), ({"num_random_sample": 4, "beam_size": 0}, 4)):
        loss, mean_r, seq = tr.scst_step(att, boxes, scorer=scorer, opt=opt, lr=1e-3)
        assert loss.numel() == 1 and torch.isfinite(loss).all() and mean_r.numel() == 1
        assert tuple(seq.shape) == (B, S, L) and seq.is_cuda
    m.sync_from_trainer()
    sd = tr.state_dict()
    for k, v in m.state_dict().items():
        if k in sd:
            assert torch.equal(v, sd[k].to(v.device)), k
    assert m.trainer() is tr   # the module now holds the trainer's parameters
