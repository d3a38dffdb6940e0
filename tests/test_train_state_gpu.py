"""Resumable training on the device: the trainer a fresh model builds from model_last.pth + optimizer_last.pth is bitwise the
trainer that saved them, and it continues the run as the uninterrupted trainer does (OrtTrainer in fp32 / bf16, eager / graph
mode, across a gradual pruning event and SCST steps; ModuleTrainer on ACORT); the state loads into and out of torch.optim.Adam
built like the reference's optimizer; a pending SNIP saliency is refused; with >= 2 GPUs the ShardedExchange export equals the
all-reduce run's state.

The continuation is compared within tolerances, not bitwise: the training step itself is not bitwise reproducible.  It sums the
loss and the bias, LayerNorm and embedding gradients with float atomics, so two runs of the same steps from the same state differ
in the last bits, and Adam's sign-like update turns a last-bit change of a near-zero gradient into a change of up to 2 lr in that
weight.  Measured on a B200, two uninterrupted 6-step runs of the fp32 eager setup below: losses 1 ulp apart, m_w up to 5.6e-9,
flat_s up to 1.4e-5, and 12915 weights up to 1.5e-3; the module path (ACORT) differs the same way.  So the two continuations start
from one bitwise-equal state and are held to tolerances far below what a wrong restore causes: measured, the continuations of
this file stay within 3.3e-7 of each other (losses, moments, logits, relative), while a Philox seed off by one or lost moments
move the losses by 1e-3 to 6e-2 and the moments by 0.3 to 1.2 (test_continuation_check_detects_a_wrong_restore)."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests import golden_io

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUFFIX = "_pruning_mask"


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _model(name, mask_type, sd=None, precision="fp32"):
    import sparse_caption_b200.relation_transformer as R
    z = golden_io.load(name)
    torch.manual_seed(0)
    m = R.get_model("relation_transformer_prune")(dict(z["cfg_dict"], prune_type=mask_type))
    if sd is None:   # the golden weights, and supermask logits spread over both sides of 0 (masks that really sample)
        sd = m.state_dict()
        sd.update({k: v for k, v in z["w"].items() if k in sd})
        g = torch.Generator().manual_seed(1)
        for k in sd:
            if k.endswith(SUFFIX) and mask_type == "supermask":
                sd[k] = torch.randn(sd[k].shape, generator=g) * 2 + 1
    m.load_state_dict(sd)
    m.precision = precision
    return m.to(DEV), z


def _params(m):
    named = list(m.named_parameters())
    return [p for n, p in named if not n.endswith(SUFFIX)], [p for n, p in named if n.endswith(SUFFIX)]


def _bitwise_differences(sa, sb):
    """[(key, differing elements or values)] of two state dicts of tensors and numbers."""
    out = []
    for k in sa:
        if torch.is_tensor(sa[k]) and not torch.equal(sa[k], sb[k]):
            out.append((k, int((sa[k] != sb[k]).sum())))
        elif not torch.is_tensor(sa[k]) and sa[k] != sb[k]:
            out.append((k, sa[k], sb[k]))
    return out


def _beyond_tolerance(a, b, weights):
    """[(what, error)] where the continuation ``b`` = (per-step losses, final state) leaves the tolerances around ``a``: losses and
    rewards 1e-4 relative, every other state tensor 1e-4 of its largest element, except the weights (``weights``: their keys),
    held to 5e-3 in mean absolute difference over mean magnitude (the sign-like update, see the module docstring); counters exact."""
    (la, sa), (lb, sb) = a, b
    err = {f"step {i + 4}": float((x - y).abs().max() / x.abs().max()) for i, (x, y) in enumerate(zip(la, lb))}
    limit = dict.fromkeys(err, 1e-4)
    out = []
    for k in sa:
        if not torch.is_tensor(sa[k]):
            if sa[k] != sb[k]:
                out.append((k, (sa[k], sb[k])))
        elif k in weights:
            err[k], limit[k] = float((sa[k] - sb[k]).abs().mean() / sa[k].abs().mean()), 5e-3
        else:
            err[k], limit[k] = rel_err(sb[k], sa[k]), 1e-4
    print("continuation errors (limit):", {k: f"{v:.1e} ({limit[k]:.0e})" for k, v in err.items() if v > 0})
    return out + [(k, v) for k, v in err.items() if v > limit[k]]


# ---- OrtTrainer ------------------------------------------------------------------------------------------------------------------
def _ort_step(tr, z, i, kind, scorer):
    """Step i + 1: (loss [, mean reward]) and, for SCST, the sampled captions."""
    att, boxes = z["att_feats"].to(DEV), z["boxes"].to(DEV)
    if kind == "prune":   # an event at step 4 only (the first step after the restart): mag_grad_blind to 50 %
        tr.update_masks_gradual(0.8, current_step=i, start_step=3, prune_steps=1, initial_sparsity=0.5, prune_frequency=10)
    if kind == "scst" and i >= 3:
        loss, reward, seq = tr.scst_step(att, boxes, scorer=scorer, opt={"num_random_sample": 2, "beam_size": 0}, lr=1e-3)
        return torch.cat([loss.reshape(1), reward.reshape(1)]), seq
    S = z["seqs"].shape[0] // att.shape[0]
    sp = dict(sparsity_target=0.5, sparsity_weight=1.0, current_step=i, max_step=10) if tr.mask_type == "supermask" else {}
    return tr.train_step(att, boxes, z["seqs"], z["masks"], seq_per_img=S, lr=1e-3, **sp).reshape(1).clone(), None


def _ort_state(tr):
    """The trainer's state.  The logit moments outside the parameters are left out: the sparsity-loss term gives the generator's
    padded logit rows moments, but every update resets those logits to -1, so those moments never reach a parameter (a loaded
    trainer has zeros there).  The weights without the generator's padding (its bias is -1e9)."""
    torch.cuda.synchronize()
    live = ~tr._s_pad_mask
    return dict(weights=torch.cat([tr.p[k].reshape(-1) for k in tr.names]), flat_s=tr.flat_s.clone(), m_w=tr.m_w.clone(), v_w=tr.v_w.clone(), m_s=tr.m_s[live].clone(),
                v_s=tr.v_s[live].clone(), opt_step=tr.opt_step, step_id=tr.step_id, seed=tr.seed, sparsity_target=tr.sparsity_target)


def _ort_resume(precision, graph, kind, scorer, tmp, tamper=None):
    """3 steps; model_last.pth + optimizer_last.pth through torch.save; a fresh model and trainer built from the two files (checked
    bitwise against the saved trainer, then ``tamper``-ed) and the original trainer each take steps 4-6.  Returns the two runs'
    (per-step outputs, sampled captions, final state)."""
    mask_type = "mag_grad_blind" if kind == "prune" else "supermask"
    m, z = _model("ort_tiny", mask_type, precision=precision)
    tr = m.trainer(seed=5, use_graph=graph)
    for i in range(3):
        _ort_step(tr, z, i, kind, scorer)
    saved = _ort_state(tr)
    m.sync_from_trainer()
    torch.save(m.state_dict(), os.path.join(tmp, "model_last.pth"))
    torch.save(tr.optimizer_state_dict(), os.path.join(tmp, "optimizer_last.pth"))
    m2, _ = _model("ort_tiny", mask_type, sd=torch.load(os.path.join(tmp, "model_last.pth")), precision=precision)
    tr2 = m2.trainer(seed=123, use_graph=graph)    # (the seed comes from the optimizer state)
    tr2.load_optimizer_state_dict(torch.load(os.path.join(tmp, "optimizer_last.pth")))
    assert not _bitwise_differences(saved, _ort_state(tr2)), _bitwise_differences(saved, _ort_state(tr2))
    if tamper is not None:
        tamper(tr2)
    runs = []
    for t in (tr, tr2):
        out = [_ort_step(t, z, i, kind, scorer) for i in range(3, 6)]
        runs.append(([o[0] for o in out], [o[1] for o in out], _ort_state(t)))
    return runs


@pytest.fixture(scope="module")
def scorer():
    from sparse_caption_b200.cider import CiderD
    z = golden_io.load("ort_tiny")
    refs = [[[int(t) for t in row[1:] if t not in (0, 3)] for row in z["seqs"][i * 2: (i + 1) * 2]] for i in range(z["att_feats"].shape[0])]
    return CiderD.from_corpus(refs, device=DEV)


@pytest.mark.parametrize("kind", ["train", "prune", "scst"])
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_ort_resume_restores_the_trainer_and_continues_the_run(precision, graph, kind, scorer, tmp_path):
    (la, qa, sa), (lb, qb, sb) = _ort_resume(precision, graph, kind, scorer, str(tmp_path))
    assert sb["opt_step"] == 6 and sb["step_id"] == 6
    assert not _beyond_tolerance((la, sa), (lb, sb), ("weights",)), _beyond_tolerance((la, sa), (lb, sb), ("weights",))
    if kind == "scst":   # step 4 samples from one bitwise state with one Philox position: the same captions
        assert torch.equal(qa[0], qb[0])
    if kind == "prune":  # the masks of the step-4 event, selected from one bitwise state; later steps leave them alone
        assert torch.equal(sa["flat_s"], sb["flat_s"]) and sb["sparsity_target"] == 0.5


def test_continuation_check_detects_a_wrong_restore(scorer, tmp_path):
    """The tolerances of the continuation check against what a wrong restore does: the Philox seed one off (other masks and
    dropout), or the moments lost (a restart with a fresh optimizer)."""
    def seed_off(tr):
        tr.seed += 1

    def moments_lost(tr):
        for buf in (tr.m_w, tr.v_w, tr.m_s, tr.v_s):
            buf.zero_()
        tr.opt_step = 0

    for tamper in (seed_off, moments_lost):
        (la, _, sa), (lb, _, sb) = _ort_resume("fp32", False, "train", scorer, str(tmp_path), tamper=tamper)
        sa, sb = dict(sa, opt_step=0, step_id=0, seed=0), dict(sb, opt_step=0, step_id=0, seed=0)   # (the values, not the counters)
        assert _beyond_tolerance((la, sa), (lb, sb), ("weights",)), tamper.__name__


# ---- ModuleTrainer (ACORT) ----------------------------------------------------------------------------------------------------------
def _acort_step(tr, z, i):
    S = z["seqs"].shape[0] // z["att_feats"].shape[0]
    return tr.train_step(z["att_feats"], z["boxes"], z["seqs"], z["masks"], seq_per_img=S, lr=1e-3, mask_lr=10.0, sparsity_target=0.5,
                         sparsity_weight=1.0, current_step=i, max_step=10).reshape(1).clone()


def _acort_state(m, tr):
    from sparse_caption_b200 import sampler
    torch.cuda.synchronize()
    state = {n: p.detach().clone() for n, p in m.named_parameters()}
    state.update({f"{n}/{j}": t.clone() for n, mv in tr._mv.items() for j, t in enumerate(mv)})
    return dict(state, opt_step=tr.opt_step, **{f"sampler.{k}": sampler._state[k] for k in ("seed", "stream", "drop")})


def test_acort_module_trainer_restores_and_continues(tmp_path):
    """fp32 (the module path's bf16 backward needs out_features % 8 == 0; the tiny ACORT vocabulary has 35 words).  The sampler's
    streams are process-wide: each continuation starts from the position it had when the state was saved, as a new process
    would after loading the file."""
    from sparse_caption_b200 import sampler
    sampler.set_mask_seed(11)
    sampler._state["drop"] = 0
    m, z = _model("acort_tiny", "supermask")
    tr = m.trainer()
    for i in range(3):
        _acort_step(tr, z, i)
    saved = _acort_state(m, tr)
    torch.save(m.state_dict(), os.path.join(tmp_path, "model_last.pth"))
    torch.save(tr.optimizer_state_dict(), os.path.join(tmp_path, "optimizer_last.pth"))
    runs = [([_acort_step(tr, z, i) for i in range(3, 6)], _acort_state(m, tr))]
    sampler.set_mask_seed(999)
    sampler._state["drop"] = 0
    m2, _ = _model("acort_tiny", "supermask", sd=torch.load(os.path.join(tmp_path, "model_last.pth")))
    tr2 = m2.trainer()
    tr2.load_optimizer_state_dict(torch.load(os.path.join(tmp_path, "optimizer_last.pth")))
    assert not _bitwise_differences(saved, _acort_state(m2, tr2)), _bitwise_differences(saved, _acort_state(m2, tr2))
    runs.append(([_acort_step(tr2, z, i) for i in range(3, 6)], _acort_state(m2, tr2)))
    weights = [n for n, _ in m.named_parameters() if not n.endswith(SUFFIX)]
    assert runs[1][1]["opt_step"] == 6 and runs[1][1]["sampler.stream"] == runs[0][1]["sampler.stream"]
    assert not _beyond_tolerance(runs[0], runs[1], weights), _beyond_tolerance(runs[0], runs[1], weights)


# ---- torch.optim.Adam interoperability -------------------------------------------------------------------------------------------
def _views(tr):
    """{module parameter: (trainer parameter view, exp_avg view, exp_avg_sq view, gradient view)} in the trainer's buffers."""
    out = {}
    for k in tr.names:
        o, n = tr._offs_w[k], tr.p[k].numel()
        out[k] = (tr.p[k], tr.m_w[o: o + n].view(tr.p[k].shape), tr.v_w[o: o + n].view(tr.p[k].shape), tr.g[k])
    for k in tr.masked:
        o, n = tr._offs_s[k], tr.s[k].numel()
        out[k + SUFFIX] = (tr.s[k], tr.m_s[o: o + n].view(tr.s[k].shape), tr.v_s[o: o + n].view(tr.s[k].shape), tr.gs[k])
    return out


def test_torch_adam_loads_the_trainer_state_and_takes_the_same_step():
    m, z = _model("ort_tiny", "supermask")
    tr = m.trainer(seed=5, fused_st=False)
    S = z["seqs"].shape[0] // z["att_feats"].shape[0]
    for _ in range(2):
        tr.train_step(z["att_feats"].to(DEV), z["boxes"].to(DEV), z["seqs"], z["masks"], seq_per_img=S, lr=1e-3)
    m.sync_from_trainer()
    w, s = _params(m)
    opt = torch.optim.Adam([{"params": w}, {"params": s, "lr": 100.0, "eps": 1e-2}], lr=1e-3, betas=(0.9, 0.98), eps=1e-9)
    opt.load_state_dict(tr.optimizer_state_dict())
    views = _views(tr)
    named = dict(m.named_parameters())
    for n, p in named.items():
        assert torch.equal(opt.state[p]["exp_avg"], views[n][1]) and torch.equal(opt.state[p]["exp_avg_sq"], views[n][2]), n
        assert float(opt.state[p]["step"]) == 2.0
    # the same random gradients (some beyond the 0.1 clip) -> clip_grad_value_ + Adam against the trainer's two-group update
    g = torch.Generator().manual_seed(3)
    tr.flat_gw.zero_()
    tr.flat_gs.zero_()
    for n, p in named.items():
        p.grad = (torch.randn(p.shape, generator=g) * 0.08).to(DEV)
        views[n][3].copy_(p.grad)
    torch.nn.utils.clip_grad_value_(list(named.values()), 0.1)
    opt.step()
    tr.optimizer_step(lr=1e-3, mask_lr=100.0)
    # (the update kernel forms 1 - beta2 in fp32, 0.01999998, where torch rounds 0.02 from double: exp_avg_sq differs by up to
    # 9.5e-7 relative from that constant alone)
    for n, p in named.items():
        assert rel_err(views[n][0], p.detach()) < 1e-6, n
        assert rel_err(views[n][1], opt.state[p]["exp_avg"]) < 1e-6 and rel_err(views[n][2], opt.state[p]["exp_avg_sq"]) < 2e-6, n


def test_trainer_loads_a_torch_adam_state_bit_for_bit():
    m, _ = _model("ort_tiny", "supermask")
    w, s = _params(m)
    opt = torch.optim.Adam([{"params": w}, {"params": s, "lr": 100.0, "eps": 1e-2, "pruning_mask": True}], lr=1e-3, betas=(0.9, 0.98),
                           eps=1e-9)
    g = torch.Generator().manual_seed(4)
    for _ in range(3):
        for p in w + s:
            p.grad = (torch.randn(p.shape, generator=g) * 0.05).to(DEV)
        opt.step()
    tr = m.trainer(seed=5)
    tr.load_optimizer_state_dict(opt.state_dict())
    views = _views(tr)
    for n, p in m.named_parameters():
        assert torch.equal(views[n][1], opt.state[p]["exp_avg"]) and torch.equal(views[n][2], opt.state[p]["exp_avg_sq"]), n
    assert tr.opt_step == 3 and tr.step_id == 3
    assert tr._hyper["mask_lr"] == 100.0 and tr._hyper["mask_eps"] == 1e-2 and tr._hyper["lr"] == 1e-3


def test_pending_snip_saliency_is_refused():
    m, z = _model("ort_tiny", "snip")
    tr = m.trainer(seed=5)
    S = z["seqs"].shape[0] // z["att_feats"].shape[0]
    tr.snip_saliency(z["att_feats"].to(DEV), z["boxes"].to(DEV), z["seqs"], z["masks"], seq_per_img=S)
    with pytest.raises(ValueError, match="SNIP"):
        tr.optimizer_state_dict()
    tr.update_masks_once(0.5)
    sd = tr.optimizer_state_dict()
    assert sd["trainer"]["sparsity_target"] == 0.5 and len(sd["param_groups"]) == 2


# ---- data parallel, NCCL: the ShardedExchange export equals the all-reduce run's state ---------------------------------------------
def _nccl_worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from sparse_caption_b200 import distributed as D
    from sparse_caption_b200.engine import ModelCfg
    from sparse_caption_b200.trainer import OrtTrainer
    m, z = _model("ort_tiny", "supermask")
    sd = {k: v.to(dev) for k, v in m.state_dict().items()}
    B = z["att_feats"].shape[0]
    S = z["seqs"].shape[0] // B
    lo, hi = D.shard_range(B, rank, world)
    att, boxes = z["att_feats"][lo:hi].to(dev), z["boxes"][lo:hi].to(dev)
    seqs, masks = z["seqs"][lo * S: hi * S], z["masks"][lo * S: hi * S]
    gtok = D.global_token_count(masks.to(dev), seqs.shape[1] - 1)
    res = {}
    for mode in ("all_reduce", "exchange"):
        tr = OrtTrainer(sd, ModelCfg(z["cfg_dict"]), mask_type="supermask", precision="fp32", device=dev, seed=5, dropout=0.0,
                        drop_prob_src=0.0, fused_st=False)
        ex = D.ShardedExchange(device=dev) if mode == "exchange" else None
        kw = dict(exchange=ex) if ex is not None else dict(all_reduce=D.make_all_reduce(async_op=True))
        for _ in range(2):
            tr.train_step(att, boxes, seqs, masks, seq_per_img=S, lr=1e-3, global_tokens=gtok, **kw)
        res[mode] = tr.optimizer_state_dict(exchange=ex)
    torch.save(res, f"{out}.{rank}")
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_exchange_export_equals_all_reduce_state(tmp_path):
    out = str(tmp_path / "nccl.pt")
    mp.spawn(_nccl_worker, args=(2, 37500 + os.getpid() % 2000, out), nprocs=2, join=True)
    got = [torch.load(f"{out}.{r}") for r in range(2)]
    for r in range(2):
        ex, ar = got[r]["exchange"], got[r]["all_reduce"]
        assert ex["trainer"] == ar["trainer"] and ex["param_groups"] == ar["param_groups"] and sorted(ex["state"]) == sorted(ar["state"])
        for i, st in ar["state"].items():
            for key in ("exp_avg", "exp_avg_sq"):
                assert torch.equal(ex["state"][i][key], got[0]["exchange"]["state"][i][key])   # every rank returns the same state
                assert rel_err(ex["state"][i][key], st[key]) < 1e-5, (r, i, key)
