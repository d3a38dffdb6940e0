"""CPU tier of the resumable optimizer state: the layout of ``OrtTrainer.optimizer_state_dict`` against ``torch.optim.Adam`` built over
the drop-in module's parameters in the reference's two groups, the round trip through ``torch.save``, the load errors, and - world
size 3 over gloo - the all-gather of the moments a ``ShardedExchange`` run keeps on the shard owners only.  The trainer is built
on the CPU for its parameter layout; no kernel runs here."""
import io
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests import golden_io

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUFFIX = "_pruning_mask"


def _module(mask_type="supermask"):
    import sparse_caption_b200.relation_transformer as R
    z = golden_io.load("ort_tiny")
    torch.manual_seed(0)
    return R.get_model("relation_transformer_prune")(dict(z["cfg_dict"], prune_type=mask_type))


def _trainer(m, **kw):
    from sparse_caption_b200.trainer import OrtTrainer
    kw = dict(dict(mask_type=m.mask_type if m.MASKED else None, precision="fp32", device="cpu", seed=7), **kw)
    return OrtTrainer(m.state_dict(), m.cfg, **kw)


def _fill(tr, seed=1):
    """Seeded moments in every parameter's view (the padding stays zero, as after real steps), opt_step / step_id as after 5 steps."""
    g = torch.Generator().manual_seed(seed)
    for buf in (tr.m_w, tr.v_w, tr.m_s, tr.v_s):
        buf.copy_(torch.rand(buf.shape, generator=g))
    keep_w = torch.zeros_like(tr.m_w, dtype=torch.bool)
    for k in tr.names:
        keep_w[tr._offs_w[k]: tr._offs_w[k] + tr.p[k].numel()] = True
    for buf in (tr.m_w, tr.v_w):
        buf[~keep_w] = 0.0
    for buf in (tr.m_s, tr.v_s):
        buf[tr._s_pad_mask] = 0.0
    tr.opt_step, tr.step_id = 5, 6


def _groups(m):
    named = [(n, p) for n, p in m.named_parameters()]
    return [[p for n, p in named if not n.endswith(SUFFIX)], [p for n, p in named if n.endswith(SUFFIX)]]


def test_layout_loads_into_torch_adam_of_the_reference_groups():
    m = _module()
    tr = _trainer(m)
    _fill(tr)
    tr._hyper.update(lr=3e-4, mask_lr=50.0)
    sd = tr.optimizer_state_dict()
    w, s = _groups(m)
    assert [len(g["params"]) for g in sd["param_groups"]] == [len(w), len(s)]
    assert sd["param_groups"][0]["params"] == list(range(len(w)))
    assert sd["param_groups"][1]["params"] == list(range(len(w), len(w) + len(s)))
    assert sd["param_groups"][1]["pruning_mask"] is True and sd["param_groups"][1]["lr"] == 50.0
    assert sd["param_groups"][1]["eps"] == 1e-2 and sd["param_groups"][0]["eps"] == 1e-9
    assert sd["trainer"] == {"step_id": 6, "seed": 7, "mask_type": "supermask", "sparsity_target": 0.0}
    # every entry: a CPU tensor of the parameter's shape that owns exactly its elements, step = opt_step
    for i, p in enumerate(w + s):
        st = sd["state"][i]
        assert st["exp_avg"].shape == p.shape and st["exp_avg_sq"].shape == p.shape and st["exp_avg"].device.type == "cpu"
        assert st["exp_avg"].untyped_storage().nbytes() == 4 * p.numel()
        assert st["step"].dtype == torch.float32 and float(st["step"]) == 5.0
    # the generator's padded rows are not exported; the per-parameter views are
    gen = "model.generator.proj.weight"
    i = [n for n, _ in m.named_parameters() if not n.endswith(SUFFIX)].index(gen)
    assert tr.Vp > tr.cfg.vocab_size or sd["state"][i]["exp_avg"].shape[0] == tr.cfg.vocab_size
    o = tr._offs_w[gen]
    assert torch.equal(sd["state"][i]["exp_avg"].reshape(-1), tr.m_w[o: o + tr.p[gen].numel()])
    opt = torch.optim.Adam([{"params": w}, {"params": s, "lr": 100.0, "eps": 1e-2, "pruning_mask": True}], lr=1e-3, betas=(0.9, 0.98),
                           eps=1e-9)
    opt.load_state_dict(sd)
    for i, p in enumerate(w + s):
        assert torch.equal(opt.state[p]["exp_avg"], sd["state"][i]["exp_avg"])
    assert opt.param_groups[1]["lr"] == 50.0 and opt.param_groups[0]["lr"] == 3e-4
    # back into a fresh trainer, through torch.save
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    tr2 = _trainer(m, seed=0)
    tr2.load_optimizer_state_dict(torch.load(buf))
    for a, b in ((tr.m_w, tr2.m_w), (tr.v_w, tr2.v_w), (tr.m_s, tr2.m_s), (tr.v_s, tr2.v_s)):
        assert torch.equal(a, b)
    assert (tr2.opt_step, tr2.step_id, tr2.seed) == (5, 6, 7) and tr2._hyper == tr._hyper
    # torch Adam's own state dict: no "trainer" key, the Philox position continues at step_id = opt_step
    tr3 = _trainer(m)
    tr3.load_optimizer_state_dict(opt.state_dict())
    assert torch.equal(tr3.m_s, tr.m_s) and (tr3.opt_step, tr3.step_id) == (5, 5)


@pytest.mark.parametrize("mask_type", [None, "mag_blind"])
def test_groups_without_logit_updates(mask_type):
    """Dense: one group.  Masks the trainer does not update: listed in group 1 without state, as torch.optim.Adam lists parameters
    that never received a gradient; loading needs no entry for them."""
    import sparse_caption_b200.relation_transformer as R
    if mask_type is None:
        z = golden_io.load("ort_tiny")
        m = R.get_model("relation_transformer")(z["cfg_dict"])
    else:
        m = _module(mask_type)
    tr = _trainer(m, mask_type=mask_type)
    _fill(tr)
    sd = tr.optimizer_state_dict()
    n_w = len([n for n, _ in m.named_parameters() if not n.endswith(SUFFIX)])
    assert len(sd["param_groups"]) == (1 if mask_type is None else 2) and sorted(sd["state"]) == list(range(n_w))
    if mask_type:
        assert len(sd["param_groups"][1]["params"]) == len(tr.masked)
    tr2 = _trainer(m, mask_type=mask_type)
    tr2.load_optimizer_state_dict(sd)
    assert torch.equal(tr2.m_w, tr.m_w) and float(tr2.m_s.abs().sum()) == 0.0


def test_load_errors_name_the_parameter():
    m = _module()
    tr = _trainer(m)
    _fill(tr)
    names = [n for n, _ in m.named_parameters() if not n.endswith(SUFFIX)]
    i = names.index("model.decoder.layers.1.feed_forward.w_1.weight")

    def fresh():
        return _trainer(m), tr.optimizer_state_dict()

    t, sd = fresh()
    sd["state"][i]["exp_avg"] = sd["state"][i]["exp_avg"][:, :-1]
    with pytest.raises(ValueError, match="model.decoder.layers.1.feed_forward.w_1.weight"):
        t.load_optimizer_state_dict(sd)
    t, sd = fresh()
    del sd["state"][i]
    with pytest.raises(ValueError, match="feed_forward.w_1.weight: no optimizer state"):
        t.load_optimizer_state_dict(sd)
    t, sd = fresh()
    j = len(names) + 3
    del sd["state"][j]                        # a supermask logit: the trainer updates it
    with pytest.raises(ValueError, match=SUFFIX):
        t.load_optimizer_state_dict(sd)
    t, sd = fresh()
    sd["state"][i]["step"] = torch.tensor(4.0)
    with pytest.raises(ValueError, match="step 4.0 differs"):
        t.load_optimizer_state_dict(sd)
    t, sd = fresh()
    sd["param_groups"][0]["params"] = sd["param_groups"][0]["params"][:-1]
    with pytest.raises(ValueError, match="parameters"):
        t.load_optimizer_state_dict(sd)
    t, sd = fresh()
    sd["trainer"]["mask_type"] = "mag_blind"
    with pytest.raises(ValueError, match="mask_type"):
        t.load_optimizer_state_dict(sd)
    # nothing was loaded by the failed calls
    assert t.opt_step == 0 and float(t.m_w.abs().sum()) == 0.0
    # a pending SNIP saliency is not part of the resumable state
    ts = _trainer(_module("snip"), mask_type="snip")
    ts._has_saliency = True
    with pytest.raises(ValueError, match="SNIP"):
        ts.optimizer_state_dict()


# ---- ShardedExchange: the moments of the shard owners, all-gathered ------------------------------------------------------------------
def _adam_moments(tr, grads, lo, hi, which):
    """Stand-in for the update: Adam's moment recurrences on [lo, hi) of the weight ("w") or logit ("s") buffers."""
    m, v = (tr.m_w, tr.v_w) if which == "w" else (tr.m_s, tr.v_s)
    g = grads[which][lo:hi]
    m[lo:hi].mul_(0.9).add_(0.1 * g)
    v[lo:hi].mul_(0.98).add_(0.02 * g * g)


def _run(tr, ex, rank, world, steps=2):
    """``steps`` sharded updates over the trainer's buckets with rank-local gradients (their sum over the ranks is the gradient of the
    step), as OrtTrainer._sharded_step issues them."""
    for step in range(steps):
        grads = {}
        for which, flat in (("w", tr.flat_gw), ("s", tr.flat_gs)):
            g = torch.zeros_like(flat)
            for r in (range(world) if ex is None else [rank]):
                g += torch.randn(flat.shape, generator=torch.Generator().manual_seed(1000 * step + 10 * r + (which == "s")))
            flat.copy_(g)
            grads[which] = flat
        for phase in range(tr.N_PHASES):
            for flat, a, b in tr.grad_buckets(phase):
                which = "w" if flat is tr.flat_gw else "s"
                param = tr.flat_w if which == "w" else tr.flat_s
                if ex is None:
                    _adam_moments(tr, grads, a, b, which)
                else:
                    ex.bucket(flat, param, a, b, lambda lo, hi, w=which: _adam_moments(tr, grads, lo, hi, w))
        tr.opt_step += 1
        tr.step_id += 1


def _sharded_worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    from sparse_caption_b200 import distributed as D
    tr = _trainer(_module(), fused_st=False)
    ex = D.ShardedExchange()
    _run(tr, ex, rank, world)
    ex.finish()
    local = tr.optimizer_state_dict()                   # this rank's buffers as they are: live only on its shards
    before = (tr.m_w.clone(), tr.m_s.clone())
    sd = tr.optimizer_state_dict(exchange=ex)
    assert torch.equal(tr.m_w, before[0]) and torch.equal(tr.m_s, before[1])   # (gathered into copies)
    torch.save({"local": local, "gathered": sd}, f"{out}.{rank}")
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_exchange_gathers_the_single_process_state(tmp_path):
    out = str(tmp_path / "state.pt")
    world = 3
    port = 35500 + os.getpid() % 2000
    mp.spawn(_sharded_worker, args=(world, port, out), nprocs=world, join=True)
    tr = _trainer(_module(), fused_st=False)
    _run(tr, None, 0, world)
    want = tr.optimizer_state_dict()
    for r in range(world):
        got = torch.load(f"{out}.{r}")
        assert got["gathered"]["param_groups"] == want["param_groups"] and got["gathered"]["trainer"] == want["trainer"]
        assert sorted(got["gathered"]["state"]) == sorted(want["state"])
        differs = 0
        for i, st in want["state"].items():
            for key in ("exp_avg", "exp_avg_sq"):
                torch.testing.assert_close(got["gathered"]["state"][i][key], st[key], rtol=1e-6, atol=1e-7)
                differs += not torch.allclose(got["local"]["state"][i][key], st[key], rtol=1e-6, atol=1e-7)
        assert differs > 0   # (without the gather a rank holds only its shards)
