"""Beam search with 9 to 32 beams (group_size 1): the radix-select row pass and merge of the beam step, the cross-attention
step over more than 8 query rows per image, and every decode surface at those widths, against torch restatements and the
CPU oracle.  Beams above 32 are refused."""
import pytest
import torch

from oracle import ort_oracle as O
from tests import golden_io
from tests.test_boundary_gpu import _oracle_beam_with_rules
from tests.test_parity_baseline_gpu import ORT, _search_parity, _weights

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def K():
    import sparse_caption_b200.kernels as k
    return k


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


# ------------------------------------------------------------------------------------------------------------------
# K7: the beam step
# ------------------------------------------------------------------------------------------------------------------
class _RefBeam:
    """caption_model.py:56-111 / 195-210 restated step by step in torch: oracle.beam_select (stable descending sort: ties to
    the smaller flat index), ancestors, finished lists (stable insertion by the penalised score, in double), -1000 on finished
    beams and the forced finish at t = L - 1.  The row's log-softmax statistics are taken from the kernel's workspace, so the
    scores are the kernel's bit for bit and every comparison is exact."""

    def __init__(self, B, beam, L, eos, pad, penalty):
        self.B, self.beam, self.L, self.eos, self.pad = B, beam, L, eos, pad
        self.pen = O.length_penalty(penalty)
        self.seq = torch.full((B, beam, L), pad, dtype=torch.long)
        self.lp = torch.zeros(B, beam, L)
        self.anc = torch.arange(B * beam).view(B, beam, 1).expand(B, beam, L).clone()
        self.sum = torch.zeros(B, beam)
        self.done = [[] for _ in range(B)]

    def step(self, x, stats, t, T, constraint, sup, pen_col):
        B, beam, L = self.B, self.beam, self.L
        V = x.shape[-1]
        mx, ls, mx2, ls2 = (stats[:, i:i + 1] for i in range(4))
        lp = (x - mx) - ls
        if t > 0 and T != 1.0:
            lp = (lp / T - mx2) - ls2
        chosen_src = lp.clone()
        if constraint and t > 0:
            lp.scatter_(1, self.seq[:, :, t - 1].reshape(-1, 1), float("-inf"))
        if sup is not None and t > 0:
            rows = (sup >= 0).nonzero().flatten()
            lp[rows, sup[rows]] = float("-inf")
        if 0 <= pen_col < V:
            lp[:, pen_col] -= 1000
            chosen_src[:, pen_col] -= 1000
        if t == 0:
            lp, chosen_src = lp.view(B, beam, V)[:, :1].reshape(B, V), chosen_src.view(B, beam, V)[:, :1].reshape(B, V)
        parent, word, new_sum = O.beam_select(lp, self.sum, beam, first=(t == 0))
        nb = lp.shape[0] // B
        chosen = chosen_src.view(B, nb, V).gather(1, parent.unsqueeze(-1).expand(-1, -1, V)).gather(2, word.unsqueeze(-1)).squeeze(-1)
        gather = parent.unsqueeze(-1).expand(B, beam, L)
        self.seq, self.lp, self.anc = self.seq.gather(1, gather), self.lp.gather(1, gather), self.anc.gather(1, gather)
        self.seq[:, :, t], self.lp[:, :, t] = word, chosen
        self.seq[:, :, t + 1:], self.lp[:, :, t + 1:] = self.pad, 0.0
        self.anc[:, :, t] = parent + torch.arange(B).unsqueeze(1) * beam
        self.anc[:, :, t + 1:] = torch.arange(B * beam).view(B, beam, 1)
        self.sum = new_sum.clone()
        for b in range(B):
            for v in range(beam):
                if int(word[b, v]) == self.eos or t == L - 1:
                    self.done[b].append({"seq": self.seq[b, v].clone(), "lp": self.lp[b, v].clone(),
                                         "p": self.pen(t + 1, float(self.sum[b, v]))})
                    self.sum[b, v] -= 1000
        return parent, word

    def finished(self):
        B, beam, L = self.B, self.beam, self.L
        seq = torch.full((B, beam, L), self.pad, dtype=torch.long)
        lp, p = torch.zeros(B, beam, L), torch.zeros(B, beam, dtype=torch.float64)
        count = torch.zeros(B, dtype=torch.long)
        for b in range(B):
            ranked = sorted(self.done[b], key=lambda d: -d["p"])[:beam]
            count[b] = len(ranked)
            for v, d in enumerate(ranked):
                seq[b, v], lp[b, v], p[b, v] = d["seq"], d["lp"], d["p"]
        return seq, lp, p, count


def _tie_logits(g, R, V, eos, t):
    """Logits quantised to 1/4 (so many columns share one score exactly), EOS made likely, a few -inf columns."""
    x = torch.round(torch.randn(R, V, generator=g) * 8) / 4
    x[:, eos] += 2.0 if t > 1 else -4.0
    x[:, 7 % V] = float("-inf")
    x[1::3, 11 % V] = float("-inf")
    return x


def _run_beam_step(K, B, beam, V, L, opt, seed, logits=None):
    from sparse_caption_b200.engine import BeamState, _parse_penalty
    eos, pad = 3, 0
    g = torch.Generator().manual_seed(seed)
    T = opt.get("temperature", 1.0)
    kind, alpha = _parse_penalty(opt.get("length_penalty", ""))
    st = BeamState(B, beam, L, torch.device(DEV))
    st.reset(2, pad)
    ref = _RefBeam(B, beam, L, eos, pad, opt.get("length_penalty", ""))
    for t in range(L):
        x = _tie_logits(g, B * beam, V, eos, t) if logits is None else logits[t]
        sup = None
        if opt.get("suppress") and t > 0:
            sup = torch.full((B * beam,), -1, dtype=torch.int32)
            sup[::2] = 5  # remove_bad_endings: token 5 may not follow on these rows
        pen_col = opt.get("penalized_col", -1)
        K.beam_step(x.to(DEV), st, t, B=B, beam=beam, V=V, L=L, eos=eos, pad=pad, temperature=T,
                    constraint=opt.get("decoding_constraint", 0), penalty_kind=kind, penalty_alpha=alpha,
                    suppress_tok=None if sup is None else sup.to(DEV), penalized_col=pen_col)
        stats = st.ws[: B * beam * 16].view(torch.float32).view(B * beam, 4).cpu()
        if t == 0:  # only row 0 of an image is expanded (and writes statistics) at the first step
            stats = stats.view(B, beam, 4)[:, :1].expand(B, beam, 4).reshape(B * beam, 4)
        parent, word = ref.step(x, stats, t, T, opt.get("decoding_constraint", 0), None if sup is None else sup.long(), pen_col)
        o = (t + 1) & 1
        assert torch.equal(st.tokens.cpu().long().view(B, beam), word), t
        assert torch.equal(st.anc[o].cpu().long()[:, t].view(B, beam), parent + torch.arange(B).unsqueeze(1) * beam), t
        assert torch.equal(st.anc[o].cpu().long().view(B, beam, L), ref.anc), t
        assert torch.equal(st.seq[o].cpu().long().view(B, beam, L), ref.seq), t
        assert torch.equal(st.lp[o].cpu().view(B, beam, L), ref.lp), t
        assert torch.equal(st.sum.cpu().view(B, beam), ref.sum), t
    seq, lp, p, count = ref.finished()
    assert torch.equal(st.done_count.cpu().long(), count)
    assert torch.equal(st.done_seq.cpu().long(), seq)
    assert torch.equal(st.done_lp.cpu(), lp)
    if kind == 1:  # (5 + len)^alpha in double: the device pow and Python's may differ in the last bit
        torch.testing.assert_close(st.done_p.cpu(), p, rtol=1e-14, atol=0)
    else:
        assert torch.equal(st.done_p.cpu(), p)


@pytest.mark.parametrize("beam", [9, 10, 16, 17, 31, 32])
@pytest.mark.parametrize("V", [35, 771, 10000, 10244])
def test_wide_beam_step_exact(K, beam, V):
    """Register path (V % 4 == 0, V <= 10240) and L2 path (V = 35, 10244): t = 0 with one live row per image, later steps,
    finished beams, exact ties and -inf columns; parents, words, sums, ancestors, finished lists and done_p bit for bit."""
    _run_beam_step(K, 3, beam, V, 6, {}, seed=beam * 100003 + V)


@pytest.mark.parametrize("V", [771, 10244])
@pytest.mark.parametrize("opt", [{"temperature": 0.7, "decoding_constraint": 1},
                                 {"length_penalty": "wu_0.5", "suppress": True, "penalized_col": 9},
                                 {"length_penalty": "avg_1", "temperature": 1.3, "penalized_col": 4}])
def test_wide_beam_step_options(K, V, opt):
    """Every row-pass option at beam 12 and 32: temperature, decoding constraint, length penalties, suppress_tok
    (remove_bad_endings) and penalized_col (suppress_UNK)."""
    for beam in (12, 32):
        _run_beam_step(K, 2, beam, V, 5, opt, seed=V + beam)


def test_wide_beam_step_random_logits(K):
    """Unquantised logits (no ties) over more steps: the same exact agreement."""
    g = torch.Generator().manual_seed(5)
    B, beam, V, L = 4, 20, 1000, 9
    logits = [torch.randn(B * beam, V, generator=g) * 2 for _ in range(L)]
    for t in range(L):
        logits[t][:, 3] += 2.5
    _run_beam_step(K, B, beam, V, L, {"length_penalty": "avg_1"}, seed=0, logits=logits)


def test_beam_above_32_is_refused(K):
    from sparse_caption_b200.engine import BeamState
    st = BeamState(1, 33, 4, torch.device(DEV)).reset(2, 0)
    with pytest.raises(RuntimeError, match="32"):
        K.beam_step(torch.zeros(33, 50, device=DEV), st, 0, B=1, beam=33, V=50, L=4, eos=3, pad=0)
    D, N, h = 128, 10, 2
    out = torch.zeros(33, D, device=DEV)
    with pytest.raises(RuntimeError, match="32"):
        K.cross_attn_step(torch.zeros(33, D, device=DEV), torch.zeros(N, D, device=DEV), torch.zeros(N, D, device=DEV), None, out,
                          B=1, beam=33, N=N, D=D, h=h, ldq=D, ldm=D, ldo=D)


# ------------------------------------------------------------------------------------------------------------------
# K6: the cross-attention step
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beam", [9, 12, 16, 17, 24, 32])
@pytest.mark.parametrize("dt,dk", [(torch.float32, 64), (torch.bfloat16, 64), (torch.bfloat16, 32), (torch.float32, 16)])
def test_wide_cross_attention(K, beam, dt, dk):
    """bf16 with d_k = 64 runs the mma kernel (two query m-tiles above 16 beams); the other shapes the generic kernel in
    8-row chunks over the once-staged K/V.  With and without att_mask, against fp32 softmax attention."""
    B, N, h = 3, 37, 4
    D, R = h * dk, B * beam
    g = torch.Generator().manual_seed(beam * 7 + dk)
    mem = torch.randn(B * N, 2 * D, generator=g).to(dt)
    qc = torch.randn(R, D, generator=g).to(dt)
    mask = torch.ones(B, N)
    mask[1, 20:] = 0
    md = mem.to(DEV)
    for m in (None, mask):
        out = torch.zeros(R, D, dtype=dt, device=DEV)
        K.cross_attn_step(qc.to(DEV), md[:, 0:], md[:, D:], None if m is None else m.to(DEV), out, B=B, beam=beam, N=N, D=D,
                          h=h, ldq=D, ldm=2 * D, ldo=D)
        kk = mem.float()[:, :D].view(B, N, h, dk).transpose(1, 2).repeat_interleave(beam, 0)
        vv = mem.float()[:, D:].view(B, N, h, dk).transpose(1, 2).repeat_interleave(beam, 0)
        m4 = None if m is None else m.view(B, 1, 1, N).repeat_interleave(beam, 0)
        ref = O.attention(qc.float().view(R, 1, h, dk).transpose(1, 2), kk, vv, m4).transpose(1, 2).reshape(R, D)
        assert rel_err(out.float(), ref) < (1e-5 if dt == torch.float32 else 2e-2)


# ------------------------------------------------------------------------------------------------------------------
# Engine and model surface, fp32, against the oracle
# ------------------------------------------------------------------------------------------------------------------
def _engine(sd, cfg_dict, **kw):
    from sparse_caption_b200.engine import ModelCfg, OrtEngine
    return OrtEngine(sd, ModelCfg(cfg_dict), **kw)


def _check_search(eng, z, opt, no_history=False):
    beam = opt["beam_size"]
    memory, src_mask = O.encode(z["w"], z["cfg"], z["att_feats"], z["boxes"], None)
    rseq, rlp, rp = O.beam_search(z["w"], z["cfg"], memory, src_mask, opt, no_history=no_history)
    enc = eng.encode(z["att_feats"], z["boxes"])
    for rep in range(2):  # the second call replays the captured graph
        seq, lp = eng.decode(enc, opt)
        assert tuple(seq.shape) == tuple(rseq.shape)
        assert torch.equal(seq.cpu().long(), rseq), (beam, rep)
        torch.testing.assert_close(lp.cpu(), rlp, rtol=1e-4, atol=2e-5)
        done_p = eng._get_dec_ws(enc.B, beam, enc.N, False, enc.slot).state.done_p.cpu().float()
        torch.testing.assert_close(done_p, rp, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("name", ["ort_tiny", "acort_tiny"])
@pytest.mark.parametrize("beam", [9, 10, 16, 32])
def test_engine_wide_beam_matches_oracle(name, beam):
    """OrtEngine.decode with graph capture and replay (ACORT: shared layers and key/value-shared attention, quirk Q2)."""
    z = golden_io.load(name)
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32", use_graphs=True)
    _check_search(eng, z, {"beam_size": beam})


def test_engine_wide_beam_no_history():
    z = golden_io.load("ort_tiny")
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32", no_history=True)
    _check_search(eng, z, {"beam_size": 10}, no_history=True)


@pytest.mark.parametrize("opt", [{"decoding_constraint": 1}, {"length_penalty": "wu_0.5"}, {"length_penalty": "avg_1"},
                                 {"temperature": 0.7}])
def test_engine_wide_beam_options(opt):
    z = golden_io.load("ort_tiny")
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32")
    _check_search(eng, z, dict(opt, beam_size=12))


def test_engine_wide_beam_bad_endings_and_unk():
    """remove_bad_endings and suppress_UNK at beam 12, against the oracle search with both rules restated."""
    z = golden_io.load("ort_tiny")
    V = z["cfg"].vocab_size
    bad = 5
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32")
    seq, _ = eng.sample(z["att_feats"], z["boxes"], None, {"beam_size": 12, "bad_endings_ix": [bad], "penalized_col": V - 1})
    memory, sm = O.encode(z["w"], z["cfg"], z["att_feats"], z["boxes"], None)
    ref = _oracle_beam_with_rules(z["w"], z["cfg"], memory, sm, 12, [bad], V - 1)
    assert torch.equal(seq.cpu().long(), ref)


def test_engine_wide_beam_pipeline_slots():
    """submit on pipeline slots at beam 16 gives the sequential result."""
    z = golden_io.load("ort_tiny")
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32")
    opt = {"beam_size": 16}
    want_seq, want_lp = (x.cpu() for x in eng.sample(z["att_feats"], z["boxes"], None, opt))
    B, L = want_seq.shape[0], want_seq.shape[-1]
    outs = [(torch.zeros(B, 16, L, dtype=torch.int32).pin_memory(), torch.zeros(B, 16, L).pin_memory()) for _ in range(2)]
    for i, out in enumerate(outs):
        eng.submit(z["att_feats"].pin_memory(), z["boxes"].pin_memory(), None, opt, slot=1 + i, out=out)
    eng.wait(host=True)
    for out in outs:
        assert torch.equal(out[0].long(), want_seq.long())
        torch.testing.assert_close(out[1], want_lp, rtol=1e-5, atol=1e-6)


def _model(name, z):
    import sparse_caption_b200.relation_transformer as R
    m = R.get_model(name)(z["cfg_dict"])
    m.load_state_dict(z["w"], strict=True)
    m = m.to(DEV).eval()
    m.precision = "fp32"
    return m


@pytest.mark.parametrize("name", ["ort_tiny", "acort_tiny"])
def test_model_sample_beam10(name):
    z = golden_io.load(name)
    m = _model("relation_transformer", z)
    seq, lp = m(att_feats=z["att_feats"].to(DEV), boxes=z["boxes"].to(DEV), opt={"beam_size": 10}, mode="sample")
    rseq, rlp = O.sample(z["w"], z["cfg"], z["att_feats"], z["boxes"], None, {"beam_size": 10})
    assert torch.equal(seq.cpu().long(), rseq)
    torch.testing.assert_close(lp.cpu(), rlp, rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("name", ["ort_tiny", "acort_tiny"])
def test_batch_beam_search_default_beam_10(name):
    """batch_beam_search(init_state, init_logprobs, memory, mask, opt={}): the reference's default of 10 beams."""
    import sparse_caption_b200.relation_transformer as R
    z = golden_io.load(name)
    m = _model("relation_transformer", z)
    c = m.cfg
    att, boxes = z["att_feats"].to(DEV), z["boxes"].to(DEV)
    B = att.shape[0]
    with torch.no_grad(), R._Precision("fp32"):
        feats, bx, _, att_masks, _ = m._prepare_feature(att, None, boxes)
        memory = m.model.encode(feats, bx, att_masks)
    it = torch.full((B,), c.bos_token_id, dtype=torch.long, device=DEV)
    logprobs, state = m.get_logprobs_state(it, memory, att_masks, None)
    mem_r, mask_r = torch.repeat_interleave(memory, 10, 0), torch.repeat_interleave(att_masks, 10, 0)
    done = m.batch_beam_search(state, logprobs, mem_r, mask_r, opt={})
    assert len(done) == B and all(len(d) == 10 for d in done)
    rseq, rlp = O.sample(z["w"], z["cfg"], z["att_feats"], z["boxes"], None, {"beam_size": 10})
    for b in range(B):
        for v in range(10):
            got = done[b][v]["seq"].cpu()
            n = got.numel()
            assert got.tolist() == rseq[b, v, :n].tolist() and bool((rseq[b, v, n:] == c.pad_token_id).all()), (name, b, v)
            torch.testing.assert_close(done[b][v]["logps"].cpu(), rlp[b, v, :n], rtol=1e-4, atol=2e-5)
        ps = [d["p"] for d in done[b]]
        assert ps == sorted(ps, reverse=True)


def test_model_beam_33_is_refused():
    z = golden_io.load("ort_tiny")
    m = _model("relation_transformer", z)
    with pytest.raises(RuntimeError, match="32"):
        m(att_feats=z["att_feats"].to(DEV), boxes=z["boxes"].to(DEV), opt={"beam_size": 33}, mode="sample")


def test_scst_step_beam10():
    """The SCST rollout at beam 10 through the trainer's engine: samples [B, 10, L] and a finite loss."""
    from tests.test_scst_gpu import _tiny
    z, tr, scorer = _tiny("supermask", "fp32")
    B, L = z["att_feats"].shape[0], tr.cfg.max_seq_length
    loss, mean_r, seq = tr.scst_step(z["att_feats"].to(DEV), z["boxes"].to(DEV), scorer=scorer, opt={"beam_size": 10}, lr=1e-4)
    assert tuple(seq.shape) == (B, 10, L)
    assert bool(torch.isfinite(loss).all()) and bool(torch.isfinite(mean_r).all())


# ------------------------------------------------------------------------------------------------------------------
# bf16 at configs[2] size (V = 10000, peaked weights, 64 images)
# ------------------------------------------------------------------------------------------------------------------
def _best_caption_tied(sd, opt, n=64):
    """The checks of _search_parity that apply at any beam width: the engine's best caption is the oracle's, or one that the
    oracle itself scores (with the search's length penalty) within twice the bf16 tolerance of its own best; the log-probs the
    engine reports along its best caption are the oracle's on those tokens within the bf16 tolerance; every image whose
    smallest decision gap in the oracle's search exceeds twice the tolerance keeps all beams identical.  (_search_parity's
    last check compares log-probs over images whose whole beam set is identical; at 32 beams no image keeps all 32 beams
    identical under bf16 rounding, so that check has nothing to compare there.)"""
    from tests.test_parity_baseline_gpu import TOL, _engine, _inputs, _oracle_forced, _valid_steps
    ocfg = O.Cfg(**ORT)
    pen = O.length_penalty(opt.get("length_penalty", ""))
    att, boxes = _inputs(n)
    margins = torch.full((n,), float("inf"))
    with torch.no_grad():
        memory, src_mask = O.encode(sd, ocfg, att, boxes, None)
        rseq, rlp, _ = O.beam_search(sd, ocfg, memory, src_mask, opt, margins=margins)
    eng = _engine(sd, ORT)
    seq, lp = eng.decode(eng.encode(att, boxes), opt)
    seq, lp = seq.long().cpu(), lp.float().cpu()
    best = seq[:, 0]
    with torch.no_grad():
        w = _oracle_forced(sd, ocfg, memory, src_mask, best)
    v_eng = _valid_steps(best, ocfg.eos_token_id, ocfg.pad_token_id)
    v_orc = _valid_steps(rseq[:, 0], ocfg.eos_token_id, ocfg.pad_token_id)
    chosen = w.gather(2, best.t().unsqueeze(-1)).squeeze(-1).t()  # [n, L]: oracle log-probs of the engine's tokens
    scale = max(1.0, float(((w.amax(-1) - w.amin(-1)) * 0.5).t()[v_eng].max()))
    lp_err = float((lp[:, 0] - chosen)[v_eng].abs().max())
    safe = margins > 2 * TOL
    all_same = (seq == rseq).all(-1).all(-1)
    s_eng = (chosen * v_eng).sum(-1)
    s_orc = (rlp[:, 0] * v_orc).sum(-1)
    p_eng = torch.tensor([pen(int(v_eng[i].sum()), float(s_eng[i])) for i in range(n)])
    p_orc = torch.tensor([pen(int(v_orc[i].sum()), float(s_orc[i])) for i in range(n)])
    same = (best == rseq[:, 0]).all(-1)
    tied = same | (p_orc - p_eng <= 2 * TOL)
    print(f"\n[configs[2] peaked weights, {opt}] best caption identical {float(same.float().mean()):.4f}, identical or tied "
          f"{float(tied.float().mean()):.4f}, mean caption length {float(v_orc.sum(-1).float().mean()):.1f}; best-caption "
          f"log-probs within {lp_err:.2e} of the oracle's (logit scale {scale:.2f}); images with min decision gap > {2 * TOL:g}: "
          f"{int(safe.sum())}/{n}")
    assert bool(tied.all()), (p_orc - p_eng)[~tied]
    assert lp_err <= TOL * scale, (lp_err, scale)
    assert bool(all_same[safe].all())


@pytest.mark.parametrize("beam", [10, 32])
def test_config2_bf16_wide_beam(beam):
    """Best caption identical or tied within the bf16 envelope on every image, graph replays bitwise deterministic, beams
    sorted by score."""
    sd = _weights(ORT, 0.95, peaked=True)
    if beam <= 10:
        _search_parity(ORT, sd, {"beam_size": beam}, f"configs[2] peaked weights, beam {beam}", floor_top=0.9, floor_all=0.0)
    _best_caption_tied(sd, {"beam_size": beam})
    _best_caption_tied(sd, {"beam_size": beam, "length_penalty": "avg_1"})
    from sparse_caption_b200.engine import ModelCfg, OrtEngine
    from tests.test_parity_baseline_gpu import _inputs
    eng = OrtEngine(sd, ModelCfg(ORT), precision="bf16", device=DEV)
    att, boxes = _inputs(64)
    enc = eng.encode(att, boxes)
    opt = {"beam_size": beam}
    s1, l1 = (x.clone() for x in eng.decode(enc, opt))
    s2, l2 = eng.decode(enc, opt)
    assert torch.equal(s1, s2) and torch.equal(l1, l2)
    p = eng._get_dec_ws(enc.B, beam, enc.N, False, enc.slot).state.done_p
    assert bool((p[:, :-1] >= p[:, 1:]).all())
