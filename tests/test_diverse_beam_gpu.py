"""Diverse beam search (group_size > 1) on the device: the diverse beam-step kernels against the CPU restatement
(tests/diverse_oracle.py) on scripted logits, the records path against the materialised-logits path, the engine's
staggered group schedule (graphs off / on, pipeline slot 1), the model surface, and full-size bf16 properties.  GPU tier."""
import pytest
import torch

from oracle import ort_oracle as O
from tests import diverse_oracle as D
from tests import golden_io

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def K():
    from sparse_caption_b200 import kernels, lib
    lib.load()
    return kernels


def _engine(sd, cfg_dict, **kw):
    from sparse_caption_b200.engine import ModelCfg, OrtEngine
    return OrtEngine(sd, ModelCfg(cfg_dict), **kw)


def _states(B, G, bdash, L):
    from sparse_caption_b200.engine import BeamState
    hist = torch.zeros(G, 2, B * bdash, L, dtype=torch.int32, device=DEV)
    sts = []
    for g in range(G):
        st = BeamState(B, bdash, L, torch.device(DEV))
        st.seq = [hist[g, 0], hist[g, 1]]
        st.reset(2, 0)
        sts.append(st)
    return hist, sts


def _schedule(G, L):
    """(group, local step) in the order of caption_model.py:151-153."""
    return [(g, t - g) for t in range(L + G - 1) for g in range(G) if 0 <= t - g <= L - 1]


@pytest.mark.parametrize("V,bdash,G", [(10000, 3, 2), (12000, 2, 3), (771, 1, 3)])
@pytest.mark.parametrize("lam", [0.5, 3.0])
@pytest.mark.parametrize("opt", [{}, {"decoding_constraint": 1, "length_penalty": "wu_0.7"},
                                 {"temperature": 0.8, "suppress": True, "penalized_col": 7}])
def test_diverse_beam_step_matches_oracle(K, V, bdash, G, lam, opt):
    """sc_beam_step_diverse over the staggered schedule on scripted logits (register path V = 10000, L2 path V = 12000 and
    V = 771) == the restated bookkeeping: tokens exact, log-probs within 1e-5.  EOS made likely; the two bad endings 8 and 9
    are the rows' leading columns and are exactly tied in every other row, so ties between candidates (penalised or not)
    decide beams."""
    from sparse_caption_b200.engine import _parse_penalty, _suppress_bad
    B, L, eos = 5, 7, 3
    R = B * bdash
    T = opt.get("temperature", 1.0)
    pen_col = opt.get("penalized_col", -1)
    bad = [8, 9] if opt.get("suppress") else None
    gen = torch.Generator().manual_seed(V + 10 * bdash + G)
    logits = [[torch.randn(R, V, generator=gen) * 2 for _ in range(L)] for _ in range(G)]
    for g in range(G):
        for t in range(L):
            x = logits[g][t]
            x[:, eos] += 2.0
            x[:, [8, 9]] += 2.5    # bad endings show up, token 0 is attractive after them
            x[:, 0] += 2.0
            x[::2, 9] = x[::2, 8]  # exact ties inside a row, on columns that win
        logits[g][0] = logits[0][0]  # every group starts from the same BOS-step row

    def lp_of(x, t):
        lp = torch.log_softmax(x, -1)
        if t > 0:
            lp = torch.log_softmax(lp / T, -1)
        return lp

    def advance(g, state_ix, it, tau):
        return lp_of(logits[g][tau + 1], tau + 1) if tau + 1 < L else torch.zeros(R, V)

    init = lp_of(logits[0][0], 0).view(B, bdash, V)[:, 0]
    ropt = dict(opt, beam_size=G * bdash, group_size=G, diversity_lambda=lam, bad_endings_ix=bad)
    rseq, rlp, rp, _ = D.diverse_beam_core(init, advance, B, V, L, eos, 0, ropt)
    hist, sts = _states(B, G, bdash, L)
    kind, alpha = _parse_penalty(opt.get("length_penalty", ""))
    bad_d = torch.tensor(bad, dtype=torch.int32, device=DEV) if bad else None
    for g, tau in _schedule(G, L):
        st = sts[g]
        K.beam_step(logits[g][tau].to(DEV), st, tau, B=B, beam=bdash, V=V, L=L, eos=eos, pad=0, temperature=T,
                    constraint=opt.get("decoding_constraint", 0), penalty_kind=kind, penalty_alpha=alpha,
                    suppress_tok=_suppress_bad(st, bad_d, tau), penalized_col=pen_col, diverse=(hist, g, lam))
    seq = torch.cat([st.done_seq for st in sts], 1).cpu().long()
    lp = torch.cat([st.done_lp for st in sts], 1).cpu()
    p = torch.cat([st.done_p for st in sts], 1).cpu().float()
    assert torch.equal(seq, rseq)
    torch.testing.assert_close(lp, rlp, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(p, rp, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("G,bdash", [(3, 1), (2, 2), (5, 1)])
def test_diverse_partials_match_diverse_beam_step(K, G, bdash):
    """sc_linear_topk (candidates = the whole beam size) + sc_beam_step_partials_diverse == sc_linear + sc_beam_step_diverse
    over the staggered schedule (same tokens, parents, finished beams; log-probs within fp32 summation-order noise)."""
    gen = torch.Generator().manual_seed(23)
    B, V, L, Kd = 9, 1000, 6, 128
    R = B * bdash
    w = (torch.randn(V, Kd, generator=gen) * 0.3).bfloat16().cuda()
    b = torch.randn(V, generator=gen).cuda()
    b[3] += 2.0
    ha, sa = _states(B, G, bdash, L)
    hb, sb = _states(B, G, bdash, L)
    part = torch.empty(R, K.linear_topk_parts(V), 12, device=DEV)
    x0 = torch.randn(B, 1, Kd, generator=gen).expand(B, bdash, Kd).reshape(R, Kd).bfloat16().cuda()
    for g, tau in _schedule(G, L):
        x = x0 if tau == 0 else torch.randn(R, Kd, generator=gen).bfloat16().cuda()
        logits = K.linear(x, w, b)
        K.beam_step(logits, sa[g], tau, B=B, beam=bdash, V=V, L=L, eos=3, pad=0, penalty_kind=1, penalty_alpha=0.7,
                    diverse=(ha, g, 0.5))
        K.linear_topk(x, w, b, part, candidates=G * bdash)
        K.beam_step_partials(part, sb[g], tau, B=B, beam=bdash, V=V, L=L, eos=3, pad=0, penalty_kind=1, penalty_alpha=0.7,
                             diverse=(hb, g, 0.5))
        o = (tau + 1) & 1
        assert torch.equal(sa[g].tokens, sb[g].tokens), (g, tau)
        assert torch.equal(sa[g].seq[o], sb[g].seq[o]) and torch.equal(sa[g].anc[o], sb[g].anc[o]), (g, tau)
        torch.testing.assert_close(sa[g].lp[o], sb[g].lp[o], rtol=1e-5, atol=2e-5)
        torch.testing.assert_close(sa[g].sum, sb[g].sum, rtol=1e-5, atol=1e-4)
    for g in range(G):
        assert torch.equal(sa[g].done_seq, sb[g].done_seq) and torch.equal(sa[g].done_count, sb[g].done_count)
        torch.testing.assert_close(sa[g].done_lp, sb[g].done_lp, rtol=1e-5, atol=2e-5)


def test_diverse_entry_points_reject_bad_arguments(K):
    hist, sts = _states(2, 2, 3, 4)
    logits = torch.zeros(6, 100, device=DEV)
    with pytest.raises(RuntimeError, match="sc_beam_step_diverse"):
        K.lib.call("sc_beam_step_diverse", K.lib.ptr(logits), 2, 3, 100, 4, 0, 3, 0, 1.0, 0, 0, 0.0, None, -1, None, 1, 0.5,
                   *([K.lib.ptr(logits)] * 12), K.lib.ptr(sts[0].ws), sts[0].ws.numel(), K.lib.stream())
    part = torch.zeros(6, K.linear_topk_parts(100), 12, device=DEV)
    with pytest.raises(RuntimeError, match="sc_beam_step_partials_diverse"):
        K.beam_step_partials(part, sts[1], 0, B=2, beam=3, V=100, L=4, eos=3, pad=0, diverse=(hist, 1, 0.5))


_GOLDEN_OPTS = (("beam3", {"beam_size": 6, "group_size": 2}), ("beam2", {"beam_size": 6, "group_size": 3}),
                ("beam3c", {"beam_size": 6, "group_size": 2, "decoding_constraint": 1, "length_penalty": "wu_0.5"}))


@pytest.mark.parametrize("name", ["ort_tiny", "ort_tiny_masks", "acort_tiny"])
@pytest.mark.parametrize("graphs", [False, True])
def test_engine_fp32_goldens_and_oracle(name, graphs):
    """fp32 engine, two calls each (the second replays the graph): lambda = 0 reproduces the reference goldens group by
    group; lambda 0.5 / 2.0 are token-exact against the restated search; the same through submit() on pipeline slot 1."""
    z = golden_io.load(name)
    am = z.get("att_masks")
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32", use_graphs=graphs)
    memory, src_mask = O.encode(z["w"], z["cfg"], z["att_feats"], z["boxes"], am)
    for key, opt in _GOLDEN_OPTS:
        G = opt["group_size"]
        bdash = 6 // G
        for lam in (0.0, 0.5, 2.0):
            o = dict(opt, diversity_lambda=lam)
            if lam == 0.0:
                want = z[key + "_seq"].repeat(1, G, 1), z[key + "_lp"].repeat(1, G, 1)
            else:
                want = D.diverse_beam_search(z["w"], z["cfg"], memory, src_mask, o)[:2]
            for rep in range(2):
                seq, lp = eng.sample(z["att_feats"], z["boxes"], am, o)
                assert tuple(seq.shape) == (z["att_feats"].shape[0], G * bdash, z["cfg"].max_seq_length)
                assert torch.equal(seq.cpu(), want[0]), (name, key, lam, rep)
                torch.testing.assert_close(lp.cpu(), want[1], rtol=1e-4, atol=2e-5)
            if am is None and lam == 0.5:
                seq, lp = eng.submit(z["att_feats"].pin_memory(), z["boxes"].pin_memory(), None, o, slot=1)
                eng.wait(1)
                assert torch.equal(seq.cpu().long(), want[0]), (name, key, "slot 1")
                torch.testing.assert_close(lp.cpu(), want[1], rtol=1e-4, atol=2e-5)


def test_engine_group_size_ignored_by_greedy_and_checked():
    z = golden_io.load("ort_tiny")
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32")
    seq, lp = eng.sample(z["att_feats"], z["boxes"], None, {"beam_size": 1, "group_size": 3})
    assert torch.equal(seq.cpu(), z["greedy_seq"])                       # greedy decoding never reads group_size
    with pytest.raises(ValueError, match="group_size"):
        eng.sample(z["att_feats"], z["boxes"], None, {"beam_size": 2, "group_size": 3})
    with pytest.raises(ValueError, match="group_size"):
        eng.sample(z["att_feats"], z["boxes"], None, {"beam_size": 18, "group_size": 2})


def test_engine_no_history_and_dec_ctas():
    """Quirk Q1 (no self-attention history) and the sized decode grids (dec_ctas) under the diverse schedule."""
    z = golden_io.load("acort_tiny")
    opt = {"beam_size": 6, "group_size": 3, "diversity_lambda": 0.5}
    memory, src_mask = O.encode(z["w"], z["cfg"], z["att_feats"], z["boxes"], None)
    want = D.diverse_beam_search(z["w"], z["cfg"], memory, src_mask, opt, no_history=True)
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32", no_history=True)
    seq, lp = eng.sample(z["att_feats"], z["boxes"], None, opt)
    assert torch.equal(seq.cpu(), want[0])
    torch.testing.assert_close(lp.cpu(), want[1], rtol=1e-4, atol=2e-5)
    want = D.diverse_beam_search(z["w"], z["cfg"], memory, src_mask, opt)
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32", dec_ctas=(2, 1))
    seq, lp = eng.sample(z["att_feats"], z["boxes"], None, opt)
    assert torch.equal(seq.cpu(), want[0])
    torch.testing.assert_close(lp.cpu(), want[1], rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("cls", ["relation_transformer", "relation_transformer_prune"])
def test_model_surface(cls):
    """mode="sample" and the step-wise batch_beam_search with group_size 3: the graphed engine's result, the restated
    search's, and the done_beams structure (groups in order, each best first by p)."""
    import sparse_caption_b200.relation_transformer as R
    for name in ("ort_tiny", "acort_tiny"):
        z = golden_io.load(name)
        cfg = dict(z["cfg_dict"], prune_type="supermask") if cls.endswith("prune") else z["cfg_dict"]
        m = R.get_model(cls)(cfg)
        sd = m.state_dict()
        for k in sd:
            if k.endswith("_pruning_mask"):
                sd[k] = torch.full_like(sd[k], 10.0)   # every mask bit on: the weights of the dense fixture
            elif k in z["w"]:
                sd[k] = z["w"][k]
        m.load_state_dict(sd, strict=True)
        m = m.to(DEV).eval()
        m.precision = "fp32"
        opt = {"beam_size": 6, "group_size": 3, "diversity_lambda": 0.5}
        att, boxes = z["att_feats"].to(DEV), z["boxes"].to(DEV)
        seq, lp = m(att, boxes, opt=opt, mode="sample")
        memory, src_mask = O.encode(z["w"], z["cfg"], z["att_feats"], z["boxes"], None)
        want_seq, want_lp, want_p = D.diverse_beam_search(z["w"], z["cfg"], memory, src_mask, opt)
        B = att.shape[0]
        assert tuple(seq.shape) == (B, 6, z["cfg"].max_seq_length)
        assert torch.equal(seq.cpu(), want_seq), (cls, name)
        torch.testing.assert_close(lp.cpu(), want_lp, rtol=1e-4, atol=2e-5)
        with torch.no_grad(), R._Precision("fp32"):
            feats, bx, _, att_masks, _ = m._prepare_feature(att, None, boxes)
            mem = m.model.encode(feats, bx, att_masks)
        it = torch.full((B,), m.cfg.bos_token_id, dtype=torch.long, device=DEV)
        logprobs, state = m.get_logprobs_state(it, mem, att_masks, None)
        mem_r, mask_r = torch.repeat_interleave(mem, 6, 0), torch.repeat_interleave(att_masks, 6, 0)
        done = m.batch_beam_search(state, logprobs, mem_r, mask_r, opt=opt)
        assert len(done) == B and all(len(d) == 6 for d in done)
        for b in range(B):
            for v in range(6):
                n = int((want_seq[b, v] != 0).sum())
                assert done[b][v]["seq"].cpu().tolist() == want_seq[b, v, :n].tolist(), (cls, name, b, v)
                torch.testing.assert_close(done[b][v]["logps"].cpu(), want_lp[b, v, :n], rtol=1e-4, atol=2e-5)
                assert done[b][v]["p"] == pytest.approx(float(want_p[b, v]), rel=1e-4, abs=1e-4)
                assert done[b][v]["unaug_p"] == pytest.approx(float(want_lp[b, v, :n].sum()), rel=1e-4, abs=1e-4)
            for g in range(3):
                ps = [d["p"] for d in done[b][2 * g:2 * g + 2]]
                assert ps == sorted(ps, reverse=True)


def test_full_size_bf16_properties():
    """configs[2] (ORT 6x512, V=10000, 95 % sparse) at 512 images, beam 3 / group_size 3: deterministic replays, the fused
    records path against fuse_topk=False, and a permutation of the images permutes the captions."""
    import bench
    from sparse_caption_b200 import synthetic
    from sparse_caption_b200.engine import ModelCfg
    cfg = ModelCfg(bench.CFG)
    sd = synthetic.random_state_dict(cfg, seed=1234, sparsity=bench.SPARSITY, device="cuda")
    att, boxes = synthetic.synthetic_inputs(512, 36, 2048, seed=8888)
    opt = {"beam_size": 3, "group_size": 3, "diversity_lambda": 0.5}
    eng = _engine(sd, bench.CFG, precision="bf16")
    seq, lp = eng.sample(att, boxes, None, opt)
    seq2, lp2 = eng.sample(att, boxes, None, opt)
    assert torch.equal(seq, seq2) and torch.equal(lp, lp2)
    assert tuple(seq.shape) == (512, 3, 16) and torch.isfinite(lp).all() and bool((lp <= 0).all())
    ref = _engine(sd, bench.CFG, precision="bf16", fuse_topk=False)
    rseq, rlp = ref.sample(att, boxes, None, opt)
    same = (seq == rseq).all(-1).all(-1).float().mean()
    assert float(same) >= 0.99, float(same)
    perm = torch.randperm(512, generator=torch.Generator().manual_seed(0))
    pseq, _ = eng.sample(att[perm], boxes[perm], None, opt)
    same_p = (pseq == seq[perm.cuda()]).all(-1).all(-1).float().mean()
    assert float(same_p) >= 0.995, float(same_p)


@pytest.mark.parametrize("graphs", [False, True])
def test_engine_bad_endings_and_unk(graphs):
    """remove_bad_endings (the id tensor the workspace holds, read by every graph replay) and suppress_UNK under the diverse
    schedule against the restated search: two calls, a call with other ids (new graph), then the first ids again."""
    z = golden_io.load("ort_tiny")
    V = z["cfg"].vocab_size
    memory, src_mask = O.encode(z["w"], z["cfg"], z["att_feats"], z["boxes"], None)
    eng = _engine(z["w"], z["cfg_dict"], precision="fp32", use_graphs=graphs)
    toks = sorted({int(t) for t in z["beam3_seq"][:, :, 0].reshape(-1)} - {0, 3})
    opts = [{"beam_size": 6, "group_size": 3, "diversity_lambda": 0.5, "bad_endings_ix": toks, "penalized_col": V - 1},
            {"beam_size": 6, "group_size": 3, "diversity_lambda": 0.5, "bad_endings_ix": toks[:1] + [V - 2], "penalized_col": V - 1}]
    wants = [D.diverse_beam_search(z["w"], z["cfg"], memory, src_mask, o)[:2] for o in opts]
    for i in (0, 0, 1, 0):
        seq, lp = eng.sample(z["att_feats"], z["boxes"], None, opts[i])
        torch.empty(1 << 22, device=DEV).fill_(7.0)   # reuse any freed allocation before the next replay
        assert torch.equal(seq.cpu(), wants[i][0]), i
        torch.testing.assert_close(lp.cpu(), wants[i][1], rtol=1e-4, atol=2e-5)


def _diverse_parity(cfg_dict, sd, opt, name, n=64):
    """bf16 engine vs the restated search on an n-image slice, per (image, group), tie-adjusted as
    tests/test_parity_baseline_gpu._search_parity does for group_size 1:
      * bit-exact given equal scores: where no decision of group g or of the groups before it (whose tokens set g's
        penalties) had a score gap within twice the bf16 tolerance, group g's beams must equal the oracle's;
      * identical-or-tied best caption >= 0.99: identical; or a caption the oracle itself scores (unaugmented,
        teacher-forced) within twice the tolerance of the oracle group's best one; or a group whose decisions (its own or
        an earlier group's) include such a near-tie - the search went another way at a tie, like a greedy flip (with
        bdash = 1 a group is a beam-1 search and cannot come back either)."""
    from tests.test_parity_baseline_gpu import TOL, _inputs, _oracle_forced, _valid_steps
    from tests.test_parity_baseline_gpu import _engine as _bf16_engine
    ocfg = O.Cfg(**cfg_dict)
    att, boxes = _inputs(n)
    G, bdash, _ = D.diverse_groups(opt)
    margins = torch.full((n, G), float("inf"))
    with torch.no_grad():
        memory, src_mask = O.encode(sd, ocfg, att, boxes, None)
        rseq, rlp, _ = D.diverse_beam_search(sd, ocfg, memory, src_mask, opt, margins=margins)
    eng = _bf16_engine(sd, cfg_dict)
    seq, _ = eng.decode(eng.encode(att, boxes), opt)
    seq = seq.long().cpu()
    eos, pad = ocfg.eos_token_id, ocfg.pad_token_id
    heads = [g * bdash for g in range(G)]
    top_same = torch.stack([(seq[:, h] == rseq[:, h]).all(-1) for h in heads], 1)                           # [n, G]
    group_same = torch.stack([(seq[:, h:h + bdash] == rseq[:, h:h + bdash]).all(-1).all(-1) for h in heads], 1)
    s_eng, s_orc = torch.zeros(n, G), torch.zeros(n, G)
    with torch.no_grad():
        for gi, h in enumerate(heads):
            w2 = _oracle_forced(sd, ocfg, memory, src_mask, seq[:, h])
            s_eng[:, gi] = (w2.gather(2, seq[:, h].t().unsqueeze(-1)).squeeze(-1).t() * _valid_steps(seq[:, h], eos, pad)).sum(-1)
            s_orc[:, gi] = (rlp[:, h] * _valid_steps(rseq[:, h], eos, pad)).sum(-1)
    near_tie = torch.cummin(margins, 1).values <= 2 * TOL        # a near-tie in group g or before it
    score_tie = (s_orc - s_eng) <= 2 * TOL
    tie_ok = top_same | score_tie | near_tie
    deficit = (s_orc - s_eng)[~top_same]
    print(f"\n[{name}] images {n} {opt}: per-(image, group) identical-or-tied best caption {float(tie_ok.float().mean()):.4f} "
          f"(identical {float(top_same.float().mean()):.4f}, + within the oracle-score tolerance "
          f"{float((top_same | score_tie).float().mean()):.4f}); whole group identical {float(group_same.float().mean()):.4f}; "
          f"(image, group) pairs without a near-tie up to their group: {int((~near_tie).sum())}/{n * G} (of those whole group "
          f"identical: {int((group_same & ~near_tie).sum())}); differing best captions {int((~top_same).sum())}, of those on a "
          f"near-tie {int((~top_same & near_tie).sum())}; oracle-score deficit max "
          f"{float(deficit.max()) if deficit.numel() else 0.0:.3g} nats; median smallest gap {float(margins.median()):.3g}")
    assert bool(group_same[~near_tie].all()), torch.nonzero(~group_same & ~near_tie)[:4]
    assert float(tie_ok.float().mean()) >= 0.99, float(tie_ok.float().mean())


def test_bf16_config2_peaked_against_oracle():
    """configs[2] (ORT 6x512, V = 10000, 95 % sparse) with peaked weights, beam 3 / group_size 3: the fused records path."""
    from tests.test_parity_baseline_gpu import ORT, _weights
    _diverse_parity(ORT, _weights(ORT, 0.95, peaked=True), {"beam_size": 3, "group_size": 3, "diversity_lambda": 0.5},
                    "configs[2] peaked weights, diverse")


def test_bf16_config3_acort_peaked_against_oracle():
    """configs[3] (ACORT shared layers, V = 771, L = 26, 99.1 % sparse) with peaked weights, beam 6 / group_size 2: the
    materialised-logits path and the L2 row pass, shared-layer cache slots at each group's local step."""
    from tests.test_parity_baseline_gpu import ACORT, _weights
    _diverse_parity(ACORT, _weights(ACORT, 0.991, peaked=True), {"beam_size": 6, "group_size": 2, "diversity_lambda": 0.5},
                    "configs[3] ACORT peaked weights, diverse")
