"""Kernel-level parity: every C-ABI entry point against the CPU oracle / plain torch fp32 on the same inputs.
GPU tier (`-m gpu`).  Tolerances: fp32 kernels 1e-5 relative (north_star), bf16 tensor path 2e-2;
integer / index / mask results bit-exact."""
import math

import pytest
import torch

from oracle import ort_oracle as O
from tests import golden_io

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def K():
    import sparse_caption_b200.kernels as k
    return k


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _mk(M, N, Kd, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, Kd, generator=g)
    w = torch.randn(N, Kd, generator=g) / math.sqrt(Kd)
    s = torch.randn(N, Kd, generator=g) * 2
    s.view(-1)[:4] = torch.tensor([0.0, 5e-8, 1e-7, -0.0])
    u = torch.rand(N, Kd, generator=g)
    b = torch.randn(N, generator=g)
    r = torch.randn(M, N, generator=g)
    return x, w, s, u, b, r


def _ref_linear(x, w, s, u, b, r, mode, relu):
    if mode == 1:
        w = w * O.binarize_logits(s)
    elif mode == 3:
        w = w * s
    elif mode == 4:
        w = w * O.bernoulli_from_uniform(s, u)
    y = torch.nn.functional.linear(x.double(), w.double(), b.double())
    if relu:
        y = torch.relu(y)
    return y + r.double()


@pytest.mark.parametrize("shape", [(7, 5, 8), (64, 64, 16), (130, 70, 96), (300, 771, 512), (50, 1, 64)])
@pytest.mark.parametrize("mode", [0, 1, 3, 4])
def test_linear_fp32(K, shape, mode):
    M, N, Kd = shape
    x, w, s, u, b, r = _mk(M, N, Kd)
    dev = "cuda"
    y = K.linear(x.to(dev), w.to(dev), b.to(dev), mask=s.to(dev), mask_mode=mode, uniforms=u.to(dev), residual=r.to(dev),
                 relu=True)
    assert rel_err(y, _ref_linear(x, w, s, u, b, r, mode, True)) < 1e-5


@pytest.mark.parametrize("tile_n", [64, 128, 256])
@pytest.mark.parametrize("shape", [(128, 128, 64), (128, 256, 512), (300, 200, 512), (1536, 512, 512), (1800, 2048, 512),
                                   (257, 1000, 2048), (100, 771, 512), (36, 64, 96)])
def test_linear_bf16_dense(K, shape, tile_n):
    """tcgen05 GEMM, bf16 operands via TMA.  Checked against a float64 product of the SAME bf16-rounded operands,
    so the tolerance only covers fp32 accumulation order (tight), not quantisation."""
    M, N, Kd = shape
    x, w, s, u, b, r = _mk(M, N, Kd, seed=1)
    xb, wb = x.bfloat16(), w.bfloat16()
    dev = "cuda"
    y = K.linear(xb.to(dev), wb.to(dev), b.to(dev), residual=r.to(dev), relu=False, tile_n=tile_n)
    ref = torch.nn.functional.linear(xb.double(), wb.double(), b.double()) + r.double()
    assert rel_err(y, ref) < 2e-5, shape
    yb = K.linear(xb.to(dev), wb.to(dev), b.to(dev), relu=True, out_dtype=torch.bfloat16, tile_n=tile_n)
    ref = torch.relu(torch.nn.functional.linear(xb.double(), wb.double(), b.double()))
    assert rel_err(yb.float(), ref) < 1e-2


@pytest.mark.parametrize("shape,tile_n", [((19000, 1024, 256), 0), ((19000, 1024, 256), 5128), ((40000, 512, 128), 64),
                                          ((5000, 2304, 192), 0)])
def test_linear_bf16_persistent(K, shape, tile_n):
    """More output tiles than resident CTAs: every CTA loops over several tiles with the double-buffered TMEM
    accumulator (epilogue of tile i overlapping the main loop of tile i+1)."""
    M, N, Kd = shape
    x, w, s, u, b, r = _mk(M, N, Kd, seed=5)
    xb, wb = x.bfloat16(), w.bfloat16()
    dev = "cuda"
    for rep in range(2):
        y = K.linear(xb.to(dev), wb.to(dev), b.to(dev), residual=r.to(dev), relu=False, tile_n=tile_n)
    ref = torch.nn.functional.linear(xb.float(), wb.float(), b) + r
    assert rel_err(y, ref) < 2e-5, shape


@pytest.mark.parametrize("shape", [(1536, 512, 512), (300, 1536, 512), (130, 96, 64)])
def test_linear_ln_fold(K, shape):
    """LayerNorm folded around the GEMM: a producer GEMM emits the fp32 residual stream, its bf16 copy and the chunk
    statistics; the consumer GEMM applies a*(x-mean)/(std+eps)+b through pre-scaled weights (transformer.py:329-358)."""
    M, N, D = shape
    g = torch.Generator().manual_seed(11)
    h = torch.randn(M, 256, generator=g)
    wp = torch.randn(D, 256, generator=g) / 16
    bp = torch.randn(D, generator=g)
    res = torch.randn(M, D, generator=g) * 2 + 0.5
    a2, b2 = torch.rand(D, generator=g) + 0.5, torch.randn(D, generator=g) * 0.1
    w = torch.randn(N, D, generator=g) / math.sqrt(D)
    bias = torch.randn(N, generator=g)
    dev = "cuda"
    x32 = torch.empty(M, D, device=dev)
    xb = torch.empty(M, D, device=dev, dtype=torch.bfloat16)
    stats = torch.zeros(M, D // 32, 2, device=dev)
    K.linear_ln(h.bfloat16().to(dev), wp.bfloat16().to(dev), bp.to(dev), residual=res.to(dev), out=x32, out_bf16=xb, stats_out=stats)
    x_ref = torch.nn.functional.linear(h.bfloat16().double(), wp.bfloat16().double(), bp.double()) + res.double()
    assert rel_err(x32, x_ref) < 2e-5
    assert torch.equal(xb.cpu(), x32.cpu().bfloat16())
    mean_ref = x_ref.mean(1)
    st = stats.double().cpu()
    assert rel_err(st[:, :, 0].sum(1) / D, mean_ref) < 1e-5
    # consumer
    wf = (w * a2).bfloat16()
    ln_c = wf.float().sum(1)
    bias_f = w @ b2 + bias
    y = torch.empty(M, N, device=dev)
    K.linear_ln(xb, wf.to(dev), bias_f.to(dev), out=y, ln_stats=stats, ln_c=ln_c.to(dev), relu=False)
    xn = a2.double() * (x_ref - mean_ref[:, None]) / (x_ref.std(1, keepdim=True) + 1e-6) + b2.double()
    y_ref = xn @ w.double().t() + bias.double()
    # operands are bf16 (x copy and scaled weights): bf16-level agreement with the fp64 LayerNorm + linear
    assert rel_err(y, y_ref) < 2e-2
    # exactness of the algebra: same quantised operands, float64 arithmetic
    xq = xb.cpu().double()
    rstd = 1.0 / (x_ref.std(1) + 1e-6)
    y_alg = rstd[:, None] * (xq @ wf.double().t()) - (rstd * mean_ref)[:, None] * ln_c.double() + bias_f.double()
    assert rel_err(y, y_alg) < 5e-5


@pytest.mark.parametrize("mode", [0, 1, 3, 4])
@pytest.mark.parametrize("shape", [(128, 128, 64), (300, 200, 512), (1536, 512, 2048), (100, 771, 512)])
def test_linear_bf16_masked_prologue(K, shape, mode):
    """fp32 master weights + fp32 mask logits, mask applied while building the UMMA operand tile."""
    M, N, Kd = shape
    x, w, s, u, b, r = _mk(M, N, Kd, seed=2)
    xb = x.bfloat16()
    dev = "cuda"
    y = K.linear(xb.to(dev), w.to(dev), b.to(dev), mask=s.to(dev), mask_mode=mode, uniforms=u.to(dev), residual=r.to(dev))
    if mode == 1:
        wm = w * O.binarize_logits(s)
    elif mode == 3:
        wm = w * s
    elif mode == 4:
        wm = w * O.bernoulli_from_uniform(s, u)
    else:
        wm = w
    ref = torch.nn.functional.linear(xb.double(), wm.bfloat16().double(), b.double()) + r.double()
    assert rel_err(y, ref) < 2e-5, (shape, mode)


def test_bernoulli_mask_consistency(K):
    """Philox masks: the tensor-core prologue, the fp32 kernel and sc_apply_mask regenerate the SAME mask from
    (seed, stream_id, element); the keep-rate matches sigmoid(S)."""
    M, N, Kd = 256, 384, 512
    x, w, s, u, b, r = _mk(M, N, Kd, seed=3)
    s = s * 0 + 1.0  # p = sigmoid(1) = 0.731
    dev = "cuda"
    wm = K.apply_mask(w.to(dev), s.to(dev), K.MASK_BERNOULLI, seed=1234, stream_id=7)
    keep = float((wm != 0).float().mean())
    assert abs(keep - 0.7311) < 0.01
    wm2 = K.apply_mask(w.to(dev), s.to(dev), K.MASK_BERNOULLI, seed=1234, stream_id=8)
    assert float(((wm != 0) != (wm2 != 0)).float().mean()) > 0.2  # different stream -> different mask
    y32 = K.linear(x.to(dev), w.to(dev), b.to(dev), mask=s.to(dev), mask_mode=K.MASK_BERNOULLI, seed=1234, stream_id=7)
    ref = torch.nn.functional.linear(x.double(), wm.cpu().double(), b.double())
    assert rel_err(y32, ref) < 1e-5
    xb = x.bfloat16()
    yb = K.linear(xb.to(dev), w.to(dev), b.to(dev), mask=s.to(dev), mask_mode=K.MASK_BERNOULLI, seed=1234, stream_id=7)
    ref = torch.nn.functional.linear(xb.double(), wm.cpu().bfloat16().double(), b.double())
    assert rel_err(yb, ref) < 2e-5


def test_binarize_bit_exact(K):
    z = golden_io.load("binarize")
    s = z["s"].cuda()
    m = K.apply_mask(torch.ones_like(s), s, K.MASK_ROUND)
    assert torch.equal(m.cpu(), z["m"])
    assert int(K.mask_count([s])) == int(z["m"].sum())
    big = torch.randn(1_000_003) * 3
    assert int(K.mask_count([big.cuda()])) == int(O.binarize_logits(big).sum())


@pytest.mark.parametrize("D", [64, 512, 2048])
def test_layernorm(K, D):
    g = torch.Generator().manual_seed(0)
    x = torch.randn(77, D, generator=g) * 3 + 1
    a, b = torch.randn(D, generator=g), torch.randn(D, generator=g)
    y = K.layernorm(x.cuda(), a.cuda(), b.cuda())
    assert rel_err(y, O.layer_norm(x.double(), a.double(), b.double())) < 1e-5
    yb = K.layernorm(x.cuda(), a.cuda(), b.cuda(), out_dtype=torch.bfloat16)
    assert rel_err(yb.float(), O.layer_norm(x, a, b)) < 1e-2


def test_embed_pe(K):
    g = torch.Generator().manual_seed(0)
    V, D, T, R = 50, 64, 7, 5
    table = torch.randn(V, D, generator=g)
    s = torch.randn(V, D, generator=g)
    pe = O.positional_encoding(D, 20)
    tok = torch.randint(0, V, (R, T), generator=g)
    out = K.embed_pe(tok.int().cuda().view(-1), table.cuda(), pe.cuda(), T=T, pos0=0, mask=s.cuda(), mask_mode=K.MASK_ROUND)
    ref = (table * O.binarize_logits(s))[tok] * math.sqrt(D) + pe[:T]
    assert rel_err(out.view(R, T, D), ref) < 1e-6
    out = K.embed_pe(tok[:, 0].int().cuda().contiguous(), table.cuda(), pe.cuda(), T=1, pos0=3)
    assert rel_err(out, table[tok[:, 0]] * math.sqrt(D) + pe[3]) < 1e-6


@pytest.mark.parametrize("cfg", [(2, 9, 4, 16), (3, 36, 8, 64), (2, 47, 8, 64), (1, 100, 8, 64)])
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_box_attention(K, cfg, dt):
    B, N, h, dk = cfg
    g = torch.Generator().manual_seed(5)
    D = h * dk
    data = O.synthetic_inputs(B, N, 8, seed=11)
    boxes = data["boxes"]
    mask = torch.ones(B, N)
    if N > 10:
        mask[0, N - 3:] = 0
        boxes[0, N - 3:] = 0
    qkv = (torch.randn(B * N, 3 * D, generator=g)).to(dt)
    wg_w = torch.randn(h, 64, generator=g) * 0.3
    wg_b = torch.randn(h, generator=g) * 0.3
    out = torch.zeros(B * N, D, dtype=dt, device="cuda")
    qkv_d = qkv.cuda()
    K.box_attention(qkv_d[:, 0:], qkv_d[:, D:], qkv_d[:, 2 * D:], boxes.cuda(), wg_w.cuda(), wg_b.cuda(), mask.cuda(), out,
                    B=B, N=N, h=h, dk=dk, ldq=3 * D, ldk=3 * D, ldv=3 * D, ldo=D)
    emb = O.box_relational_embedding(boxes)
    q, k, v = (qkv.float()[:, i * D:(i + 1) * D].view(B, N, h, dk).transpose(1, 2) for i in range(3))
    gw = torch.relu(torch.einsum("bijf,hf->bhij", emb, wg_w) + wg_b.view(1, h, 1, 1))
    scores = (q @ k.transpose(-2, -1)) / math.sqrt(dk)
    scores = scores.masked_fill(mask.view(B, 1, 1, N) == 0, -1e9)
    ref = torch.softmax(torch.log(torch.clamp(gw, min=1e-6)) + scores, -1) @ v
    ref = ref.transpose(1, 2).reshape(B * N, D)
    tol = 3e-4 if dt == torch.float32 else 2e-2  # fp32: logf/sincosf ulp differences are amplified by 100x angles (SURVEY Q-notes)
    assert rel_err(out.float(), ref) < tol


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_decode_attention_steps(K, dt):
    g = torch.Generator().manual_seed(9)
    B, beam, N, h, dk, L = 3, 3, 11, 4, 16, 6
    D, R = h * dk, B * beam
    dev = "cuda"
    ck = torch.zeros(L, R, D, dtype=dt, device=dev)
    cv = torch.zeros(L, R, D, dtype=dt, device=dev)
    hist_k, hist_v = [], []
    anc = torch.arange(R, dtype=torch.int32).unsqueeze(1).expand(R, L).contiguous()
    for t in range(4):
        qkv = torch.randn(R, 3 * D, generator=g).to(dt)
        if t > 0:  # shuffle beams inside each image like a beam step would
            perm = torch.cat([torch.randperm(beam, generator=g) + b * beam for b in range(B)])
            anc = anc[perm].clone()
            anc[:, t:] = torch.arange(R, dtype=torch.int32).unsqueeze(1)
            hist_k = [x[perm] for x in hist_k]
            hist_v = [x[perm] for x in hist_v]
        out = torch.zeros(R, D, dtype=dt, device=dev)
        qd = qkv.to(dev)
        K.self_attn_step(qd[:, 0:], qd[:, D:], qd[:, 2 * D:], ck, cv, anc.to(dev), out, R=R, D=D, h=h, n_prev=t, write_slot=t,
                         ldq=3 * D, ldk=3 * D, ldv=3 * D, ldo=D, anc_ld=L)
        q, k, v = (qkv.float()[:, i * D:(i + 1) * D] for i in range(3))
        hist_k.append(k)
        hist_v.append(v)
        kk = torch.stack(hist_k, 1).view(R, t + 1, h, dk).transpose(1, 2)
        vv = torch.stack(hist_v, 1).view(R, t + 1, h, dk).transpose(1, 2)
        ref = O.attention(q.view(R, 1, h, dk).transpose(1, 2), kk, vv, None).transpose(1, 2).reshape(R, D)
        assert rel_err(out.float(), ref) < (1e-5 if dt == torch.float32 else 2e-2), t
    # cross attention
    mem = torch.randn(B * N, 2 * D, generator=g).to(dt)
    qc = torch.randn(R, D, generator=g).to(dt)
    mask = torch.ones(B, N)
    mask[1, 7:] = 0
    out = torch.zeros(R, D, dtype=dt, device=dev)
    md = mem.to(dev)
    K.cross_attn_step(qc.to(dev), md[:, 0:], md[:, D:], mask.to(dev), out, B=B, beam=beam, N=N, D=D, h=h, ldq=D, ldm=2 * D, ldo=D)
    kk = mem.float()[:, :D].view(B, N, h, dk).transpose(1, 2).repeat_interleave(beam, 0)
    vv = mem.float()[:, D:].view(B, N, h, dk).transpose(1, 2).repeat_interleave(beam, 0)
    m4 = mask.view(B, 1, 1, N).repeat_interleave(beam, 0)
    ref = O.attention(qc.float().view(R, 1, h, dk).transpose(1, 2), kk, vv, m4).transpose(1, 2).reshape(R, D)
    assert rel_err(out.float(), ref) < (1e-5 if dt == torch.float32 else 2e-2)


@pytest.mark.parametrize("cfg", [(3, 36, 8, 2), (2, 47, 8, 3), (1, 100, 8, 1), (2, 17, 4, 2), (1, 128, 2, 1)])
@pytest.mark.parametrize("masked", [False, True])
def test_box_bias_all_and_tensor_attention(K, cfg, masked):
    """Inference split of K4: geometry bias of all layers in one pass (fp32, vs the oracle embedding), then the
    mma.sync attention of each layer (bf16, d_k = 64) vs plain fp32 softmax attention with that bias."""
    B, N, h, layers = cfg
    dk = 64
    g = torch.Generator().manual_seed(17)
    D = h * dk
    data = O.synthetic_inputs(B, N, 8, seed=13)
    boxes = data["boxes"]
    mask = torch.ones(B, N)
    if masked and N > 10:
        mask[0, N - 5:] = 0
        boxes[0, N - 5:] = 0
    wg_w = torch.randn(layers * h, 64, generator=g) * 0.3
    wg_b = torch.randn(layers * h, generator=g) * 0.3
    bias = torch.zeros(layers, B, h, N, N, device="cuda")
    K.box_bias_all(boxes.cuda(), wg_w.cuda(), wg_b.cuda(), bias, B=B, N=N, layers=layers, h=h)
    emb = O.box_relational_embedding(boxes)
    gw = torch.relu(torch.einsum("bijf,lhf->lbhij", emb, wg_w.view(layers, h, 64)) + wg_b.view(layers, 1, h, 1, 1))
    ref_bias = torch.log(torch.clamp(gw, min=1e-6))
    # relu/log amplify fp32 rounding of the 100x angles where WG.emb crosses 0: compare g = exp(bias) (SURVEY hard parts)
    assert float((bias.cpu().exp() - ref_bias.exp()).abs().max()) < 2e-4
    for l in range(layers):
        qkv = torch.randn(B * N, 3 * D, generator=g).bfloat16()
        out = torch.zeros(B * N, D, dtype=torch.bfloat16, device="cuda")
        qd = qkv.cuda()
        K.bias_attention(qd[:, 0:], qd[:, D:], qd[:, 2 * D:], bias[l], mask.cuda() if masked else None, out, B=B, N=N, h=h,
                         dk=dk, ldq=3 * D, ldk=3 * D, ldv=3 * D, ldo=D)
        q, k, v = (qkv.float()[:, i * D:(i + 1) * D].view(B, N, h, dk).transpose(1, 2) for i in range(3))
        scores = (q @ k.transpose(-2, -1)) / math.sqrt(dk)
        if masked:
            scores = scores.masked_fill(mask.view(B, 1, 1, N) == 0, -1e9)
        ref = torch.softmax(bias[l].cpu() + scores, -1) @ v
        ref = ref.transpose(1, 2).reshape(B * N, D)
        assert rel_err(out.float(), ref) < 2e-2, l


@pytest.mark.parametrize("cfg", [(3, 36, 8, 6), (2, 47, 8, 2), (1, 100, 8, 1), (2, 17, 4, 2), (5, 36, 8, 3)])
def test_box_bias_all_tensor_cores(K, cfg):
    """sc_box_bias_all_tc (mma.sync tiles over bf16 hi + lo operand splits, SFU sin / cos / log: the bf16 engine's encoder) vs the
    fp64 geometry weights of the oracle embedding: the attention multiplier g = exp(bias) within 2e-4 absolute - the bound the
    exact fp32 kernel is held to (the 100x angles amplify fp32 rounding where WG.emb crosses 0) - and bias within 2e-3 wherever
    g >= 1e-2; non-multiple-of-16 pair counts and ragged tiles covered by N = 47 / 17."""
    B, N, h, layers = cfg
    g = torch.Generator().manual_seed(23)
    boxes = O.synthetic_inputs(B, N, 8, seed=31)["boxes"]
    wg_w = torch.randn(layers * h, 64, generator=g) * 0.3
    wg_b = torch.randn(layers * h, generator=g) * 0.3
    bias = torch.full((layers, B, h, N, N), float("nan"), device="cuda")
    K.box_bias_all(boxes.cuda(), wg_w.cuda(), wg_b.cuda(), bias, B=B, N=N, layers=layers, h=h, tensor_cores=True)
    exact = torch.zeros_like(bias)
    K.box_bias_all(boxes.cuda(), wg_w.cuda(), wg_b.cuda(), exact, B=B, N=N, layers=layers, h=h)
    emb = O.box_relational_embedding(boxes).double()
    gw = torch.relu(torch.einsum("bijf,lhf->lbhij", emb, wg_w.double().view(layers, h, 64)) + wg_b.double().view(layers, 1, h, 1, 1))
    ref = torch.log(torch.clamp(gw, min=1e-6))
    got = bias.cpu().double()
    assert torch.isfinite(got).all()
    assert float((got.exp() - ref.exp()).abs().max()) < 2e-4
    big = gw >= 1e-2
    assert float((got - ref)[big].abs().max()) < 2e-3
    assert float((got.exp() - exact.cpu().double().exp()).abs().max()) < 2e-4


@pytest.mark.parametrize("cfg", [(5, 3, 36, 8), (3, 5, 47, 4), (2, 1, 100, 8), (4, 8, 7, 2)])
def test_cross_attention_tensor_path(K, cfg):
    """K6 on the mma.sync path (bf16, d_k = 64): the beam rows of an image share one read of its memory K/V."""
    B, beam, N, h = cfg
    dk = 64
    D, R = h * dk, B * beam
    g = torch.Generator().manual_seed(23)
    mem = torch.randn(B * N, 2 * D, generator=g).bfloat16()
    qc = torch.randn(R, D, generator=g).bfloat16()
    mask = torch.ones(B, N)
    mask[B - 1, N - 2:] = 0
    for m in (None, mask):
        out = torch.zeros(R, D, dtype=torch.bfloat16, device="cuda")
        md = mem.cuda()
        K.cross_attn_step(qc.cuda(), md[:, 0:], md[:, D:], None if m is None else m.cuda(), out, B=B, beam=beam, N=N, D=D, h=h,
                          ldq=D, ldm=2 * D, ldo=D)
        kk = mem.float()[:, :D].view(B, N, h, dk).transpose(1, 2).repeat_interleave(beam, 0)
        vv = mem.float()[:, D:].view(B, N, h, dk).transpose(1, 2).repeat_interleave(beam, 0)
        m4 = None if m is None else m.view(B, 1, 1, N).repeat_interleave(beam, 0)
        ref = O.attention(qc.float().view(R, 1, h, dk).transpose(1, 2), kk, vv, m4).transpose(1, 2).reshape(R, D)
        assert rel_err(out.float(), ref) < 2e-2


def test_cache_reorder(K):
    src = torch.randn(12, 4, 5, 8).cuda()
    idx = torch.tensor([3, 3, 0, 11, 7, 1, 2, 2, 2, 9, 10, 4], dtype=torch.int32).cuda()
    assert torch.equal(K.cache_reorder(src, idx), src[idx.long()])


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(1536, 512, 512, 0.95), (100, 771, 512, 0.99), (300, 512, 2048, 0.9), (20, 64, 96, 0.5)])
def test_csr_spmm(K, dt, shape):
    M, N, Kd, sp = shape
    x, w, s, u, b, r = _mk(M, N, Kd, seed=4)
    w = w * (torch.rand(N, Kd) >= sp)
    w[min(3, N - 1)] = 0  # an empty row
    dev = "cuda"
    csr = K.CsrWeight(w.to(dev), dt)
    y = K.csr_spmm(x.to(dt).to(dev), csr, b.to(dev), residual=r.to(dev), relu=True)
    ref = torch.relu(torch.nn.functional.linear(x.to(dt).double(), w.to(dt).double(), b.double())) + r.double()
    assert rel_err(y, ref) < 2e-5


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(1536, 512, 512, 0.95), (100, 771, 512, 0.99), (300, 512, 2048, 0.9), (20, 64, 96, 0.5),
                                   (1, 10000, 512, 0.95)])
def test_sell_spmm(K, dt, shape):
    """Sliced-ELL product (K3b'): ragged rows, an empty feature row, N not a multiple of the 32-feature slab, M not a
    multiple of the 8-row tile; fp32 accumulation of exactly representable operands -> 2e-5."""
    M, N, Kd, sp = shape
    x, w, s, u, b, r = _mk(M, N, Kd, seed=4)
    w = w * (torch.rand(N, Kd) >= sp)
    w[min(3, N - 1)] = 0  # an empty row
    dev = "cuda"
    sw = K.SellWeight(w.to(dt).float().to(dev), dt)
    assert sw.nnz == int((w.to(dt) != 0).sum())
    for out_dt in (torch.float32, torch.bfloat16):
        y = K.sell_spmm(x.to(dt).to(dev), sw, b.to(dev), residual=r.to(dev), relu=True, out_dtype=out_dt)
        ref = torch.relu(torch.nn.functional.linear(x.to(dt).double(), w.to(dt).double(), b.double())) + r.double()
        assert rel_err(y.float(), ref) < (2e-5 if out_dt == torch.float32 else 1e-2)
    y2 = K.sell_spmm(x.to(dt).to(dev), sw, None)
    assert rel_err(y2, torch.nn.functional.linear(x.to(dt).double(), w.to(dt).double())) < 2e-5


@pytest.mark.parametrize("shape", [(1536, 512, 512, 0.95), (100, 771, 512, 0.99), (300, 512, 2048, 0.9), (20, 64, 96, 0.5),
                                   (130, 10000, 512, 0.95), (2560, 2048, 512, 0.991), (257, 512, 1024, 0.8)])
def test_gspmm(K, shape):
    """Gather SpMM on the tensor cores (K3b''): ragged feature groups, an empty feature row, N not a multiple of 8, M not a
    multiple of the 128-row slab, K chunks (K > 512) with accumulators carried across them, x with a leading dimension > K;
    bf16 operands, fp32 accumulation -> 2e-5 against the fp64 product of the same bf16 values."""
    M, N, Kd, sp = shape
    x, w, s, u, b, r = _mk(M, N, Kd, seed=4)
    w = w * (torch.rand(N, Kd) >= sp)
    w[min(3, N - 1)] = 0  # an empty row
    dev = "cuda"
    dt = torch.bfloat16
    gw = K.GsWeight(w.to(dt).float().to(dev))
    assert gw.nnz == int((w.to(dt) != 0).sum()) and gw.padded % 16 == 0
    xb = x.to(dt).to(dev)
    ref0 = torch.nn.functional.linear(x.to(dt).double(), w.to(dt).double(), b.double())
    for out_dt in (torch.float32, torch.bfloat16):
        y = K.gspmm(xb, gw, b.to(dev), residual=r.to(dev), relu=True, out_dtype=out_dt)
        assert rel_err(y.float(), torch.relu(ref0) + r.double()) < (2e-5 if out_dt == torch.float32 else 1e-2)
    y2 = K.gspmm(xb, gw, None)
    assert rel_err(y2, torch.nn.functional.linear(x.to(dt).double(), w.to(dt).double())) < 2e-5
    # activations inside a wider buffer (the fused q|k|v projection output): leading dimension 2 * K
    wide = torch.zeros(M, 2 * Kd, device=dev, dtype=dt)
    wide[:, Kd:] = xb
    y3 = K.gspmm(wide[:, Kd:], gw, b.to(dev))
    assert rel_err(y3, ref0) < 2e-5
    # the COO tensors of state_dict_sparse pack to the same words
    gw2 = K.GsWeight(w.to(dt).float().to_sparse().to(dev))
    assert torch.equal(gw2.entries, gw.entries) and torch.equal(gw2.grp_ptr, gw.grp_ptr)


def _beam_ref(logits, B, beam, V, L, eos, opt):
    """Drive oracle.beam_select + the bookkeeping of oracle.beam_search on a fixed logits sequence."""
    pen = O.length_penalty(opt.get("length_penalty", ""))
    T = opt.get("temperature", 1.0)
    beam_seq = torch.zeros(B, beam, 0, dtype=torch.long)
    beam_lp = torch.zeros(B, beam, 0)
    beam_sum = torch.zeros(B, beam)
    done = [[] for _ in range(B)]
    for t in range(L):
        lp = torch.log_softmax(logits[t], -1)
        if t > 0:  # caption_model.py:218 (init_logprobs at t == 0 are used as returned by the model)
            lp = torch.log_softmax(lp / T, -1)
        if t == 0:
            lp = lp.view(B, beam, V)[:, 0]
        if opt.get("decoding_constraint", 0) and t > 0:
            lp = lp.clone()
            lp.scatter_(1, beam_seq[:, :, t - 1].reshape(-1, 1), float("-inf"))
        parent, word, new_sum = O.beam_select(lp, beam_sum, beam, first=(t == 0))
        nb = lp.size(0) // B
        chosen = lp.view(B, nb, V).gather(1, parent.unsqueeze(-1).expand(-1, -1, V)).gather(2, word.unsqueeze(-1)).squeeze(-1)
        if t > 0:
            beam_seq = beam_seq.gather(1, parent.unsqueeze(-1).expand_as(beam_seq))
            beam_lp = beam_lp.gather(1, parent.unsqueeze(-1).expand_as(beam_lp))
        beam_seq = torch.cat([beam_seq, word.unsqueeze(-1)], -1)
        beam_lp = torch.cat([beam_lp, chosen.unsqueeze(-1)], -1)
        beam_sum = new_sum.clone()
        for b in range(B):
            is_end = beam_seq[b, :, t] == eos
            if t == L - 1:
                is_end = torch.ones_like(is_end)
            for v in range(beam):
                if is_end[v]:
                    done[b].append({"seq": beam_seq[b, v].clone(), "lp": beam_lp[b, v].clone(), "p": pen(t + 1, float(beam_sum[b, v]))})
            beam_sum[b, is_end] -= 1000
    seq = torch.zeros(B, beam, L, dtype=torch.long)
    slp = torch.zeros(B, beam, L)
    for b in range(B):
        for v, d in enumerate(sorted(done[b], key=lambda d: -d["p"])[:beam]):
            seq[b, v, : d["seq"].numel()] = d["seq"]
            slp[b, v, : d["lp"].numel()] = d["lp"]
    return seq, slp


@pytest.mark.parametrize("beam,V", [(3, 10000), (5, 771), (2, 37), (8, 300)])
@pytest.mark.parametrize("opt", [{}, {"decoding_constraint": 1, "length_penalty": "wu_0.7"}, {"temperature": 0.8, "length_penalty": "avg_0"}])
def test_beam_step(K, beam, V, opt):
    """K7 against the oracle's beam bookkeeping on a fixed sequence of logits (EOS made likely so beams finish)."""
    from sparse_caption_b200.engine import BeamState, _parse_penalty
    B, L, eos = 7, 9, 3
    g = torch.Generator().manual_seed(beam * 1000 + V)
    logits = [torch.randn(B * beam, V, generator=g) * 2 for _ in range(L)]
    for t in range(L):
        logits[t][:, eos] += 2.5
        logits[t][::2, 5] = logits[t][::2, 6]  # exact ties inside a row
    ref_seq, ref_lp = _beam_ref(logits, B, beam, V, L, eos, opt)
    st = BeamState(B, beam, L, torch.device("cuda"))
    st.reset(2, 0)
    kind, alpha = _parse_penalty(opt.get("length_penalty", ""))
    for t in range(L):
        K.beam_step(logits[t].cuda(), st, t, B=B, beam=beam, V=V, L=L, eos=eos, pad=0, temperature=opt.get("temperature", 1.0),
                    constraint=opt.get("decoding_constraint", 0), penalty_kind=kind, penalty_alpha=alpha)
    assert torch.equal(st.done_seq.cpu().long(), ref_seq)
    torch.testing.assert_close(st.done_lp.cpu(), ref_lp, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("cand", [5, 3])
@pytest.mark.parametrize("shape", [(1536, 10000, 512), (77, 771, 512), (300, 256, 64), (5, 1000, 128)])
def test_linear_topk_records(K, shape, cand):
    """Generator GEMM with the fused row pass: merged records == log-sum-exp and top-5 of the materialised logits."""
    M, N, Kd = shape
    g = torch.Generator().manual_seed(21)
    x = torch.randn(M, Kd, generator=g).bfloat16().cuda()
    w = (torch.randn(N, Kd, generator=g) * 0.2).bfloat16().cuda()
    b = torch.randn(N, generator=g).cuda()
    logits = K.linear(x, w, b)  # fp32 logits from the same tensor-core kernel
    P = K.linear_topk_parts(N)
    part = torch.full((M, P, 12), float("nan"), device="cuda")
    K.linear_topk(x, w, b, part, candidates=cand)
    torch.cuda.synchronize()
    assert not torch.isnan(part[:, :, :7]).any()  # (the column slots hold int bits; an empty slot is 0x7fffffff)
    m, s = part[:, :, 0], part[:, :, 1]
    Mx = m.max(1).values
    lse = Mx + torch.log((s * torch.exp(m - Mx[:, None])).sum(1))
    torch.testing.assert_close(lse, torch.logsumexp(logits, 1), rtol=1e-5, atol=1e-5)
    vals = part[:, :, 2:7].reshape(M, -1)
    idx = part[:, :, 7:12].contiguous().view(torch.int32).reshape(M, -1)
    k = min(cand, N)
    top = vals.topk(k, 1)
    ref = logits.topk(k, 1)
    assert torch.equal(top.values, ref.values)  # same accumulator values, only the selection differs
    got_idx = idx.gather(1, top.indices)
    # ties between equal logits may be listed in either order by torch.topk: compare through the values they point at
    assert torch.equal(logits.gather(1, got_idx.long()), ref.values)
    assert int(got_idx.min()) >= 0 and int(got_idx.max()) < N


def test_beam_step_partials_matches_beam_step(K):
    """sc_linear_topk + sc_beam_step_partials == sc_linear + sc_beam_step over several steps (same tokens, parents,
    finished beams; log-probs within fp32 summation-order noise)."""
    from sparse_caption_b200.engine import BeamState
    g = torch.Generator().manual_seed(22)
    B, beam, V, L, Kd = 9, 3, 1000, 6, 128
    R = B * beam
    w = (torch.randn(V, Kd, generator=g) * 0.3).bfloat16().cuda()
    b = torch.randn(V, generator=g).cuda()
    b[3] += 2.0  # EOS shows up among the candidates
    sa, sb = BeamState(B, beam, L, "cuda"), BeamState(B, beam, L, "cuda")
    sa.reset(2, 0); sb.reset(2, 0)
    part = torch.empty(R, K.linear_topk_parts(V), 12, device="cuda")
    for t in range(L):
        x = torch.randn(R, Kd, generator=g).bfloat16().cuda()
        if t == 0:
            x = x.view(B, beam, Kd)[:, :1].expand(B, beam, Kd).reshape(R, Kd).contiguous()
        logits = K.linear(x, w, b)
        K.beam_step(logits, sa, t, B=B, beam=beam, V=V, L=L, eos=3, pad=0, penalty_kind=1, penalty_alpha=0.7)
        K.linear_topk(x, w, b, part, candidates=beam)
        K.beam_step_partials(part, sb, t, B=B, beam=beam, V=V, L=L, eos=3, pad=0, penalty_kind=1, penalty_alpha=0.7)
        o = (t + 1) & 1
        assert torch.equal(sa.tokens, sb.tokens), t
        assert torch.equal(sa.seq[o], sb.seq[o]) and torch.equal(sa.anc[o], sb.anc[o]), t
        torch.testing.assert_close(sa.lp[o], sb.lp[o], rtol=1e-5, atol=2e-5)
        torch.testing.assert_close(sa.sum, sb.sum, rtol=1e-5, atol=1e-4)
    assert torch.equal(sa.done_seq, sb.done_seq) and torch.equal(sa.done_count, sb.done_count)
    torch.testing.assert_close(sa.done_lp, sb.done_lp, rtol=1e-5, atol=2e-5)


@pytest.mark.parametrize("temperature,constraint", [(1.0, 0), (0.7, 1)])
def test_sample_step_inverse_cdf(K, temperature, constraint):
    """Multinomial step with injected uniforms == inverse CDF of exp(log_softmax(x) / T) in index order (what
    torch.multinomial samples from, models/transformer.py:531-538); stored log-prob = un-tempered log_softmax entry."""
    from sparse_caption_b200.engine import GreedyState
    g = torch.Generator().manual_seed(31)
    R, V, L, t = 700, 1000, 6, 2
    logits = (torch.randn(R, V, generator=g) * 2).cuda()
    u = torch.rand(R, generator=g).cuda()
    st = GreedyState(R, L, "cuda")
    st.reset(2, 0)
    prevtok = torch.randint(0, V, (R,), generator=g).int().cuda()
    st.seq[:, t - 1] = prevtok
    st.live[t - 1] = R
    K.sample_step(logits, st, t, R=R, V=V, L=L, eos=3, constraint=constraint, temperature=temperature, uniforms=u)
    lp = torch.log_softmax(logits.double(), 1)
    w = torch.exp(lp / temperature)
    if constraint:
        w.scatter_(1, prevtok.long().unsqueeze(1), 0.0)
    cdf = torch.cumsum(w, 1)
    ref = torch.searchsorted(cdf, (u.double() * cdf[:, -1]).unsqueeze(1), right=True).squeeze(1).clamp_max(V - 1)
    got = st.tokens.long()
    # fp32 vs fp64 prefix sums may disagree when u lands within rounding of a CDF step
    assert float((got == ref).float().mean()) > 0.995
    same = got == ref
    torch.testing.assert_close(st.lp[:, t][same], lp.gather(1, got.unsqueeze(1)).squeeze(1).float()[same], rtol=1e-5, atol=1e-5)
    if constraint:
        assert bool((got != prevtok.long()).all())
    assert torch.equal(st.seq[:, t].long(), got) and int(st.live[t]) == int((got != 3).sum())


def test_sample_step_distribution(K):
    """Philox-driven sampling reproduces the categorical distribution (20 000 rows sharing one logits row) and is
    deterministic for a given seed."""
    from sparse_caption_b200.engine import GreedyState
    g = torch.Generator().manual_seed(32)
    R, V, L = 20000, 40, 4
    row = torch.randn(V, generator=g) * 1.5
    logits = row.unsqueeze(0).expand(R, V).contiguous().cuda()
    outs = []
    for seed in (7, 7, 8):
        st = GreedyState(R, L, "cuda")
        st.reset(2, 0)
        K.sample_step(logits, st, 0, R=R, V=V, L=L, eos=3, seed=seed)
        outs.append(st.tokens.clone())
    assert torch.equal(outs[0], outs[1]) and not torch.equal(outs[0], outs[2])
    freq = torch.bincount(outs[0].long().cpu(), minlength=V).double() / R
    p = torch.softmax(row.double(), 0)
    assert float((freq - p).abs().max()) < 4 * float(torch.sqrt(p.max() * (1 - p.max()) / R)) + 2e-3


def test_ingest_pinned_host_features(K):
    """Fused ingest: the kernel reads pinned host fp32 over PCIe and writes bf16 - bit-identical to copy + cast."""
    g = torch.Generator().manual_seed(51)
    x = (torch.randn(37, 36, 2048, generator=g) * 3).pin_memory()
    out = torch.zeros(x.numel(), device="cuda", dtype=torch.bfloat16)
    K.ingest_f32_bf16(x, out, ctas=8)
    assert torch.equal(out, x.cuda().bfloat16().view(-1))


def test_new_entry_points_report_library_errors(K):
    """Error behaviour of the entry points added this round: negative status -> RuntimeError with the library's message,
    nothing launched."""
    from sparse_caption_b200.engine import BeamState
    x = torch.randn(16, 36, device="cuda").bfloat16()          # K = 36 is not a multiple of 8
    w = torch.randn(40, 36) * (torch.rand(40, 36) > 0.5)
    sw = K.SellWeight(w.cuda(), torch.bfloat16)
    with pytest.raises(RuntimeError, match="sc_sell_spmm"):
        K.sell_spmm(x, sw, None)
    xb = torch.randn(8, 64, device="cuda").bfloat16()
    wb = torch.randn(300, 64, device="cuda").bfloat16()
    part = torch.empty(8, K.linear_topk_parts(300), 12, device="cuda")
    with pytest.raises(RuntimeError, match="candidates"):
        K.linear_topk(xb, wb, None, part, candidates=9)
    st = BeamState(2, 7, 4, "cuda")
    st.reset(2, 0)
    with pytest.raises(RuntimeError, match="beam=7"):
        K.beam_step_partials(torch.empty(14, 4, 12, device="cuda"), st, 0, B=2, beam=7, V=300, L=4, eos=3, pad=0)
    with pytest.raises(RuntimeError, match="sc_ingest_f32_bf16"):
        K.lib.call("sc_ingest_f32_bf16", torch.randn(16, device="cuda").data_ptr(), torch.empty(16, device="cuda", dtype=torch.bfloat16),
                   16, 0)                                       # a raw device address is not pinned host memory


def test_pointer_arguments_are_checked_before_the_launch(K):
    """lib.call refuses, in Python and before anything is enqueued, a CUDA or pageable tensor for the pinned host pointer of
    sc_ingest_f32_bf16, a CPU tensor for a device pointer and a non-contiguous tensor; the launch count does not move."""
    out = torch.empty(16, device="cuda", dtype=torch.bfloat16)
    before = K.lib.launch_count
    with pytest.raises(RuntimeError, match="^sc_ingest_f32_bf16: pinned_host must be a pinned CPU tensor, got a CUDA tensor"):
        K.ingest_f32_bf16(torch.randn(16, device="cuda"), out)
    with pytest.raises(RuntimeError, match="^sc_ingest_f32_bf16: pinned_host must be a pinned CPU tensor, got a pageable CPU tensor"):
        K.ingest_f32_bf16(torch.randn(16), out)
    with pytest.raises(RuntimeError, match="^sc_ingest_f32_bf16: y must be a CUDA tensor, got a cpu tensor"):
        K.ingest_f32_bf16(torch.randn(16).pin_memory(), out.cpu())
    with pytest.raises(RuntimeError, match="^sc_cast_f32_bf16: x must be contiguous"):
        K.cast_bf16(torch.randn(8, 2, device="cuda").t())
    assert K.lib.launch_count == before


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_tensor_on_another_device_is_refused(K):
    x = torch.randn(16, device="cuda:1")
    with torch.cuda.device(0):
        with pytest.raises(RuntimeError, match=r"^sc_cast_f32_bf16: x is on cuda:1, not on the current device cuda:0"):
            K.cast_bf16(x, out=torch.empty(16, device="cuda:0", dtype=torch.bfloat16))
        with pytest.raises(RuntimeError, match=r"^sc_apply_mask_batched: descs\[0\]\.w is on cuda:1"):
            K.mask_descriptors([(x.view(4, 4), None, None, None, None, 0)], "cuda:0")


@pytest.mark.parametrize("mode", ["0", "1", "3"])
def test_cluster_gemm_variants(mode):
    """SC_GEMM_MULTICAST (read once per process, hence the subprocess): 0 = no clusters, 1 = 2-CTA clusters with a multicast B
    tile, 3 = CTA pairs (tcgen05.mma.cta_group::2, the default for >= 64 M blocks) forced for every size.  Same results as
    torch for an even and an odd number of M blocks, fp32 and bf16 (staged, coalesced stores) outputs, and a 72-block problem
    that takes the pair path by default."""
    import os
    import subprocess
    import sys
    code = r"""
import torch, sys
sys.path.insert(0, %r)
import sparse_caption_b200.kernels as K
for (M, N, Kd) in ((1536, 1000, 512), (1400, 520, 136), (9216, 1024, 512)):   # 12 / 11 (phantom block in the last pair) / 72 M blocks
    g = torch.Generator().manual_seed(M)
    x = torch.randn(M, Kd, generator=g).bfloat16().cuda(); w = (torch.randn(N, Kd, generator=g) * 0.1).bfloat16().cuda(); b = torch.randn(N, generator=g).cuda()
    ref = x.float() @ w.float().t() + b
    out = torch.full((M, N), 7.0, device="cuda")
    K.linear(x, w, b, out=out, tile_n=3256)
    err = float((out - ref).abs().max() / ref.abs().max())
    assert err < 1e-5, (M, N, Kd, err)
    out16 = torch.full((M, N), 7.0, device="cuda", dtype=torch.bfloat16)
    K.linear(x, w, b, out=out16, tile_n=3256, relu=True)
    assert torch.equal(out16, torch.relu(out).bfloat16()), (M, N, Kd, "bf16")
print("variants ok")
""" % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SC_GEMM_MULTICAST=mode)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "variants ok" in r.stdout, r.stdout + r.stderr
