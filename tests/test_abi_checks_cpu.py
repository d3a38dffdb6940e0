"""CPU tier: lib.call checks every pointer argument against the header before the library is reached.  Every kernel wrapper
called with CPU tensors raises a RuntimeError naming its entry point and the refused parameter (the loaded functions are
replaced by ones that fail if called); with the device check satisfied by a stand-in, contiguity, row-strided views, raw
addresses, NULL and the appended stream are checked on the arguments the library would receive."""
import inspect
import os

import pytest
import torch

from sparse_caption_b200 import kernels as K, lib
from sparse_caption_b200.engine import BeamState, GreedyState


@pytest.fixture
def so(monkeypatch):
    """The loaded library with every entry point that enqueues work (its last parameter is the stream) replaced by a function
    that fails the test if it is reached; the host-side queries stay."""
    if not os.path.exists(lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    so = lib.load()

    def reached(*a):
        raise AssertionError("the library was reached")
    for name, (_, stream) in lib._params.items():
        if stream:
            monkeypatch.setattr(so, name, reached)
    return so


def _f(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype)


def _i(*shape):
    return torch.zeros(*shape, dtype=torch.int32)


def _b(*shape):
    return torch.zeros(*shape, dtype=torch.bfloat16)


_BEAM = dict(B=1, beam=2, V=8, L=4, eos=3, pad=0)
_ATT = dict(ldq=64, ldk=64, ldv=64, ldo=64)
_BWD = dict(G=1, Tq=2, Tk=2, h=1, dk=64, ldq=64, ldk=64, ldv=64, ldd=64, ldgq=64, ldgk=64, ldgv=64)
_ADAM = dict(lr=1e-3, betas=(0.9, 0.98), eps=1e-9, weight_decay=0.0, clip=0.1, grad_scale=1.0, step=1)

# wrapper -> (call with CPU tensors, entry point, first pointer parameter of the header that the call fills with a tensor)
CASES = {
    "linear": (lambda: K.linear(_b(2, 8), _b(4, 8)), "sc_linear", "x"),
    "linear_ln": (lambda: K.linear_ln(_b(2, 8), _b(4, 8), out=_f(2, 4)), "sc_linear_ln", "x"),
    "csr_spmm": (lambda: K.csr_spmm(_f(2, 8), K.CsrWeight(torch.eye(4, 8), torch.float32)), "sc_csr_spmm", "x"),
    "sell_spmm": (lambda: K.sell_spmm(_f(2, 8), K.SellWeight(torch.eye(4, 8), torch.float32)), "sc_sell_spmm", "x"),
    "gspmm": (lambda: K.gspmm(_b(2, 8), K.GsWeight(torch.eye(4, 8))), "sc_gspmm", "x"),
    "ingest_f32_bf16": (lambda: K.ingest_f32_bf16(_f(8), _b(8)), "sc_ingest_f32_bf16", "pinned_host"),
    "layernorm": (lambda: K.layernorm(_f(2, 8), _f(8), _f(8)), "sc_layernorm", "x"),
    "embed_pe": (lambda: K.embed_pe(_i(2), _f(8, 4), _f(4, 4)), "sc_embed_pe", "tokens"),
    "embed_pe_stats": (lambda: K.embed_pe_stats(_i(2), _f(8, 32), _f(4, 32), _f(2, 32), _b(2, 32), _f(2, 1, 2)), "sc_embed_pe_stats",
                       "tokens"),
    "apply_mask": (lambda: K.apply_mask(_f(4, 8), _f(4, 8), K.MASK_ROUND), "sc_apply_mask", "w"),
    "mask_count": (lambda: K.mask_count([_f(4, 8)]), "sc_mask_count", "logits"),
    "cast_bf16": (lambda: K.cast_bf16(_f(4, 8)), "sc_cast_f32_bf16", "x"),
    "mask_rows": (lambda: K.mask_rows(_f(4, 8), _f(4)), "sc_mask_rows", "x"),
    "box_attention": (lambda: K.box_attention(_f(2, 64), _f(2, 64), _f(2, 64), _f(1, 2, 4), _f(1, 64), _f(1), None, _f(2, 64),
                                              B=1, N=2, h=1, dk=64, **_ATT), "sc_box_attention_fwd", "q"),
    "box_bias_all": (lambda: K.box_bias_all(_f(1, 4, 4), _f(8, 64), _f(8), _f(1, 1, 8, 4, 4), B=1, N=4, layers=1, h=8),
                     "sc_box_bias_all", "boxes"),
    "box_bias_all_tc": (lambda: K.box_bias_all(_f(1, 4, 4), _f(8, 64), _f(8), _f(1, 1, 8, 4, 4), B=1, N=4, layers=1, h=8,
                                               tensor_cores=True), "sc_box_bias_all_tc", "boxes"),
    "bias_attention": (lambda: K.bias_attention(_b(2, 64), _b(2, 64), _b(2, 64), _f(1, 1, 2, 2), None, _b(2, 64), B=1, N=2, h=1,
                                                dk=64, **_ATT), "sc_bias_attention_fwd", "q"),
    "self_attn_step": (lambda: K.self_attn_step(_f(2, 64), _f(2, 64), _f(2, 64), _f(4, 2, 64), _f(4, 2, 64), _i(2, 4), _f(2, 64),
                                                R=2, D=64, h=1, n_prev=0, write_slot=0, anc_ld=4, **_ATT),
                       "sc_decode_self_attn_step", "q"),
    "cross_attn_step": (lambda: K.cross_attn_step(_f(2, 64), _f(2, 64), _f(2, 64), None, _f(2, 64), B=1, beam=2, N=2, D=64, h=1,
                                                  ldq=64, ldm=64, ldo=64), "sc_decode_cross_attn_step", "q"),
    "beam_step": (lambda: K.beam_step(_f(2, 8), BeamState(1, 2, 4, "cpu"), 0, **_BEAM), "sc_beam_step", "logits"),
    "beam_step_diverse": (lambda: K.beam_step(_f(2, 8), BeamState(1, 2, 4, "cpu"), 0, diverse=(_i(2, 2, 2, 4), 1, 0.5), **_BEAM),
                          "sc_beam_step_diverse", "logits"),
    "linear_hmask": (lambda: K.linear_hmask(_b(2, 8), _b(4, 8), _b(2, 4), _b(2, 4)), "sc_linear_hmask", "x"),
    "linear_topk": (lambda: K.linear_topk(_b(2, 8), _b(4, 8), None, _f(2, K.linear_topk_parts(4), 12)), "sc_linear_topk", "x"),
    "beam_step_partials": (lambda: K.beam_step_partials(_f(2, 2, 12), BeamState(1, 2, 4, "cpu"), 0, **_BEAM),
                           "sc_beam_step_partials", "partials"),
    "beam_step_partials_diverse": (lambda: K.beam_step_partials(_f(2, 2, 12), BeamState(1, 2, 4, "cpu"), 0,
                                                                diverse=(_i(2, 2, 2, 4), 1, 0.5), **_BEAM),
                                   "sc_beam_step_partials_diverse", "partials"),
    "greedy_step": (lambda: K.greedy_step(_f(2, 8), GreedyState(2, 4, "cpu"), 0, R=2, V=8, L=4, eos=3), "sc_greedy_step", "logits"),
    "sample_step": (lambda: K.sample_step(_f(2, 8), GreedyState(2, 4, "cpu"), 0, R=2, V=8, L=4, eos=3), "sc_sample_step", "logits"),
    "cache_reorder": (lambda: K.cache_reorder(_f(4, 8), _i(4)), "sc_cache_reorder", "src"),
    "linear_dropout": (lambda: K.linear_dropout(_f(2, 8), _f(4, 8), p=0.1), "sc_linear_dropout", "x"),
    "linear_wgrad": (lambda: K.linear_wgrad(_f(4, 8), _f(8, 8), _f(4, 8), None, K.MASK_NONE, _f(4, 8), None, M=8), "sc_linear_wgrad",
                     "dyT"),
    "linear_wgrad_rowmajor": (lambda: K.linear_wgrad_rowmajor(_b(2, 4), _b(2, 8), _f(4, 8), None, K.MASK_NONE, _f(4, 8), None,
                                                              workspace=_f(32)), "sc_linear_wgrad_rowmajor", "dy"),
    "prep_grad": (lambda: K.prep_grad(_f(2, 8), out=_b(2, 8)), "sc_prep_grad", "g"),
    "transpose": (lambda: K.transpose(_f(2, 8), _f(8, 2)), "sc_transpose", "x"),
    "apply_mask_transposed": (lambda: K.apply_mask_transposed(_f(4, 8), _f(4, 8), K.MASK_ROUND, _b(8, 4)), "sc_apply_mask_transposed",
                              "w"),
    "mask_descriptors": (lambda: K.mask_descriptors([(_f(4, 8), _f(4, 8), None, _b(4, 8), None, 0)], "cpu"), "sc_apply_mask_batched",
                         r"descs\[0\]\.w"),
    "apply_mask_batched": (lambda: K.apply_mask_batched(torch.zeros(1, 10, dtype=torch.int64), 1, K.MASK_ROUND),
                           "sc_apply_mask_batched", "descs"),
    "mask_grad": (lambda: K.mask_grad(_f(4, 8), _f(4, 8), _f(4, 8), K.MASK_ROUND, _f(4, 8), _f(4, 8)), "sc_mask_grad", "dwm"),
    "colsum": (lambda: K.colsum(_f(2, 8), _f(8)), "sc_colsum", "x"),
    "layernorm_bwd": (lambda: K.layernorm_bwd(_f(2, 8), _f(8), _f(2, 8), _f(2, 8), _f(8), _f(8)), "sc_layernorm_bwd", "x"),
    "layernorm_bwd_fused": (lambda: K.layernorm_bwd(_f(2, 8), _f(8), _f(2, 8), _f(2, 8), _f(8), _f(8), next_gb=_b(2, 8)),
                            "sc_layernorm_bwd_fused", "x"),
    "logsoftmax_nll": (lambda: K.logsoftmax_nll(_f(2, 8), logprobs=_f(2, 8)), "sc_logsoftmax_nll", "logits"),
    "scst_targets": (lambda: K.scst_targets(_i(2, 4), _f(2, dtype=torch.float64), None, S=2, cider_weight=1.0, bos=2, pad=0,
                                            tokens=_i(8), targets=_i(8), tok_w=_f(8), key_valid=_f(8), inv_norm=_f(1)),
                     "sc_scst_targets", "seq"),
    "embedding_bwd": (lambda: K.embedding_bwd(_i(2), _f(2, 8), _f(4, 8), 1.0), "sc_embedding_bwd", "tokens"),
    "adam_clip": (lambda: K.adam_clip(_f(8), _f(8), _f(8), _f(8), **_ADAM), "sc_adam_clip", "param"),
    "adam_clip_st": (lambda: K.adam_clip_st(torch.zeros(1, 5, dtype=torch.int64), 1, _f(8), _f(8), _f(8), _f(8), _f(8), _f(8), _f(8),
                                            uniforms=None, mask_mode=K.MASK_ROUND, bypass=False, update_logits=True, seed=0,
                                            stream_base=0, mask_lr=1e-2, mask_eps=1e-8, **_ADAM), "sc_adam_clip_st", "descs"),
    "prune_stats": (lambda: K.prune_stats(torch.zeros(1, 6, dtype=torch.int64), 1, _f(8)), "sc_prune_stats", "descs"),
    "prune_select": (lambda: K.prune_select(torch.zeros(1, 6, dtype=torch.int64), 1, [2], K.PRUNE_ABS, _f(8), _f(8)),
                     "sc_prune_select", "descs"),
    "sparsity_coeff": (lambda: K.sparsity_coeff(torch.zeros(1, dtype=torch.int64), 8, 0.5, 1.0, _f(3)), "sc_sparsity_coeff", "count"),
    "attention_fwd": (lambda: K.attention_fwd(_f(2, 64), _f(2, 64), _f(2, 64), _f(2, 64), _f(1, 2, 2), G=1, Tq=2, Tk=2, h=1, dk=64,
                                              **_ATT), "sc_attention_fwd", "q"),
    "attention_bwd": (lambda: K.attention_bwd(_f(2, 64), _f(2, 64), _f(2, 64), _f(1, 2, 2), _f(2, 64), _f(2, 64), _f(2, 64), _f(2, 64),
                                              dtype=torch.float32, **_BWD), "sc_attention_bwd", "q"),
    "attention_bwd_bf16out": (lambda: K.attention_bwd_bf16out(_b(2, 64), _b(2, 64), _b(2, 64), _f(1, 2, 2), _f(2, 64), _b(2, 64),
                                                              _b(2, 64), _b(2, 64), **_BWD), "sc_attention_bwd_bf16out", "q"),
    "box_bias_fwd": (lambda: K.box_bias_fwd(_f(1, 2, 4), _f(1, 64), _f(1), _f(1, 1, 2, 2), B=1, N=2, h=1), "sc_box_bias_fwd", "boxes"),
    "box_bias_bwd": (lambda: K.box_bias_bwd(_f(1, 2, 4), _f(1, 1, 2, 2), _f(1, 1, 2, 2), _f(1, 64), _f(1), B=1, N=2, h=1),
                     "sc_box_bias_bwd", "boxes"),
    "box_embedding": (lambda: K.box_embedding(_f(1, 2, 4)), "sc_box_embedding", "boxes"),
    "log_clamp": (lambda: K.log_clamp(_f(8)), "sc_log_clamp", "x"),
    "logsoftmax_bwd": (lambda: K.logsoftmax_bwd(_f(2, 8), _f(2, 8)), "sc_logsoftmax_bwd", "logprobs"),
}


def test_every_launching_wrapper_is_covered():
    launching = {name for name, f in vars(K).items() if inspect.isfunction(f) and f.__module__ == K.__name__
                 and not name.startswith("_") and ("lib.call(" in inspect.getsource(f) or "lib.address(" in inspect.getsource(f))}
    covered = {name.replace("_diverse", "").replace("_fused", "").replace("_tc", "") for name in CASES}
    assert launching == covered


@pytest.mark.parametrize("case", sorted(CASES))
def test_cpu_tensors_are_refused_before_the_library(so, case):
    run, entry, param = CASES[case]
    with pytest.raises(RuntimeError, match=rf"^{entry}: {param} must be a CUDA tensor, got a cpu tensor: .*no CPU fallback"
                       if entry != "sc_ingest_f32_bf16" else rf"^{entry}: {param} must be a pinned CPU tensor"):
        run()


@pytest.fixture
def fake_device(so, monkeypatch):
    """Every tensor counts as a CUDA tensor on device 0 (= the current device) and the current stream is 0x5eed; the library
    functions record the arguments they receive."""
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda t: True))
    monkeypatch.setattr(torch.Tensor, "get_device", lambda t: 0)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    monkeypatch.setattr(lib, "_current", lambda: (0, 0x5eed))
    calls = []

    def recorder(name):
        return lambda *a: calls.append((name, a)) or 0
    for name, (_, stream) in lib._params.items():
        if stream:
            monkeypatch.setattr(so, name, recorder(name))
    return calls


def test_non_contiguous_tensor_is_refused(fake_device):
    x = _f(8, 2).t()
    with pytest.raises(RuntimeError, match=r"^sc_layernorm: x must be contiguous"):
        K.layernorm(x, _f(8), _f(8))
    with pytest.raises(RuntimeError, match=r"^sc_cast_f32_bf16: y must be contiguous"):
        K.cast_bf16(_f(8), out=_b(4, 4).t())
    with pytest.raises(RuntimeError, match=r"^sc_apply_mask_batched: descs\[0\]\.out must be contiguous"):
        K.mask_descriptors([(_f(4, 8), None, None, _b(8, 4).t(), None, 0)], "cpu")
    assert fake_device == []


def test_row_strided_views_and_pass_through_values(fake_device):
    qkv, out, probs, kv = _f(2, 192), _f(2, 64), _f(1, 2, 2), _f(2)
    K.attention_fwd(qkv[:, 0:], qkv[:, 64:], qkv[:, 128:], out, probs, G=1, Tq=2, Tk=2, h=1, dk=64, ldq=192, ldk=192, ldv=192, ldo=64,
                    key_valid=kv, seed=(1 << 63) | 0x1000, stream_id=7)
    (name, args), = fake_device
    assert name == "sc_attention_fwd"
    assert args == (qkv.data_ptr(), qkv.data_ptr() + 256, qkv.data_ptr() + 512, 192, 192, 192, lib.F32, kv.data_ptr(), None,
                    probs.data_ptr(), out.data_ptr(), 64, 1, 2, 2, 1, 64, 0, 0.0, (1 << 63) | 0x1000, 7, 0x5eed)
    with pytest.raises(RuntimeError, match=r"^sc_attention_fwd: q must have a unit inner stride"):
        K.attention_fwd(qkv[:, ::2], qkv[:, 64:], qkv[:, 128:], out, probs, G=1, Tq=2, Tk=2, h=1, dk=64, ldq=192, ldk=192, ldv=192,
                        ldo=64)
    lib.call("sc_cast_f32_bf16", 0x1234, None, 8)                      # raw addresses and NULL pass unchanged
    assert fake_device[-1] == ("sc_cast_f32_bf16", (0x1234, None, 8, 0x5eed))
    assert len(fake_device) == 2


def test_wrong_device_and_argument_count_are_refused(fake_device, monkeypatch):
    monkeypatch.setattr(torch.Tensor, "get_device", lambda t: 1)
    with pytest.raises(RuntimeError, match=r"^sc_cast_f32_bf16: x is on cuda:1, not on the current device cuda:0"):
        K.cast_bf16(_f(8))
    with pytest.raises(TypeError, match=r"sc_cast_f32_bf16 takes 3 arguments \(x, y, n\), got 2"):
        lib.call("sc_cast_f32_bf16", 0, 0)
    assert fake_device == []
