"""ctypes binding of the C ABI in include/sc_b200.h (built as csrc/libsc_b200.so).

There is deliberately NO fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

import torch  # noqa: F401  (loads libcudart into the process before our library)

_HERE = os.path.dirname(os.path.abspath(__file__))
# SC_LIB_PATH: diagnostic override (same-box A/B of two builds of the library, scripts/); the product path is the in-tree build
LIB_PATH = os.environ.get("SC_LIB_PATH") or os.path.join(_HERE, "csrc", "libsc_b200.so")

F32, BF16 = 0, 1
MASK_NONE, MASK_ROUND, MASK_BERNOULLI, MASK_RAW, MASK_UNIFORM = 0, 1, 2, 3, 4

_p, _i, _f, _u64, _sz, _l = C.c_void_p, C.c_int, C.c_float, C.c_ulonglong, C.c_size_t, C.c_long

# name -> argtypes (mirrors include/sc_b200.h; tests/test_abi.py checks header and table agree)
SIGNATURES = {
    "sc_linear": [_p, _i, _p, _i, _p, _i, _p, _u64, _u64, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p],
    "sc_linear_ln": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _f, _p, _p, _p],
    "sc_set_pdl": [_i],
    "sc_csr_spmm": [_p, _i, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p],
    "sc_sell_spmm": [_p, _i, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p],
    "sc_gspmm": [_p, _i, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p],
    "sc_layernorm": [_p, _p, _p, _p, _i, _i, _i, _f, _p],
    "sc_embed_pe": [_p, _p, _p, _i, _p, _u64, _u64, _p, _p, _i, _i, _i, _i, _i, _i, _f, _p],
    "sc_embed_pe_stats": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p],
    "sc_apply_mask": [_p, _p, _i, _p, _u64, _u64, _p, _i, _sz, _p],
    "sc_mask_count": [_p, _sz, _p, _p],
    "sc_cast_f32_bf16": [_p, _p, _sz, _p],
    "sc_ingest_f32_bf16": [_p, _p, _sz, _i, _p],
    "sc_mask_rows": [_p, _p, _i, _i, _p],
    "sc_box_attention_fwd": [_p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _f, _p],
    "sc_box_bias_all": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p],
    "sc_box_bias_all_tc": [_p, _p, _p, _p, _i, _i, _i, _i, _f, _p],
    "sc_bias_attention_fwd": [_p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _i, _i, _i, _i, _i, _p],
    "sc_decode_self_attn_step": [_p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _i, _i, _p, _i, _i, _i, _i, _i, _i, _p],
    "sc_decode_cross_attn_step": [_p, _i, _p, _p, _i, _i, _p, _p, _i, _i, _i, _i, _i, _i, _p],
    "sc_beam_step": [_p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _f, _p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p],
    "sc_beam_step_workspace_bytes": [_i, _i],
    "sc_linear_hmask": [_p, _p, _p, _f, _p, _p, _i, _i, _i, _p],
    "sc_linear_topk_parts": [_i],
    "sc_linear_topk": [_p, _p, _p, _i, _i, _i, _p, _i, _p],
    "sc_beam_step_partials": [_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p],
    "sc_beam_step_diverse": [_p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _f, _p, _i, _p, _i, _f, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p,
                             _p, _p, _p, _sz, _p],
    "sc_beam_step_partials_diverse": [_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p, _i, _f, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p,
                                      _p, _p, _p, _sz, _p],
    "sc_greedy_step": [_p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p],
    "sc_sample_step": [_p, _i, _i, _i, _i, _i, _i, _f, _p, _u64, _p, _p, _p, _p, _p, _p],
    "sc_cache_reorder": [_p, _p, _p, _l, _l, _p],
    # training
    "sc_linear_dropout": [_p, _i, _p, _i, _p, _i, _p, _u64, _u64, _p, _p, _p, _i, _i, _i, _i, _i, _i, _f, _u64, _u64, _p],
    "sc_linear_wgrad": [_p, _p, _i, _p, _p, _i, _p, _u64, _u64, _i, _f, _p, _p, _i, _i, _i, _i, _i, _p, _sz, _p],
    "sc_linear_wgrad_rowmajor": [_p, _p, _p, _p, _i, _p, _u64, _u64, _i, _f, _p, _p, _i, _i, _i, _i, _p, _sz, _p],
    "sc_prep_grad": [_p, _p, _i, _p, _p, _i, _i, _i, _i, _f, _f, _u64, _u64, _p, _p],
    "sc_transpose": [_p, _i, _p, _i, _i, _i, _i, _p],
    "sc_apply_mask_transposed": [_p, _p, _i, _p, _u64, _u64, _p, _i, _i, _i, _p, _p],
    "sc_apply_mask_batched": [_p, _i, _l, _i, _u64, _u64, _i, _p],
    "sc_mask_grad": [_p, _p, _p, _i, _p, _u64, _u64, _i, _f, _p, _p, _i, _sz, _p],
    "sc_colsum": [_p, _i, _p, _i, _i, _i, _p],
    "sc_layernorm_bwd": [_p, _p, _p, _i, _p, _p, _p, _p, _i, _i, _f, _p],
    "sc_layernorm_bwd_fused": [_p, _p, _p, _i, _p, _p, _p, _p, _i, _i, _f, _p, _p, _f, _u64, _u64, _p],
    "sc_logsoftmax_nll": [_p, _p, _p, _p, _p, _p, _i, _p, _i, _i, _p],
    "sc_embedding_bwd": [_p, _p, _p, _i, _i, _i, _f, _p],
    "sc_adam_clip": [_p, _p, _p, _p, _sz, _f, _f, _f, _f, _f, _f, _f, _i, _p, _p, _p],
    "sc_sparsity_coeff": [_p, C.c_double, _f, _f, _p, _p, _p],
    "sc_adam_clip_st_chunk": [],
    "sc_adam_clip_st": [_p, _i, _l, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _u64, _u64, _f, _f, _f, _f, _f, _f, _f, _f, _f, _i, _p, _p, _p],
    "sc_attention_fwd": [_p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _u64, _u64, _p],
    "sc_attention_bwd": [_p, _p, _p, _i, _i, _i, _i, _p, _p, _i, _p, _p, _p, _i, _i, _i, _p, _i, _i, _i, _i, _i, _f, _u64, _u64, _p],
    "sc_attention_bwd_bf16out": [_p, _p, _p, _i, _i, _i, _p, _p, _i, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _u64, _u64, _p],
    "sc_box_bias_fwd": [_p, _p, _p, _p, _i, _i, _i, _i, _f, _p],
    "sc_box_bias_bwd": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _p],
    "sc_box_embedding": [_p, _p, _i, _i, _i, _f, _p],
    "sc_log_clamp": [_p, _p, _p, _sz, _f, _p],
    "sc_logsoftmax_bwd": [_p, _p, _p, _i, _i, _p],
    "sc_ciderd_score": [_p, _i, _i, _p, _i, _i, _p, _p, _l, C.c_double, C.c_double, _p, _p, _p, _p, _p, _p, _p, _p],
    "sc_cider_score": [_p, _i, _i, _p, _i, _i, _i, _p, _p, _l, C.c_double, _p, _p, _p, _p, _p, _p, _p],
    "sc_bleu_stats": [_p, _i, _i, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "sc_rouge_l": [_p, _i, _i, _p, _i, _i, _i, _p, _p, _p, _p, _p],
    "sc_caption_metrics_reduce": [_p, _p, _p, _p, _p, _i, _p, _p],
    "sc_scst_targets": [_p, _i, _i, _i, _p, _p, _f, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "sc_prune_chunk": [],
    "sc_prune_stats": [_p, _i, _l, _p, _i, _p, _p, _p, _p],
    "sc_prune_select": [_p, _i, _l, _i, _p, _i, _p, _p, _p, _p, _sz, _p],
}

_lib = None


def load():
    """Load the shared library (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"(or `make -C {os.path.dirname(LIB_PATH)}`).  There is no CPU/PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.sc_last_error.restype = C.c_char_p
    lib.sc_last_error.argtypes = []
    lib.sc_version.restype = C.c_int
    lib.sc_version.argtypes = []
    _lib = lib
    return lib


def ptr(t):
    """Device pointer of a tensor (or NULL)."""
    return None if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def resolve_device(device):
    """The kernels launch on the CURRENT device's current stream and cache function attributes / the SM count per process:
    an engine or trainer therefore lives on the current CUDA device (one process per GPU; call torch.cuda.set_device first)."""
    dev = torch.device(device)
    if dev.type != "cuda":
        return dev  # (parameter-layout bookkeeping only, e.g. the CPU tier's bucket tests: every kernel wrapper rejects CPU tensors)
    cur = torch.cuda.current_device()
    if dev.index is not None and dev.index != cur:
        raise RuntimeError(f"device {dev} is not the current CUDA device (cuda:{cur}): call torch.cuda.set_device({dev.index}) "
                           f"first - kernels launch on the current device's stream")
    return torch.device("cuda", cur)


def dtype_code(dt):
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported dtype {dt}")


launch_count = 0  # kernels launched through this binding (bench.py reports it as gpu_launches)
profile = None    # set to a list to record (name, meta, start_event, end_event) per launch (bench.py roofline leg)


def call(name, *args, meta=None):
    global launch_count
    lib = load()
    if profile is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed (status {rc}): {lib.sc_last_error().decode()}")
    if profile is not None:
        ev1.record()
        profile.append((name, meta, ev0, ev1))
    launch_count += 1
