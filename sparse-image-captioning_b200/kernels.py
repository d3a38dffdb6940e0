"""Tensor-level wrappers over the C ABI (one Python function per entry point of include/sc_b200.h).

All tensors must be CUDA tensors on the current device (lib.call checks every pointer argument); outputs are allocated by
the caller or here with torch (plumbing only).  Every function launches on torch's current stream, so calls are CUDA-graph
capturable.
"""
import contextlib
import math

import torch

from . import lib
from .lib import F32, BF16, MASK_NONE, MASK_ROUND, MASK_BERNOULLI, MASK_RAW, MASK_UNIFORM  # noqa: F401


def linear(x, w, bias=None, *, mask=None, mask_mode=MASK_NONE, uniforms=None, seed=0, stream_id=0, residual=None,
           relu=False, out=None, out_dtype=None, tile_n=0):
    """y = epilogue(x @ (w (.) mask)^T): sc_linear.  x [M,K] bf16|fp32, w [N,K] bf16|fp32."""
    M, K = x.shape
    N = w.shape[0]
    assert w.shape[1] == K, (w.shape, x.shape)
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=out_dtype or torch.float32)
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_linear", x, lib.dtype_code(x.dtype), w, lib.dtype_code(w.dtype), mask, mask_mode, uniforms, seed, stream_id,
             bias, residual, out, lib.dtype_code(out.dtype), M, N, K, int(relu), tile_n,
             meta=("gemm_bf16" if x.dtype == torch.bfloat16 else "gemm_f32", M, N, K, x.element_size(), w.element_size(),
                   out.element_size(), mask is not None, residual is not None, bool(relu), tile_n))
    return out


def linear_ln(x, w, bias=None, *, residual=None, relu=False, out=None, tile_n=0, ln_stats=None, ln_c=None, eps=1e-6,
              out_bf16=None, stats_out=None):
    """sc_linear_ln: bf16 tensor-core GEMM with a folded LayerNorm on its input (``ln_stats``/``ln_c``) and/or the
    residual-stream producer epilogue (``out_bf16`` copy + ``stats_out`` row statistics).  x, w bf16."""
    M, K = x.shape
    N = w.shape[0]
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and w.shape[1] == K
    lib.call("sc_linear_ln", x, w, bias, residual, out, lib.dtype_code(out.dtype), M, N, K, int(relu), tile_n, ln_stats, ln_c,
             float(eps), out_bf16, stats_out,
             meta=("gemm_bf16", M, N, K, 2, 2, out.element_size(), False, residual is not None, bool(relu)))
    return out


def set_pdl(enabled):
    """Programmatic dependent launch between consecutive kernels of a stream (on by default).  True / False, or a mask:
    bit 0 = GEMM + inference kernels, bit 1 = training row / attention kernels, bit 2 = early trigger inside the GEMM."""
    global _pdl_mask
    prev = _pdl_mask
    _pdl_mask = 7 if enabled is True or enabled == 1 else int(enabled) & 7
    lib.load().sc_set_pdl(_pdl_mask)
    return prev


_pdl_mask = 7


@contextlib.contextmanager
def pdl(mask):
    """``with pdl(mask):`` the block launches with set_pdl(mask), then the previous mask is restored."""
    prev = set_pdl(mask)
    try:
        yield
    finally:
        set_pdl(prev)


class CsrWeight:
    """CSR form of a pruned [N,K] weight: row_ptr int32 [N+1], col uint16 [nnz] (stored in an int16 tensor),
    values in the activation dtype.  Built from a dense (already masked) tensor; also accepts the reference's
    COO ``to_sparse()`` tensors (pruning/prune.py:200-221)."""

    def __init__(self, w, dtype):
        if w.is_sparse:
            w = w.to_dense()
        w = w.detach()
        N, K = w.shape
        assert K <= 65536
        nz = w != 0
        counts = nz.sum(1)
        row_ptr = torch.zeros(N + 1, dtype=torch.int64, device=w.device)
        row_ptr[1:] = torch.cumsum(counts, 0)
        idx = nz.nonzero(as_tuple=False)  # row-major order -> already grouped by row, columns ascending
        self.row_ptr = row_ptr.to(torch.int32).contiguous()
        self.col = idx[:, 1].to(torch.int32).to(torch.int16).contiguous()  # bit pattern of uint16
        self.val = w[nz].to(dtype).contiguous()
        self.shape = (N, K)
        self.nnz = int(self.val.numel())
        if self.nnz == 0:  # keep pointers valid
            self.col = torch.zeros(1, dtype=torch.int16, device=w.device)
            self.val = torch.zeros(1, dtype=dtype, device=w.device)


def csr_spmm(x, csr, bias=None, *, residual=None, relu=False, out=None, out_dtype=None):
    M, K = x.shape
    N = csr.shape[0]
    assert csr.shape[1] == K and csr.val.dtype == x.dtype
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=out_dtype or torch.float32)
    lib.call("sc_csr_spmm", x, lib.dtype_code(x.dtype), csr.row_ptr, csr.col, csr.val, bias, residual, out,
             lib.dtype_code(out.dtype), M, N, K, int(relu),
             meta=("csr_spmm", M, N, K, x.element_size(), csr.nnz, out.element_size()))
    return out


class SellWeight:
    """Sliced-ELL form (slab = 32 output features) of a pruned [N,K] weight for sc_sell_spmm: ``slab_ptr`` int32
    [slabs+1] in entries, ``entries`` int32 [total] = (column << 16) | bf16 bits, or int32 [total, 2] = {column, fp32 bits}
    in fp32 mode.  Built once from the dense (already masked) tensor or the reference's COO ``to_sparse()`` tensors."""

    def __init__(self, w, dtype):
        if w.is_sparse:
            w = w.to_dense()
        w = w.detach().float()
        N, K = w.shape
        assert K <= 65536
        dev = w.device
        slabs = (N + 31) // 32
        Np = slabs * 32
        wp = torch.zeros(Np, K, device=dev)
        wp[:N] = w
        nz = wp != 0
        counts = nz.sum(1)                                              # [Np]
        width = counts.view(slabs, 32).max(1).values                    # widest row of each slab
        width = ((width + 3) // 4 * 4).clamp_min(4)
        slab_ptr = torch.zeros(slabs + 1, dtype=torch.int64, device=dev)
        slab_ptr[1:] = torch.cumsum(width * 32, 0)
        total = int(slab_ptr[-1])
        # rank of every non-zero inside its row (columns ascending)
        rows, cols = nz.nonzero(as_tuple=True)
        row_start = torch.cumsum(counts, 0) - counts
        rank = torch.arange(rows.numel(), device=dev) - row_start[rows]
        pos = slab_ptr[rows // 32] + rank * 32 + (rows % 32)
        vals = wp[rows, cols]
        if dtype == torch.bfloat16:
            bits = vals.to(torch.bfloat16).view(torch.int16).to(torch.int64) & 0xFFFF
            packed = (cols << 16) | bits
            packed = torch.where(packed >= (1 << 31), packed - (1 << 32), packed)
            ent = torch.zeros(total, dtype=torch.int64, device=dev)
            ent[pos] = packed
            self.entries = ent.to(torch.int32).contiguous()
        else:
            ent = torch.zeros(total, 2, dtype=torch.int32, device=dev)
            ent[pos, 0] = cols.to(torch.int32)
            ent[pos, 1] = vals.contiguous().view(torch.int32)
            self.entries = ent.contiguous()
        self.slab_ptr = slab_ptr.to(torch.int32).contiguous()
        self.shape = (N, K)
        self.dtype = dtype
        self.nnz = int(rows.numel())
        self.padded = total


def sell_spmm(x, sw, bias=None, *, residual=None, relu=False, out=None, out_dtype=None):
    M, K = x.shape
    N = sw.shape[0]
    assert sw.shape[1] == K and sw.dtype == x.dtype
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=out_dtype or torch.float32)
    lib.call("sc_sell_spmm", x, lib.dtype_code(x.dtype), sw.slab_ptr, sw.entries, bias, residual, out, lib.dtype_code(out.dtype),
             M, N, K, int(relu),
             meta=("sell_spmm", M, N, K, x.element_size(), sw.nnz, out.element_size()))
    return out


class GsWeight:
    """Gather-SpMM form of a pruned [N, K] weight for sc_gspmm (tensor-core SpMM, bf16): per K chunk of 512 columns and per
    group of 8 output features, the group's non-zeros as 32-bit words ``(col_in_chunk << 19) | (feature_in_group << 16) | bf16
    bits``, padded with zero-valued words to a multiple of 16 (one m16n8k16 MMA step).  Inside a step the two octets are
    ordered so that their columns differ mod 8 wherever the group's columns allow it: the eight ldmatrix row pointers of an
    octet then fall into eight different shared-memory bank groups.  Built once from the dense (already masked) tensor or the
    reference's COO ``to_sparse()`` tensors (pruning/prune.py:200-221)."""

    KC = 512

    def __init__(self, w):
        import numpy as np
        if w.is_sparse:
            w = w.to_dense()
        dev = w.device
        wn = w.detach().float().cpu()
        N, K = wn.shape
        assert K % 8 == 0
        bits_all = (wn.to(torch.bfloat16).view(torch.int16).to(torch.int32) & 0xFFFF).numpy()
        nzmask = (wn != 0).numpy()
        ngroups, nchunks = (N + 7) // 8, (K + self.KC - 1) // self.KC
        ptr = np.zeros((nchunks, ngroups + 1), dtype=np.int32)
        words, off = [], 0
        for c in range(nchunks):
            k0, k1 = c * self.KC, min(K, (c + 1) * self.KC)
            for g in range(ngroups):
                ptr[c, g] = off
                sub = nzmask[g * 8: (g + 1) * 8, k0:k1]
                f, col = np.nonzero(sub)
                if f.size:
                    val = bits_all[g * 8 + f, k0 + col]
                    ent = ((col.astype(np.int64) << 19) | (f.astype(np.int64) << 16) | val.astype(np.int64))
                    ent = self._order(ent, col)
                    words.append(ent)
                    off += ent.size
            ptr[c, ngroups] = off
        ent = np.concatenate(words) if words else np.zeros(16, dtype=np.int64)
        ent = np.where(ent >= (1 << 31), ent - (1 << 32), ent).astype(np.int32)
        self.entries = torch.from_numpy(ent).to(dev).contiguous()
        self.grp_ptr = torch.from_numpy(ptr.reshape(-1)).to(dev).contiguous()
        self.shape = (N, K)
        self.nnz = int(nzmask.sum())
        self.padded = int(off)

    @staticmethod
    def _order(ent, col):
        """Entries of one (chunk, group) -> ceil(n / 8) octets (no octet of padding is ever added: shared-memory traffic is the
        kernel's bound) with the columns of every residue class mod 8 spread evenly over the octets, so that as few ldmatrix
        phases as the column set allows see two rows in one bank group; the tail is padded with zero-valued words to 16."""
        import numpy as np
        n = ent.size
        n_oct = (n + 7) // 8
        octets = [[] for _ in range(n_oct)]
        per_res = [[0] * 8 for _ in range(n_oct)]
        res = (col & 7)
        for r in sorted(range(8), key=lambda r: -int((res == r).sum())):
            for e in ent[res == r]:
                k = min((o for o in range(n_oct) if len(octets[o]) < 8), key=lambda o: (per_res[o][r], len(octets[o])))
                octets[k].append(int(e))
                per_res[k][r] += 1
        out = []
        for o in range(n_oct):
            free = [r for r in range(8) if per_res[o][r] == 0]
            while len(octets[o]) < 8:
                octets[o].append((free.pop() if free else 0) << 19)   # zero-valued padding word (column r < 8 of the chunk)
            out += octets[o]
        if len(out) % 16:
            out += [r << 19 for r in range(8)]
        return np.array(out, dtype=np.int64)


def gspmm(x, gw, bias=None, *, residual=None, relu=False, out=None, out_dtype=None):
    """y = act(x W^T + b) + residual with W in gather-SpMM form (sc_gspmm: mma.sync over gathered activation columns)."""
    M, K = x.shape
    N = gw.shape[0]
    assert gw.shape[1] == K and x.dtype == torch.bfloat16
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=out_dtype or torch.float32)
    lib.call("sc_gspmm", lib.Strided(x), x.stride(0), gw.grp_ptr, gw.entries, bias, residual, out, lib.dtype_code(out.dtype),
             M, N, K, int(relu),
             meta=("gspmm", M, N, K, 2, gw.nnz, out.element_size()))
    return out


def ingest_f32_bf16(host_pinned, out, ctas=0):
    """out (device bf16) = cast(host_pinned fp32): the kernel reads the pinned host tensor over PCIe itself (sc_ingest_f32_bf16)."""
    assert host_pinned.dtype == torch.float32 and out.dtype == torch.bfloat16 and out.numel() == host_pinned.numel()
    lib.call("sc_ingest_f32_bf16", host_pinned, out, host_pinned.numel(), int(ctas))
    return out


def layernorm(x, a, b, *, eps=1e-6, out=None, out_dtype=None):
    rows, D = x.shape
    assert x.dtype == torch.float32
    if out is None:
        out = torch.empty(rows, D, device=x.device, dtype=out_dtype or torch.float32)
    lib.call("sc_layernorm", x, a, b, out, lib.dtype_code(out.dtype), rows, D, eps)
    return out


def embed_pe(tokens, table, pe, *, T=1, pos0=0, mask=None, mask_mode=MASK_NONE, uniforms=None, seed=0, stream_id=0,
             out=None, out_dtype=None):
    rows = tokens.numel()
    V, D = table.shape
    assert tokens.dtype == torch.int32
    if out is None:
        out = torch.empty(rows, D, device=table.device, dtype=out_dtype or torch.float32)
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_embed_pe", tokens, table, mask, mask_mode, uniforms, seed, stream_id, pe, out, lib.dtype_code(out.dtype), rows, D,
             V, T, pos0, math.sqrt(D))
    return out


def embed_pe_stats(tokens, table, pe, x32, xb, stats, *, T=1, pos0=0):
    """sc_embed_pe_stats: embedding + positional encoding -> fp32 stream, bf16 copy, chunk statistics."""
    rows = tokens.numel()
    V, D = table.shape
    assert tokens.dtype == torch.int32 and xb.dtype == torch.bfloat16 and x32.dtype == torch.float32
    lib.call("sc_embed_pe_stats", tokens, table, pe, x32, xb, stats, rows, D, V, T, pos0, math.sqrt(D))
    return x32


def apply_mask(w, mask, mask_mode, *, uniforms=None, seed=0, stream_id=0, out_dtype=torch.float32, out=None):
    if out is None:
        out = torch.empty(w.shape, device=w.device, dtype=out_dtype)
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_apply_mask", w, mask, mask_mode, uniforms, seed, stream_id, out, lib.dtype_code(out.dtype), w.numel())
    return out


def mask_count(logits_list, out=None):
    """sum over tensors of sum(rint(sigmoid(S))) -> int64 CUDA scalar tensor (``out``: zeroed, then counted into)."""
    dev = logits_list[0].device
    cnt = torch.zeros(1, dtype=torch.int64, device=dev) if out is None else out.zero_()
    for s in logits_list:
        lib.call("sc_mask_count", s, s.numel(), cnt)
    return cnt


def cast_bf16(x, out=None):
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    lib.call("sc_cast_f32_bf16", x, out, x.numel())
    return out


def mask_rows(x, row_mask):
    rows, D = x.shape
    lib.call("sc_mask_rows", x, row_mask, rows, D)
    return x


def box_attention(q, k, v, boxes, wg_w, wg_b, att_mask, out, *, B, N, h, dk, ldq, ldk, ldv, ldo, trig=True,
                  wave_len=1000.0):
    lib.call("sc_box_attention_fwd", lib.Strided(q), lib.Strided(k), lib.Strided(v), ldq, ldk, ldv, lib.dtype_code(out.dtype),
             boxes, wg_w, wg_b, att_mask, lib.Strided(out), ldo, B, N, h, dk, int(trig), wave_len)
    return out


def box_bias_all(boxes, wg_w, wg_b, out, *, B, N, layers, h, trig=True, wave_len=1000.0, tensor_cores=False):
    """Geometry bias of every encoder layer at once: out fp32 [layers, B, h, N, N] (sc_box_bias_all).
    ``tensor_cores``: the TF32 mma variant of the bf16 inference path (sc_box_bias_all_tc) when the shape is served."""
    if (tensor_cores and trig and (layers * h) % 8 == 0 and layers * h <= 64 and 4 <= N <= 2048
            and layers * h * B * N * N * 4 < 2 ** 32):
        lib.call("sc_box_bias_all_tc", boxes, wg_w, wg_b, out, B, N, layers, h, wave_len)
        return out
    lib.call("sc_box_bias_all", boxes, wg_w, wg_b, out, B, N, layers, h, int(trig), wave_len)
    return out


def bias_attention(q, k, v, bias, att_mask, out, *, B, N, h, dk, ldq, ldk, ldv, ldo):
    """box_attention of one layer given its geometry bias [B,h,N,N] (bf16 tensor path, sc_bias_attention_fwd)."""
    lib.call("sc_bias_attention_fwd", lib.Strided(q), lib.Strided(k), lib.Strided(v), ldq, ldk, ldv, lib.dtype_code(out.dtype),
             bias, att_mask, lib.Strided(out), ldo, B, N, h, dk)
    return out


def self_attn_step(q, k, v, cache_k, cache_v, anc, out, *, R, D, h, n_prev, write_slot, ldq, ldk, ldv, ldo, anc_ld,
                   slot_div=1):
    lib.call("sc_decode_self_attn_step", lib.Strided(q), lib.Strided(k), lib.Strided(v), ldq, ldk, ldv, lib.dtype_code(out.dtype),
             cache_k, cache_v, anc, anc_ld, slot_div, lib.Strided(out), ldo, R, D, h, n_prev, write_slot)
    return out


def cross_attn_step(q, mem_k, mem_v, att_mask, out, *, B, beam, N, D, h, ldq, ldm, ldo):
    lib.call("sc_decode_cross_attn_step", lib.Strided(q), ldq, lib.Strided(mem_k), lib.Strided(mem_v), ldm, lib.dtype_code(out.dtype),
             att_mask, lib.Strided(out), ldo, B, beam, N, D, h)
    return out


def beam_step(logits, st, t, *, B, beam, V, L, eos, pad, temperature=1.0, constraint=0, penalty_kind=0, penalty_alpha=0.0,
              suppress_tok=None, penalized_col=-1, diverse=None):
    """``st``: BeamState.  Reads buffers ``t % 2`` and writes ``(t+1) % 2``.  ``suppress_tok`` (int32 [B*beam], -1 = none):
    per-row token that cannot be chosen at this step (remove_bad_endings); ``penalized_col``: column whose log-prob is
    lowered by 1000 (suppress_UNK).  ``diverse = (group_seq, group, diversity_lambda)``: the diverse-beam step of group
    ``group`` at its local step ``t`` (sc_beam_step_diverse; group_seq int32 [G, 2, B*beam, L] holds every group's seq)."""
    i, o = t & 1, (t + 1) & 1
    assert suppress_tok is None or (suppress_tok.dtype == torch.int32 and suppress_tok.numel() == B * beam)
    head = [logits, B, beam, V, L, t, eos, pad, float(temperature), int(constraint), int(penalty_kind), float(penalty_alpha),
            suppress_tok, int(penalized_col)]
    tail = [st.seq[i], st.seq[o], st.lp[i], st.lp[o], st.sum, st.anc[i], st.anc[o], st.tokens, st.done_seq, st.done_lp, st.done_p,
            st.done_count, st.ws, st.ws.numel()]
    if diverse is None:
        lib.call("sc_beam_step", *head, *tail)
    else:
        lib.call("sc_beam_step_diverse", *head, *_diverse_args(diverse, B, beam, L), *tail)


def _diverse_args(diverse, B, beam, L):
    hist, group, lam = diverse
    assert hist.dtype == torch.int32 and tuple(hist.shape[1:]) == (2, B * beam, L) and group < hist.shape[0]
    return [hist, int(group), float(lam)]


def linear_hmask(x, w, h, out, *, scale=1.0, colsum=None):
    """out (bf16 [M,N]) = (x @ w^T) * scale where h != 0 else 0; colsum (fp32 [N]) += column sums of out (sc_linear_hmask)."""
    M, K = x.shape
    N = w.shape[0]
    assert x.dtype == w.dtype == h.dtype == out.dtype == torch.bfloat16 and tuple(h.shape) == tuple(out.shape) == (M, N)
    lib.call("sc_linear_hmask", x, w, h, float(scale), colsum, out, M, N, K,
             meta=("gemm_bf16", M, N, K, 2, 2, 2, False, False, False))
    return out


def linear_topk_parts(N):
    """Records per row that sc_linear_topk writes for an N-column generator."""
    return 2 * ((N + 255) // 256)


def linear_topk(x, w, bias, partials, candidates=5):
    """Generator GEMM whose epilogue keeps only the per-row log-sum-exp partials and top-5 candidates (no logits):
    partials fp32 [M, linear_topk_parts(N), 12]."""
    M, K = x.shape
    N = w.shape[0]
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and w.shape[1] == K
    assert tuple(partials.shape) == (M, linear_topk_parts(N), 12) and partials.dtype == torch.float32
    lib.call("sc_linear_topk", x, w, bias, M, N, K, partials, int(candidates),
             meta=("gemm_bf16", M, N, K, 2, 2, 0, False, False, False))
    return partials


def beam_step_partials(partials, st, t, *, B, beam, V, L, eos, pad, penalty_kind=0, penalty_alpha=0.0, diverse=None):
    """Beam step from sc_linear_topk records (temperature 1, no decoding constraint, beam <= 5).  ``diverse``: as in
    ``beam_step`` (the records must hold (group + 1) * beam candidates per row)."""
    i, o = t & 1, (t + 1) & 1
    head = [partials, partials.shape[1], B, beam, V, L, t, eos, pad, int(penalty_kind), float(penalty_alpha)]
    tail = [st.seq[i], st.seq[o], st.lp[i], st.lp[o], st.sum, st.anc[i], st.anc[o], st.tokens, st.done_seq, st.done_lp, st.done_p,
            st.done_count, st.ws, st.ws.numel()]
    if diverse is None:
        lib.call("sc_beam_step_partials", *head, *tail)
    else:
        lib.call("sc_beam_step_partials_diverse", *head, *_diverse_args(diverse, B, beam, L), *tail)


def beam_step_workspace_bytes(B, beam):
    return int(lib.load().sc_beam_step_workspace_bytes(B, beam))


def greedy_step(logits, st, t, *, R, V, L, eos, constraint=0):
    lib.call("sc_greedy_step", logits, R, V, L, t, eos, int(constraint), st.seq, st.lp, st.tokens, st.unfinished, st.live)


def sample_step(logits, st, t, *, R, V, L, eos, constraint=0, temperature=1.0, uniforms=None, seed=0):
    """Multinomial step on a GreedyState (one row per sample): sc_sample_step."""
    lib.call("sc_sample_step", logits, R, V, L, t, eos, int(constraint), float(temperature), uniforms, seed,
             st.seq, st.lp, st.tokens, st.unfinished, st.live)


def cache_reorder(src, idx, out=None):
    """dst[r] = src[idx[r]] along dim 0 (K8)."""
    rows = idx.numel()
    row_bytes = src[0].numel() * src.element_size()
    if out is None:
        out = torch.empty((rows,) + tuple(src.shape[1:]), device=src.device, dtype=src.dtype)
    assert idx.dtype == torch.int32
    lib.call("sc_cache_reorder", src, out, idx, rows, row_bytes)
    return out


# ------------------------------------------------------------------------------------------------------------------
# training-side wrappers
# ------------------------------------------------------------------------------------------------------------------
def pad8(n):
    return (n + 7) // 8 * 8


def linear_dropout(x, w, bias=None, *, mask=None, mask_mode=MASK_NONE, uniforms=None, seed=0, stream_id=0, residual=None,
                   relu=False, out=None, out_dtype=None, p=0.0, drop_seed=0, drop_stream=0, tile_n=0):
    """Training forward of a (masked) linear: y = dropout(act(x (W.m)^T + b), p) + residual."""
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=out_dtype or torch.float32)
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_linear_dropout", x, lib.dtype_code(x.dtype), w, lib.dtype_code(w.dtype), mask, mask_mode, uniforms, seed,
             stream_id, bias, residual, out, lib.dtype_code(out.dtype), M, N, K, int(relu), tile_n, float(p), drop_seed, drop_stream,
             meta=("gemm_bf16" if x.dtype == torch.bfloat16 else "gemm_f32", M, N, K, x.element_size(), w.element_size(),
                   out.element_size(), mask is not None, residual is not None, bool(relu), p > 0, tile_n))
    return out


def linear_wgrad(dyT, xT, w, mask, mask_mode, dw, ds, *, M, uniforms=None, seed=0, stream_id=0, bypass=False, sp_coeff=0.0,
                 accumulate=False, tile_n=0, workspace=None):
    """dWm = dyT[N,Mp] @ xT[K,Mp]^T with the fused straight-through epilogue into dw / ds (either may be None).
    ``M`` = padded token count (columns of dyT / xT, multiple of 8 in bf16)."""
    N, K = w.shape
    assert dyT.shape[0] == N and xT.shape[0] == K and dyT.shape[1] == xT.shape[1] == M
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_linear_wgrad", dyT, xT, lib.dtype_code(dyT.dtype), w, mask, mask_mode, uniforms, seed, stream_id, int(bypass),
             float(sp_coeff), dw, ds, int(accumulate), N, K, M, tile_n, workspace,
             0 if workspace is None else workspace.numel() * workspace.element_size(),
             meta=("gemm_bf16" if dyT.dtype == torch.bfloat16 else "gemm_f32", N, K, M, dyT.element_size(), xT.element_size(), 4, False))


def linear_wgrad_rowmajor(dy, x, w, mask, mask_mode, dw, ds, *, workspace, uniforms=None, seed=0, stream_id=0, bypass=False,
                          sp_coeff=0.0, accumulate=False):
    """Weight gradient from the row-major bf16 activations dy [M,N], x [M,K] (no transposed copies): sc_linear_wgrad_rowmajor."""
    N, K = w.shape
    M = dy.shape[0]
    assert dy.shape[1] == N and tuple(x.shape) == (M, K) and dy.dtype == x.dtype == torch.bfloat16
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_linear_wgrad_rowmajor", dy, x, w, mask, mask_mode, uniforms, seed, stream_id, int(bypass), float(sp_coeff), dw,
             ds, int(accumulate), N, K, M, workspace, workspace.numel() * workspace.element_size(),
             meta=("gemm_bf16", N, K, M, 2, 2, 4, False))


def prep_grad(g, *, h=None, out=None, outT=None, scale=1.0, p=0.0, seed=0, stream_id=0, colsum=None):
    """out = g * keep * scale (cast), outT = its transpose with leading dim outT.shape[1] (zero padded);
    ``colsum`` (fp32 [cols]) accumulates the column sums of out (bias gradient)."""
    rows, cols = g.shape
    assert g.dtype == torch.float32
    ref = out if out is not None else outT
    ldT = outT.shape[1] if outT is not None else rows
    lib.call("sc_prep_grad", g, h, lib.dtype_code(h.dtype) if h is not None else F32, out, outT, ldT, lib.dtype_code(ref.dtype), rows,
             cols, float(scale), float(p), seed, stream_id, colsum)


def transpose(x, outT):
    rows, cols = x.shape
    lib.call("sc_transpose", x, lib.dtype_code(x.dtype), outT, outT.shape[1], lib.dtype_code(outT.dtype), rows, cols)
    return outT


def apply_mask_transposed(w, mask, mask_mode, outT, *, uniforms=None, seed=0, stream_id=0, out=None):
    """outT [K,N] = (w (.) mask)^T; ``out`` [N,K] (optional, same dtype) = w (.) mask from the same pass."""
    N, K = w.shape
    assert tuple(outT.shape) == (K, N) and (out is None or (tuple(out.shape) == (N, K) and out.dtype == outT.dtype))
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_apply_mask_transposed", w, mask, mask_mode, uniforms, seed, stream_id, outT, lib.dtype_code(outT.dtype), N, K, out)
    return outT


def mask_descriptors(items, device):
    """Descriptor table of sc_apply_mask_batched.  items: (w [N,K] fp32, s | None, u | None, out | None, outT | None, stream_id).
    Returns (int64 device tensor [n, 10], total 64x64 tiles)."""
    rows, start = [], 0
    for i, (w, s, u, out, outT, sid) in enumerate(items):
        N, K = w.shape
        assert K % 4 == 0
        tk = (K + 63) // 64
        rows.append([lib.address(t, "sc_apply_mask_batched", f"descs[{i}].{f}") for t, f in
                     ((w, "w"), (s, "s"), (u, "uniforms"), (out, "out"), (outT, "outT"))] + [N, K, int(sid), start, tk])
        start += tk * ((N + 63) // 64)
    return torch.tensor(rows, dtype=torch.int64).to(device), start


def apply_mask_batched(desc, total_tiles, mask_mode, *, seed=0, stream_base=0, out_dtype=torch.bfloat16):
    lib.call("sc_apply_mask_batched", desc, desc.shape[0], total_tiles, mask_mode, seed, stream_base, lib.dtype_code(out_dtype))


def mask_grad(dwm, w, mask, mask_mode, dw, ds, *, uniforms=None, seed=0, stream_id=0, bypass=False, sp_coeff=0.0,
              accumulate=False):
    if mask is None:
        mask_mode = MASK_NONE
    lib.call("sc_mask_grad", dwm, w, mask, mask_mode, uniforms, seed, stream_id, int(bypass), float(sp_coeff), dw, ds,
             int(accumulate), w.numel())


def colsum(x, out, accumulate=False):
    rows, cols = x.shape
    lib.call("sc_colsum", x, lib.dtype_code(x.dtype), out, rows, cols, int(accumulate))
    return out


def layernorm_bwd(x, a, dy, dx, da, db, *, dres=None, eps=1e-6, next_gb=None, next_colsum=None, next_p=0.0, seed=0, stream_id=0):
    """LayerNorm backward; ``next_gb`` (bf16 [rows, D], D == 512): also emit dx (.) dropout mask as the gradient operand of
    the next linear in the backward chain and add its column sums to ``next_colsum`` (sc_layernorm_bwd_fused)."""
    rows, D = x.shape
    if next_gb is None:
        lib.call("sc_layernorm_bwd", x, a, dy, lib.dtype_code(dy.dtype), dres, dx, da, db, rows, D, eps)
    else:
        assert next_gb.dtype == torch.bfloat16 and tuple(next_gb.shape) == (rows, D)
        lib.call("sc_layernorm_bwd_fused", x, a, dy, lib.dtype_code(dy.dtype), dres, dx, da, db, rows, D, eps, next_gb, next_colsum,
                 float(next_p), seed, stream_id)
    return dx


def logsoftmax_nll(logits, target=None, weight=None, inv_norm=None, loss_sum=None, dlogits=None, logprobs=None):
    rows, V = logits.shape
    lib.call("sc_logsoftmax_nll", logits, target, weight, inv_norm, loss_sum, dlogits,
             lib.dtype_code(dlogits.dtype) if dlogits is not None else F32, logprobs, rows, V)


def scst_targets(seq, score, base_score, *, S, cider_weight, bos, pad, tokens, targets, tok_w, key_valid, inv_norm, mask_sum=None,
                 norm_in=None, mean_reward=None):
    """SCST rollout seq int32 [R, L] + CIDEr-D scores float64 [R] (+ greedy baseline scores float64 [R // S], or None: mean of
    the image's other samples) -> the training step's tokens / targets / tok_w / key_valid [R * L] and inv_norm (sc_scst_targets)."""
    R, L = seq.shape
    assert seq.dtype == torch.int32 and score.dtype == torch.float64 and score.numel() == R
    assert base_score is None or (base_score.dtype == torch.float64 and base_score.numel() == R // S)
    for t, dt in ((tokens, torch.int32), (targets, torch.int32), (tok_w, torch.float32), (key_valid, torch.float32)):
        assert t.dtype == dt and t.numel() == R * L
    lib.call("sc_scst_targets", seq, R, L, int(S), score, base_score, float(cider_weight), int(bos), int(pad), tokens, targets, tok_w,
             key_valid, mask_sum, inv_norm, norm_in, mean_reward)


def embedding_bwd(tokens, dy, dtable, scale):
    rows, D = dy.shape
    lib.call("sc_embedding_bwd", tokens, dy, dtable, rows, D, dtable.shape[0], float(scale))


def adam_clip(param, grad, m, v, *, lr, betas, eps, weight_decay, clip, grad_scale, step, sigmoid_grad_coeff=None, dyn=None):
    """``dyn``: optional device fp32 [3] = {lr, 1 - b1^step, sqrt(1 - b2^step)} read at run time (CUDA-graph replay)."""
    lib.call("sc_adam_clip", param, grad, m, v, param.numel(), float(lr), float(betas[0]), float(betas[1]), float(eps),
             float(weight_decay), float(clip), float(grad_scale), int(step), sigmoid_grad_coeff, dyn)


def st_descriptors(segments, device):
    """Descriptor table of sc_adam_clip_st.  segments: (w_off, s_off | -1, n, stream_id) in flat-buffer elements.
    Returns (int64 device tensor [n, 5], total blocks)."""
    chunk = int(lib.load().sc_adam_clip_st_chunk())
    rows, start = [], 0
    for w_off, s_off, n, sid in segments:
        rows.append([int(w_off), int(s_off), int(n), int(sid), start])
        start += (int(n) + chunk - 1) // chunk
    return torch.tensor(rows, dtype=torch.int64).to(device), start


def adam_clip_st(desc, blocks, w, g, m_w, v_w, s, m_s, v_s, *, uniforms, mask_mode, bypass, update_logits, seed, stream_base, lr, eps,
                 weight_decay, mask_lr, mask_eps, betas, clip, grad_scale, step, sigmoid_grad_coeff=None, dyn=None):
    """One-launch optimizer step over a descriptor table (sc_adam_clip_st): straight-through dW / dS from the exchanged dWm
    with the mask sample regenerated, then clip + Adam for the weight and the mask-logit groups."""
    lib.call("sc_adam_clip_st", desc, desc.shape[0], blocks, w, g, m_w, v_w, s, m_s, v_s, uniforms, int(mask_mode), int(bypass),
             int(update_logits), seed, stream_base, float(lr), float(eps), float(weight_decay), float(mask_lr), float(mask_eps),
             float(betas[0]), float(betas[1]), float(clip), float(grad_scale), int(step), sigmoid_grad_coeff, dyn)


PRUNE_ABS, PRUNE_DIST, PRUNE_SNIP = 0, 1, 2


def prune_descriptors(segments, device):
    """Descriptor table of sc_prune_stats / sc_prune_select.  segments: (src_off, dst_off, n, group, pos_base) in flat-buffer
    elements.  Returns (int64 device tensor [n, 6], total blocks)."""
    chunk = int(lib.load().sc_prune_chunk())
    rows, start = [], 0
    for src_off, dst_off, n, group, pos_base in segments:
        assert n > 0 and 0 <= pos_base and pos_base + n <= 1 << 32, (n, pos_base)
        rows.append([int(src_off), int(dst_off), int(n), int(group), int(pos_base), start])
        start += (int(n) + chunk - 1) // chunk
    return _to_device(torch.tensor(rows, dtype=torch.int64), device), start


def _to_device(t, device):
    """Host tensor -> device without a host synchronisation: staged in pinned memory, copied asynchronously on the current
    stream (the caching host allocator keeps the staging block until the copy has run)."""
    device = torch.device(device)
    if device.type != "cuda":
        return t.to(device)
    return t.pin_memory().to(device, non_blocking=True)


def prune_stats(desc, blocks, src, *, binarize=False, centered=False):
    """Per-segment {sum x, sum x^2} (float64 [n_desc, 2]) of ``src`` (or of rint(sigmoid(src)) with ``binarize``); ``centered``:
    {sum x, sum (x - mean)^2} from a second pass (the two-pass variance of mag_dist)."""
    assert src.dtype == torch.float32
    partials = torch.empty(blocks, 2, dtype=torch.float64, device=src.device)

    def run(center):
        sums = torch.empty(desc.shape[0], 2, dtype=torch.float64, device=src.device)
        lib.call("sc_prune_stats", desc, desc.shape[0], blocks, src, int(binarize), center, partials, sums)
        return sums

    sums = run(None)
    return run(sums) if centered else sums


def prune_select(desc, blocks, group_k, criterion, src, mask_out, *, sums=None):
    """0/1 masks into ``mask_out``: per group, the first group_k[g] elements in (criterion, position) order are pruned
    (sc_prune_select).  group_k: a list of ints (uploaded without a host synchronisation) or a device int64 tensor.  ``sums``:
    prune_stats of ``src`` for PRUNE_SNIP, prune_stats(centered=True) for PRUNE_DIST."""
    if not torch.is_tensor(group_k):
        group_k = _to_device(torch.tensor(group_k, dtype=torch.int64), src.device)
    assert src.dtype == mask_out.dtype == torch.float32 and group_k.dtype == torch.int64
    n_groups = group_k.numel()
    ws = torch.empty(n_groups * 1056 + desc.shape[0] * 8, dtype=torch.uint8, device=src.device)
    lib.call("sc_prune_select", desc, desc.shape[0], blocks, n_groups, group_k, int(criterion), src, sums, mask_out, ws, ws.numel())
    return mask_out


def sparsity_coeff(count, total, target, scale, out3, scale_dev=None):
    """out3 = [|target - sparsity|, d(scaled loss)/d(nnz), sparsity] from the device-side binarized-mask count."""
    lib.call("sc_sparsity_coeff", count, float(total), float(target), float(scale), scale_dev, out3)
    return out3


def attention_fwd(q, k, v, out, probs, *, G, Tq, Tk, h, dk, ldq, ldk, ldv, ldo, key_valid=None, bias=None, causal_T=0, p=0.0,
                  seed=0, stream_id=0):
    lib.call("sc_attention_fwd", lib.Strided(q), lib.Strided(k), lib.Strided(v), ldq, ldk, ldv, lib.dtype_code(out.dtype), key_valid,
             bias, probs, lib.Strided(out), ldo, G, Tq, Tk, h, dk, causal_T, float(p), seed, stream_id)
    return out


def attention_bwd(q, k, v, probs, d_out, dq, dk_, dv, *, dtype, G, Tq, Tk, h, dk, ldq, ldk, ldv, ldd, ldgq, ldgk, ldgv, dbias=None,
                  p=0.0, seed=0, stream_id=0):
    lib.call("sc_attention_bwd", lib.Strided(q), lib.Strided(k), lib.Strided(v), ldq, ldk, ldv, lib.dtype_code(dtype), probs,
             lib.Strided(d_out), ldd, lib.Strided(dq), lib.Strided(dk_), lib.Strided(dv), ldgq, ldgk, ldgv, dbias, G, Tq, Tk, h, dk,
             float(p), seed, stream_id)


def attention_bwd_bf16out(q, k, v, probs, d_out, dq, dk_, dv, *, G, Tq, Tk, h, dk, ldq, ldk, ldv, ldd, ldgq, ldgk, ldgv, bq=None, bk=None,
                          bv=None, dbias=None, p=0.0, seed=0, stream_id=0):
    """attention_bwd whose dq / dk / dv are bf16 GEMM operands and whose bias gradients (column sums) go to bq / bk / bv."""
    assert dq.dtype == dk_.dtype == dv.dtype == torch.bfloat16
    lib.call("sc_attention_bwd_bf16out", lib.Strided(q), lib.Strided(k), lib.Strided(v), ldq, ldk, ldv, probs, lib.Strided(d_out),
             ldd, lib.Strided(dq), lib.Strided(dk_), lib.Strided(dv), ldgq, ldgk, ldgv, bq, bk, bv, dbias, G, Tq, Tk, h, dk, float(p),
             seed, stream_id)


def box_bias_fwd(boxes, wg_w, wg_b, bias, *, B, N, h, trig=True, wave_len=1000.0):
    lib.call("sc_box_bias_fwd", boxes, wg_w, wg_b, bias, B, N, h, int(trig), wave_len)
    return bias


def box_bias_bwd(boxes, bias, dbias, dwg_w, dwg_b, *, B, N, h, trig=True, wave_len=1000.0):
    lib.call("sc_box_bias_bwd", boxes, bias, dbias, dwg_w, dwg_b, B, N, h, int(trig), wave_len)


def box_embedding(boxes, *, trig=True, wave_len=1000.0, out=None):
    """BoxRelationalEmbedding (relation_transformer.py:196-256): boxes fp32 [B,N,4] -> fp32 [B,N,N,64] (or [B,N,N,4])."""
    B, N = boxes.shape[:2]
    assert boxes.dtype == torch.float32
    if out is None:
        out = torch.empty(B, N, N, 64 if trig else 4, device=boxes.device)
    lib.call("sc_box_embedding", boxes, out, B, N, int(trig), float(wave_len))
    return out


def log_clamp(x, *, lo=1e-6, dy=None, out=None):
    """out = log(max(x, lo)); with ``dy``: out = dy / x where x > lo else 0 (its gradient).  fp32."""
    if out is None:
        out = torch.empty_like(x)
    lib.call("sc_log_clamp", x, dy, out, x.numel(), float(lo))
    return out


def logsoftmax_bwd(logprobs, dy, out=None):
    """dx = dy - exp(logprobs) * rowsum(dy): backward of log_softmax (sc_logsoftmax_bwd)."""
    rows, V = logprobs.shape
    if out is None:
        out = torch.empty_like(logprobs)
    lib.call("sc_logsoftmax_bwd", logprobs, dy, out, rows, V)
    return out
