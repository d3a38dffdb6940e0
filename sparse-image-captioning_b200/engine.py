"""Inference engine for the ORT / ACORT captioner: encoder, KV-cached incremental decoding, beam / greedy search.

Host-side orchestration only — every arithmetic step is one of the sm_100a kernels behind include/sc_b200.h.
The whole encoder and the whole L-step decode loop are each captured into ONE CUDA graph per (batch, boxes, beam)
configuration, so a batch costs two graph launches and no host synchronisation (the reference does B*beam
``bool(tensor)`` syncs per step, sparse_caption/models/caption_model.py:195-210).

Reference call stack replaced (SURVEY.md section 3.2):
  RelationTransformerModel._sample          sparse_caption/models/relation_transformer.py:390-396
  CachedTransformerBase._generate_captions  sparse_caption/models/transformer.py:471-561
  CaptionModel.batch_beam_search            sparse_caption/models/caption_model.py:30-226
"""
import math
import os
import types
from typing import Dict, Optional

import torch

from . import kernels as K
from . import lib


class ModelCfg:
    """Hyper-parameters the model reads from the reference Config (models/transformer.py:418-437)."""

    FIELDS = ("d_model", "dim_feedforward", "num_layers", "num_heads", "max_seq_length", "att_feat_size", "vocab_size",
              "eos_token_id", "bos_token_id", "unk_token_id", "pad_token_id", "share_att_encoder", "share_att_decoder",
              "share_layer_encoder", "share_layer_decoder", "no_box_trigonometric_embedding")
    DEFAULTS = dict(d_model=512, dim_feedforward=2048, num_layers=6, num_heads=8, max_seq_length=16, att_feat_size=2048,
                    eos_token_id=3, bos_token_id=2, unk_token_id=1, pad_token_id=0, share_att_encoder=None,
                    share_att_decoder=None, share_layer_encoder=None, share_layer_decoder=None,
                    no_box_trigonometric_embedding=False)

    def __init__(self, config=None, **kw):
        for f in self.FIELDS:
            if f in kw:
                v = kw[f]
            elif config is not None and hasattr(config, f):
                v = getattr(config, f)
            elif config is not None and isinstance(config, dict) and f in config:
                v = config[f]
            elif f in self.DEFAULTS:
                v = self.DEFAULTS[f]
            else:
                raise ValueError(f"missing config field `{f}`")
            setattr(self, f, v)
        assert self.d_model % self.num_heads == 0

    def uids(self, which):
        share = self.share_layer_encoder if which == "enc" else self.share_layer_decoder
        return list(share) if share else list(range(self.num_layers))


def _att_parts(share_att):
    """(q, k, v, out) linear indices per share mode (relation_transformer.py:162-176, transformer.py:256-263)."""
    if share_att is None:
        return 0, 1, 2, 3
    if share_att == "kv":
        return 0, 1, 1, 2
    if share_att == "qk":
        return 0, 0, 1, 2
    raise ValueError(f"Invalid `share_att`: {share_att}")


class _Lin:
    """One packed linear: dense weight in the activation dtype and/or CSR, fp32 bias.

    ``norm=(a_2, b_2)``: the LayerNorm in front of this linear (SublayerConnection, transformer.py:345-358) is folded
    into it for the bf16 tensor path: ``wf = (W (.) a_2)`` in bf16, ``ln_c = rowsum(wf)``, ``bias_f = W b_2 + bias``;
    ``ln()`` then consumes the un-normalised bf16 residual stream + its row statistics (sc_linear_ln)."""

    def __init__(self, w, b, adt, backend, csr_threshold, norm=None):
        w = w.detach().float().contiguous()
        self.N, self.K = w.shape
        self.tile_n = 0  # GEMM tile hint (1000 * stages + block_n; 0 = the kernel's own heuristic)
        self.bias = None if b is None else b.detach().float().contiguous()
        self.sparsity = float((w == 0).sum()) / w.numel()
        use_csr = backend == "csr"
        # sliced-ELL (K3b'): the measured winner over the dense tensor-core GEMM at decode sizes from `csr_threshold` up
        # (DESIGN.md, "K3a vs K3b"); its X tile [K][8] fp32 must fit in shared memory
        use_sell = (backend == "sell" or (backend == "auto" and self.sparsity >= csr_threshold)) and self.K * 32 <= 200 * 1024 \
            and self.K % 8 == 0
        # "gs": gather SpMM on the tensor cores (sc_gspmm, bf16); "auto": from `csr_threshold` sparsity up (measured winner table:
        # DESIGN.md "K3a vs K3b")
        use_gs = (backend == "gs" or (backend == "auto" and self.sparsity >= csr_threshold)) and adt == torch.bfloat16 and self.K % 8 == 0
        use_sell = use_sell and not use_gs
        self.csr = K.CsrWeight(w, adt) if use_csr else None
        self.sell = K.SellWeight(w, adt) if use_sell else None
        self.gs = K.GsWeight(w) if use_gs else None
        use_csr = use_csr or use_sell or use_gs  # "not on the dense path"
        self.w = None
        if not use_csr:
            self.w = K.cast_bf16(w) if adt == torch.bfloat16 else w
        self.wf = None
        if norm is not None and not use_csr and adt == torch.bfloat16 and self.K % 32 == 0:
            a2, b2 = norm
            self.wf = (w * a2.float()[None, :]).to(torch.bfloat16).contiguous()
            self.ln_c = self.wf.float().sum(1).contiguous()
            self.bias_f = (w @ b2.float() + (self.bias if self.bias is not None else 0.0)).contiguous()

    def ln(self, xb, stats, out, relu=False, tile_n=None):
        """out = act(LayerNorm(x) W^T + b) from the bf16 copy of x and its chunk statistics."""
        return K.linear_ln(xb, self.wf, self.bias_f, out=out, relu=relu, ln_stats=stats, ln_c=self.ln_c,
                           tile_n=self.tile_n if tile_n is None else tile_n)

    def produce(self, x, out, out_bf16, stats, residual=None, relu=False, tile_n=None):
        """out (fp32 residual stream) = act(x W^T + b) + residual, plus its bf16 copy and chunk statistics."""
        return K.linear_ln(x, self.w, self.bias, residual=residual, relu=relu, out=out, out_bf16=out_bf16, stats_out=stats,
                           tile_n=self.tile_n if tile_n is None else tile_n)

    def __call__(self, x, out, residual=None, relu=False, tile_n=None):
        if self.gs is not None:
            return K.gspmm(x, self.gs, self.bias, residual=residual, relu=relu, out=out)
        if self.sell is not None:
            return K.sell_spmm(x, self.sell, self.bias, residual=residual, relu=relu, out=out)
        if self.csr is not None:
            return K.csr_spmm(x, self.csr, self.bias, residual=residual, relu=relu, out=out)
        return K.linear(x, self.w, self.bias, residual=residual, relu=relu, out=out, tile_n=self.tile_n if tile_n is None else tile_n)


class _Norm:
    def __init__(self, sd, prefix):
        self.a = sd[prefix + ".a_2"].detach().float().contiguous()
        self.b = sd[prefix + ".b_2"].detach().float().contiguous()

    def __call__(self, x, out):
        return K.layernorm(x, self.a, self.b, out=out)


class BeamState:
    def __init__(self, B, beam, L, dev):
        R = B * beam
        i32, f32 = dict(dtype=torch.int32, device=dev), dict(dtype=torch.float32, device=dev)
        self.seq = [torch.zeros(R, L, **i32) for _ in range(2)]
        self.lp = [torch.zeros(R, L, **f32) for _ in range(2)]
        self.anc = [torch.zeros(R, L, **i32) for _ in range(2)]
        self.sum = torch.zeros(R, **f32)
        self.tokens = torch.zeros(R, **i32)
        self.done_seq = torch.zeros(B, beam, L, **i32)
        self.done_lp = torch.zeros(B, beam, L, **f32)
        self.done_p = torch.zeros(B, beam, dtype=torch.float64, device=dev)
        self.done_count = torch.zeros(B, **i32)
        self.rows = torch.arange(R, **i32).unsqueeze(1).expand(R, L).contiguous()
        self.ws = torch.zeros(K.beam_step_workspace_bytes(B, beam), dtype=torch.uint8, device=dev)  # sc_beam_step scratch

    def reset(self, bos, pad):
        self.anc[0].copy_(self.rows)
        self.sum.zero_()
        self.tokens.fill_(bos)
        self.done_count.zero_()
        self.done_seq.fill_(pad)
        self.done_lp.zero_()
        self.done_p.zero_()
        return self


def shared_history(states):
    """Points the seq ping-pong buffers of a diverse beam search's G group BeamStates into one int32 [G, 2, rows, L] tensor,
    from which each group's beam step reads the earlier groups' tokens (sc_beam_step_diverse); returns it."""
    seq = states[0].seq[0]
    hist = torch.zeros(len(states), 2, *seq.shape, dtype=torch.int32, device=seq.device)
    for g, st in enumerate(states):
        st.seq = [hist[g, 0], hist[g, 1]]
    return hist


class GreedyState:
    def __init__(self, R, L, dev):
        i32 = dict(dtype=torch.int32, device=dev)
        self.seq = torch.zeros(R, L, **i32)
        self.lp = torch.zeros(R, L, dtype=torch.float32, device=dev)
        self.tokens = torch.zeros(R, **i32)
        self.unfinished = torch.ones(R, **i32)
        self.live = torch.zeros(L, **i32)
        self.anc = torch.arange(R, **i32).unsqueeze(1).expand(R, L).contiguous()

    def reset(self, bos, pad):
        self.seq.fill_(pad)
        self.lp.zero_()
        self.tokens.fill_(bos)
        self.unfinished.fill_(1)
        self.live.zero_()


class OrtEngine:
    """Packed weights + workspaces + CUDA graphs for one model.

    ``state_dict``: dense-class parameter names (``relation_transformer``); masked weights must already be folded
    (``prune.fold_masks`` does that on device).  ``precision``: "bf16" (tcgen05 tensor-core GEMMs, bf16 activations)
    or "fp32" (fp32 verification kernels).  ``sparse_backend``: "dense" | "csr" | "sell" | "auto" for the decoder linears
    (K3a vs K3b / K3b'; "auto" = sliced-ELL for tensors at or above ``csr_threshold`` sparsity); the encoder always runs
    the dense tensor path (M = B*N rows is large).
    """

    def __init__(self, state_dict: Dict[str, torch.Tensor], cfg: ModelCfg, *, precision="bf16", sparse_backend="dense",
                 csr_threshold=0.995, device="cuda", use_graphs=True, no_history=False, ln_fold=False, fuse_topk=True,
                 dec_tiles=None, dec_ctas=None):
        if not torch.cuda.is_available():
            raise RuntimeError("OrtEngine needs a CUDA device: the B200 path has no CPU fallback")
        lib.load()
        assert precision in ("bf16", "fp32")
        self.cfg = cfg
        self.dev = lib.resolve_device(device)
        self.adt = torch.bfloat16 if precision == "bf16" else torch.float32
        self.precision = precision
        self.use_graphs = use_graphs
        # generator GEMM fused with the beam step's row pass (sc_linear_topk + sc_beam_step_partials): the [R, V] fp32
        # logits (61 MB per step at 512 images x beam 3) are never written or re-read
        self.fuse_topk = bool(fuse_topk)
        self.no_history = no_history  # reference quirk Q1 (relation_transformer_prune never enables its KV cache)
        self.sparse_backend = sparse_backend
        sd = {k: v.to(self.dev) for k, v in state_dict.items() if torch.is_tensor(v) and not v.is_sparse}
        sd.update({k: v.to(self.dev).to_dense() for k, v in state_dict.items() if torch.is_tensor(v) and v.is_sparse})
        d, adt = cfg.d_model, self.adt

        # LayerNorm folding (bf16 tensor path only): every pre-norm is absorbed by the GEMM that consumes it
        self.ln_fold = bool(ln_fold) and adt == torch.bfloat16 and d % 32 == 0

        def lin(prefixes, backend="dense", norm=None):
            ws = torch.cat([sd[p + ".weight"].float() for p in prefixes], 0)
            bs = torch.cat([sd[p + ".bias"].float() for p in prefixes], 0)
            nrm = (sd[norm + ".a_2"], sd[norm + ".b_2"]) if (norm and self.ln_fold) else None
            return _Lin(ws, bs, adt, backend, csr_threshold, norm=nrm)

        def layer(p, share_att, backend, n_norms):
            """The entries both stacks share: self-attention projections (qkv fused per share mode, then o), feed-forward and
            the sublayer LayerNorms n0 .. n{n_norms-1}; the last one feeds ff1."""
            qi, ki, vi, oi = _att_parts(share_att)
            parts = sorted(set((qi, ki, vi)))
            e = {"qkv": lin([f"{p}.self_attn.linears.{j}" for j in parts], backend, norm=f"{p}.sublayer.0.norm"),
                 "offs": tuple(parts.index(j) * d for j in (qi, ki, vi)),
                 "ld": len(parts) * d,
                 "o": lin([f"{p}.self_attn.linears.{oi}"], backend),
                 "ff1": lin([f"{p}.feed_forward.w_1"], backend, norm=f"{p}.sublayer.{n_norms - 1}.norm"),
                 "ff2": lin([f"{p}.feed_forward.w_2"], backend)}
            e.update({f"n{j}": _Norm(sd, f"{p}.sublayer.{j}.norm") for j in range(n_norms)})
            return e

        self.att_embed = lin(["att_embed.0"])
        # ---- encoder (unique modules only; shared layers re-use the pack) ----
        self.enc_uids = cfg.uids("enc")
        self.enc = {}
        for pos, u in enumerate(self.enc_uids):
            if u in self.enc:
                continue
            p = f"model.encoder.layers.{pos}"
            e = layer(p, cfg.share_att_encoder, "dense", 2)
            e["wg_w"] = torch.cat([sd[f"{p}.self_attn.WGs.{j}.weight"].float() for j in range(cfg.num_heads)], 0).contiguous()
            e["wg_b"] = torch.cat([sd[f"{p}.self_attn.WGs.{j}.bias"].float() for j in range(cfg.num_heads)], 0).contiguous()
            self.enc[u] = e
        self.enc_norm = _Norm(sd, "model.encoder.norm")
        # all unique encoder layers' WG rows stacked: the geometry bias of every layer comes from ONE pass over the boxes
        self.enc_slot = {u: i for i, u in enumerate(self.enc)}
        self.wg_w_all = torch.cat([self.enc[u]["wg_w"] for u in self.enc], 0).contiguous()
        self.wg_b_all = torch.cat([self.enc[u]["wg_b"] for u in self.enc], 0).contiguous()
        # tensor-path attention (mma tiles) serves bf16, d_k = 64, N <= 128; fp32 mode keeps the exact fused kernel
        self.split_box_attn = (adt == torch.bfloat16 and d // cfg.num_heads == 64)
        # CTA-per-(image, head) encoder attention (the training forward kernel without saved probabilities): 43 vs 50 us per
        # launch, no difference on the whole step -> the warp-per-(image, head) kernel stays the default
        self.enc_attn_cta = os.environ.get("SC_ENC_ATTN_CTA") == "1"
        # > 0: fused ingest (sc_ingest_f32_bf16: the kernel reads the pinned fp32 features over PCIe and writes the bf16 operand,
        # 51 GB/s vs 45.5 GB/s for cudaMemcpyAsync) with that many CTAs, queued FIFO on one ingest stream.  Off: its CTAs sit on
        # SMs for the ~3 ms a batch takes to cross PCIe, and an SM that hosts one cannot take a full-register GEMM CTA (end to end,
        # ms/step: DMA copy + cast 6.84; ingest with 8 / 16 / 32 CTAs 7.05 / 7.31 / 7.66) - the copy engines are the better tool
        self.zero_copy_ingest = int(os.environ.get("SC_INGEST_CTAS", "0"))
        # ---- decoder ----
        self.dec_uids = cfg.uids("dec")
        self.dec = {}
        qi, ki, vi, oi = _att_parts(cfg.share_att_decoder)
        be = sparse_backend
        for pos, u in enumerate(self.dec_uids):
            if u in self.dec:
                continue
            p = f"model.decoder.layers.{pos}"
            kv_parts = sorted(set((ki, vi)))
            if cfg.share_att_decoder == "qk":
                # cross-attention: key = linears.0(memory), value = linears.1(memory)
                kv_parts = [0, 1]
            e = layer(p, cfg.share_att_decoder, be, 3)
            e.update({
                "cq": lin([f"{p}.src_attn.linears.{qi}"], be, norm=f"{p}.sublayer.1.norm"),
                "ckv": lin([f"{p}.src_attn.linears.{j}" for j in kv_parts], norm="model.encoder.norm"),
                "ckv_offs": tuple(kv_parts.index(j) * d for j in (ki, vi)),
                "ckv_ld": len(kv_parts) * d,
                "co": lin([f"{p}.src_attn.linears.{oi}"], be),
                "apps": self.dec_uids.count(u),
            })
            self.dec[u] = e
        self.dec_norm = _Norm(sd, "model.decoder.norm")
        self.table = sd["model.tgt_embed.0.lut.weight"].float().contiguous()
        L = cfg.max_seq_length
        pe = sd.get("model.tgt_embed.1.pe")
        self.pe = (pe[0, : L + 2] if pe is not None else _positional_encoding(d, L + 2, self.dev)).float().contiguous()
        self.generator = lin(["model.generator.proj"], be, norm="model.decoder.norm")
        # the folded decode path needs every decoder linear on the dense tensor path
        self.fold_dec = self.ln_fold and os.environ.get("SC_LN_FOLD_ENC_ONLY") != "1" and all(
            e[k].w is not None for e in self.dec.values() for k in ("qkv", "o", "cq", "co", "ff1", "ff2")) and self.generator.w is not None
        # decode-GEMM tile hints {"o": 3256, ...} (1000 * stages + block_n).  With >= 8 batches in flight the wide tiles
        # give a little more aggregate throughput than the latency-oriented 64-wide default (scripts/gemm_concurrency.py)
        hints = dict(dec_tiles or {})
        for kv in filter(None, os.environ.get("SC_DEC_TILES", "").split(",")):
            name, val = kv.split("=")
            hints[name] = int(val)
        for name, val in hints.items():
            for e in self.dec.values():
                e[name].tile_n = int(val)
        # throughput regime (several device launches in flight): ``dec_ctas = (wide, narrow)`` sizes the persistent grids of the
        # decode GEMMs per workspace - ~wide CTAs for N > d_model (qkv, ff1), ~narrow for the N = d_model GEMMs with the fp32
        # residual epilogue - by giving each CTA ceil(tiles / target) tiles.  Measured (scripts/gpu_cap_ab*.sh): the 360- / 480-tile
        # GEMMs on 148 CTAs monopolise the SMs for their whole duration; on ~48 CTAs (8 - 10 tiles each, epilogues hidden under the
        # next main loops) the GEMMs of the other launches and their HBM-bound attention kernels run beside them: 4.95 -> 4.75 ms/step
        self.dec_ctas = tuple(dec_ctas) if dec_ctas else None
        self._ingest_stream = None
        self._sample_seed = torch.zeros(1, dtype=torch.int64, device=self.dev)  # re-seeds captured sampling graphs
        self._sample_count = 0
        self._enc_ws = {}
        self._dec_ws = {}
        self._streams = {}
        self._done = {}
        torch.cuda.synchronize(self.dev)

    # ------------------------------------------------------------------------------------------------
    def stream(self, slot):
        """CUDA stream of pipeline slot `slot` (slot 0 = the caller's current stream)."""
        if slot == 0:
            return torch.cuda.current_stream(self.dev)
        if slot not in self._streams:
            self._streams[slot] = torch.cuda.Stream(self.dev)
        return self._streams[slot]

    def _get_enc_ws(self, B, N, masked, slot=0, bf16_in=False):
        key = (B, N, masked, slot, bf16_in)
        if key in self._enc_ws:
            return self._enc_ws[key]
        c, dev, adt = self.cfg, self.dev, self.adt
        d, ff, M = c.d_model, c.dim_feedforward, B * N
        ws = type("EncWs", (), {})()
        ws.B, ws.N, ws.masked, ws.slot = B, N, masked, slot
        # bf16_in: the caller hands bf16 features (half the H2D bytes); they land directly in the GEMM operand buffer
        ws.bf16_in = bool(bf16_in) and adt == torch.bfloat16
        ws.att_in = torch.zeros(M, c.att_feat_size, device=dev) if not ws.bf16_in else None
        ws.att_a = torch.zeros(M, c.att_feat_size, device=dev, dtype=adt) if adt != torch.float32 else ws.att_in
        ws.boxes = torch.zeros(B, N, 4, device=dev)
        ws.att_mask = torch.ones(B, N, device=dev) if masked else None
        ws.x = torch.zeros(M, d, device=dev)
        ws.xn = torch.zeros(M, d, device=dev, dtype=adt)
        ws.qkv = torch.zeros(M, 3 * d, device=dev, dtype=adt)
        ws.att = torch.zeros(M, d, device=dev, dtype=adt)
        ws.hid = torch.zeros(M, ff, device=dev, dtype=adt)
        ws.mem = torch.zeros(M, d, device=dev, dtype=adt)
        ws.memkv = {u: torch.zeros(M, e["ckv_ld"], device=dev, dtype=adt) for u, e in self.dec.items()}
        ws.fold = self.ln_fold and not masked
        if ws.fold:
            ws.xb = torch.zeros(M, d, device=dev, dtype=adt)
            ws.stats = torch.zeros(M, d // 32, 2, device=dev)
        ws.box_bias = (torch.zeros(len(self.enc), B, c.num_heads, N, N, device=dev)
                       if self.split_box_attn and N <= 128 else None)
        ws.tile = {}
        ws.graph = None
        ws.opt_key = None
        self._enc_ws[key] = ws
        return ws

    # ---- the pre-norm sublayers of both stacks: ``ws.fold`` selects the LayerNorm folded into the GEMMs (bf16 copy of the
    # residual stream + its row statistics, written by the previous residual GEMM) or a LayerNorm kernel into ``ws.xn`` ----
    @staticmethod
    def _norm_linear(ws, u, e, norm, name, out, relu=False):
        """out = act(LayerNorm(x) W^T + b) of linear ``e[name]`` behind LayerNorm ``e[norm]``."""
        tile_n = ws.tile.get((u, name))
        if ws.fold:
            e[name].ln(ws.xb, ws.stats, out, relu=relu, tile_n=tile_n)
        else:
            e[norm](ws.x, ws.xn)
            e[name](ws.xn, out, relu=relu, tile_n=tile_n)

    @staticmethod
    def _residual_linear(ws, u, e, name, src):
        """x += src W^T + b of linear ``e[name]``."""
        tile_n = ws.tile.get((u, name))
        if ws.fold:
            e[name].produce(src, ws.x, ws.xb, ws.stats, residual=ws.x, tile_n=tile_n)
        else:
            e[name](src, ws.x, residual=ws.x, tile_n=tile_n)

    def _feed_forward(self, ws, u, e, norm):
        self._norm_linear(ws, u, e, norm, "ff1", ws.hid, relu=True)
        self._residual_linear(ws, u, e, "ff2", ws.hid)

    def _encode_body(self, ws):
        c = self.cfg
        B, N, d, h = ws.B, ws.N, c.d_model, c.num_heads
        dk = d // h
        if ws.att_a is not ws.att_in and not ws.bf16_in:
            K.cast_bf16(ws.att_in, out=ws.att_a)
        if ws.fold:
            self.att_embed.produce(ws.att_a, ws.x, ws.xb, ws.stats, relu=True)
        else:
            self.att_embed(ws.att_a, ws.x, relu=True)
        if ws.att_mask is not None:
            K.mask_rows(ws.x, ws.att_mask.view(-1))
        trig = not c.no_box_trigonometric_embedding
        if ws.box_bias is not None:
            K.box_bias_all(ws.boxes, self.wg_w_all, self.wg_b_all, ws.box_bias, B=B, N=N, layers=len(self.enc), h=h, trig=trig,
                           tensor_cores=True)  # (bf16 path only: ws.box_bias exists when split_box_attn)
        for u in self.enc_uids:
            e = self.enc[u]
            ld = e["ld"]
            qkv = ws.qkv.view(-1)[: B * N * ld].view(B * N, ld)
            self._norm_linear(ws, u, e, "n0", "qkv", qkv)
            qo, ko, vo = e["offs"]
            if ws.box_bias is not None and self.enc_attn_cta:
                # CTA = (image, head) with one warp per 16-query tile sharing the staged K / V (sc_attention_fwd's tensor path
                # without saved probabilities): 3x the warps per SM of the warp-per-(image, head) kernel below
                K.attention_fwd(qkv[:, qo:], qkv[:, ko:], qkv[:, vo:], ws.att, None, G=B, Tq=N, Tk=N, h=h, dk=dk, ldq=ld, ldk=ld,
                                ldv=ld, ldo=d, key_valid=ws.att_mask, bias=ws.box_bias[self.enc_slot[u]])
            elif ws.box_bias is not None:
                K.bias_attention(qkv[:, qo:], qkv[:, ko:], qkv[:, vo:], ws.box_bias[self.enc_slot[u]], ws.att_mask, ws.att,
                                 B=B, N=N, h=h, dk=dk, ldq=ld, ldk=ld, ldv=ld, ldo=d)
            else:
                K.box_attention(qkv[:, qo:], qkv[:, ko:], qkv[:, vo:], ws.boxes, e["wg_w"], e["wg_b"], ws.att_mask, ws.att,
                                B=B, N=N, h=h, dk=dk, ldq=ld, ldk=ld, ldv=ld, ldo=d, trig=trig)
            self._residual_linear(ws, u, e, "o", ws.att)
            self._feed_forward(ws, u, e, "n1")
        if ws.fold:
            for u, e in self.dec.items():
                e["ckv"].ln(ws.xb, ws.stats, ws.memkv[u])
        else:
            self.enc_norm(ws.x, ws.mem)
            for u, e in self.dec.items():
                e["ckv"](ws.mem, ws.memkv[u])

    def encode(self, att_feats, boxes, att_masks=None, slot=0, prefetch=False):
        """Runs att_embed + encoder + cross K/V projections; returns the workspace holding memory K/V.
        ``slot`` selects an independent set of workspaces/graphs so that several batches can be in flight.
        ``prefetch`` (host inputs): the H2D copy runs on the slot's own copy stream and only waits for the previous ENCODER on
        this slot (the only reader of the input buffers), so it overlaps the batch that is still decoding on this slot.
        Measured SLOWER with 5-8 slots in flight (7.10 vs 6.85 ms/step end to end; a variant through staging buffers: 7.08): the
        other slots already hide the copy - off by default (bench.py --prefetch)."""
        B, N, F = att_feats.shape
        masked = att_masks is not None
        host = att_feats.device.type == "cpu"
        if (self.zero_copy_ingest and self.adt == torch.bfloat16 and host and att_feats.dtype == torch.float32
                and att_feats.is_pinned() and att_feats.is_contiguous() and (B * N * F) % 4 == 0):
            # fused ingest: one kernel reads the pinned fp32 features over PCIe and writes the bf16 operand (no fp32 staging, no cast)
            ws = self._get_enc_ws(B, N, masked, slot, True)
            # one engine-wide ingest stream: the ingest kernels of all slots queue FIFO on the PCIe link like DMA copies would
            # (launched on the slots' own streams they all share the link and every encoder starts late)
            if self._ingest_stream is None:
                self._ingest_stream = torch.cuda.Stream(self.dev)
            # (after the current stream: the previous batch of this slot is done with the operand buffer)
            self._fork_join(self._ingest_stream, lambda: K.ingest_f32_bf16(att_feats, ws.att_a.view(-1), ctas=self.zero_copy_ingest),
                            after_stream=torch.cuda.current_stream(self.dev))
            prefetch = False
        else:
            bf16_in = att_feats.dtype == torch.bfloat16 and self.adt == torch.bfloat16
            ws = self._get_enc_ws(B, N, masked, slot, bf16_in)
            dst = ws.att_a if ws.bf16_in else ws.att_in
            src = att_feats.reshape(B * N, F)
            prefetch = prefetch and host and boxes.device.type == "cpu" and not masked
            if prefetch:
                # the input buffers are only read by the encoder graph: the next batch's H2D may start as soon as the previous
                # ENCODER on this slot is done (event), on the slot's copy stream, underneath the previous batch's decode
                if getattr(ws, "copy_stream", None) is None:
                    ws.copy_stream, ws.enc_done = torch.cuda.Stream(self.dev), None
                self._fork_join(ws.copy_stream, lambda: (dst.copy_(src, non_blocking=True), ws.boxes.copy_(boxes, non_blocking=True)),
                                after_event=ws.enc_done)
            else:
                dst.copy_(src, non_blocking=True)
        if not prefetch:
            ws.boxes.copy_(boxes, non_blocking=True)
        if masked:
            ws.att_mask.copy_(att_masks.float(), non_blocking=True)
        self.run_encoder(ws)
        if prefetch:
            ws.enc_done = torch.cuda.Event()
            ws.enc_done.record(torch.cuda.current_stream(self.dev))
        return ws

    def _fork_join(self, side, work, after_stream=None, after_event=None):
        """Runs ``work()`` on stream ``side`` once it has waited for ``after_stream`` / ``after_event`` (when given); the
        current stream waits for it."""
        cur = torch.cuda.current_stream(self.dev)
        if after_stream is not None:
            side.wait_stream(after_stream)
        if after_event is not None:
            side.wait_event(after_event)
        with torch.cuda.stream(side):
            work()
            ready = torch.cuda.Event()
            ready.record(side)
        cur.wait_event(ready)

    def run_encoder(self, ws):
        self._run(ws, lambda: self._encode_body(ws), None)

    def _run(self, ws, body, key, eager=False):
        """Runs a body eagerly, or as the workspace's CUDA graph (captured again when ``key`` changes)."""
        if eager or not self.use_graphs:
            body()
            return
        if ws.graph is None or ws.opt_key != key:
            # warm-up on a side stream (lazy module loading, cudaFuncSetAttribute) before capture
            s = torch.cuda.Stream(self.dev)
            s.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(s):
                body()
            torch.cuda.current_stream(self.dev).wait_stream(s)
            torch.cuda.synchronize(self.dev)
            g = torch.cuda.CUDAGraph()
            before = lib.launch_count
            with torch.cuda.graph(g):
                body()
            ws.graph, ws.opt_key = g, key
            ws.launches = lib.launch_count - before
        ws.graph.replay()

    # ------------------------------------------------------------------------------------------------
    def _new_dec_ws(self, key, kind, R, topk=False):
        """A decode workspace (type name ``kind``) registered under ``key``: the step's activation buffers at R rows, the fused
        generator's top-k records when ``topk``, and the folded LayerNorms' bf16 stream copy and row statistics."""
        c, dev, adt = self.cfg, self.dev, self.adt
        d = c.d_model
        ws = type(kind, (), {})()
        ws.R, ws.fold, ws.tile = R, self.fold_dec, {}
        ws.x = torch.zeros(R, d, device=dev)
        ws.xn = torch.zeros(R, d, device=dev, dtype=adt)
        ws.qkv = torch.zeros(R, 3 * d, device=dev, dtype=adt)
        ws.att = torch.zeros(R, d, device=dev, dtype=adt)
        ws.qc = torch.zeros(R, d, device=dev, dtype=adt)
        ws.hid = torch.zeros(R, c.dim_feedforward, device=dev, dtype=adt)
        ws.logits = torch.zeros(R, c.vocab_size, device=dev)
        ws.topk_part = torch.zeros(R, K.linear_topk_parts(c.vocab_size), 12, device=dev) if topk else None
        if ws.fold:
            ws.xb = torch.zeros(R, d, device=dev, dtype=adt)
            ws.stats = torch.zeros(R, d // 32, 2, device=dev)
        self._dec_ws[key] = ws
        return ws

    def _get_dec_ws(self, B, beam, N, greedy, slot=0, tag=None):
        key = (B, beam, N, greedy, slot, tag)
        if key in self._dec_ws:
            return self._dec_ws[key]
        c, dev = self.cfg, self.dev
        L, R = c.max_seq_length, B * beam
        ws = self._new_dec_ws(key, "DecWs", R, topk=not greedy and self._topk_ok(beam))
        ws.B, ws.beam, ws.N, ws.greedy = B, beam, N, greedy
        ws.cache = {u: (torch.zeros(L * e["apps"], R, c.d_model, device=dev, dtype=self.adt),
                        torch.zeros(L * e["apps"], R, c.d_model, device=dev, dtype=self.adt)) for u, e in self.dec.items()}
        ws.state = GreedyState(R, L, dev) if greedy else BeamState(B, beam, L, dev)
        ws.tile = self._dec_hints(R)
        ws.graph = None
        ws.opt_key = None
        return ws

    def _dec_hints(self, R):
        """{(unique layer, linear): tile hint} of the decode GEMMs at R rows (None: the linear's own hint); see ``dec_ctas``."""
        hints = {}
        if not self.dec_ctas:
            return hints
        for u, e in self.dec.items():
            for name in ("qkv", "o", "cq", "co", "ff1", "ff2"):
                lin = e[name]
                if lin.w is None or lin.tile_n:   # sparse backends / an explicit hint win
                    continue
                hint = decode_grid_hint(R, lin.N, self.cfg.d_model, self.dec_ctas)
                if hint:
                    hints[(u, name)] = hint
        return hints

    def _topk_ok(self, beam):
        """The fused generator + beam row pass serves the dense bf16 tensor path, beam <= 5 (options are checked per call)."""
        g = self.generator
        return (self.fuse_topk and self.adt == torch.bfloat16 and g.w is not None and g.w.dtype == torch.bfloat16 and beam <= 5
                and g.K % 8 == 0)

    def _decode_step(self, ws, enc, t, anc, topk=None):
        """One decode step of every row; ``topk``: candidates per row of the fused generator + top-k records (None: the
        generator writes the logits)."""
        c = self.cfg
        R, d, h, N = ws.R, c.d_model, c.num_heads, ws.N
        if ws.fold:
            K.embed_pe_stats(ws.state.tokens, self.table, self.pe, ws.x, ws.xb, ws.stats, T=1, pos0=t)
        else:
            K.embed_pe(ws.state.tokens, self.table, self.pe, T=1, pos0=t, out=ws.x)
        used = {u: 0 for u in self.dec}
        for u in self.dec_uids:
            e = self.dec[u]
            ld = e["ld"]
            qkv = ws.qkv.view(-1)[: R * ld].view(R, ld)
            self._norm_linear(ws, u, e, "n0", "qkv", qkv)
            qo, ko, vo = e["offs"]
            apps = e["apps"]
            slot = t * apps + used[u]
            used[u] += 1
            ck, cv = ws.cache[u]
            K.self_attn_step(qkv[:, qo:], qkv[:, ko:], qkv[:, vo:], ck, cv, anc, ws.att, R=R, D=d, h=h,
                             n_prev=0 if self.no_history else slot, write_slot=-1 if self.no_history else slot,
                             ldq=ld, ldk=ld, ldv=ld, ldo=d, anc_ld=anc.shape[1], slot_div=apps)
            self._residual_linear(ws, u, e, "o", ws.att)
            self._norm_linear(ws, u, e, "n1", "cq", ws.qc)
            mkv = enc.memkv[u]
            ko2, vo2 = e["ckv_offs"]
            K.cross_attn_step(ws.qc, mkv[:, ko2:], mkv[:, vo2:], enc.att_mask, ws.att, B=ws.B, beam=ws.beam, N=N, D=d, h=h,
                              ldq=d, ldm=e["ckv_ld"], ldo=d)
            self._residual_linear(ws, u, e, "co", ws.att)
            self._feed_forward(ws, u, e, "n2")
        # (the final norm stays a kernel also when the layers' norms are folded: the fused generator + top-k epilogue has no
        # folded-LayerNorm variant, and one LayerNorm per step is 1/19 of them)
        self.dec_norm(ws.x, ws.xn)
        if topk:
            K.linear_topk(ws.xn, self.generator.w, self.generator.bias, ws.topk_part, candidates=topk)
        else:
            self.generator(ws.xn, ws.logits)

    def _bad_endings(self, ws, so):
        """remove_bad_endings (caption_model.py:161-168): the ids as a device tensor held by the workspace, made outside any
        graph capture, so that a captured decode reads live memory on every replay (None when the option is off)."""
        if so.bad is None:
            return None
        if getattr(ws, "bad_ids", None) != so.bad:
            ws.bad_ids, ws.bad_t = so.bad, torch.tensor(so.bad, dtype=torch.int32, device=self.dev)
        return ws.bad_t

    def _beam_step(self, scores, st, t, B, beam, so, bad_t, fused=False, diverse=None):
        """sc_beam_step on one group's log-probs ``scores`` [B*beam, V], or (``fused``) sc_beam_step_partials on its top-k
        records; ``diverse``: (hist, group, diversity_lambda) of a diverse beam search."""
        c = self.cfg
        kw = dict(B=B, beam=beam, V=c.vocab_size, L=c.max_seq_length, eos=c.eos_token_id, pad=c.pad_token_id,
                  penalty_kind=so.kind, penalty_alpha=so.alpha, diverse=diverse)
        if fused:
            K.beam_step_partials(scores, st, t, **kw)
        else:
            K.beam_step(scores, st, t, temperature=so.temperature, constraint=so.constraint,
                        suppress_tok=_suppress_bad(st, bad_t, t), penalized_col=so.pen_col, **kw)

    def _get_diverse_ws(self, B, N, G, bdash, slot):
        """Diverse beam search: one decode workspace + BeamState per group (B*bdash rows each) over one seq history
        (``shared_history``)."""
        key = (B, G * bdash, N, "diverse", G, slot)
        dv = self._dec_ws.get(key)
        if dv is not None:
            return dv
        L = self.cfg.max_seq_length
        dv = type("DiverseWs", (), {})()
        dv.B, dv.G, dv.bdash = B, G, bdash
        dv.groups = [self._get_dec_ws(B, bdash, N, False, slot, tag=("diverse", G, g)) for g in range(G)]
        dv.hist = shared_history([ws.state for ws in dv.groups])
        dv.seq = torch.zeros(B, G * bdash, L, dtype=torch.int32, device=self.dev)
        dv.lp = torch.zeros(B, G * bdash, L, device=self.dev)
        dv.graph = None
        dv.opt_key = None
        self._dec_ws[key] = dv
        return dv

    def _search_body(self, groups, enc, opt, dv=None):
        """batch_beam_search (caption_model.py:30-226) over the workspaces of G = len(groups) groups of beams.  G > 1 (diverse
        beam search, ``dv``, :126-226): global step t = 0 .. L+G-2, group g decodes and steps at its local step t - g while that
        lies in [0, L-1], groups in ascending order; finished beams stay per group and are concatenated group by group into
        ``dv.seq`` / ``dv.lp`` (:221-225)."""
        c = self.cfg
        L, G = c.max_seq_length, len(groups)
        so = search_options(opt)
        bad_t = self._bad_endings(dv or groups[0], so)
        # fused generator + row pass: group g needs its bdash + g*bdash <= beam_size best raw candidates per row
        cands = G * groups[0].beam
        fused = so.fusable and all(ws.topk_part is not None for ws in groups) and self._topk_ok(cands)
        for ws in groups:
            ws.state.reset(c.bos_token_id, c.pad_token_id)
        for t in range(L + G - 1):
            for g, ws in enumerate(groups):
                tau = t - g
                if not 0 <= tau <= L - 1:
                    continue
                st = ws.state
                self._decode_step(ws, enc, tau, st.anc[tau & 1], topk=cands if fused else None)
                self._beam_step(ws.topk_part if fused else ws.logits, st, tau, ws.B, ws.beam, so, bad_t, fused,
                                None if dv is None else (dv.hist, g, so.lam))
        if dv is not None:
            for g, ws in enumerate(groups):
                dv.seq[:, g * dv.bdash:(g + 1) * dv.bdash].copy_(ws.state.done_seq)
                dv.lp[:, g * dv.bdash:(g + 1) * dv.bdash].copy_(ws.state.done_lp)

    def _greedy_body(self, ws, enc, opt):
        c = self.cfg
        L, V = c.max_seq_length, c.vocab_size
        st = ws.state
        st.reset(c.bos_token_id, c.pad_token_id)
        for t in range(L):
            self._decode_step(ws, enc, t, st.anc)
            K.greedy_step(ws.logits, st, t, R=ws.R, V=V, L=L, eos=c.eos_token_id,
                          constraint=opt.get("decoding_constraint", 0))

    def _sample_body(self, ws, enc, opt):
        c = self.cfg
        L, V = c.max_seq_length, c.vocab_size
        st = ws.state
        st.reset(c.bos_token_id, c.pad_token_id)
        for t in range(L):
            self._decode_step(ws, enc, t, st.anc)
            K.sample_step(ws.logits, st, t, R=ws.R, V=V, L=L, eos=c.eos_token_id, constraint=opt.get("decoding_constraint", 0),
                          temperature=opt.get("temperature", 1.0), uniforms=ws.uniforms[t] if ws.uniforms is not None else None,
                          seed=(1 << 63) | self._sample_seed.data_ptr())

    def decode(self, enc, opt):
        """Beam (beam_size > 1), greedy (beam_size == 1) or multinomial (num_random_sample > 0, models/transformer.py:
        507-561) decoding over an encoded batch.  Returns (seq int32 [B,b,L], lp [B,b,L]); b = num_random_sample when sampling.
        ``opt["sample_seed"]`` re-seeds the sampler (default: a counter), ``opt["sample_uniforms"]`` (fp32 [L, B*n], tests)
        replaces the Philox draws.  ``group_size`` G > 1 with beam_size > 1: diverse beam search (``diversity_lambda``,
        default 0.5), b = G * (beam_size // G) beams per image in group-major order."""
        beam = int(opt.get("beam_size", 1))
        n_rand = int(opt.get("num_random_sample", 0))
        if n_rand > 0:
            assert beam < 1, f"Beam size must be < 1, saw {beam}"  # transformer.py:509
            opt = dict(opt)
            seed = opt.pop("sample_seed", None)
            uni = opt.pop("sample_uniforms", None)
            self._sample_count += 1
            self._sample_seed.fill_(int(seed) if seed is not None else 0x5CB200 + self._sample_count)
            ws = self._get_dec_ws(enc.B, n_rand, enc.N, True, enc.slot, tag="sample")
            ws.uniforms = None
            if uni is not None:
                ws.uniforms = uni.to(self.dev, torch.float32).contiguous()
                assert tuple(ws.uniforms.shape) == (self.cfg.max_seq_length, enc.B * n_rand)
            opt_key = (id(enc), "sample", uni is not None, tuple(sorted((k, str(v)) for k, v in opt.items())))
            self._run(ws, lambda: self._sample_body(ws, enc, opt), opt_key, eager=uni is not None)
            return ws.state.seq.view(enc.B, n_rand, -1), ws.state.lp.view(enc.B, n_rand, -1)
        assert beam <= self.cfg.vocab_size
        opt_key = (id(enc), tuple(sorted((k, str(v)) for k, v in opt.items())))
        if beam == 1:
            ws = self._get_dec_ws(enc.B, beam, enc.N, True, enc.slot)
            self._run(ws, lambda: self._greedy_body(ws, enc, opt), opt_key)
            return ws.state.seq.view(enc.B, 1, -1), ws.state.lp.view(enc.B, 1, -1)
        if int(opt.get("group_size", 1)) > 1:
            G, bdash, _ = diverse_groups(opt)
            dv = self._get_diverse_ws(enc.B, enc.N, G, bdash, enc.slot)
            self._run(dv, lambda: self._search_body(dv.groups, enc, opt, dv), opt_key)
            return dv.seq, dv.lp
        ws = self._get_dec_ws(enc.B, beam, enc.N, False, enc.slot)
        self._run(ws, lambda: self._search_body([ws], enc, opt), opt_key)
        return ws.state.done_seq, ws.state.done_lp

    def teacher_force(self, enc, tokens, beam=1, out=None):
        """Incremental (KV-cached) decoding along GIVEN token paths: row r = image r // beam feeds BOS, tokens[r, 0], ...,
        tokens[r, L-2] and every step's full log-softmax is returned (fp32 [L, B*beam, V]).  Each row keeps its own KV
        history (identity ancestors) and shares its image's cross K/V - the per-step arithmetic of ``decode`` without the
        search, i.e. ``get_logprobs_state`` (relation_transformer.py:374-387) unrolled over a fixed path.  Used by the
        parity tests at the BASELINE sizes and by ``get_logprobs_state``-style callers that score given captions."""
        c = self.cfg
        L, V = c.max_seq_length, c.vocab_size
        R = enc.B * beam
        tokens = tokens.to(self.dev).to(torch.int32).reshape(R, tokens.shape[-1])
        ws = self._get_dec_ws(enc.B, beam, enc.N, True, enc.slot, tag="force")
        st = ws.state
        st.reset(c.bos_token_id, c.pad_token_id)
        steps = min(L, tokens.shape[1] + 1)
        if out is None:
            out = torch.empty(steps, R, V, device=self.dev)
        for t in range(steps):
            if t > 0:
                st.tokens.copy_(tokens[:, t - 1])
            self._decode_step(ws, enc, t, st.anc)
            K.logsoftmax_nll(ws.logits, logprobs=out[t])
        return out

    # ---- step-wise entry points (get_logprobs_state / batch_beam_search of the reference) over an explicit state ----
    def logprobs_step(self, it, memory, att_mask, caches, t):
        """One ``get_logprobs_state`` step (relation_transformer.py:374-387).  ``it`` [R] tokens; ``memory`` [R, N, d] encoder
        output (final norm applied); ``att_mask`` [R, 1, N] / [R, N] / None; ``caches`` None at t = 0 or, per unique decoder
        layer, (self K [slots, R, d], self V [slots, R, d], cross K|V [1, R, N * ld]) - row dimension at dim 1, so the caller
        may reorder / repeat beams with ``x[:, ix]``.  Returns (log-softmax fp32 [R, V], caches)."""
        c = self.cfg
        R = it.numel()
        N = memory.shape[1]
        d, L = c.d_model, c.max_seq_length
        assert 0 <= t <= L, f"step {t} beyond max_seq_length {L}"
        ws = self._dec_ws.get(("step", R, N))
        if ws is None:
            ws = self._new_dec_ws(("step", R, N), "StepWs", R)
            ws.B, ws.beam, ws.N = R, 1, N   # every row carries its own memory K/V
            ws.state = type("Tok", (), {})()
            ws.state.tokens = torch.zeros(R, dtype=torch.int32, device=self.dev)
            ws.anc = torch.arange(R, dtype=torch.int32, device=self.dev).unsqueeze(1).expand(R, L * max(e["apps"] for e in self.dec.values())).contiguous()
        uids = list(self.dec)
        if caches is None:
            mem = memory.reshape(-1, d)
            mem = (K.cast_bf16(mem.float().contiguous()) if self.adt == torch.bfloat16 else mem.float().contiguous()) if mem.dtype != self.adt else mem.contiguous()
            caches = []
            for u in uids:
                e = self.dec[u]
                slots = L * e["apps"] + e["apps"]  # (+ one spare step: the reference calls the model once more after the last step)
                ckv = torch.empty(1, memory.shape[0], N * e["ckv_ld"], device=self.dev, dtype=self.adt)
                e["ckv"](mem, ckv.view(-1, e["ckv_ld"]))
                caches += [torch.zeros(slots, memory.shape[0], d, device=self.dev, dtype=self.adt),
                           torch.zeros(slots, memory.shape[0], d, device=self.dev, dtype=self.adt), ckv]
        caches = list(caches)
        rows = caches[0].shape[1]
        if rows != R:  # first beam step: every cached row is repeated `beam` times (transformer.py:240-252)
            assert R % rows == 0 and rows < R, (rows, R)
            caches = [x.repeat_interleave(R // rows, 1) for x in caches]
        caches = [x.contiguous() for x in caches]
        enc = type("StepEnc", (), {})()
        enc.memkv = {u: caches[3 * i + 2].view(R * N, self.dec[u]["ckv_ld"]) for i, u in enumerate(uids)}
        m = None
        if att_mask is not None:
            m = att_mask.reshape(R, N).float().contiguous()
            if bool((m != 0).all()):
                m = None
        enc.att_mask = m
        ws.cache = {u: (caches[3 * i], caches[3 * i + 1]) for i, u in enumerate(uids)}
        ws.state.tokens.copy_(it.reshape(-1).to(torch.int32))
        self._decode_step(ws, enc, t, ws.anc)
        out = torch.empty(R, c.vocab_size, device=self.dev)
        K.logsoftmax_nll(ws.logits, logprobs=out)
        return out, caches

    def beam_search_stepwise(self, init_state, init_logprobs, args, opt, get_logprobs_state):
        """``batch_beam_search`` (caption_model.py:30-226) driven step by step: sc_beam_step ranks the b*V candidates, keeps
        the beam / finished-beam state on the device and yields the parent rows; the model state is reordered with
        ``state[i][:, parents]`` and advanced through ``get_logprobs_state`` - the reference's own control flow.  With
        group_size G > 1 (diverse beam search) every group has its own state list cloned from ``init_state``, its share of
        ``args`` (row r of the B*b repeated rows goes to group r % G, model_utils.split_tensors) and its own staggered
        steps (sc_beam_step_diverse).  Returns done_beams [B][G*bdash] dicts {seq, logps, unaug_p, p}, group-major."""
        c = self.cfg
        beam = int(opt.get("beam_size", 10))
        G, bdash, _ = diverse_groups(opt) if int(opt.get("group_size", 1)) > 1 else (1, beam, 0.0)
        L, V = c.max_seq_length, c.vocab_size
        B = init_logprobs.shape[0]
        sts = [BeamState(B, bdash, L, self.dev).reset(c.bos_token_id, c.pad_token_id) for _ in range(G)]
        hist = shared_history(sts) if G > 1 else None
        so = search_options(opt)
        bad_t = None if so.bad is None else torch.tensor(so.bad, dtype=torch.int32, device=self.dev)
        args = list(args)
        group_args = [[None if a is None else a.reshape(a.shape[0] // G, G, *a.shape[1:])[:, g] for a in args] for g in range(G)]
        logits, state = [], []
        for g in range(G):
            lg = torch.zeros(B * bdash, V, device=self.dev)
            lg.view(B, bdash, V)[:, 0] = init_logprobs.float()   # local step 0: only beam 0 of an image is expanded
            logits.append(lg)
            state.append([x.clone() for x in init_state])
        for t in range(L + G - 1):
            for g in range(G):
                tau = t - g
                if not 0 <= tau <= L - 1:
                    continue
                st = sts[g]
                self._beam_step(logits[g], st, tau, B, bdash, so, bad_t, diverse=None if hist is None else (hist, g, so.lam))
                parents = st.anc[(tau + 1) & 1][:, tau].long()      # row each new beam descends from (b*bdash + parent)
                if tau == 0:
                    parents = parents // bdash                       # the first state holds one row per image
                state[g] = [x[:, parents] for x in state[g]]
                logprobs, state[g] = get_logprobs_state(st.tokens.long(), *(group_args[g] + [state[g]]))
                logits[g] = logprobs.contiguous()                    # (sc_beam_step re-normalises: log_softmax is idempotent)
        out = [[] for _ in range(B)]
        for st in sts:
            done_seq, done_lp, done_p = st.done_seq.long().cpu(), st.done_lp.cpu(), st.done_p.cpu()
            for b in range(B):
                for v in range(bdash):
                    n = int((done_seq[b, v] != c.pad_token_id).sum())
                    eos = (done_seq[b, v] == c.eos_token_id).nonzero()
                    if eos.numel():
                        n = int(eos[0]) + 1
                    out[b].append({"seq": done_seq[b, v, :n].to(self.dev), "logps": done_lp[b, v, :n].to(self.dev),
                                   "unaug_p": float(done_lp[b, v, :n].sum()), "p": float(done_p[b, v])})
        return out

    # ---- batch pipelining: slot s owns a stream + workspaces + graphs; batches in different slots overlap on the GPU
    # (the decode loop is a chain of ~70 short dependent kernels per step that leaves most SMs idle; a second
    # batch fills them, and its H2D copy hides behind the first batch's compute) ----
    def submit(self, att_feats, boxes, att_masks=None, opt=None, slot=0, out=None, prefetch=False):
        """Enqueue encode + decode of one batch on slot `slot` without waiting.  ``out``: optional pinned host tensors
        (seq int32 [B,b,L], lp fp32 [B,b,L]) that receive the result asynchronously.  Returns (seq, lp) device views
        that are valid after ``wait(slot)``.  ``opt`` may be a LIST of option dicts: several decodes over ONE encoder pass
        (SCST: a beam / multinomial rollout plus the greedy baseline, utils/training.py:216-237); ``out`` and the result are
        then lists."""
        many = isinstance(opt, (list, tuple))
        opts = [dict(o or {}) for o in (opt if many else [opt])]
        outs = out if many else [out]
        cur = torch.cuda.current_stream(self.dev)
        st = self.stream(slot)
        if st is not cur:
            st.wait_stream(cur)
        res = []
        with torch.cuda.stream(st):
            enc = self.encode(att_feats, boxes, att_masks, slot=slot, prefetch=prefetch)
            for i, o in enumerate(opts):
                seq, lp = self.decode(enc, o)
                if outs is not None and outs[i] is not None:
                    outs[i][0].copy_(seq, non_blocking=True)
                    outs[i][1].copy_(lp, non_blocking=True)
                res.append((seq, lp))
            ev = torch.cuda.Event()
            ev.record(st)
        self._done[slot] = ev
        return res if many else res[0]

    def wait(self, slot=None, host=False):
        """Make the current stream (or the host when ``host``) wait for slot `slot` (all slots when None)."""
        for s, ev in list(self._done.items()):
            if slot is None or s == slot:
                if host:
                    ev.synchronize()
                else:
                    torch.cuda.current_stream(self.dev).wait_event(ev)

    def sample(self, att_feats, boxes, att_masks=None, opt=None):
        """Drop-in for ``model(att_feats=..., boxes=..., att_masks=..., opt=..., mode="sample")``:
        returns (seq int64 [B,b,L], seq_logprobs fp32 [B,b,L]) on the device."""
        opt = dict(opt or {})
        if att_masks is not None:
            # clip_att (relation_transformer.py:398-405): host-side length, no device sync for CPU masks
            max_len = int(att_masks.long().sum(1).max())
            att_feats, boxes, att_masks = att_feats[:, :max_len], boxes[:, :max_len], att_masks[:, :max_len]
        enc = self.encode(att_feats, boxes, att_masks)
        seq, lp = self.decode(enc, opt)
        return seq.long(), lp.clone()


def decode_grid_hint(rows, n_out, d_model, dec_ctas):
    """Tile hint (10^7 * tiles per persistent CTA + 3256: 256-wide tiles) that holds the persistent grid of a decode GEMM with
    ``rows`` x ``n_out`` outputs to about ``dec_ctas[0]`` CTAs (N > d_model: qkv, ff1) or ``dec_ctas[1]`` (the N <= d_model GEMMs
    with the fp32 residual epilogue); 0 when one tile per CTA already stays below the target (small batches: the kernel's own
    heuristic)."""
    tiles = -(-rows // 128) * -(-n_out // 256)
    target = dec_ctas[1] if n_out <= d_model else dec_ctas[0]
    tpc = -(-tiles // max(1, target))
    return min(tpc, 200) * 10000000 + 3256 if tpc >= 2 else 0


MAX_GROUP_BEAMS = 8  # beams per group: the beam-step kernel's per-image limit


def diverse_groups(opt):
    """(G, bdash, diversity_lambda) of a diverse beam search (caption_model.py:114-123: bdash = beam_size // group_size beams
    per group, diversity_lambda default 0.5).  ValueError when a group would hold no beam or more than the kernel serves."""
    beam, G = int(opt.get("beam_size", 10)), int(opt.get("group_size", 1))
    bdash = beam // G if G > 0 else 0
    if bdash < 1 or bdash > MAX_GROUP_BEAMS:
        raise ValueError(f"diverse beam search: beam_size={beam} // group_size={G} = {bdash} beams per group; "
                         f"it must lie in [1, {MAX_GROUP_BEAMS}]")
    if (G - 1) * bdash > 256:
        raise ValueError(f"diverse beam search: (group_size - 1) * (beam_size // group_size) = {(G - 1) * bdash} "
                         f"earlier-group beams; at most 256")
    return G, bdash, float(opt.get("diversity_lambda", 0.5))


def _suppress_bad(st, bad_t, t):
    """remove_bad_endings at step t > 0: int32 [rows], 0 where the row's previous token (the token just fed) is a bad ending
    (token 0 may not follow it), -1 elsewhere; None when the option is off."""
    if bad_t is None or t == 0:
        return None
    return torch.where(torch.isin(st.tokens, bad_t), 0, -1).to(torch.int32)


def search_options(opt):
    """The beam-step options of a search (caption_model.py:114-172): length penalty kind and alpha, the column suppressed by
    suppress_UNK (``pen_col``), temperature, decoding constraint, the sorted bad-ending ids (None: off), the diversity lambda,
    and whether the fused generator + top-k row pass can serve them (temperature 1, no constraint, no bad endings, no
    suppressed column)."""
    kind, alpha = _parse_penalty(opt.get("length_penalty", ""))
    bad = opt.get("bad_endings_ix")
    so = types.SimpleNamespace(kind=kind, alpha=alpha, pen_col=int(opt.get("penalized_col", -1)),
                               temperature=float(opt.get("temperature", 1.0)), constraint=opt.get("decoding_constraint", 0),
                               bad=sorted(int(i) for i in bad) if bad else None, lam=float(opt.get("diversity_lambda", 0.5)))
    so.fusable = so.temperature == 1.0 and not so.constraint and so.bad is None and so.pen_col < 0
    return so


def _parse_penalty(s):
    if not s:
        return 0, 0.0
    kind, alpha = s.split("_")
    return {"wu": 1, "avg": 2}[kind], float(alpha)


def _positional_encoding(d_model, max_len, dev):
    pe = torch.zeros(max_len, d_model)
    position = torch.arange(0, max_len).unsqueeze(1).float()
    div_term = torch.exp(torch.arange(0, d_model, 2).float() * -(math.log(10000.0) / d_model))
    pe[:, 0::2] = torch.sin(position * div_term)
    pe[:, 1::2] = torch.cos(position * div_term)
    return pe.to(dev)
