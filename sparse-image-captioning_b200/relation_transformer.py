"""Drop-in model classes for the ORT / ACORT hot path — mirrors the public surface of
sparse_caption/models/{__init__,caption_model,transformer,relation_transformer,relation_transformer_prune}.py.

* ``get_model("relation_transformer")(config)`` / ``get_model("relation_transformer_prune")(config)`` build modules whose
  parameter names equal the reference's (``model.encoder.layers.0.self_attn.WGs.3.weight_pruning_mask`` ...), so
  reference checkpoints load with ``strict=True`` (SURVEY.md section 8b).
* ``model(att_feats=, boxes=, seqs=, att_masks=)`` returns teacher-forcing log-probs ``[B*S, T, V]`` WITH an autograd
  graph: every module of the tree has a kernel-backed ``forward`` (autograd_ops.py), so the reference training loop
  ``loss.backward(); clip_gradient(); optimizer.step()`` (scripts/train_n_prune_transformer.py:136-153) and SCST's
  teacher-forced re-scoring run unmodified, for any weight-sharing pattern (ACORT ``share_att_*`` / ``share_layer_*``).
* ``model(att_feats=, boxes=, att_masks=, opt=, mode="sample")`` returns ``(seq [B,b,L] int64, seq_logprobs [B,b,L])``
  from the fused inference engine (OrtEngine: CUDA graphs, per-image cross K/V, parent-pointer KV cache).
* ``get_logprobs_state`` / ``batch_beam_search`` are the step-wise entry points of the reference
  (relation_transformer.py:374-387, caption_model.py:30-226) over the same decode kernels with an explicit state list.
* ``trainer()`` is the fused SMP training engine (trainer.OrtTrainer) - the fast path for the non-shared ORT.

There is no PyTorch arithmetic to fall back to: calling a model that lives on the CPU raises.
"""
import logging
import math
from argparse import ArgumentParser, _ArgumentGroup
from typing import Any, Union

import torch
from torch import nn

from . import autograd_ops as A
from . import kernels as K
from . import masked_layer, prune
from .engine import ModelCfg, OrtEngine
from .masked_layer import MaskedEmbedding, MaskedLinear
from .prune import PruningMixin

logger = logging.getLogger(__name__)

MODEL_REGISTRY = {}


def register_model(name):
    """Same decorator contract as sparse_caption/models/__init__.py:16-36."""

    def deco(cls):
        if name.lower() in MODEL_REGISTRY:
            raise ValueError(f"Cannot register duplicate model: `{name}`.")
        MODEL_REGISTRY[name.lower()] = cls
        return cls

    return deco


def get_model(name: str) -> Any:
    try:
        return MODEL_REGISTRY[name.lower()]
    except KeyError:
        raise ValueError(f"Model specified `{name}` is invalid. Available options are: \n" + "\n".join(MODEL_REGISTRY))


def str_to_none(v):
    """argparse type of the reference's ``--share_att_*`` flags (utils/config.py): "none" / "" -> None."""
    if v is None or str(v).lower() in ("none", ""):
        return None
    return str(v)


def str_to_sequence(v):
    """argparse type of ``--share_layer_*``: "0,0,1,1" -> (0, 0, 1, 1); "none" -> None."""
    if v is None or isinstance(v, (tuple, list)):
        return v
    if str(v).lower() in ("none", ""):
        return None
    return tuple(int(x) for x in str(v).split(","))


def repeat_tensors(n, x, dim=0):
    """utils/model_utils.py:34-47."""
    if torch.is_tensor(x):
        return torch.repeat_interleave(x, repeats=n, dim=dim)
    if isinstance(x, (list, tuple)):
        return [repeat_tensors(n, v, dim) for v in x]
    return x


# ---- kernel-backed building blocks (names follow the reference module tree) ------------------------------------------
def _apply_linear(layer, x, relu=False):
    """nn.Linear / MaskedLinear through sc_linear (mask in the operand prologue)."""
    prec = masked_layer.get_precision()
    if isinstance(layer, MaskedLinear):
        return A.masked_linear(x, layer.weight, layer.weight_pruning_mask, layer.bias, layer.mask_mode(),
                               layer.bypass_sigmoid_grad or layer.mask_type not in prune.SUPER_MASKS, prec, relu=relu)
    return A.linear(x, layer.weight, layer.bias, prec, relu=relu)


class LayerNorm(nn.Module):
    """a_2 * (x - mean) / (std_unbiased + eps) + b_2 (transformer.py:329-341)."""

    def __init__(self, features, eps=1e-6):
        super().__init__()
        self.a_2 = nn.Parameter(torch.ones(features))
        self.b_2 = nn.Parameter(torch.zeros(features))
        self.eps = eps

    def forward(self, x):
        return A.layer_norm(x, self.a_2, self.b_2, self.eps)


class SublayerConnection(nn.Module):
    def __init__(self, size, dropout):
        super().__init__()
        self.norm = LayerNorm(size)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x, sublayer):
        return x + A.dropout(sublayer(self.norm(x)), self.dropout.p, self.training)


def _linear(mask, i, o):
    return MaskedLinear(i, o, mask[0], mask[1]) if mask else nn.Linear(i, o)


def _key_mask(mask, B, Tq, Tk):
    """Reference attention masks -> (key_valid fp32 [B, Tk] | None, causal_T).  [B,1,Tk] = key padding (encoder / cross
    attention); [B,Tq,Tk] = padding & subsequent_mask (decoder self-attention, relation_transformer.py:356-361)."""
    if mask is None:
        return None, 0
    m = mask.reshape(B, -1, Tk)
    if m.shape[1] == 1:
        return m[:, 0].float().contiguous(), 0
    assert m.shape[1] == Tq == Tk, f"unsupported attention mask shape {tuple(mask.shape)}"
    # the last query row of (padding & lower-triangular) is the padding mask itself
    return m[:, -1].float().contiguous(), Tq


def _heads(x, h):
    """[B, T, h*dk] -> [B, h, T, dk] (the reference's cache layout)."""
    B, T, d = x.shape
    return x.view(B, T, h, d // h).transpose(1, 2)


def _rows(x):
    """[B, h, T, dk] -> [B*T, h*dk]."""
    B, h, T, dk = x.shape
    return x.transpose(1, 2).reshape(B * T, h * dk)


class MultiHeadedAttention(nn.Module):
    """transformer.py:214-295, including the incremental-decoding cache protocol (``cache`` = [K, V] as [B, h, T, d_k],
    ``cache_size``, batch-repeat of the cache on the first beam step, cross-attention re-use, self-attention concat)."""

    def __init__(self, h, d_model, dropout=0.1, self_attention=False, share_att=None, mask=None):
        super().__init__()
        assert d_model % h == 0
        self.d_k = d_model // h
        self.h = h
        self.self_attention = self_attention
        assert share_att in (None, "kv", "qk"), f"Invalid `share_att`: {share_att}"
        self.share_att = share_att
        self.linears = nn.ModuleList([_linear(mask, d_model, d_model) for _ in range(3 if share_att else 4)])
        self.dropout = nn.Dropout(p=dropout)
        self.cache = [None, None]
        self.cache_size = 2

    def forward(self, query, key, value, mask=None):
        B, Tq = query.shape[:2]
        h = self.h
        q = _apply_linear(self.linears[0], query)
        if torch.is_tensor(self.cache[0]) and self.cache[0].size(0) != key.size(0):
            cb = self.cache[0].size(0)
            assert cb < key.size(0) and key.size(0) % cb == 0, (self.cache[0].shape, key.shape)
            self.cache = repeat_tensors(key.size(0) // cb, self.cache)
        if not self.self_attention and torch.is_tensor(self.cache[0]):
            k4, v4 = self.cache  # encoder-attention re-uses its projections
        else:
            if self.share_att == "qk":
                k = _apply_linear(self.linears[0], key)
                v = _apply_linear(self.linears[1], value)
            else:
                k = _apply_linear(self.linears[1], key)
                v = k if self.share_att else _apply_linear(self.linears[2], value)
            k4, v4 = _heads(k, h), _heads(v, h)
        if self.self_attention and torch.is_tensor(self.cache[0]):
            k4 = torch.cat((self.cache[0], k4), dim=2)
            v4 = torch.cat((self.cache[1], v4), dim=2)
            mask = None
        if getattr(self, "incremental_decoding", False):
            self.cache = [k4, v4]
        Tk = k4.shape[2]
        kv, causal = _key_mask(mask, B, Tq, Tk)
        out, _ = A.attention(q.reshape(B * Tq, -1), _rows(k4), _rows(v4), G=B, Tq=Tq, Tk=Tk, h=h, key_valid=kv, causal_T=causal,
                             p=self.dropout.p, training=self.training, precision=masked_layer.get_precision())
        return _apply_linear(self.linears[-1], out.view(B, Tq, -1))

    @staticmethod
    def attention(query, key, value, mask=None, dropout=None):
        """'Scaled Dot Product Attention' on [B, h, T, d_k] tensors (transformer.py:285-295) -> (output, p_attn)."""
        B, h, Tq, dk = query.shape
        Tk = key.shape[2]
        kv, causal = _key_mask(mask, B, Tq, Tk)
        p = dropout.p if (dropout is not None and dropout.training) else 0.0
        out, probs = A.attention(_rows(query), _rows(key), _rows(value), G=B, Tq=Tq, Tk=Tk, h=h, key_valid=kv, causal_T=causal, p=p,
                                 training=p > 0, precision=masked_layer.get_precision())
        return out.view(B, Tq, h, dk).transpose(1, 2), probs


class CachedMultiHeadedAttention(MultiHeadedAttention):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.incremental_decoding = False

    def reset_cache(self):
        self.cache = [None, None]


class BoxMultiHeadedAttention(nn.Module):
    """Self-attention with relative-geometry weights (relation_transformer.py:117-293).  ``forward`` never materialises the
    [B,N,N,64] embedding: the log-geometry bias of all heads comes straight from the boxes (sc_box_bias_fwd / _bwd) and
    enters the fused attention kernel as an additive term."""

    def __init__(self, h, d_model, trigonometric_embedding=True, dropout=0.1, share_att=None, mask=None):
        super().__init__()
        assert d_model % h == 0
        self.trigonometric_embedding = trigonometric_embedding
        self.h = h
        self.d_k = d_model // h
        self.dim_g = 64 if trigonometric_embedding else 4
        assert share_att in (None, "kv", "qk"), f"Invalid `share_att`: {share_att}"
        self.share_att = share_att
        self.linears = nn.ModuleList([_linear(mask, d_model, d_model) for _ in range(3 if share_att else 4)])
        self.WGs = nn.ModuleList([_linear(mask, self.dim_g, 1) for _ in range(h)])
        self.dropout = nn.Dropout(p=dropout)

    def geometry_weights(self):
        """([h, dim_g] effective WG weights, [h] biases) of this layer (masks applied, straight-through gradients)."""
        ws = []
        for ly in self.WGs:
            if isinstance(ly, MaskedLinear):
                ws.append(A.masked_weight(ly.weight, ly.weight_pruning_mask, ly.mask_mode(),
                                          ly.bypass_sigmoid_grad or ly.mask_type not in prune.SUPER_MASKS))
            else:
                ws.append(ly.weight)
        return torch.cat(ws, 0), torch.cat([ly.bias for ly in self.WGs], 0)

    def forward(self, input_query, input_key, input_value, input_box, mask=None):
        B, N = input_query.shape[:2]
        q = _apply_linear(self.linears[0], input_query)
        if self.share_att == "kv":
            k = _apply_linear(self.linears[1], input_key)
            v = k
        elif self.share_att == "qk":
            k = _apply_linear(self.linears[0], input_key)
            v = _apply_linear(self.linears[1], input_value)
        else:
            k = _apply_linear(self.linears[1], input_key)
            v = _apply_linear(self.linears[2], input_value)
        wg_w, wg_b = self.geometry_weights()
        bias = A.box_bias(input_box, wg_w, wg_b, self.trigonometric_embedding)  # log(clamp(relu(WG emb + b), 1e-6))
        kv, _ = _key_mask(mask, B, N, N)
        out, _ = A.attention(q.reshape(B * N, -1), k.reshape(B * N, -1), v.reshape(B * N, -1), G=B, Tq=N, Tk=N, h=self.h, bias=bias,
                             key_valid=kv, p=self.dropout.p, training=self.training, precision=masked_layer.get_precision())
        return _apply_linear(self.linears[-1], out.view(B, N, -1))

    @staticmethod
    def BoxRelationalEmbedding(f_g, dim_g=64, wave_len=1000, trigonometric_embedding=True):
        """[B, N, 4] boxes -> [B, N, N, dim_g] relational embedding (sc_box_embedding)."""
        if not f_g.is_cuda:
            raise RuntimeError("BoxRelationalEmbedding: the B200 path runs on CUDA tensors only (there is no CPU fallback)")
        assert dim_g == 64 or not trigonometric_embedding, "the trigonometric embedding has dim_g = 64 (4 deltas x 8 wavelengths x sin/cos)"
        return K.box_embedding(f_g.detach().float().contiguous(), trig=bool(trigonometric_embedding), wave_len=float(wave_len))

    @staticmethod
    def box_attention(query, key, value, box_relation_embds_matrix, mask=None, dropout=None):
        """softmax(log(clamp(w_g, 1e-6)) + QK^T / sqrt(d_k)) V on [B, h, N, d_k] tensors; ``box_relation_embds_matrix`` is the
        relu'd geometry weight tensor w_g [B, h, N, N] (relation_transformer.py:258-293).  Returns (output, w_mn)."""
        B, h, N, dk = query.shape
        bias = A.log_clamp(box_relation_embds_matrix.reshape(B, h, N, N), 1e-6)
        kv, _ = _key_mask(mask, B, N, N)
        p = dropout.p if (dropout is not None and dropout.training) else 0.0
        out, probs = A.attention(_rows(query), _rows(key), _rows(value), G=B, Tq=N, Tk=N, h=h, bias=bias, key_valid=kv, p=p,
                                 training=p > 0, precision=masked_layer.get_precision())
        return out.view(B, N, h, dk).transpose(1, 2), probs


class PositionwiseFeedForward(nn.Module):
    def __init__(self, mask, d_model, d_ff, dropout):
        super().__init__()
        self.w_1 = _linear(mask, d_model, d_ff)
        self.w_2 = _linear(mask, d_ff, d_model)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x):
        return _apply_linear(self.w_2, A.dropout(_apply_linear(self.w_1, x, relu=True), self.dropout.p, self.training))


class EncoderLayer(nn.Module):
    def __init__(self, mask, cfg, dropout):
        super().__init__()
        d = cfg.d_model
        self.self_attn = BoxMultiHeadedAttention(cfg.num_heads, d, not cfg.no_box_trigonometric_embedding, dropout,
                                                 cfg.share_att_encoder, mask=mask)
        self.feed_forward = PositionwiseFeedForward(mask, d, cfg.dim_feedforward, dropout)
        self.sublayer = nn.ModuleList([SublayerConnection(d, dropout) for _ in range(2)])
        self.size = d

    def forward(self, x, box, mask):
        x = self.sublayer[0](x, lambda y: self.self_attn(y, y, y, box, mask))
        return self.sublayer[1](x, self.feed_forward)


class DecoderLayer(nn.Module):
    def __init__(self, mask, cfg, dropout):
        super().__init__()
        d = cfg.d_model
        self.size = d
        self.self_attn = CachedMultiHeadedAttention(cfg.num_heads, d, dropout, True, cfg.share_att_decoder, mask=mask)
        self.src_attn = CachedMultiHeadedAttention(cfg.num_heads, d, dropout, False, cfg.share_att_decoder, mask=mask)
        self.feed_forward = PositionwiseFeedForward(mask, d, cfg.dim_feedforward, dropout)
        self.sublayer = nn.ModuleList([SublayerConnection(d, dropout) for _ in range(3)])

    def forward(self, x, memory, src_mask, tgt_mask):
        m = memory
        x = self.sublayer[0](x, lambda y: self.self_attn(y, y, y, tgt_mask))
        x = self.sublayer[1](x, lambda y: self.src_attn(y, m, m, src_mask))
        return self.sublayer[2](x, self.feed_forward)


class _Stack(nn.Module):
    """N layers (shared according to ``share_layer``) + final norm (relation_transformer.py:77-96, transformer.py:172-190)."""

    def __init__(self, make_layer, N, size, share_layer=None):
        super().__init__()
        if share_layer:
            if not isinstance(share_layer, (tuple, list)):
                raise TypeError(f"`share_layer` must be a tuple or list, saw {type(share_layer)}")
            uniq = [make_layer() for _ in range(len(set(share_layer)))]
            layers = [uniq[i] for i in share_layer]
        else:
            layers = [make_layer() for _ in range(N)]
        self.layers = nn.ModuleList(layers)
        self.norm = LayerNorm(size)


class Encoder(_Stack):
    def forward(self, x, box, mask):
        for layer in self.layers:
            x = layer(x, box, mask)
        return self.norm(x)


class Decoder(_Stack):
    def forward(self, x, memory, src_mask, tgt_mask):
        for layer in self.layers:
            x = layer(x, memory, src_mask, tgt_mask)
        return self.norm(x)


class InputEmbedding(nn.Module):
    def __init__(self, mask, d_model, vocab):
        super().__init__()
        self.lut = MaskedEmbedding(vocab, d_model, mask[0], mask[1]) if mask else nn.Embedding(vocab, d_model)
        self.d_model = d_model

    def forward(self, x):
        e = self.lut(x) if isinstance(self.lut, MaskedEmbedding) else A.embedding(x, self.lut.weight)
        return e * math.sqrt(self.d_model)


class PositionalEncoding(nn.Module):
    def __init__(self, d_model, dropout, max_len=5000):
        super().__init__()
        self.dropout = nn.Dropout(p=dropout)
        pe = torch.zeros(max_len, d_model)
        position = torch.arange(0, max_len).unsqueeze(1).float()
        div_term = torch.exp(torch.arange(0, d_model, 2).float() * -(math.log(10000.0) / d_model))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer("pe", pe.unsqueeze(0))
        self.incremental_decoding = False
        self.current_time_step = 0

    def reset_cache(self):
        self.current_time_step = 0

    def forward(self, x):
        if self.incremental_decoding:
            assert x.size(1) == 1, f"{self.__class__.__name__}: Expected input to have shape (M, 1, N), saw {x.shape}"
            x = x + self.pe[:, self.current_time_step: self.current_time_step + 1]
            self.current_time_step += 1
        else:
            x = x + self.pe[:, : x.size(1)]
        return A.dropout(x, self.dropout.p, self.training)


class OutputEmbedding(nn.Module):
    def __init__(self, mask, d_model, vocab):
        super().__init__()
        self.proj = _linear(mask, d_model, vocab)

    def forward(self, x):
        return A.log_softmax(_apply_linear(self.proj, x))


Embeddings, Generator = InputEmbedding, OutputEmbedding  # names used by relation_transformer_prune.py:97-105, 31-37


class EncoderDecoder(nn.Module):
    """relation_transformer.py:39-73 (``src_embed`` is the identity for this model family)."""

    def __init__(self, encoder, decoder, tgt_embed, generator):
        super().__init__()
        self.encoder, self.decoder, self.tgt_embed, self.generator = encoder, decoder, tgt_embed, generator

    def forward(self, src, boxes, tgt, src_mask, tgt_mask):
        enc_out = self.encode(src, boxes, src_mask)
        assert enc_out.size(0) == src_mask.size(0)
        if enc_out.size(0) != tgt.size(0):
            assert tgt.size(0) % enc_out.size(0) == 0
            seq_per_img = tgt.size(0) // enc_out.size(0)
            enc_out, src_mask = repeat_tensors(seq_per_img, (enc_out, src_mask))
        return self.decode(enc_out, src_mask, tgt, tgt_mask)

    def encode(self, src, boxes, src_mask):
        return self.encoder(src, boxes, src_mask)

    def decode(self, memory, src_mask, tgt, tgt_mask):
        return self.decoder(self.tgt_embed(tgt), memory, src_mask, tgt_mask)


class PrunedEncoderDecoder(PruningMixin, EncoderDecoder):
    pass


class _Precision:
    """Numeric mode of the module-level kernels for the duration of one model call ("bf16" | "fp32")."""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        self.prev = masked_layer.get_precision()
        masked_layer.set_precision(self.mode)

    def __exit__(self, *exc):
        masked_layer.set_precision(self.prev)


# ---- models -------------------------------------------------------------------------------------------------------
class _OrtBase(nn.Module):
    """CaptionModel.forward dispatch (caption_model.py:24-28) + the kernel-backed entry points."""

    MASKED = False

    def _init_common(self, config):
        self.config = config
        self.cfg = ModelCfg(config)
        for f in ModelCfg.FIELDS:
            setattr(self, {"eos_token_id": "eos_idx", "bos_token_id": "bos_idx", "unk_token_id": "unk_idx",
                           "pad_token_id": "pad_idx", "max_seq_length": "seq_length"}.get(f, f), getattr(self.cfg, f))
        self.drop_prob_src = getattr(config, "drop_prob_src", 0.5) if not isinstance(config, dict) else config.get("drop_prob_src", 0.5)
        self.precision = "bf16"
        self._engine = None
        self._engine_key = None
        self._trainer = None
        self._trainer_key = None

    def make_model(self, mask, dropout):
        c = self.cfg
        enc = Encoder(lambda: EncoderLayer(mask, c, dropout), c.num_layers, c.d_model, c.share_layer_encoder)
        dec = Decoder(lambda: DecoderLayer(mask, c, dropout), c.num_layers, c.d_model, c.share_layer_decoder)
        tgt = nn.Sequential(InputEmbedding(mask, c.d_model, c.vocab_size), PositionalEncoding(c.d_model, dropout))
        gen = OutputEmbedding(mask, c.d_model, c.vocab_size)
        if mask:
            model = PrunedEncoderDecoder(mask_type=mask[0], mask_freeze_scope="", encoder=enc, decoder=dec, tgt_embed=tgt, generator=gen)
            weights = model.all_weights(named=False)
        else:
            model = EncoderDecoder(enc, dec, tgt, gen)
            weights = list(model.parameters())
        self.att_embed = nn.Sequential(_linear(mask, c.att_feat_size, c.d_model), nn.ReLU(), nn.Dropout(self.drop_prob_src))
        for p in weights:  # Glorot / fan_avg on the inner model only (relation_transformer.py:333-337)
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)
        self.model = model
        self.dropout_p = dropout

    # -- dispatch ----------------------------------------------------------------------------------------------
    def forward(self, *args, **kwargs):
        mode = kwargs.pop("mode", "forward")
        return getattr(self, "_" + mode)(*args, **kwargs)

    def _device(self):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("the B200 captioning path runs on CUDA only (no CPU fallback): call model.cuda() first")
        return dev

    def _effective_state_dict(self):
        sd = self.state_dict()
        if self.MASKED:
            return prune.fold_masks(sd, self.mask_type)
        return sd

    def _param_key(self):
        return (tuple(p._version for p in self.parameters()), tuple(p.data_ptr() for p in self.parameters()), self.precision)

    def _get_engine(self):
        dev = self._device()
        key = self._param_key() + (self.training if self.MASKED else False,)
        if self._engine is None or self._engine_key != key:
            self._engine = OrtEngine(self._effective_state_dict(), self.cfg, precision=self.precision, device=dev,
                                     no_history=self.MASKED and getattr(self, "compat_no_history", False))
            self._engine_key = key
        return self._engine

    # -- teacher forcing (autograd) ----------------------------------------------------------------------------------
    def _embed_features(self, att_feats, att_masks):
        """att_embed = Linear + ReLU + Dropout(drop_prob_src) applied through pack_wrapper (model_utils.py:163-168): rows of
        padded regions come back as zeros."""
        x = _apply_linear(self.att_embed[0], att_feats.float(), relu=True)
        x = A.dropout(x, self.att_embed[2].p, self.training)
        if att_masks is not None:
            x = x * (att_masks > 0).unsqueeze(-1).to(x.dtype)
        return x

    def _prepare_feature(self, att_feats, att_masks=None, boxes=None, seq=None):
        """relation_transformer.py:341-365."""
        self._device()
        att_feats, att_masks = self.clip_att(att_feats, att_masks)
        if boxes is not None and att_masks is not None:
            boxes = boxes[:, : att_masks.shape[1]].contiguous()
        att_feats = self._embed_features(att_feats, att_masks)
        if att_masks is None:
            att_masks = att_feats.new_ones(att_feats.shape[:2], dtype=torch.long)
        att_masks = att_masks.unsqueeze(-2)
        if seq is not None:
            seq = seq[:, :-1]
            seq_mask = (seq.data != self.pad_idx).unsqueeze(-2)
            seq_mask = seq_mask & self.subsequent_mask(seq.size(-1)).to(seq_mask)
        else:
            seq_mask = None
        return att_feats, boxes, seq, att_masks, seq_mask

    def _forward(self, att_feats, boxes, seqs, att_masks=None, **kwargs):
        """Teacher-forcing log-probs [B*S, T, V] (relation_transformer.py:368-372) through the kernel-backed module tree:
        differentiable with respect to every weight and mask logit."""
        with _Precision(self.precision):
            att_feats, boxes, seq, att_masks, seq_mask = self._prepare_feature(att_feats, att_masks, boxes, seqs)
            out = self.model(att_feats, boxes.float(), seq, att_masks, seq_mask)
            return self.model.generator(out)

    def trainer(self, **kw):
        """The fused training engine bound to a COPY of this module's parameters (rebuilt when they change).
        ``trainer().train_step(...)`` replaces loss.backward() + clip_gradient + optimizer.step() of the reference
        loop (scripts/train_n_prune_transformer.py:136-153); ``sync_from_trainer()`` copies the result back."""
        from .trainer import ModuleTrainer, OrtTrainer
        c = self.cfg
        if c.share_att_encoder or c.share_att_decoder or c.share_layer_encoder or c.share_layer_decoder:
            # ACORT weight sharing: the module tree under autograd + the fused clip / Adam kernel (trainer.ModuleTrainer)
            if not isinstance(self._trainer, ModuleTrainer):
                self._trainer = ModuleTrainer(self)
            return self._trainer
        key = self._param_key()
        if self._trainer is None or self._trainer_key != key:
            if self.MASKED:
                kw.setdefault("mask_freeze_scope", self.mask_freeze_scope)
            self._trainer = OrtTrainer(self.state_dict(), self.cfg, mask_type=self.mask_type if self.MASKED else None,
                                       precision=self.precision, device=self._device(), dropout=self.dropout_p,
                                       drop_prob_src=self.drop_prob_src, **kw)
            self._trainer_key = key
        return self._trainer

    @torch.no_grad()
    def sync_from_trainer(self):
        from .trainer import ModuleTrainer
        if isinstance(self._trainer, ModuleTrainer):
            return  # (it updates this module's parameters in place)
        self.load_state_dict(self._trainer.state_dict(), strict=False)
        self._trainer_key = self._param_key()  # the trainer's parameters ARE the module's now

    # -- inference ---------------------------------------------------------------------------------------------
    def _decode_opts(self, opt):
        """Options of caption_model.py:114-123 that need model attributes."""
        opt = dict(opt or {})
        if opt.get("remove_bad_endings", 0):
            opt["bad_endings_ix"] = list(self.bad_endings_ix)  # AttributeError when the model defines none, like the reference
        if opt.get("suppress_UNK", 0) and hasattr(self, "vocab") and self.vocab[str(self.cfg.vocab_size - 1)] == "UNK":
            opt["penalized_col"] = self.cfg.vocab_size - 1
        return opt

    @torch.no_grad()
    def _sample(self, att_feats, boxes, att_masks=None, opt=None, **kwargs):
        """relation_transformer.py:390-396 -> OrtEngine.sample (encoder + KV-cached beam / greedy / multinomial search).
        The pruned class samples with binarized masks in eval mode and with ONE Bernoulli mask draw per call in train mode
        (SCST rollouts, utils/training.py:224-237; the reference draws a new mask per layer call)."""
        return self._get_engine().sample(att_feats, boxes, att_masks, self._decode_opts(opt))

    @torch.no_grad()
    def get_logprobs_state(self, it, memory, mask, state):
        """One decoding step (relation_transformer.py:374-387): ``it`` [R] tokens, ``memory`` [R, N, d] encoder output,
        ``mask`` [R, 1, N]; ``state`` None (first step) or the list returned by the previous call - the tokens fed so far
        [1, R, t] (ys[None]) followed, per unique decoder layer, by self K [slots, R, d], self V, and the cross K|V
        [1, R, N*ld] of the row's image, all with the row dimension at dim 1 so that ``state[i][:, ix]`` reorders beams
        exactly as caption_model.py:106-110 does.  The decode position is the length of that token history, so several
        searches (the groups of a diverse beam search) may advance their own states in any interleaving.
        Returns (log-probs fp32 [R, V], new state)."""
        eng = self._get_engine() if (state is None or self._engine is None) else self._engine
        ys = it.reshape(1, -1, 1)
        if state is None:
            t, caches = 0, None
        else:
            t, caches, prev = state[0].shape[-1], state[1:], state[0]
            if prev.shape[1] != ys.shape[1]:  # first beam step: rows repeated `beam` times (transformer.py:240-252)
                prev = prev.repeat_interleave(ys.shape[1] // prev.shape[1], 1)
            ys = torch.cat([prev.to(ys.dtype), ys], -1)
        logprobs, caches = eng.logprobs_step(it, memory, mask, caches, t)
        return logprobs, [ys] + caches

    @torch.no_grad()
    def batch_beam_search(self, init_state, init_logprobs, *args, **kwargs):
        """caption_model.py:30-226: the per-step candidate ranking, beam bookkeeping and finished-beam handling run in
        sc_beam_step (sc_beam_step_diverse for group_size > 1) on device state; ``get_logprobs_state`` advances the model.
        Returns ``done_beams``: per image a list of dicts {seq, logps (chosen-token log-probs [len]), unaug_p, p} - beam_size
        of them best first, or with group_size G > 1 each group's beam_size // G best, groups in order."""
        opt = self._decode_opts(kwargs["opt"])
        eng = self._engine if self._engine is not None else self._get_engine()
        self.done_beams = eng.beam_search_stepwise(init_state, init_logprobs, list(args), opt, self.get_logprobs_state)
        return self.done_beams

    @staticmethod
    def clip_att(att_feats, att_masks):
        if att_masks is not None:
            max_len = att_masks.data.long().sum(1).max()
            att_feats = att_feats[:, :max_len].contiguous()
            att_masks = att_masks[:, :max_len].contiguous()
        return att_feats, att_masks

    @staticmethod
    def subsequent_mask(size):
        return torch.triu(torch.ones((1, size, size)), diagonal=1).eq(0)

    @staticmethod
    def add_argparse_args(parser: Union[_ArgumentGroup, ArgumentParser]):
        parser.add_argument("--d_model", type=int, default=512)
        parser.add_argument("--dim_feedforward", type=int, default=2048)
        parser.add_argument("--num_layers", type=int, default=6)
        parser.add_argument("--num_heads", type=int, default=8)
        parser.add_argument("--drop_prob_src", type=float, default=0.5)
        parser.add_argument("--att_feat_size", type=int, default=2048)
        parser.add_argument("--share_att_encoder", type=str_to_none, default=None)
        parser.add_argument("--share_att_decoder", type=str_to_none, default=None)
        parser.add_argument("--share_layer_encoder", type=str_to_sequence, default=None)
        parser.add_argument("--share_layer_decoder", type=str_to_sequence, default=None)
        parser.add_argument("--no_box_trigonometric_embedding", action="store_true")


@register_model("relation_transformer")
class RelationTransformerModel(_OrtBase):
    def __init__(self, config):
        super().__init__()
        self._init_common(config)
        self.make_model(None, 0.1)


@register_model("relation_transformer_prune")
class RelationTransformerPruneModel(PruningMixin, _OrtBase):
    MASKED = True

    def __init__(self, config):
        get = (lambda k, d=None: config.get(k, d)) if isinstance(config, dict) else (lambda k, d=None: getattr(config, k, d))
        super().__init__(mask_type=get("prune_type"), mask_freeze_scope=get("prune_mask_freeze_scope", ""))
        self._init_common(config)
        self.make_model((get("prune_type"), get("prune_supermask_init", 5.0)), 0.1 / 3)

    def _effective_state_dict(self):
        """Eval: binarized masks folded into the weights.  Train (SCST rollouts): one Bernoulli(sigmoid(S)) draw per call."""
        if self.training and self.mask_type in prune.SUPER_MASKS:
            from . import sampler
            sd = self.state_dict()
            out = {}
            for k, v in sd.items():
                if k.endswith("_pruning_mask"):
                    continue
                m = sd.get(k + "_pruning_mask")
                if m is None:
                    out[k] = v
                else:
                    seed, stream = sampler.next_mask_stream()
                    out[k] = K.apply_mask(v.detach().float().contiguous(), m.detach().float().contiguous(), K.MASK_BERNOULLI,
                                          seed=seed, stream_id=stream)
            return out
        return super()._effective_state_dict()

    def _get_engine(self):
        if self.training and self.mask_type in prune.SUPER_MASKS:
            self._engine = None  # a fresh mask sample (and weight pack) per rollout call
        return super()._get_engine()

    @staticmethod
    def add_argparse_args(parser):
        _OrtBase.add_argparse_args(parser)
        PruningMixin.add_argparse_args(parser)
