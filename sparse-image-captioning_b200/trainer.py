"""Supermask (SMP) training step of the ORT captioner on the B200 kernels.

Replaces the reference's hot loop body (scripts/train_n_prune_transformer.py:132-156):
    model(**data) -> LanguageModelCriterion -> + compute_sparsity_loss -> backward -> clip_gradient(0.1) -> Adam
for `relation_transformer_prune` (sparse_caption/models/relation_transformer_prune.py) and, with mask_type=None, for the
dense `relation_transformer`.  The encoder runs once per image; the S captions of an image share its memory K/V
(the reference repeats the memory S times before the cross K/V projections, relation_transformer.py:63-66).

All parameters live in two flat fp32 buffers (weights+biases+norms | mask logits) with views per reference parameter
name, so the optimizer is two fused kernels and the data-parallel gradient exchange is an NCCL all-reduce over flat
gradient buffers (mask-logit gradients included).  Forward and backward are explicit sequences of kernel launches;
no autograd graph is built.
"""
import math
from typing import Dict, Optional

import torch

from . import kernels as K
from .engine import ModelCfg


def _round_up(n, m):
    return (n + m - 1) // m * m


# A layer's linears in parameter order.  Each entry is one storage block - consecutive linears of a module, their weights then
# their biases - and the fused groups the forward runs on it: (count, OrtEngine slot).  The cross-attention stores q, k, v like
# the self-attention's [q;k;v] but projects q alone and [k;v] once from the memory.
_ATT = (("self_attn.linears.0", (3, "qkv")), ("self_attn.linears.3", (1, "o")))
_FF = (("feed_forward.w_1", (1, "ff1")), ("feed_forward.w_2", (1, "ff2")))
_CROSS = (("src_attn.linears.0", (1, "cq"), (2, "ckv")), ("src_attn.linears.3", (1, "co")))
_LINEARS = {"encoder": _ATT + _FF, "decoder": _ATT + _CROSS + _FF}

# Philox dropout sites (_drop_stream): the backward regenerates each dropout mask of the forward from its site.  att_embed 1, the
# target embedding 2, and per layer l: site + l of the dropout after a linear (by OrtEngine slot) or of an attention's probabilities
_SITES = {"att_embed": 1, "embed": 2, "encoder": dict(attn=10, o=20, ff1=30, ff2=40),
          "decoder": dict(attn=50, o=60, cattn=70, co=80, ff1=90, ff2=100)}
_DEC0 = "model.decoder.layers.0.self_attn.linears.0.weight"   # first decoder parameter: the decoder / encoder cut of the layout


def _member(first, i):
    """Name of the i-th linear of a block that starts at `first` ("self_attn.linears.0", 2 -> "self_attn.linears.2")."""
    stem, j = first.rsplit(".", 1)
    return first if i == 0 else f"{stem}.{int(j) + i}"


def _layer_linears(p, stack):
    """(first weight name, fused count, OrtEngine slot) of every fused group of layer `p`, and its linears' parameter names."""
    groups, names = [], []
    for first, *fused in _LINEARS[stack]:
        members = [f"{p}.{_member(first, i)}" for i in range(sum(n for n, _ in fused))]
        names += [m + ".weight" for m in members] + [m + ".bias" for m in members]
        i = 0
        for n, slot in fused:
            groups.append((f"{members[i]}.weight", n, slot))
            i += n
    return groups, names


def _anneal(current_step, max_step):
    """Cosine anneal of the sparsity-loss weight (prune.py:246): 1 at step 0, 0 from max_step on."""
    return (1.0 + math.cos(min(1.0, current_step / max_step) * math.pi)) / 2.0


def _part(n, cut, part):
    """[lo, hi) of an optimizer `part` of a layout of n: "all", "hi" (decoder, embedding, generator: from `cut`) or "lo"."""
    return {"all": (0, n), "hi": (cut, n), "lo": (0, cut)}[part]


# ---- optimizer state in the layout of torch.optim.Adam.state_dict() (train_n_prune_transformer.py:67-82: group 0 the weights, group 1
# the mask logits with their own lr / eps, "pruning_mask": True) ------------------------------------------------------------------------
_ADAM = dict(mask_lr=100.0, betas=(0.9, 0.98), eps=1e-9, mask_eps=1e-2, weight_decay=0.0)


def _adam_hyper(lr, opt):
    """The Adam hyper-parameters of a step (its optimizer keywords, defaults filled in): the param_groups of the exported state."""
    return dict(_ADAM, **{k: opt[k] for k in _ADAM if k in opt}, lr=float(lr))


def _export_adam(groups, hyper, step, trainer):
    """torch.optim.Adam.state_dict() of ``groups`` = [[(name, (exp_avg, exp_avg_sq) or None)]]: parameter indices run over the groups
    in order, a parameter without moments gets no state entry, every entry's step is ``float(step)``.  ``trainer``: the extra
    top-level key (Adam.load_state_dict ignores it)."""
    state, param_groups, i = {}, [], 0
    for gi, entries in enumerate(groups):
        ids = []
        for _, mv in entries:
            if mv is not None:
                state[i] = {"step": torch.tensor(float(step), dtype=torch.float32), "exp_avg": mv[0], "exp_avg_sq": mv[1]}
            ids.append(i)
            i += 1
        g = dict(lr=hyper["lr"], betas=tuple(hyper["betas"]), eps=hyper["eps"], weight_decay=hyper["weight_decay"], amsgrad=False,
                 maximize=False)
        if gi == 1:
            g.update(lr=hyper["mask_lr"], eps=hyper["mask_eps"], weight_decay=0.0, pruning_mask=True)
        param_groups.append(dict(g, params=ids))
    return {"state": state, "param_groups": param_groups, "trainer": trainer}


def _import_adam(sd, groups, mask_type):
    """Checks an Adam state dict against ``groups`` = [[(name, shape, has_state)]] (``has_state``: the trainer updates it, so its
    entry must be there).  Returns ({name: (exp_avg, exp_avg_sq)}, step, hyper-parameters, the "trainer" key or None); ValueError,
    naming the parameter, for a different parameter count or shape, a missing entry, unequal steps or another mask type."""
    pgs, state, extra = sd["param_groups"], sd["state"], sd.get("trainer")
    if extra is not None and extra.get("mask_type") != mask_type:
        raise ValueError(f"the state was saved by a trainer with mask_type {extra.get('mask_type')!r}, this one has {mask_type!r}")
    if len(pgs) != len(groups):
        raise ValueError(f"the state has {len(pgs)} parameter groups, the trainer {len(groups)}")
    moments, step, first = {}, None, None
    for gi, (pg, entries) in enumerate(zip(pgs, groups)):
        if len(pg["params"]) != len(entries):
            raise ValueError(f"parameter group {gi} has {len(pg['params'])} parameters in the state, {len(entries)} in the trainer "
                             f"(first of them: {entries[0][0] if entries else None})")
        for idx, (name, shape, has_state) in zip(pg["params"], entries):
            st = state.get(idx)
            if st is None:
                if has_state:
                    raise ValueError(f"{name}: no optimizer state entry (parameter {idx})")
                continue
            for key in ("exp_avg", "exp_avg_sq"):
                if tuple(st[key].shape) != tuple(shape):
                    raise ValueError(f"{name}: {key} has shape {tuple(st[key].shape)}, the parameter {tuple(shape)}")
            s = float(st["step"])
            if step is None:
                step, first = s, name
            elif s != step:
                raise ValueError(f"{name}: step {s} differs from the step {step} of {first}")
            moments[name] = (st["exp_avg"], st["exp_avg_sq"])
    g0 = pgs[0]
    hyper = dict(lr=g0["lr"], betas=tuple(g0["betas"]), eps=g0["eps"], weight_decay=g0["weight_decay"])
    if len(pgs) > 1:
        hyper.update(mask_lr=pgs[1]["lr"], mask_eps=pgs[1]["eps"])
    return moments, int(step or 0), hyper, extra


def scst_samples(opt, baseline, bleu_weight=0.0):
    """Captions per image S of an SCST rollout ``opt`` (beam_size b, G * (b // G) for diverse beam search, or num_random_sample);
    ValueError for the options the device step does not support."""
    from .engine import diverse_groups
    if baseline not in ("greedy", "sample"):
        raise ValueError(f"SCST baseline must be 'greedy' or 'sample', got {baseline!r}")
    if bleu_weight:
        raise ValueError("bleu_weight > 0: the BLEU scorer does not run on the device (CIDEr-D only)")
    if float(opt.get("temperature", 1.0)) != 1.0:
        raise ValueError("SCST re-scores the plain log-softmax of the sampled tokens: temperature must be 1")
    beam, n_rand = int(opt.get("beam_size", 1)), int(opt.get("num_random_sample", 0))
    if n_rand > 0:
        assert beam < 1, f"Beam size must be < 1, saw {beam}"  # transformer.py:509
        S = n_rand
    elif beam == 1:
        raise ValueError("beam_size == 1 is the greedy baseline, not a rollout: use beam_size > 1 or num_random_sample > 0")
    elif beam < 1:
        raise ValueError(f"SCST rollout needs beam_size > 1 or num_random_sample > 0 (got beam_size={beam})")
    else:
        S = beam
        if int(opt.get("group_size", 1)) > 1:
            G, bdash, _ = diverse_groups(opt)
            S = G * bdash
    if baseline == "sample" and S < 2:
        raise ValueError(f"baseline='sample' averages the image's other samples: it needs at least 2 per image (got {S})")
    return S


class OrtTrainer:
    def __init__(self, state_dict: Dict[str, torch.Tensor], cfg: ModelCfg, *, mask_type: Optional[str] = "supermask",
                 precision="bf16", device="cuda", dropout=0.1 / 3, drop_prob_src=0.5, bypass_sigmoid_grad=False, seed=0,
                 mask_init_value=5.0, uniforms: Optional[Dict[str, torch.Tensor]] = None, use_graph=False, fused_st=True,
                 mask_freeze_scope=None):
        assert cfg.share_att_encoder is None and cfg.share_att_decoder is None and not cfg.share_layer_encoder \
            and not cfg.share_layer_decoder, "the fused engine lays out the ORT stack; ACORT weight sharing trains through ModuleTrainer (model.trainer() picks it)"
        self.cfg = cfg
        self.dev = K.lib.resolve_device(device)
        self.adt = torch.bfloat16 if precision == "bf16" else torch.float32
        self.mask_type = mask_type
        # prefixes of the frozen masks (PruningMixin.mask_freeze_scope: a list, or the comma-separated string of its constructor);
        # magnitude / SNIP updates leave those masks alone
        if isinstance(mask_freeze_scope, str):
            mask_freeze_scope = [x for x in mask_freeze_scope.split(",") if x != ""] if mask_freeze_scope != "" else None
        self.mask_freeze_scope = None if mask_freeze_scope is None else list(mask_freeze_scope)
        self.sparsity_target = 0.0
        self.p_drop, self.p_src = float(dropout), float(drop_prob_src)
        self.bypass = bool(bypass_sigmoid_grad)
        self.seed = int(seed)
        self.step_id = 0
        self.training = True
        # CUDA-graph mode: the whole step (forward, backward, optimizer) is captured once per batch shape and replayed;
        # everything that changes per step (Philox seeds, lr, Adam bias corrections, sparsity-loss scale) is read from
        # small device buffers that the host rewrites before each replay (sc_b200.h: seed pointers, `dyn`)
        self.use_graph = bool(use_graph)
        # straight-through epilogue inside the optimizer kernel (sc_adam_clip_st): the backward leaves dWm = dL/d(W.m) in flat_gw,
        # which is ALL a data-parallel run exchanges (half the bytes of dW + dS); dW = dWm.m and dS = dWm.W.sigmoid'(S) are formed
        # per element inside the update with the step's mask sample regenerated.  False: the weight-gradient epilogue writes dW and
        # dS (needed by the ZeRO-style ShardedExchange, whose shards cut through tensors).
        self.fused_st = bool(fused_st)
        self._materialized = False
        self._st_desc = {}
        self._seeds_host = torch.zeros(3, dtype=torch.int64).pin_memory() if self.use_graph else None
        self._seeds_dev = torch.zeros(3, dtype=torch.int64, device=self.dev)
        self._dyn_host = torch.zeros(8, dtype=torch.float32).pin_memory() if self.use_graph else None
        self._dyn_dev = torch.zeros(8, dtype=torch.float32, device=self.dev)
        d, L, h = cfg.d_model, cfg.num_layers, cfg.num_heads
        sd = state_dict
        # ---- parameter layout: fused groups are contiguous so that [q;k;v] / [k;v] / WG blocks are single views ----
        # the one-element WG biases of ALL encoder layers come first, contiguous: the geometry bias of every layer is then
        # one kernel (sc_box_bias_all) over a single [L*h] bias vector
        order = [f"model.encoder.layers.{i}.self_attn.WGs.{j}.bias" for i in range(L) for j in range(h)]
        order += ["att_embed.0.weight", "att_embed.0.bias"]
        self._groups = {}   # (stack, layer) -> [(first weight name, fused count, OrtEngine slot)] of its linears, in forward order
        for stack, n_norms in (("encoder", 2), ("decoder", 3)):
            for i in range(L):
                p = f"model.{stack}.layers.{i}"
                self._groups[stack, i], names = _layer_linears(p, stack)
                if stack == "encoder":   # the geometry heads' weights follow the self-attention's linears
                    at = names.index(f"{p}.self_attn.linears.3.bias") + 1
                    names[at:at] = [f"{p}.self_attn.WGs.{j}.weight" for j in range(h)]
                order += names + [f"{p}.sublayer.{j}.norm.{ab}" for j in range(n_norms) for ab in ("a_2", "b_2")]
            order += [f"model.{stack}.norm.a_2", f"model.{stack}.norm.b_2"]
        order += ["model.tgt_embed.0.lut.weight", "model.generator.proj.weight", "model.generator.proj.bias"]
        self.names = order
        # the generator is stored with its vocabulary padded to a multiple of 8 rows (zero weights, bias -1e9, masked
        # out) so that dlogits can be a 16-byte-aligned bf16 GEMM operand for any V (e.g. the 771-token radix vocab)
        V = cfg.vocab_size
        self.Vp = K.pad8(V)
        self._pad_rows = {"model.generator.proj.weight": self.Vp, "model.generator.proj.bias": self.Vp}

        def alloc(k):
            if k in self._pad_rows:
                return sd[k].numel() // V * self.Vp
            return sd[k].numel()

        def layout(keys):
            # every view 16-byte aligned, except that the h one-element WG biases of a layer are packed into one [h] block
            offs, n = {}, 0
            for k in keys:
                offs[k] = n
                n += alloc(k)
                if not (".WGs." in k and k.endswith(".bias") and not k.endswith(f".WGs.{cfg.num_heads - 1}.bias")):
                    n = _round_up(n, 4)
            return offs, n

        offs, n = layout(order)
        self.flat_w = torch.zeros(n, device=self.dev)
        self.flat_gw = torch.zeros(n, device=self.dev)
        self.p = {k: self.flat_w[offs[k]: offs[k] + sd[k].numel()].view(sd[k].shape) for k in order}
        self.g = {k: self.flat_gw[offs[k]: offs[k] + sd[k].numel()].view(sd[k].shape) for k in order}
        for k in order:
            self.p[k].copy_(sd[k])
        self._offs_w = offs
        # all WG biases as one [L*h] view when the layout packed them without padding (h % 4 == 0)
        b0 = offs["model.encoder.layers.0.self_attn.WGs.0.bias"]
        packed = all(offs[f"model.encoder.layers.{l}.self_attn.WGs.{j}.bias"] == b0 + l * h + j for l in range(L) for j in range(h))
        self._wg_b_all = self.flat_w[b0: b0 + L * h] if packed else None
        if self.Vp != V:
            ob = offs["model.generator.proj.bias"]
            self.flat_w[ob + V: ob + self.Vp] = -1e9
        # mask logits for every 2-D weight
        self.masked = [k for k in order if k.endswith(".weight") and sd[k].dim() == 2] if mask_type else []
        offs_s, n = layout(self.masked)
        self.flat_s = torch.zeros(max(n, 4), device=self.dev)
        self.flat_gs = torch.zeros(max(n, 4), device=self.dev)
        self.n_logits = sum(sd[k].numel() for k in self.masked)
        self.s = {k: self.flat_s[offs_s[k]: offs_s[k] + sd[k].numel()].view(sd[k].shape) for k in self.masked}
        self.gs = {k: self.flat_gs[offs_s[k]: offs_s[k] + sd[k].numel()].view(sd[k].shape) for k in self.masked}
        for k in self.masked:
            mk = k + "_pruning_mask"
            if mk in sd:
                self.s[k].copy_(sd[mk])
            else:
                self.s[k].fill_(mask_init_value)
        self._offs_s = offs_s
        # parameter order of optimizer_state_dict: the key order of `state_dict` (named_parameters() order for the drop-in module); a
        # mask logit sits where its "_pruning_mask" key is, or where its weight is when the logit was initialised here
        pos = {k: i for i, k in enumerate(sd)}
        self._adam_order = sorted(order, key=pos.__getitem__)
        self._adam_masks = sorted(self.masked, key=lambda k: pos.get(k + "_pruning_mask", pos[k]))
        self._cut, self._cut_w, self._cut_s = order.index(_DEC0), offs[_DEC0], offs_s.get(_DEC0)
        # padding elements of flat_s must never count as "kept" in the sparsity statistics
        pad = torch.ones_like(self.flat_s, dtype=torch.bool)
        for k in self.masked:
            pad[offs_s[k]: offs_s[k] + sd[k].numel()] = False
        self.flat_s[pad] = -1.0
        self._s_pad_mask = pad
        self._s_pad_idx = pad.nonzero().view(-1)  # index form: index_fill_ is CUDA-graph capturable
        self.stream_of = {k: i + 1 for i, k in enumerate(order)}
        # injected uniforms (parity tests): same layout as flat_s
        self.flat_u = None
        if uniforms is not None:
            self.flat_u = torch.zeros_like(self.flat_s)
            for k in self.masked:
                self.flat_u[offs_s[k]: offs_s[k] + sd[k].numel()].view(sd[k].shape).copy_(uniforms[k])
        pe = sd.get("model.tgt_embed.1.pe")
        from .engine import _positional_encoding
        self.pe = (pe[0, : cfg.max_seq_length + 2].to(self.dev) if pe is not None
                   else _positional_encoding(d, cfg.max_seq_length + 2, self.dev)).float().contiguous()
        # optimizer state
        self.m_w, self.v_w = torch.zeros_like(self.flat_w), torch.zeros_like(self.flat_w)
        self.m_s, self.v_s = torch.zeros_like(self.flat_s), torch.zeros_like(self.flat_s)
        self.opt_step = 0
        self._hyper = _adam_hyper(0.0, {})   # hyper-parameters of the last optimizer step (optimizer_state_dict's param_groups)
        self.sp_out = torch.zeros(3, device=self.dev)
        self.sp_count = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self._ws = {}
        self.premask = True   # False: mask inside the GEMM operand prologue (K1 fused variant)
        self._wm, self._wmT, self._wm_step = {}, {}, {}
        self._premask_desc = None
        # timing diagnostic (scripts/profile_train.py SC_SKIP_WGRAD=1: wrong gradients): the main chain alone - measured 4.95 of the
        # 5.35 ms step, i.e. the weight-gradient side stream costs 0.4 ms and the step is bound by the ~290 dependent launches
        self._diag_skip_wgrad = False
        self.pdl_mask = 3            # sc_set_pdl mask while the step is launched / captured (see train_step)
        self.wgrad_ring = 4          # 1: weight gradients stay on the main stream
        import os
        self.fuse_hmask = os.environ.get("SC_NO_HMASK") != "1"      # ff2's dX GEMM prepares ff1's gradient operand
        # attention backward emitting bf16 operands + bias gradients itself (sc_attention_bwd_bf16out): parity-tested, but
        # measured SLOWER (5.66 vs 5.58 ms/step: ~640k same-address atomics for the bias sums) - off unless SC_ATTN16=1
        self.fuse_attn_bwd = os.environ.get("SC_ATTN16") == "1"
        self._side = None
        self._ost = None
        # decoder-side Adam on its own stream underneath the encoder backward: measured slower (5.42 vs 5.35 ms/step, the
        # HBM-bound update slows the backward kernels more than it hides) - off unless SC_OPT_OVERLAP=1
        self.overlap_opt = os.environ.get("SC_OPT_OVERLAP") == "1"
        # SCST step in progress: its masks were applied before the rollouts (scst_step), the forward must reuse that sample
        self._scst = False
        self._rollout = self._baseline = None
        # magnitude / SNIP mask updates: cached sc_prune descriptor tables, the accumulated SNIP saliency (flat_s layout)
        self._prune_desc = {}
        self._saliency = None
        self._has_saliency = False

    # ---------------------------------------------------------------------------------------------------------
    def _view(self, flat, offs, first, count):
        """View of a flat buffer over `count` consecutive same-shape parameters starting at `first` (e.g. [q;k;v]); the
        generator alone spans its padded Vp rows."""
        shp = self.p[first].shape
        rows = self._pad_rows.get(first, shp[0]) if count == 1 else shp[0] * count
        return flat[offs[first]: offs[first] + self.p[first].numel() // shp[0] * rows].view((rows,) + tuple(shp[1:]))

    def _group(self, table, first, count):
        """_view of the flat buffer behind `table` (self.p, self.g, self.s or self.gs)."""
        flat, offs = {id(self.p): (self.flat_w, self._offs_w), id(self.g): (self.flat_gw, self._offs_w),
                      id(self.s): (self.flat_s, self._offs_s), id(self.gs): (self.flat_gs, self._offs_s)}[id(table)]
        return self._view(flat, offs, first, count)

    def _u(self, first, count=1):
        return None if self.flat_u is None else self._view(self.flat_u, self._offs_s, first, count)

    def mask_mode(self):
        if not self.mask_type:
            return K.MASK_NONE
        if self.mask_type == "supermask":
            if not self.training:
                return K.MASK_ROUND
            return K.MASK_UNIFORM if self.flat_u is not None else K.MASK_BERNOULLI
        return K.MASK_RAW

    def _sd(self, i):
        """Philox seed i (0 masks, 1 dropout, 2 attention dropout): an immediate value, or in graph mode a device pointer
        (bit 63 set) to the seed word the host rewrites every step."""
        if self.use_graph:
            return (1 << 63) | (self._seeds_dev.data_ptr() + 8 * i)
        return self.seed + i

    def _step_base(self):
        return 0 if self.use_graph else self.step_id * 4096

    def _mask_args(self, wname, count=1):
        """(weight view, logits view, mode, uniforms view, seed, stream) of a (fused) masked weight."""
        W = self._group(self.p, wname, count)
        if not self.mask_type:
            return W, None, K.MASK_NONE, None, 0, 0
        return (W, self._group(self.s, wname, count), self.mask_mode(), self._u(wname, count), self._sd(0),
                self._step_base() + self.stream_of[wname])

    def _premask_keys(self):
        """(first weight name, fused count) of every linear the teacher-forcing forward runs, in launch order."""
        L = self.cfg.num_layers
        enc = [(w, n) for l in range(L) for w, n, _ in self._groups["encoder", l]]
        dec = [(w, n, slot) for l in range(L) for w, n, slot in self._groups["decoder", l]]
        # (the memory's [k;v] of every decoder layer is projected right after the encoder)
        return ([("att_embed.0.weight", 1)] + enc + [(w, n) for w, n, slot in dec if slot == "ckv"]
                + [(w, n) for w, n, slot in dec if slot != "ckv"] + [("model.generator.proj.weight", 1)])

    def _premask_all(self):
        """W (.) m (bf16) and its transpose for EVERY linear of the step in one launch (sc_apply_mask_batched): the forward
        operand, the dX operand and the weight-gradient epilogue all see the same Philox sample."""
        if self._premask_desc is None:
            items = []
            for key in self._premask_keys():
                wname, count = key
                W, S, mode, U, seed, stream = self._mask_args(wname, count)
                wm = self._wm[key] = torch.empty(W.shape, device=self.dev, dtype=torch.bfloat16)
                wT = self._wmT[key] = torch.empty(W.shape[1], W.shape[0], device=self.dev, dtype=torch.bfloat16)
                items.append((W, S, U, wm, wT, self.stream_of[wname]))
            self._premask_desc = K.mask_descriptors(items, self.dev) + ([k for k in self._premask_keys()],)
        desc, tiles, keys = self._premask_desc
        K.apply_mask_batched(desc, tiles, self.mask_mode(), seed=self._sd(0), stream_base=self._step_base())
        for key in keys:
            self._wm_step[key] = (self.step_id, self.training)

    def _drop_stream(self, site):
        return self._step_base() + 2048 + site

    # ---------------------------------------------------------------------------------------------------------
    def _get_ws(self, B, N, S, T, masked):
        key = (B, N, S, T, masked)
        if key in self._ws:
            return self._ws[key]
        c, dev, adt = self.cfg, self.dev, self.adt
        d, ff, V, L, h, F = c.d_model, c.dim_feedforward, c.vocab_size, c.num_layers, c.num_heads, c.att_feat_size
        ME, R = B * N, B * S
        MD = R * T
        Mp = K.pad8(max(ME, MD))
        f32 = dict(device=dev, dtype=torch.float32)
        a = dict(device=dev, dtype=adt)
        ws = type("TrainWs", (), {})()
        ws.B, ws.N, ws.S, ws.T, ws.ME, ws.MD, ws.R, ws.Mp = B, N, S, T, ME, MD, R, Mp
        ws.att_in = torch.zeros(ME, F, **f32)
        ws.att_a = torch.zeros(ME, F, **a) if adt != torch.float32 else ws.att_in
        ws.boxes = torch.zeros(B, N, 4, **f32)
        ws.att_mask = torch.ones(B, N, **f32) if masked else None
        ws.tokens = torch.zeros(MD, device=dev, dtype=torch.int32)
        ws.targets = torch.zeros(MD, device=dev, dtype=torch.int32)
        ws.tok_w = torch.zeros(MD, **f32)
        ws.key_valid = torch.zeros(R, T, **f32)
        ws.inv_norm = torch.zeros(1, **f32)
        ws.loss_sum = torch.zeros(1, **f32)
        ws.xe = [torch.zeros(ME, d, **f32) for _ in range(2 * L + 1)]
        ws.e_xn1 = [torch.zeros(ME, d, **a) for _ in range(L)]
        ws.e_qkv = [torch.zeros(ME, 3 * d, **a) for _ in range(L)]
        ws.e_bias_all = torch.zeros(L, B, h, N, N, **f32)
        ws.e_bias = [ws.e_bias_all[l] for l in range(L)]
        ws.e_probs = [torch.zeros(B, h, N, N, **f32) for _ in range(L)]
        ws.e_att = [torch.zeros(ME, d, **a) for _ in range(L)]
        ws.e_xn2 = [torch.zeros(ME, d, **a) for _ in range(L)]
        ws.e_hid = [torch.zeros(ME, ff, **a) for _ in range(L)]
        dim_g = 64 if not c.no_box_trigonometric_embedding else 4
        ws.wg_eff_all = torch.zeros(L * h, dim_g, **f32)
        ws.wg_eff = [ws.wg_eff_all[l * h: (l + 1) * h] for l in range(L)]
        ws.wg_b_all = self._wg_b_all
        ws.mem = torch.zeros(ME, d, **a)
        ws.memkv = [torch.zeros(ME, 2 * d, **a) for _ in range(L)]
        ws.y = [torch.zeros(MD, d, **f32) for _ in range(3 * L + 1)]
        ws.d_yn1 = [torch.zeros(MD, d, **a) for _ in range(L)]
        ws.d_qkv = [torch.zeros(MD, 3 * d, **a) for _ in range(L)]
        ws.d_probs = [torch.zeros(R, h, T, T, **f32) for _ in range(L)]
        ws.d_att = [torch.zeros(MD, d, **a) for _ in range(L)]
        ws.d_yn2 = [torch.zeros(MD, d, **a) for _ in range(L)]
        ws.d_qc = [torch.zeros(MD, d, **a) for _ in range(L)]
        ws.c_probs = [torch.zeros(B, h, S * T, N, **f32) for _ in range(L)]
        ws.d_catt = [torch.zeros(MD, d, **a) for _ in range(L)]
        ws.d_yn3 = [torch.zeros(MD, d, **a) for _ in range(L)]
        ws.d_hid = [torch.zeros(MD, ff, **a) for _ in range(L)]
        ws.yf = torch.zeros(MD, d, **a)
        ws.logits = torch.zeros(MD, self.Vp, **f32)
        ws.dlogits = torch.zeros(MD, self.Vp, **a)
        # backward scratch
        nmax = max(self.Vp, ff, 3 * d, F)
        ws.gb = torch.zeros(max(ME, MD) * max(ff, 3 * d), **a)         # grad operand [M, N]
        # bf16: the weight-gradient GEMMs (+ their split-K reductions) run on a side stream next to the dX chain; the
        # gradient operand they read lives in a ring so that the next layers can already overwrite "their" buffer
        ws.gb_ring = [ws.gb] + [torch.zeros_like(ws.gb) for _ in range(self.wgrad_ring - 1)] if self._side_wgrad() else [ws.gb]
        ws.gb_free = [None] * len(ws.gb_ring)   # event: the side-stream consumer of ring slot i has finished
        ws.gb_next = 0
        ws.gT = torch.zeros(nmax * Mp, **a)                            # grad operand transposed [N, Mp]
        ws.xT = torch.zeros(max(ff, F, d) * Mp, **a)                   # activation transposed [K, Mp]
        ws.wT = torch.zeros(max(self.Vp * d, ff * d, F * d, 3 * d * d), **a)  # (W.m)^T [K, N]
        ws.ga = torch.zeros(max(ME, MD), max(ff, 3 * d), **f32)        # fp32 activation gradient scratch
        ws.gq = torch.zeros(max(ME, MD), 3 * d, **f32)                 # dq|dk|dv
        ws.dres = [torch.zeros(max(ME, MD), d, **f32) for _ in range(2)]  # running residual-stream gradient (ping-pong)
        ws.dmem = torch.zeros(ME, d, **f32)
        ws.dmemkv = torch.zeros(ME, 2 * d, **f32)
        ws.dbias = torch.zeros(B, h, N, N, **f32)
        ws.dwg = torch.zeros(h, ws.wg_eff[0].shape[1], **f32)
        ws.dtable = torch.zeros(V, d, **f32)
        # split-K partial products of the weight-gradient GEMMs (sc_linear_wgrad workspace): up to 8 fp32 copies of the
        # largest non-vocabulary weight, at least 2 of the generator
        ws.wgrad_ws = torch.zeros(max(8 * max(ff * d, F * d, 3 * d * d), 2 * self.Vp * d), **f32)
        self._ws[key] = ws
        return ws

    def _side_wgrad(self):
        return self.adt == torch.bfloat16 and self.wgrad_ring > 1

    def _opt_stream(self):
        if self._ost is None:
            self._ost = torch.cuda.Stream(self.dev)
        return self._ost

    def _side_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(self.dev)
        return self._side

    # ---- linear forward / backward helpers ------------------------------------------------------------------
    def _lin(self, wname, x, out, *, count=1, relu=False, residual=None, p=0.0, site=0, bias=True):
        W, S, mode, U, seed, stream = self._mask_args(wname, count)
        b = self._group(self.p, wname.replace(".weight", ".bias"), count) if bias else None
        p = p if self.training else 0.0
        if self.adt == torch.bfloat16 and self.premask:
            # bf16 training at M >= 1800 rows: W (.) m is materialised ONCE per step as a bf16 TMA operand; masking in
            # the operand prologue would redo sigmoid + Philox for every 128-row tile (DESIGN.md, "K1: where to mask")
            key = (wname, count)
            wm = self._wm.get(key)
            if wm is None:
                wm = self._wm[key] = torch.empty(W.shape, device=self.dev, dtype=torch.bfloat16)
                self._wmT[key] = torch.empty(W.shape[1], W.shape[0], device=self.dev, dtype=torch.bfloat16)
            if self._wm_step.get(key) != (self.step_id, self.training):
                if self.training:
                    # one pass over W and S: the forward operand W (.) m and the dX operand (W (.) m)^T, same mask sample
                    K.apply_mask_transposed(W, S, mode, self._wmT[key], uniforms=U, seed=seed, stream_id=stream, out=wm)
                else:
                    K.apply_mask(W, S, mode, uniforms=U, seed=seed, stream_id=stream, out=wm)
                self._wm_step[key] = (self.step_id, self.training)
            K.linear_dropout(x, wm, b, residual=residual, relu=relu, out=out, p=p, drop_seed=self._sd(1),
                             drop_stream=self._drop_stream(site), tile_n=self._fwd_tile(x.shape[0], wm.shape[0], wm.shape[1], residual is not None))
            return out
        K.linear_dropout(x, W, b, mask=S, mask_mode=mode, uniforms=U, seed=seed, stream_id=stream, residual=residual,
                         relu=relu, out=out, p=p, drop_seed=self._sd(1), drop_stream=self._drop_stream(site))
        return out

    @staticmethod
    def _fwd_tile(M, N, Kd, has_res):
        """Tile hints (1000 * stages + block_n) where the sweep over the training shapes (scripts/train_gemm_sweep.py,
        profiles/r01b_train_gemm_sweep.txt) beat the kernel's own heuristic: the fp32-residual + dropout epilogue is the long
        pole of the d x d GEMMs and likes the 8-epilogue-warp configurations."""
        if has_res and N <= 512:
            return 5128 if M >= 3000 else 6064
        if not has_res and N >= 2048 and M < 3000:
            return 3256
        return 0

    def _lin_bwd(self, ws, wname, x_saved, g, *, count=1, h=None, p=0.0, site=0, dx=None, dx_residual=None, g_ready=None, pre=None,
                 dx_next=None):
        """Backward of y = drop(act(x W^T + b)).  g: fp32 [M,N] gradient wrt the layer output (after dropout);
        h: saved post-activation output when the layer has ReLU (mask = h != 0, which also covers its dropout);
        p/site: dropout to regenerate when h is None.  g_ready: (gb, None) when the gradient is already in the
        activation dtype and needs no masking (generator).  dx (fp32 [M,K]) receives g' (W.m) [+ dx_residual]."""
        W, S, mode, U, seed, stream = self._mask_args(wname, count)
        N, Kd = W.shape
        M = x_saved.shape[0]
        Mp = K.pad8(M)
        p = p if self.training else 0.0
        bname = wname.replace(".weight", ".bias")
        gbias = self._group(self.g, bname, count) if bname in self.g else None
        # bf16: the weight-gradient GEMM reads dy [M,N] and x [M,K] as MN-major tiles - no transposed copies, no padding
        rowmajor = self.adt == torch.bfloat16 and N % 8 == 0 and Kd % 8 == 0
        gT = None if rowmajor else ws.gT[: N * Mp].view(N, Mp)
        side = rowmajor and len(ws.gb_ring) > 1
        slot = None
        if pre is not None:
            # the LayerNorm backward that produced g already wrote the masked bf16 operand and the bias gradient (_ln_bwd)
            gb, slot = pre
        elif g_ready is not None:
            gb = g_ready
            if not rowmajor:
                if Mp != M:
                    gT[:, M:].zero_()
                K.transpose(gb, gT)
            if gbias is not None:
                K.colsum(gb, gbias)
        else:
            if side:
                gb, slot = self._take_gb(ws, M, N)
            else:
                gb = ws.gb[: M * N].view(M, N)
            if not rowmajor and Mp != M:
                gT[:, M:].zero_()
            # the bias gradient (column sums) is accumulated by the same pass (flat_gw is zeroed at the start of the backward)
            K.prep_grad(g, h=h, out=gb, outT=gT, scale=(1.0 / (1.0 - p)) if (h is not None and p > 0) else 1.0,
                        p=0.0 if h is not None else p, seed=self._sd(1), stream_id=self._drop_stream(site), colsum=gbias)
        nxt_pre = None
        if dx is not None:
            wT = self._wmT.get((wname, count)) if (self.adt == torch.bfloat16 and self.premask and self.training) else None
            if wT is None:
                wT = ws.wT[: Kd * N].view(Kd, N)
                K.apply_mask_transposed(W, S, mode, wT, uniforms=U, seed=seed, stream_id=stream)
            if dx_next is not None and self.fuse_hmask and side and dx_residual is None and Kd % 8 == 0:
                # this linear's input was h = dropout(relu(previous linear)): the dX GEMM's epilogue applies that mask, stores
                # the bf16 gradient operand of the previous linear straight into a ring buffer and accumulates its bias
                # gradient (sc_linear_hmask) - no fp32 dX tensor, no separate sc_prep_grad pass
                hm, scale, next_wname = dx_next
                gb_next, slot_next = self._take_gb(ws, M, Kd)
                K.linear_hmask(gb, wT, hm, gb_next, scale=scale, colsum=self.g[next_wname.replace(".weight", ".bias")])
                nxt_pre = (gb_next, slot_next)
            else:
                K.linear(gb, wT, None, residual=dx_residual, out=dx, tile_n=5128 if (N >= 8192 and Kd <= 512) else 0)  # generator dX
        gW = self._group(self.g, wname, count)
        gS = self._group(self.gs, wname, count) if S is not None else None
        if self.fused_st:
            S, gS, mode, U = None, None, K.MASK_NONE, None  # the weight gradient stays dWm; sc_adam_clip_st applies the mask
        if side:
            # fork after the gradient operand exists (the dX GEMM above only reads it), join before the optimizer
            main, st = torch.cuda.current_stream(self.dev), self._side_stream()
            ev = torch.cuda.Event()
            ev.record(main)
            st.wait_event(ev)
            with torch.cuda.stream(st):
                if not self._diag_skip_wgrad:
                    K.linear_wgrad_rowmajor(gb, x_saved, W, S, mode, gW, gS, workspace=ws.wgrad_ws, uniforms=U, seed=seed,
                                            stream_id=stream, bypass=self.bypass)
                if slot is not None:
                    ws.gb_free[slot] = torch.cuda.Event()
                    ws.gb_free[slot].record(st)
            ws.side_used = True
            return nxt_pre
        if rowmajor:
            K.linear_wgrad_rowmajor(gb, x_saved, W, S, mode, gW, gS, workspace=ws.wgrad_ws, uniforms=U, seed=seed, stream_id=stream,
                                    bypass=self.bypass)
            return
        xT = ws.xT[: Kd * Mp].view(Kd, Mp)
        if Mp != M:
            xT[:, M:].zero_()
        K.transpose(x_saved, xT)
        K.linear_wgrad(gT, xT, W, S, mode, gW, gS, M=Mp, uniforms=U, seed=seed, stream_id=stream, bypass=self.bypass,
                       workspace=ws.wgrad_ws if self.adt == torch.bfloat16 else None)

    def _ln(self, name, x, out):
        return K.layernorm(x, self.p[name + ".a_2"], self.p[name + ".b_2"], out=out)

    def _attn_fused(self, ws):
        """attention backward writes bf16 gradient operands + bias gradients itself (tensor path: bf16, d_k = 64, ring)."""
        c = self.cfg
        return (self.fuse_attn_bwd and self.adt == torch.bfloat16 and c.d_model // c.num_heads == 64 and len(ws.gb_ring) > 1
                and ws.N <= 128 and ws.T <= 128)

    def _take_gb(self, ws, M, N):
        """Next gradient-operand buffer of the ring (waits for the side-stream consumer that used it last)."""
        slot = ws.gb_next
        ws.gb_next = (slot + 1) % len(ws.gb_ring)
        if ws.gb_free[slot] is not None:
            torch.cuda.current_stream(self.dev).wait_event(ws.gb_free[slot])
        return ws.gb_ring[slot][: M * N].view(M, N), slot

    def _ln_bwd(self, name, x, dy, dx, dres=None, nxt=None, ws=None):
        """Backward of LayerNorm `name`.  ``nxt = (weight name, dropout site)``: the linear whose output gradient is dx
        comes next in the backward chain - its bf16 gradient operand (dropout mask regenerated) and bias gradient are
        produced by the same kernel; returns ``pre`` for ``_lin_bwd`` (None when not fused)."""
        d = x.shape[1]
        if nxt is None or self.adt != torch.bfloat16 or d != 512 or len(ws.gb_ring) < 2:
            K.layernorm_bwd(x, self.p[name + ".a_2"], dy, dx, self.g[name + ".a_2"], self.g[name + ".b_2"], dres=dres)
            return None
        wname, site = nxt
        gb, slot = self._take_gb(ws, x.shape[0], d)
        gbias = self.g[wname.replace(".weight", ".bias")]
        K.layernorm_bwd(x, self.p[name + ".a_2"], dy, dx, self.g[name + ".a_2"], self.g[name + ".b_2"], dres=dres, next_gb=gb,
                        next_colsum=gbias, next_p=self._pd(), seed=self._sd(1), stream_id=self._drop_stream(site))
        return gb, slot

    def _pd(self):
        return self.p_drop if self.training else 0.0

    # ---------------------------------------------------------------------------------------------------------
    def load_batch(self, ws, att_feats, boxes, seqs, masks, att_masks=None, global_tokens=None):
        c = self.cfg
        B, N, S, T = ws.B, ws.N, ws.S, ws.T
        ws.att_in.copy_(att_feats.reshape(B * N, -1), non_blocking=True)
        ws.boxes.copy_(boxes, non_blocking=True)
        if att_masks is not None:
            ws.att_mask.copy_(att_masks.float(), non_blocking=True)
        seqs = seqs.to(self.dev, non_blocking=True)
        masks = masks.to(self.dev, non_blocking=True).float()
        tok = seqs[:, :T].contiguous()
        ws.tokens.copy_(tok.reshape(-1).int())
        ws.targets.copy_(seqs[:, 1: T + 1].reshape(-1).int())
        ws.tok_w.copy_(masks[:, 1: T + 1].reshape(-1))
        ws.key_valid.copy_((tok != c.pad_token_id).float())
        denom = masks[:, 1: T + 1].sum() if global_tokens is None else global_tokens
        ws.inv_norm.copy_((1.0 / denom).reshape(1))

    def forward(self, ws):
        """Teacher-forcing forward; leaves logits in ws.logits and every activation the backward needs."""
        c = self.cfg
        B, N, S, T, ME, MD, R = ws.B, ws.N, ws.S, ws.T, ws.ME, ws.MD, ws.R
        d, h, L = c.d_model, c.num_heads, c.num_layers
        dk = d // h
        pd = self._pd()
        trig = not c.no_box_trigonometric_embedding
        es, ds = _SITES["encoder"], _SITES["decoder"]
        if ws.att_a is not ws.att_in:
            K.cast_bf16(ws.att_in, out=ws.att_a)
        if self.adt == torch.bfloat16 and self.premask and self.training and not self._scst:
            self._premask_all()
        self._lin("att_embed.0.weight", ws.att_a, ws.xe[0], relu=True, p=self.p_src, site=_SITES["att_embed"])
        if ws.att_mask is not None:
            K.mask_rows(ws.xe[0], ws.att_mask.view(-1))
        # effective (masked) WG weights of every layer, then the log-geometry bias of all layers and heads in ONE pass over
        # the box pairs (the sin/cos embedding only depends on the boxes; the reference rebuilds it in each layer)
        for l in range(L):
            Wg, Sg, mode, U, seed, stream = self._mask_args(f"model.encoder.layers.{l}.self_attn.WGs.0.weight", h)
            if Sg is None:
                ws.wg_eff[l].copy_(Wg)
            else:
                K.apply_mask(Wg, Sg, mode, uniforms=U, seed=seed, stream_id=stream, out=ws.wg_eff[l])
        if ws.wg_b_all is not None:
            K.box_bias_all(ws.boxes, ws.wg_eff_all, ws.wg_b_all, ws.e_bias_all, B=B, N=N, layers=L, h=h, trig=trig)
        for l in range(L):
            p = f"model.encoder.layers.{l}"
            x0, x1, x2 = ws.xe[2 * l], ws.xe[2 * l + 1], ws.xe[2 * l + 2]
            self._ln(f"{p}.sublayer.0.norm", x0, ws.e_xn1[l])
            self._lin(f"{p}.self_attn.linears.0.weight", ws.e_xn1[l], ws.e_qkv[l], count=3)
            if ws.wg_b_all is None:
                K.box_bias_fwd(ws.boxes, ws.wg_eff[l], self._group(self.p, f"{p}.self_attn.WGs.0.bias", h), ws.e_bias[l], B=B, N=N,
                               h=h, trig=trig)
            q = ws.e_qkv[l]
            K.attention_fwd(q[:, 0:], q[:, d:], q[:, 2 * d:], ws.e_att[l], ws.e_probs[l], G=B, Tq=N, Tk=N, h=h, dk=dk, ldq=3 * d,
                            ldk=3 * d, ldv=3 * d, ldo=d, key_valid=ws.att_mask, bias=ws.e_bias[l], p=pd, seed=self._sd(2),
                            stream_id=self._drop_stream(es["attn"] + l))
            self._lin(f"{p}.self_attn.linears.3.weight", ws.e_att[l], x1, residual=x0, p=pd, site=es["o"] + l)
            self._ln(f"{p}.sublayer.1.norm", x1, ws.e_xn2[l])
            self._lin(f"{p}.feed_forward.w_1.weight", ws.e_xn2[l], ws.e_hid[l], relu=True, p=pd, site=es["ff1"] + l)
            self._lin(f"{p}.feed_forward.w_2.weight", ws.e_hid[l], x2, residual=x1, p=pd, site=es["ff2"] + l)
        self._ln("model.encoder.norm", ws.xe[2 * L], ws.mem)
        for l in range(L):
            self._lin(f"model.decoder.layers.{l}.src_attn.linears.1.weight", ws.mem, ws.memkv[l], count=2)
        # ---- decoder ----
        W, S_, mode, U, seed, stream = self._mask_args("model.tgt_embed.0.lut.weight")
        K.embed_pe(ws.tokens, W, self.pe, T=T, pos0=0, mask=S_, mask_mode=mode, uniforms=U, seed=seed, stream_id=stream, out=ws.y[0])
        if pd > 0:
            K.prep_grad(ws.y[0], out=ws.y[0], p=pd, seed=self._sd(1), stream_id=self._drop_stream(_SITES["embed"]))
        for l in range(L):
            p = f"model.decoder.layers.{l}"
            y0, y1, y2, y3 = ws.y[3 * l], ws.y[3 * l + 1], ws.y[3 * l + 2], ws.y[3 * l + 3]
            self._ln(f"{p}.sublayer.0.norm", y0, ws.d_yn1[l])
            self._lin(f"{p}.self_attn.linears.0.weight", ws.d_yn1[l], ws.d_qkv[l], count=3)
            q = ws.d_qkv[l]
            K.attention_fwd(q[:, 0:], q[:, d:], q[:, 2 * d:], ws.d_att[l], ws.d_probs[l], G=R, Tq=T, Tk=T, h=h, dk=dk, ldq=3 * d,
                            ldk=3 * d, ldv=3 * d, ldo=d, key_valid=ws.key_valid, causal_T=T, p=pd, seed=self._sd(2),
                            stream_id=self._drop_stream(ds["attn"] + l))
            self._lin(f"{p}.self_attn.linears.3.weight", ws.d_att[l], y1, residual=y0, p=pd, site=ds["o"] + l)
            self._ln(f"{p}.sublayer.1.norm", y1, ws.d_yn2[l])
            self._lin(f"{p}.src_attn.linears.0.weight", ws.d_yn2[l], ws.d_qc[l])
            kv = ws.memkv[l]
            K.attention_fwd(ws.d_qc[l], kv[:, 0:], kv[:, d:], ws.d_catt[l], ws.c_probs[l], G=B, Tq=S * T, Tk=N, h=h, dk=dk, ldq=d,
                            ldk=2 * d, ldv=2 * d, ldo=d, key_valid=ws.att_mask, p=pd, seed=self._sd(2),
                            stream_id=self._drop_stream(ds["cattn"] + l))
            self._lin(f"{p}.src_attn.linears.3.weight", ws.d_catt[l], y2, residual=y1, p=pd, site=ds["co"] + l)
            self._ln(f"{p}.sublayer.2.norm", y2, ws.d_yn3[l])
            self._lin(f"{p}.feed_forward.w_1.weight", ws.d_yn3[l], ws.d_hid[l], relu=True, p=pd, site=ds["ff1"] + l)
            self._lin(f"{p}.feed_forward.w_2.weight", ws.d_hid[l], y3, residual=y2, p=pd, site=ds["ff2"] + l)
        self._ln("model.decoder.norm", ws.y[3 * L], ws.yf)
        self._lin("model.generator.proj.weight", ws.yf, ws.logits)
        return ws.logits

    def loss_and_backward(self, ws):
        """LanguageModelCriterion + full backward; gradients land in flat_gw / flat_gs (overwritten, not accumulated)."""
        for phase in range(self.N_PHASES):
            self.backward_phase(ws, phase)
        return ws.loss_sum

    # The backward in three phases whose gradients are final when the phase ends, so that a data-parallel run can start
    # the all-reduce of a finished bucket while the next phase computes (grad_buckets):
    #   0: loss, generator, decoder norm, decoder layers L-1 .. L/2     1: decoder layers L/2-1 .. 0, embedding
    #   2: encoder norm, encoder layers L-1 .. L/2                      3: encoder layers L/2-1 .. 0, att_embed
    N_PHASES = 4

    def grad_buckets(self, phase):
        """[(flat gradient buffer, start, end)] of the parameter ranges whose gradients are final after `phase`."""
        L = self.cfg.num_layers
        half = L // 2
        def rng(offs, keys, first, last):
            # [offset of `first`, offset of `last`) in a layout; names that are not in the layout (norms / biases in the
            # logit layout) move forward to the next name that is
            def at(name):
                if name is None:
                    return None
                i = self.names.index(name)
                while i < len(self.names) and self.names[i] not in offs:
                    i += 1
                return offs[self.names[i]] if i < len(self.names) else None
            return at(first), at(last)
        dec0, dech = _DEC0, f"model.decoder.layers.{half}.self_attn.linears.0.weight"
        lut, gen = "model.tgt_embed.0.lut.weight", "model.generator.proj.weight"
        ench = f"model.encoder.layers.{half}.self_attn.linears.0.weight"
        spans = {0: [(dech, lut), (gen, None)], 1: [(dec0, dech), (lut, gen)], 2: [(ench, dec0)], 3: [(self.names[0], ench)]}[phase]
        out = []
        for flat, offs in ((self.flat_gw, self._offs_w), (self.flat_gs, self._offs_s) if (self.masked and not self.fused_st) else (None, None)):
            if flat is None:
                continue
            for first, last in spans:
                a, b = rng(offs, None, first, last)
                a = 0 if a is None else a
                b = flat.numel() if b is None else b
                if b > a:
                    out.append((flat, a, b))
        return out

    def backward_phase(self, ws, phase):
        d, L = self.cfg.d_model, self.cfg.num_layers
        pd = self._pd()
        ws.gb_free = [None] * len(ws.gb_ring)
        ws.gb_next = 0
        ws.side_used = False
        stack = "decoder" if phase < 2 else "encoder"
        last_ff2 = (f"model.{stack}.layers.{L - 1}.feed_forward.w_2.weight", _SITES[stack]["ff2"] + L - 1)
        pre = None  # (a phase starts with a plain gradient preparation: the ring was reset)
        if phase == 0:
            self._materialized = False
            # norm and bias gradients accumulate through atomics: one memset of the flat buffer (weights are overwritten)
            self.flat_gw.zero_()
            ws.loss_sum.zero_()
            K.logsoftmax_nll(ws.logits, ws.targets, ws.tok_w, ws.inv_norm, ws.loss_sum, ws.dlogits)
            ga_d = ws.ga.view(-1)[: ws.MD * d].view(ws.MD, d)
            self._lin_bwd(ws, "model.generator.proj.weight", ws.yf, None, g_ready=ws.dlogits, dx=ga_d)
            ws.cur = 0
            pre = self._ln_bwd("model.decoder.norm", ws.y[3 * L], ga_d, ws.dres[0][:ws.MD], ws=ws, nxt=last_ff2)
            ws.dmem.zero_()
        elif phase == 2:
            ws.cur = 0
            pre = self._ln_bwd("model.encoder.norm", ws.xe[2 * L], ws.dmem, ws.dres[0][:ws.ME], ws=ws, nxt=last_ff2)
        cur = self._backward_layers(ws, stack, range(L // 2, L) if phase % 2 == 0 else range(L // 2), pre)
        if phase == 1:
            # embedding: its dropout mask is regenerated from the forward's Philox stream (an exact zero in the saved output is
            # not proof of a dropped element: sin(0) = 0 in the positional encoding, masked-out table entries)
            W, S_, mode, U, seed, stream = self._mask_args("model.tgt_embed.0.lut.weight")
            emb_g = ws.ga.view(-1)[: ws.MD * d].view(ws.MD, d)
            if pd > 0:
                K.prep_grad(cur, out=emb_g, p=pd, seed=self._sd(1), stream_id=self._drop_stream(_SITES["embed"]))
            else:
                emb_g = cur
            if self.fused_st:
                # (flat_gw was zeroed at the start of the backward: the scatter-add lands directly in the table's gradient view)
                K.embedding_bwd(ws.tokens, emb_g, self.g["model.tgt_embed.0.lut.weight"], math.sqrt(d))
            else:
                ws.dtable.zero_()
                K.embedding_bwd(ws.tokens, emb_g, ws.dtable, math.sqrt(d))
                K.mask_grad(ws.dtable, W, S_, mode, self.g["model.tgt_embed.0.lut.weight"],
                            self.gs.get("model.tgt_embed.0.lut.weight"), uniforms=U, seed=seed, stream_id=stream, bypass=self.bypass)
        elif phase == 3:
            if ws.att_mask is not None:
                K.mask_rows(cur, ws.att_mask.view(-1))
            self._lin_bwd(ws, "att_embed.0.weight", ws.att_a, cur, h=ws.xe[0], p=self.p_src if self.training else 0.0)
        self._join_side(ws)

    def _join_side(self, ws):
        if ws.side_used:
            torch.cuda.current_stream(self.dev).wait_stream(self._side_stream())
            ws.side_used = False

    def _backward_layers(self, ws, stack, layers, pre):
        """Backward of `layers` of a stack, last first: each sublayer reads the residual-stream gradient from `cur`, its LayerNorm
        backward writes it plus the sublayer's input gradient to `nxt` (ping-pong over ws.dres; ws.cur: the current one)."""
        s, M = _SITES[stack], ws.MD if stack == "decoder" else ws.ME
        cur, nxt = ws.dres[ws.cur][:M], ws.dres[1 - ws.cur][:M]
        for l in reversed(layers):
            p = f"model.{stack}.layers.{l}"
            o = (f"{p}.self_attn.linears.3.weight", s["o"] + l)   # (an _ln_bwd hand-off: weight, dropout site)
            if stack == "decoder":
                pre = self._ff_bwd(ws, stack, l, cur, nxt, pre, (f"{p}.src_attn.linears.3.weight", s["co"] + l))
                cur, nxt = nxt, cur
                pre = self._cross_attn_bwd(ws, l, cur, nxt, pre, o)
            else:
                pre = self._ff_bwd(ws, stack, l, cur, nxt, pre, o)
            cur, nxt = nxt, cur
            # (the previous layer's w_2 only within this phase: the next one starts with a reset ring)
            ff2 = (f"model.{stack}.layers.{l - 1}.feed_forward.w_2.weight", s["ff2"] + l - 1) if l > layers[0] else None
            pre = self._self_attn_bwd(ws, stack, l, cur, nxt, pre, ff2)
            cur, nxt = nxt, cur
        ws.cur = 0 if cur.data_ptr() == ws.dres[0].data_ptr() else 1
        return cur

    def _ff_bwd(self, ws, stack, l, cur, nxt, pre, then):
        """Feed-forward sublayer: w_2 (its dX GEMM prepares w_1's gradient operand), w_1, LayerNorm (``then``: its _ln_bwd nxt)."""
        p, pd = f"model.{stack}.layers.{l}", self._pd()
        if stack == "decoder":
            x, xn, hid, norm = ws.y[3 * l + 2], ws.d_yn3[l], ws.d_hid[l], f"{p}.sublayer.2.norm"
        else:
            x, xn, hid, norm = ws.xe[2 * l + 1], ws.e_xn2[l], ws.e_hid[l], f"{p}.sublayer.1.norm"
        (M, ff), d = hid.shape, x.shape[1]
        ga_ff = ws.ga.view(-1)[: M * ff].view(M, ff)
        pre1 = self._lin_bwd(ws, f"{p}.feed_forward.w_2.weight", hid, cur, p=pd, site=_SITES[stack]["ff2"] + l, dx=ga_ff, pre=pre,
                             dx_next=(hid, 1.0 / (1.0 - pd) if pd > 0 else 1.0, f"{p}.feed_forward.w_1.weight"))
        ga = ws.gq.view(-1)[: M * d].view(M, d)
        self._lin_bwd(ws, f"{p}.feed_forward.w_1.weight", xn, ga_ff, h=hid, p=pd, dx=ga, pre=pre1)
        return self._ln_bwd(norm, x, ga, nxt, dres=cur, ws=ws, nxt=then)

    def _self_attn_bwd(self, ws, stack, l, cur, nxt, pre, then):
        """Self-attention sublayer: output linear, attention (encoder: + the geometry bias), [q;k;v], LayerNorm."""
        p = f"model.{stack}.layers.{l}"
        enc = stack == "encoder"
        if enc:
            x, xn, qkv, probs, att, G, T = ws.xe[2 * l], ws.e_xn1[l], ws.e_qkv[l], ws.e_probs[l], ws.e_att[l], ws.B, ws.N
        else:
            x, xn, qkv, probs, att, G, T = ws.y[3 * l], ws.d_yn1[l], ws.d_qkv[l], ws.d_probs[l], ws.d_att[l], ws.R, ws.T
        M, d = x.shape
        ga, gq = ws.ga.view(-1)[: M * d].view(M, d), ws.gq[:M]
        self._lin_bwd(ws, f"{p}.self_attn.linears.3.weight", att, cur, p=self._pd(), site=_SITES[stack]["o"] + l, dx=ga, pre=pre)
        pre_qkv, = self._attn_bwd(ws, f"{p}.self_attn", qkv, qkv[:, d:], probs, ga, gq, gq[:, d:], G=G, Tq=T, Tk=T,
                                  site=_SITES[stack]["attn"] + l, dbias=ws.dbias if enc else None)
        if enc:
            self._box_bias_bwd(ws, l)
        self._lin_bwd(ws, f"{p}.self_attn.linears.0.weight", xn, gq, count=3, dx=ga, pre=pre_qkv)
        return self._ln_bwd(f"{p}.sublayer.0.norm", x, ga, nxt, dres=cur, ws=ws, nxt=then)

    def _cross_attn_bwd(self, ws, l, cur, nxt, pre, then):
        """Decoder cross-attention sublayer: output linear, attention, q, LayerNorm, then the memory's [k;v] (into ws.dmem)."""
        p, MD, d = f"model.decoder.layers.{l}", ws.MD, self.cfg.d_model
        ga, dq = ws.ga.view(-1)[: MD * d].view(MD, d), ws.gq.view(-1)[: MD * d].view(MD, d)
        self._lin_bwd(ws, f"{p}.src_attn.linears.3.weight", ws.d_catt[l], cur, p=self._pd(), site=_SITES["decoder"]["co"] + l, dx=ga,
                      pre=pre)
        pre_q, pre_kv = self._attn_bwd(ws, f"{p}.src_attn", ws.d_qc[l], ws.memkv[l], ws.c_probs[l], ga, dq, ws.dmemkv, G=ws.B,
                                       Tq=ws.S * ws.T, Tk=ws.N, site=_SITES["decoder"]["cattn"] + l)
        self._lin_bwd(ws, f"{p}.src_attn.linears.0.weight", ws.d_yn2[l], dq, dx=ga, pre=pre_q)
        pre = self._ln_bwd(f"{p}.sublayer.1.norm", ws.y[3 * l + 1], ga, nxt, dres=cur, ws=ws, nxt=then)
        self._lin_bwd(ws, f"{p}.src_attn.linears.1.weight", ws.mem, ws.dmemkv, count=2, dx=ws.dmem, dx_residual=ws.dmem, pre=pre_kv)
        return pre

    def _attn_bwd(self, ws, pa, q, kv, probs, dout, dq, dkv, *, G, Tq, Tk, site, dbias=None):
        """Attention backward of module `pa`: fp32 dq / d[k;v], or (_attn_fused) bf16 gradient operands with the bias gradients.
        Returns the _lin_bwd ``pre`` of ([q;k;v],) (self-attention: kv is a view of q) or of (q, [k;v]) (cross-attention)."""
        d, h = self.cfg.d_model, self.cfg.num_heads
        packed = pa.endswith("self_attn")
        kw = dict(G=G, Tq=Tq, Tk=Tk, h=h, dk=d // h, ldq=q.stride(0), ldk=kv.stride(0), ldv=kv.stride(0), ldd=d, dbias=dbias,
                  p=self._pd(), seed=self._sd(2), stream_id=self._drop_stream(site))
        if not self._attn_fused(ws):
            K.attention_bwd(q[:, 0:], kv[:, 0:], kv[:, d:], probs, dout, dq[:, 0:], dkv[:, 0:], dkv[:, d:], dtype=self.adt,
                            ldgq=dq.stride(0), ldgk=dkv.stride(0), ldgv=dkv.stride(0), **kw)
            return (None,) if packed else (None, None)
        if packed:
            gb, slot = self._take_gb(ws, q.shape[0], 3 * d)
            gq, gkv, pre = gb, gb[:, d:], ((gb, slot),)
        else:
            pre = self._take_gb(ws, q.shape[0], d), self._take_gb(ws, kv.shape[0], 2 * d)
            (gq, _), (gkv, _) = pre
        bkv = self._group(self.g, f"{pa}.linears.1.bias", 2)
        K.attention_bwd_bf16out(q[:, 0:], kv[:, 0:], kv[:, d:], probs, dout, gq[:, 0:], gkv[:, 0:], gkv[:, d:], ldgq=gq.stride(0),
                                ldgk=gkv.stride(0), ldgv=gkv.stride(0), bq=self.g[f"{pa}.linears.0.bias"], bk=bkv[:d], bv=bkv[d:], **kw)
        return pre

    def _box_bias_bwd(self, ws, l):
        """Geometry-bias backward of encoder layer l: WG bias gradients and dWm (fused_st) or dW / dS (sc_mask_grad) of its heads."""
        h, wg = self.cfg.num_heads, f"model.encoder.layers.{l}.self_attn.WGs.0.weight"
        gb_wg = self._group(self.g, f"model.encoder.layers.{l}.self_attn.WGs.0.bias", h)
        gb_wg.zero_()
        dwg = self._group(self.g, wg, h) if self.fused_st else ws.dwg
        dwg.zero_()
        K.box_bias_bwd(ws.boxes, ws.e_bias[l], ws.dbias, dwg, gb_wg, B=ws.B, N=ws.N, h=h, trig=not self.cfg.no_box_trigonometric_embedding)
        if not self.fused_st:
            Wg, Sg, mode, U, seed, stream = self._mask_args(wg, h)
            K.mask_grad(ws.dwg, Wg, Sg, mode, self._group(self.g, wg, h), self._group(self.gs, wg, h) if Sg is not None else None,
                        uniforms=U, seed=seed, stream_id=stream, bypass=self.bypass)

    # ---------------------------------------------------------------------------------------------------------
    def optimizer_step(self, *, lr, mask_lr=100.0, clip=0.1, betas=(0.9, 0.98), eps=1e-9, mask_eps=1e-2, weight_decay=0.0,
                       grad_scale=1.0, sparsity_target=None, sparsity_weight=0.0, current_step=0, max_step=1, _dyn=False, part="all"):
        """clip_gradient(0.1) + Adam for the two parameter groups of train_n_prune_transformer.py:67-82, with the
        sparsity-loss gradient (prune.py:228-269) folded into the mask-logit update.  ``_dyn``: graph mode - lr, the Adam
        bias corrections and the sparsity scale come from ``self._dyn_dev`` (``_upload_step``), no host bookkeeping.
        ``part``: "all", or the two halves of an overlapped update - "hi" = decoder + embedding + generator (their gradients are
        final after backward phase 1; also computes the sparsity coefficient, which must see the logits before ANY update),
        "lo" = att_embed + encoder (after the last phase; also re-pins the padding logits)."""
        if not _dyn and part != "lo":
            self.opt_step += 1
            self._hyper = _adam_hyper(lr, dict(mask_lr=mask_lr, betas=betas, eps=eps, mask_eps=mask_eps, weight_decay=weight_decay))
        dyn = self._dyn_dev if _dyn else None
        if self.fused_st and not self._materialized:
            return self._optimizer_step_st(lr=lr, mask_lr=mask_lr, clip=clip, betas=betas, eps=eps, mask_eps=mask_eps,
                                           weight_decay=weight_decay, grad_scale=grad_scale, sparsity_target=sparsity_target,
                                           sparsity_weight=sparsity_weight, current_step=current_step, max_step=max_step, dyn=dyn, part=part)
        lo_w, hi_w = _part(self.flat_w.numel(), self._cut_w, part)
        K.adam_clip(self.flat_w[lo_w:hi_w], self.flat_gw[lo_w:hi_w], self.m_w[lo_w:hi_w], self.v_w[lo_w:hi_w], lr=lr, betas=betas, eps=eps,
                    weight_decay=weight_decay, clip=clip, grad_scale=grad_scale, step=max(1, self.opt_step),
                    dyn=dyn[0:3] if _dyn else None)
        if self.masked and self.mask_type == "supermask":
            coeff = self._sparsity_coeff(sparsity_target=sparsity_target, sparsity_weight=sparsity_weight, current_step=current_step,
                                         max_step=max_step, scale_dev=dyn[6:7] if _dyn else None, part=part)
            lo_s, hi_s = _part(self.flat_s.numel(), self._cut_s, part)
            K.adam_clip(self.flat_s[lo_s:hi_s], self.flat_gs[lo_s:hi_s], self.m_s[lo_s:hi_s], self.v_s[lo_s:hi_s], lr=mask_lr, betas=betas,
                        eps=mask_eps, weight_decay=0.0, clip=clip, grad_scale=grad_scale, step=max(1, self.opt_step),
                        sigmoid_grad_coeff=coeff, dyn=dyn[3:6] if _dyn else None)
            if part != "hi" and self._s_pad_idx.numel():
                self.flat_s.index_fill_(0, self._s_pad_idx, -1.0)

    def _mask_groups(self):
        """(first weight name, fused count) of every masked tensor exactly as the forward samples it (one Philox stream and one
        element numbering per group): the linears of _premask_keys, the embedding table, the h geometry heads of each layer."""
        h = self.cfg.num_heads
        groups = list(self._premask_keys()) + [("model.tgt_embed.0.lut.weight", 1)]
        groups += [(f"model.encoder.layers.{l}.self_attn.WGs.0.weight", h) for l in range(self.cfg.num_layers)]
        return groups

    def _st_table(self, part):
        """Descriptor table of sc_adam_clip_st for "all" / "hi" (decoder, embedding, generator) / "lo" (att_embed, encoder)."""
        if part not in self._st_desc:
            first_of = {}
            member = set()
            if self.masked:
                for wname, count in self._mask_groups():
                    first_of[wname] = count
                    i = self.names.index(wname)
                    member.update(self.names[i + 1: i + count])  # (the fused members are consecutive names: [q;k;v], [k;v], WG heads)
            names = self.names[slice(*_part(len(self.names), self._cut, part))]
            segs = []
            for k in names:
                if k in member:
                    continue
                if k in first_of:
                    n = self._group(self.p, k, first_of[k]).numel()
                    segs.append((self._offs_w[k], self._offs_s[k], n, self.stream_of[k]))
                else:
                    n = self._group(self.p, k, 1).numel() if k in self._pad_rows else self.p[k].numel()
                    segs.append((self._offs_w[k], -1, n, 0))
            self._st_desc[part] = K.st_descriptors(segs, self.dev)
        return self._st_desc[part]

    def _optimizer_step_st(self, *, lr, mask_lr, clip, betas, eps, mask_eps, weight_decay, grad_scale, sparsity_target, sparsity_weight,
                           current_step, max_step, dyn, part):
        supermask = bool(self.masked) and self.mask_type == "supermask"
        coeff = self._sparsity_coeff(sparsity_target=sparsity_target, sparsity_weight=sparsity_weight, current_step=current_step,
                                     max_step=max_step, scale_dev=dyn[6:7] if dyn is not None else None, part=part)
        desc, blocks = self._st_table(part)
        mode = K.MASK_NONE  # the mask sample of the step being applied (train-mode forward)
        if self.masked:
            mode = (K.MASK_UNIFORM if self.flat_u is not None else K.MASK_BERNOULLI) if self.mask_type == "supermask" else K.MASK_RAW
        K.adam_clip_st(desc, blocks, self.flat_w, self.flat_gw, self.m_w, self.v_w, self.flat_s, self.m_s, self.v_s, uniforms=self.flat_u,
                       mask_mode=mode, bypass=self.bypass, update_logits=supermask, seed=self._sd(0), stream_base=self._step_base(),
                       lr=lr, eps=eps, weight_decay=weight_decay, mask_lr=mask_lr, mask_eps=mask_eps, betas=betas, clip=clip,
                       grad_scale=grad_scale, step=max(1, self.opt_step), sigmoid_grad_coeff=coeff, dyn=dyn)
        if supermask and part != "hi" and self._s_pad_idx.numel():
            self.flat_s.index_fill_(0, self._s_pad_idx, -1.0)

    def materialize_grads(self):
        """Reference ``.grad`` semantics for inspection: turns the dWm left by the backward into dW (in place, ``self.g``) and dS
        (``self.gs``) with the step's mask sample; a following ``optimizer_step`` then runs the plain two-group update on them."""
        if not self.fused_st or self._materialized or not self.masked:
            self._materialized = True
            return
        for wname, count in self._mask_groups():
            W, S, mode, U, seed, stream = self._mask_args(wname, count)
            gW = self._group(self.g, wname, count)
            K.mask_grad(gW, W, S, mode, gW, self._group(self.gs, wname, count), uniforms=U, seed=seed, stream_id=stream, bypass=self.bypass)
        self._materialized = True

    def _sparsity_coeff(self, *, sparsity_target=None, sparsity_weight=0.0, current_step=0, max_step=1, scale_dev=None, part="all",
                        **_):
        """Device scalar d(sparsity loss)/d(nnz) from the CURRENT logits (must run before any logit is updated; the "lo" half of
        an overlapped update reuses the one its "hi" half computed), None without a sparsity loss.  ``scale_dev``: graph mode,
        the annealed loss weight is read from the device."""
        if not (self.masked and self.mask_type == "supermask") or sparsity_target is None or not sparsity_weight:
            return None
        if part != "lo":
            K.mask_count([self.flat_s], out=self.sp_count)
            K.sparsity_coeff(self.sp_count, self.n_logits, sparsity_target, sparsity_weight * (1.0 - _anneal(current_step, max_step)),
                             self.sp_out, scale_dev=scale_dev)
        return self.sp_out[1:2]

    def _sharded_step(self, ws, exchange, opt, lr):
        """Data-parallel step with the optimizer sharded over the ranks (distributed.ShardedExchange): after each backward
        phase the finished buckets go through reduce-scatter -> Adam on the owned shard -> all-gather on the exchange's
        stream while the next phase computes."""
        assert not self.fused_st, "ShardedExchange cuts tensors into rank shards: build the trainer with fused_st=False"
        o = dict(mask_lr=100.0, clip=0.1, betas=(0.9, 0.98), eps=1e-9, mask_eps=1e-2, weight_decay=0.0, grad_scale=1.0)
        o.update({k: v for k, v in opt.items() if k in o})
        coeff = self._sparsity_coeff(**opt)
        self.opt_step += 1
        step = max(1, self.opt_step)

        def upd_w(lo, hi):
            K.adam_clip(self.flat_w[lo:hi], self.flat_gw[lo:hi], self.m_w[lo:hi], self.v_w[lo:hi], lr=lr, betas=o["betas"], eps=o["eps"],
                        weight_decay=o["weight_decay"], clip=o["clip"], grad_scale=o["grad_scale"], step=step)

        def upd_s(lo, hi):
            K.adam_clip(self.flat_s[lo:hi], self.flat_gs[lo:hi], self.m_s[lo:hi], self.v_s[lo:hi], lr=o["mask_lr"], betas=o["betas"],
                        eps=o["mask_eps"], weight_decay=0.0, clip=o["clip"], grad_scale=o["grad_scale"], step=step,
                        sigmoid_grad_coeff=coeff)

        exchange.finish()  # (the coefficient above must be ordered before the first bucket's update: same stream chain)
        for phase, part in enumerate(("fwd_p0", "p1", "p2", "p3")):
            if self.use_graph:
                self._run_graphed(ws, part, opt)
            else:
                if phase == 0:
                    self.forward(ws)
                self.backward_phase(ws, phase)
            for flat, a, b in self.grad_buckets(phase):
                if flat is self.flat_gw:
                    exchange.bucket(self.flat_gw, self.flat_w, a, b, upd_w)
                elif self.mask_type == "supermask":
                    exchange.bucket(self.flat_gs, self.flat_s, a, b, upd_s)
        exchange.finish()
        if self.masked and self.mask_type == "supermask" and self._s_pad_idx.numel():
            self.flat_s.index_fill_(0, self._s_pad_idx, -1.0)

    def _upload_step(self, *, lr, mask_lr=100.0, betas=(0.9, 0.98), sparsity_weight=0.0, current_step=0, max_step=1, **_):
        """Per-step scalars of the captured graph -> pinned host words -> device (two tiny async copies)."""
        self.opt_step += 1
        self._upload_seeds()
        bc1 = 1.0 - betas[0] ** self.opt_step
        bc2 = math.sqrt(1.0 - betas[1] ** self.opt_step)
        h = self._dyn_host
        h[0], h[1], h[2], h[3], h[4], h[5], h[6] = lr, bc1, bc2, mask_lr, bc1, bc2, sparsity_weight * (1.0 - _anneal(current_step, max_step))
        self._dyn_dev.copy_(self._dyn_host, non_blocking=True)

    def _upload_seeds(self):
        """The step's Philox seeds (masks, dropout, attention dropout) for the captured graphs."""
        for i in range(3):
            self._seeds_host[i] = self._step_seed(i)
        self._seeds_dev.copy_(self._seeds_host, non_blocking=True)

    def _step_seed(self, i):
        """Seed i of the current step (0-2: _sd's in graph mode, 3: the SCST sampler): a golden-ratio hash of the trainer seed and
        step_id, as a signed 64-bit word."""
        v = (self.seed + i + self.step_id * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        return v - (1 << 64) if v >= (1 << 63) else v

    def _graph_body(self, ws, part, opt):
        # every body (eager warm-up, capture) re-applies the masks - except an SCST body, whose masks the rollout already used
        self._wm_step = {key: (self.step_id, self.training) for key in self._premask_keys()} if self._scst else {}
        if part == "all" and self.overlap_opt:
            # the decoder-side half of the optimizer (64 % of the parameters) runs on its own stream underneath the encoder's
            # backward: its gradients are final after phase 1 and nothing the remaining phases read is touched
            self.forward(ws)
            self.backward_phase(ws, 0)
            self.backward_phase(ws, 1)
            main, ost = torch.cuda.current_stream(self.dev), self._opt_stream()
            ost.wait_stream(main)
            with torch.cuda.stream(ost):
                self.optimizer_step(_dyn=True, part="hi", **opt)
            self.backward_phase(ws, 2)
            self.backward_phase(ws, 3)
            main.wait_stream(ost)
            self.optimizer_step(_dyn=True, part="lo", **opt)
            return
        if part in ("all", "fwdbwd"):
            self.forward(ws)
            self.loss_and_backward(ws)
        if part == "fwd_p0":
            self.forward(ws)
            self.backward_phase(ws, 0)
        if part in ("p1", "p2", "p3"):
            self.backward_phase(ws, int(part[1]))
        if part in ("all", "opt"):
            self.optimizer_step(_dyn=True, **opt)
        if part in ("opt_hi", "opt_lo"):
            self.optimizer_step(_dyn=True, part=part[4:], **opt)

    def _exchange(self, all_reduce, phase, handles):
        """Start the all-reduce of every gradient bucket that `phase` finished (async: the next phase overlaps it)."""
        for flat, a, b in self.grad_buckets(phase):
            h = all_reduce(flat[a:b])
            if h is not None:
                handles.append((phase, h))

    @staticmethod
    def _wait(handles, phases):
        for ph, h in handles:
            if ph in phases:
                h.wait()

    def _run_graphed(self, ws, part, opt):
        key = (part, self._scst, tuple(sorted((k, float(v)) for k, v in opt.items() if k in ("clip", "eps", "mask_eps", "weight_decay",
                                                                                "grad_scale", "sparsity_target"))))
        graphs = ws.__dict__.setdefault("graphs", {})
        if key not in graphs:
            # the first step of a shape runs eagerly (it is a real step and also warms every kernel up), then the same
            # launch sequence is captured for all later steps
            self._graph_body(ws, part, opt)
            torch.cuda.synchronize(self.dev)
            g = torch.cuda.CUDAGraph()
            before = K.lib.launch_count
            with torch.cuda.graph(g):
                self._graph_body(ws, part, opt)
            graphs[key] = g
            # kernels of ours inside the captured graph: every replay launches this many (bench.py gpu_launches)
            ws.__dict__.setdefault("graph_launches", {})[key] = K.lib.launch_count - before
            return
        graphs[key].replay()
        K.lib.launch_count += ws.graph_launches[key]

    def train_step(self, att_feats, boxes, seqs, masks, att_masks=None, *, seq_per_img, lr, all_reduce=None, global_tokens=None,
                   exchange=None, **opt):
        """One full SMP step.  Data parallel: either ``all_reduce`` (callable applied to the gradient buckets, NCCL sum, every
        rank then runs the whole optimizer) or ``exchange`` (distributed.ShardedExchange: reduce-scatter -> Adam on the owned
        shard -> all-gather per bucket, overlapped with the backward)."""
        B, N = att_feats.shape[:2]
        T = seqs.shape[1] - 1
        ws = self._get_ws(B, N, seq_per_img, T, att_masks is not None)
        self.step_id += 1
        self._hyper = _adam_hyper(lr, opt)   # (graph mode and the sharded update do not go through optimizer_step's bookkeeping)
        # programmatic dependent launch, measured on this chain (ms/step): the GEMM's EARLY trigger (bit 2: dependents may start
        # once its loads are issued) costs time here, PDL with the implicit trigger at exit helps: mask 2 5.42, 3 5.30, 7 5.36
        with K.pdl(self.pdl_mask):
            self.load_batch(ws, att_feats, boxes, seqs, masks, att_masks, global_tokens)
            if exchange is not None and self.training:
                if self.use_graph:
                    self._upload_step(lr=lr, **opt)
                    self.opt_step -= 1  # (_sharded_step counts the step itself)
                self._sharded_step(ws, exchange, dict(opt, lr=lr) if self.use_graph else opt, lr)
                return ws.loss_sum * ws.inv_norm
            if self.use_graph and self.training:
                self._upload_step(lr=lr, **opt)
            return self._fwd_bwd_opt(ws, lr, all_reduce, opt)

    def _fwd_bwd_opt(self, ws, lr, all_reduce, opt):
        """Forward, backward (+ bucketed gradient exchange) and optimizer of a loaded workspace; graph mode expects
        ``_upload_step`` to have run for this step."""
        if self.use_graph and self.training:
            opt = dict(opt, lr=lr)
            if all_reduce is None:
                self._run_graphed(ws, "all", opt)
            else:
                # one graph per backward phase; the buckets a phase finished are exchanged while the next one computes
                # and the decoder-side half of the optimizer (its buckets arrived long ago) runs underneath the last buckets' exchange
                handles = []
                for phase, part in enumerate(("fwd_p0", "p1", "p2", "p3")):
                    self._run_graphed(ws, part, opt)
                    self._exchange(all_reduce, phase, handles)
                self._wait(handles, (0, 1))
                self._run_graphed(ws, "opt_hi", opt)
                self._wait(handles, (2, 3))
                self._run_graphed(ws, "opt_lo", opt)
            return ws.loss_sum * ws.inv_norm
        self.forward(ws)
        if all_reduce is None:
            self.loss_and_backward(ws)
        else:
            handles = []
            for phase in range(self.N_PHASES):
                self.backward_phase(ws, phase)
                self._exchange(all_reduce, phase, handles)
            self._wait(handles, (0, 1))
            self.optimizer_step(lr=lr, part="hi", **opt)
            self._wait(handles, (2, 3))
            self.optimizer_step(lr=lr, part="lo", **opt)
            return ws.loss_sum * ws.inv_norm
        self.optimizer_step(lr=lr, **opt)
        return ws.loss_sum * ws.inv_norm

    # ---- self-critical sequence training -------------------------------------------------------------------
    def rollout_engine(self, **engine_kw):
        """The inference engine of the SCST rollouts, built once and bound to this trainer's memory: bf16 linears read the
        step's pre-masked operands (``_wm``), biases and LayerNorm parameters are views of ``flat_w``; the masked embedding
        table and geometry weights (and, in fp32, every masked linear) are engine-owned and refreshed from the step's mask
        sample by ``_refresh_engine``.  The pointers never change, so its CUDA graphs replay across optimizer steps."""
        if self._rollout is None:
            self._rollout = self._bound_engine(eval_masks=False, **engine_kw)
        return self._rollout

    def _baseline_engine(self):
        """Supermask only: the greedy baseline decodes with eval-mode weights rint(sigmoid(S)), a second bound operand set."""
        if self._baseline is None:
            self._baseline = self._bound_engine(eval_masks=True)
        return self._baseline

    def _bound_engine(self, *, eval_masks, **engine_kw):
        from .engine import OrtEngine
        if engine_kw.get("ln_fold") or engine_kw.get("sparse_backend", "dense") != "dense":
            raise ValueError("the rollout engine reads the trainer's dense operands: ln_fold and the sparse backends are not supported")
        c, L, h = self.cfg, self.cfg.num_layers, self.cfg.num_heads
        sd = {k: self.p[k] for k in self.names}
        sd["model.tgt_embed.1.pe"] = self.pe[None]
        eng = OrtEngine(sd, c, precision="bf16" if self.adt == torch.bfloat16 else "fp32", device=self.dev, use_graphs=self.use_graph,
                        **engine_kw)
        lins = {("att_embed.0.weight", 1): eng.att_embed, ("model.generator.proj.weight", 1): eng.generator}
        norms = [(eng.enc_norm, "model.encoder.norm"), (eng.dec_norm, "model.decoder.norm")]
        for l in range(L):
            for stack, e, n_norms in (("encoder", eng.enc[l], 2), ("decoder", eng.dec[l], 3)):
                lins.update({(w, n): e[slot] for w, n, slot in self._groups[stack, l]})
                norms += [(e[f"n{j}"], f"model.{stack}.layers.{l}.sublayer.{j}.norm") for j in range(n_norms)]
        assert set(lins) == set(self._premask_keys())
        # bf16 rollouts read the trainer's own pre-masked operands; everything else is refreshed into engine-owned buffers
        share = self.adt == torch.bfloat16 and self.premask and not eval_masks
        if share and self._premask_desc is None:
            self._premask_all()   # (allocates _wm)
        items = {torch.bfloat16: [], torch.float32: []}

        def owned(wname, count, dtype):
            W = self._group(self.p, wname, count)
            out = torch.empty(W.shape, device=self.dev, dtype=dtype)
            S = self._group(self.s, wname, count) if self.mask_type else None
            items[dtype].append((W, S, self._u(wname, count), out, None, self.stream_of[wname]))
            return out

        for (wname, count), lin in lins.items():
            op = self._wm[(wname, count)] if share else owned(wname, count, self.adt)
            bias = self._group(self.p, wname.replace(".weight", ".bias"), count)
            assert op.shape[0] >= lin.N and op.shape[1] == lin.K and bias.shape[0] >= lin.N
            lin.w, lin.bias = op[: lin.N], bias[: lin.N]       # (generator: the first V rows of the padded operand)
        for nrm, name in norms:
            nrm.a, nrm.b = self.p[name + ".a_2"], self.p[name + ".b_2"]
        eng.table = owned("model.tgt_embed.0.lut.weight", 1, torch.float32)
        eng.wg_w_all = torch.empty_like(eng.wg_w_all)
        if self._wg_b_all is None:
            raise ValueError(f"the rollout engine needs the geometry biases packed in the trainer's layout (num_heads % 4 == 0, got {h})")
        eng.wg_b_all = self._wg_b_all
        for l in range(L):
            wname = f"model.encoder.layers.{l}.self_attn.WGs.0.weight"
            W = self._group(self.p, wname, h)
            out = eng.wg_w_all[l * h: (l + 1) * h]
            items[torch.float32].append((W, self._group(self.s, wname, h) if self.mask_type else None, self._u(wname, h), out, None,
                                         self.stream_of[wname]))
            eng.enc[l]["wg_w"], eng.enc[l]["wg_b"] = out, eng.wg_b_all[l * h: (l + 1) * h]
        eng.scst_refresh = [(K.mask_descriptors(it, self.dev), dt) for dt, it in items.items() if it]
        eng.scst_eval = eval_masks
        return eng

    def _scst_masks(self, eng):
        """Step 1 of an SCST step: the step's mask sample into the trainer's bf16 operands and the engine-owned ones (same seeds
        and Philox streams, so the rollout and the teacher-forced re-score see one network)."""
        if self.adt == torch.bfloat16 and self.premask:
            self._premask_all()
        self._refresh_engine(eng)

    def _refresh_engine(self, eng):
        """The engine-owned operands from the step's mask sample (the trainer's seeds and Philox streams), or from rint(sigmoid(S))
        for the baseline engine: one sc_apply_mask_batched launch per operand dtype."""
        mode = K.MASK_ROUND if eng.scst_eval else self.mask_mode()
        for (desc, tiles), dt in eng.scst_refresh:
            K.apply_mask_batched(desc, tiles, mode, seed=self._sd(0), stream_base=self._step_base(), out_dtype=dt)

    def scst_step(self, att_feats, boxes, att_masks=None, *, scorer, image_ids=None, opt=None, baseline="greedy", cider_weight=1.0,
                  bleu_weight=0.0, lr, all_reduce=None, **optim):
        """One self-critical step (utils/training.py:202-255 + RewardCriterion + clip + Adam) without a host synchronisation:
        premask the step's sample -> rollout (``opt``: {"beam_size": b[, "group_size": G]} or {"num_random_sample": n,
        "beam_size": 0}) and greedy baseline on the bound engine -> CIDEr-D (``scorer``: cider.CiderD; ``image_ids`` [B]: rows of
        its references, default 0 .. B-1) -> sc_scst_targets -> teacher-forcing forward / backward / optimizer (``optim``: the
        keyword arguments of ``train_step``).  ``baseline``: "greedy" or "sample" (mean of the image's other samples).  The rollout
        and the re-score share the step's ONE mask sample.  ``all_reduce``: data parallel as in ``train_step``; the token count
        is summed over the ranks before the loss.  Returns (loss, mean reward, sample_seq int32 [B, S, L]) as device tensors."""
        opt = dict(opt if opt is not None else {"beam_size": 5})
        S = scst_samples(opt, baseline, bleu_weight)
        c = self.cfg
        B, N = att_feats.shape[:2]
        L, R = c.max_seq_length, B * S
        ws = self._get_ws(B, N, S, L, att_masks is not None)
        if not hasattr(ws, "mask_sum"):
            ws.mask_sum = torch.zeros(1, device=self.dev)
            ws.mean_reward = torch.zeros(1, device=self.dev)
        self.step_id += 1
        self._hyper = _adam_hyper(lr, optim)
        if self.use_graph:
            self._upload_step(lr=lr, **optim)
        eng = self.rollout_engine()
        self._scst_masks(eng)
        # 2. rollouts; the sampler seed follows the trainer's step seed (a run is reproducible)
        if int(opt.get("num_random_sample", 0)) > 0:
            opt["sample_seed"] = self._step_seed(3)
        greedy = {"beam_size": 1}
        bseq = None
        enc = eng.encode(att_feats, boxes, att_masks)
        seq, _ = eng.decode(enc, opt)
        if baseline == "greedy":
            if self.mask_type == "supermask":
                beng = self._baseline_engine()
                self._refresh_engine(beng)
                bseq, _ = beng.decode(beng.encode(att_feats, boxes, att_masks), greedy)
            else:
                bseq, _ = eng.decode(enc, greedy)
        seq = seq.reshape(R, L)
        # 3. CIDEr-D of the samples and the baseline
        ids = (torch.arange(B, device=self.dev) if image_ids is None else torch.as_tensor(image_ids).to(self.dev)).to(torch.int32)
        score = scorer.score(seq, ids.repeat_interleave(S))
        bscore = scorer.score(bseq.reshape(B, L), ids) if bseq is not None else None
        # 4. rewards, targets and the token count
        targ = dict(S=S, cider_weight=cider_weight, bos=c.bos_token_id, pad=c.pad_token_id, tokens=ws.tokens, targets=ws.targets,
                    tok_w=ws.tok_w, key_valid=ws.key_valid, inv_norm=ws.inv_norm, mean_reward=ws.mean_reward)
        K.scst_targets(seq, score, bscore, mask_sum=ws.mask_sum, **targ)
        if all_reduce is not None:
            h = all_reduce(ws.mask_sum)
            if h is not None:
                h.wait()
            K.scst_targets(seq, score, bscore, norm_in=ws.mask_sum, **targ)   # inv_norm = 1 / global count
        ws.att_in.copy_(att_feats.reshape(B * N, -1), non_blocking=True)
        ws.boxes.copy_(boxes, non_blocking=True)
        if att_masks is not None:
            ws.att_mask.copy_(att_masks.float(), non_blocking=True)
        # 5. teacher-forcing forward on the step's operands, backward, clip + Adam
        self._scst = True
        try:
            with K.pdl(self.pdl_mask):
                loss = self._fwd_bwd_opt(ws, lr, all_reduce, optim)
        finally:
            self._scst = False
        return loss, ws.mean_reward.clone(), seq.view(B, S, L).clone()

    # ---- magnitude / SNIP mask updates (PruningMixin.update_masks_*, pruning/prune.py:259-304) ------------------------------
    # The masks of flat_s are rewritten in place by sc_prune_select; weights, Adam moments, opt_step, step_id, workspaces, captured
    # graphs and the rollout engine are untouched (every step re-reads flat_s: premask / operand prologues / _refresh_engine).
    def active_masked(self):
        """Masked tensors a mask update rewrites, in module order: PruningMixin.active_pruning_masks (mask_freeze_scope)."""
        scope = self.mask_freeze_scope
        return [k for k in self.masked if scope is None or not any((k + "_pruning_mask").startswith(s) for s in scope)]

    def _prune_table(self, from_saliency, per_tensor):
        """(descriptors, blocks, sizes) of the active masks: one segment per tensor (the generator's V rows, not the padded Vp),
        one selection group per tensor or one for all; position = index in the concatenation of the active masks (or in the
        tensor).  The criterion source is flat_w, or the saliency buffer, which has flat_s's layout."""
        key = (from_saliency, per_tensor)
        if key not in self._prune_desc:
            segs, pos = [], 0
            for i, k in enumerate(self.active_masked()):
                n = self.s[k].numel()
                segs.append((self._offs_s[k] if from_saliency else self._offs_w[k], self._offs_s[k], n, i if per_tensor else 0,
                             0 if per_tensor else pos))
                pos += n
            assert segs, "no active pruning masks (mask_freeze_scope freezes all of them)"
            self._prune_desc[key] = K.prune_descriptors(segs, self.dev) + ([sg[2] for sg in segs],)
        return self._prune_desc[key]

    @torch.no_grad()
    def update_masks_once(self, sparsity_target: float):
        """PruningMixin.update_masks_once on the trainer's own buffers, on the device and without a host synchronisation: the
        complete 0/1 mask of every active tensor from the exact k-th smallest criterion (sc_prune_select; ties in module order).
        ``snip`` consumes (and clears) the saliency accumulated by ``snip_saliency``.  Returns True."""
        from . import prune as P
        assert self.mask_type in P.MAG_PRUNE_MASKS, f"Invalid mask_type: {self.mask_type}. Must be one of {P.MAG_PRUNE_MASKS}"
        if self.mask_type == P.SNIP:
            assert self._has_saliency, "SNIP needs the mask gradients: call snip_saliency() first"
            crit, src = K.PRUNE_SNIP, self._saliency
        elif self.mask_type in P._DIST:
            crit, src = K.PRUNE_DIST, self.flat_w
        elif self.mask_type in P._BLIND or self.mask_type in P._UNIFORM:
            crit, src = K.PRUNE_ABS, self.flat_w
        else:
            raise ValueError(f"Unknown `self.mask_type`: {self.mask_type}")
        assert isinstance(sparsity_target, float) and 0 <= sparsity_target < 1.0, \
            f"`sparsity_target` must be a float >= 0 and < 1, saw {sparsity_target}"
        per_tensor = self.mask_type in P._UNIFORM
        desc, blocks, sizes = self._prune_table(crit == K.PRUNE_SNIP, per_tensor)
        groups = sizes if per_tensor else [sum(sizes)]
        ks = [int(sparsity_target * n) for n in groups]
        assert all(0 <= k < n for k, n in zip(ks, groups))
        sums = K.prune_stats(desc, blocks, src, centered=crit == K.PRUNE_DIST) if crit != K.PRUNE_ABS else None
        K.prune_select(desc, blocks, ks, crit, src, self.flat_s, sums=sums)
        if crit == K.PRUNE_SNIP:
            self._saliency.zero_()
            self._has_saliency = False
        self._wm_step = {}   # (an eval-mode operand cached for the current step_id is stale now)
        self.sparsity_target = sparsity_target
        return True

    def update_masks_gradual(self, sparsity_target: float, current_step: int, start_step: int, prune_steps: int,
                             initial_sparsity: float = 0.0, prune_frequency: int = 1000):
        """PruningMixin.update_masks_gradual (cubic schedule, prune.gradual_sparsity) through ``update_masks_once``.  Returns
        False, like the reference."""
        from . import prune as P
        assert self.mask_type in P.MAG_ANNEAL
        now = P.gradual_sparsity(sparsity_target, current_step, start_step, prune_steps, initial_sparsity, prune_frequency)
        if now is not None:
            self.update_masks_once(now)
        return False

    def snip_saliency(self, att_feats, boxes, seqs, masks, att_masks=None, *, seq_per_img, all_reduce=None, global_tokens=None):
        """SNIP: adds dL/dm = dWm (.) W of every active mask to the saliency buffer (repeated calls accumulate, the reference's
        ``prune_snip_grad_accum`` batches).  Teacher-forcing forward + backward of ``train_step`` (graph mode: the "fwdbwd"
        graph), no optimizer step.  ``all_reduce``: data parallel, the gradient buffer is summed over the ranks first (the
        weights are identical, so this sums the saliency).  Returns the batch loss (device scalar)."""
        from . import prune as P
        assert self.mask_type == P.SNIP, f"snip_saliency needs mask_type '{P.SNIP}', saw {self.mask_type!r}"
        B, N = att_feats.shape[:2]
        T = seqs.shape[1] - 1
        ws = self._get_ws(B, N, seq_per_img, T, att_masks is not None)
        self.step_id += 1
        self.load_batch(ws, att_feats, boxes, seqs, masks, att_masks, global_tokens)
        with K.pdl(self.pdl_mask):
            if self.use_graph:
                self._upload_seeds()
                self._run_graphed(ws, "fwdbwd", {})
            else:
                self.forward(ws)
                self.loss_and_backward(ws)
        grads = self.flat_gw if self.fused_st else self.flat_gs   # dWm (straight-through form) or dS = dWm (.) W (raw masks)
        if all_reduce is not None:
            h = all_reduce(grads)
            if h is not None:
                h.wait()
        if self._saliency is None:
            self._saliency = torch.zeros_like(self.flat_s)
        for k in self.active_masked():
            sal = self._saliency[self._offs_s[k]: self._offs_s[k] + self.s[k].numel()]
            if self.fused_st:
                K.mask_grad(self.g[k], self.p[k], self.s[k], K.MASK_RAW, None, sal, accumulate=True)
            else:
                sal.add_(self.gs[k].reshape(-1))
        self._has_saliency = True
        return ws.loss_sum * ws.inv_norm

    def mask_sparsities(self):
        """PruningMixin.all_mask_sparsities of the trainer's masks: (overall sparsity, nnz, per-tensor sparsities, mask names) as
        Python numbers.  Counted on the device (rint(sigmoid(S)) for supermask, the raw mask values otherwise) with one copy to
        the host."""
        assert self.masked, "the trainer has no pruning masks (mask_type=None)"
        if "count" not in self._prune_desc:
            segs = [(self._offs_s[k], self._offs_s[k], self.s[k].numel(), 0, 0) for k in self.masked]
            self._prune_desc["count"] = K.prune_descriptors(segs, self.dev)
        desc, blocks = self._prune_desc["count"]
        nnz = K.prune_stats(desc, blocks, self.flat_s, binarize=self.mask_type == "supermask")[:, 0].tolist()
        sizes = [self.s[k].numel() for k in self.masked]
        total = sum(nnz)
        return (1.0 - total / sum(sizes), total, [1.0 - c / n for c, n in zip(nnz, sizes)],
                tuple(k + "_pruning_mask" for k in self.masked))

    def state_dict(self):
        sd = {k: v.clone() for k, v in self.p.items()}
        sd.update({k + "_pruning_mask": v.clone() for k, v in self.s.items()})
        return sd

    # ---- resumable optimizer state ------------------------------------------------------------------------------------------------
    def _adam_groups(self):
        """[[(parameter name, flat moment buffers' layout, tensor name)]] of the two Adam groups: every trained weight, then (with
        masks) every mask logit, in the order of the state dict the trainer was built from."""
        groups = [[(k, self._offs_w, k) for k in self._adam_order]]
        if self.masked:
            groups.append([(k + "_pruning_mask", self._offs_s, k) for k in self._adam_masks])
        return groups

    @torch.no_grad()
    def optimizer_state_dict(self, exchange=None):
        """The optimizer state as ``torch.optim.Adam.state_dict()`` of the reference's two parameter groups: group 0 every trained
        weight, group 1 (with masks) every ``*_pruning_mask`` logit, both in the key order of the state dict the trainer was built
        from, so a ``torch.optim.Adam`` built over the drop-in module's parameters that way loads it.  Logits have moments only when
        the trainer updates them (supermask).  CPU tensors of exactly each parameter's shape (no padding); every ``step`` is
        ``opt_step``; ``param_groups`` carry the hyper-parameters of the last step.  The extra key ``"trainer"`` holds ``step_id``,
        ``seed``, ``mask_type`` and ``sparsity_target``.  ``exchange``: the ``distributed.ShardedExchange`` the steps ran with -
        the moments are all-gathered from the shard owners (a collective: every rank calls it and gets the full state).  With
        ``all_reduce`` every rank already holds the whole state.  ValueError while a SNIP saliency is pending."""
        if self._has_saliency:
            raise ValueError("a SNIP saliency accumulation is pending (snip_saliency without update_masks_once): it is consumed before "
                             "training and is not part of the resumable state")
        bufs = {"w": (self.m_w, self.v_w), "s": (self.m_s, self.v_s)}
        if exchange is not None:
            bufs = {"w": (self.m_w.clone(), self.v_w.clone()), "s": (self.m_s.clone(), self.v_s.clone())}
            for phase in range(self.N_PHASES):
                for flat, a, b in self.grad_buckets(phase):
                    if flat is self.flat_gw or self.mask_type == "supermask":   # (the update's buckets: _sharded_step)
                        for buf in bufs["w" if flat is self.flat_gw else "s"]:
                            exchange.gather(buf, a, b)
        host = {key: (m.cpu(), v.cpu()) for key, (m, v) in bufs.items()}   # (one copy per buffer, then one clone per parameter)
        groups = []
        for gi, entries in enumerate(self._adam_groups()):
            m, v = host["w" if gi == 0 else "s"]
            out = []
            for name, offs, k in entries:
                n, shp = self.p[k].numel(), self.p[k].shape
                has = gi == 0 or self.mask_type == "supermask"
                out.append((name, (m[offs[k]: offs[k] + n].view(shp).clone(), v[offs[k]: offs[k] + n].view(shp).clone()) if has else None))
            groups.append(out)
        # the host-side fields a later step reads: the Philox position and seed, the last mask update's target
        trainer = {"step_id": self.step_id, "seed": self.seed, "mask_type": self.mask_type, "sparsity_target": self.sparsity_target}
        return _export_adam(groups, self._hyper, self.opt_step, trainer)

    @torch.no_grad()
    def load_optimizer_state_dict(self, sd):
        """Loads ``optimizer_state_dict()`` - or a ``torch.optim.Adam`` state dict in that layout - in place into ``m_w`` / ``v_w``
        / ``m_s`` / ``v_s`` (operand pointers, rollout engines and captured graphs stay valid; the padding is zero - its moments
        only ever move padding logits, which every update resets) and sets
        ``opt_step``, the Adam hyper-parameters of ``optimizer_state_dict`` and, from the ``"trainer"`` key, ``step_id``, ``seed``
        and ``sparsity_target``.  A state without that key (one saved by ``torch.optim.Adam``) continues the Philox streams of
        masks, dropout and SCST sampling at ``step_id = opt_step``.  Every data-parallel rank loads the same file.  ValueError,
        naming the parameter, for a different parameter count or shape, a missing state entry of an updated parameter, unequal
        ``step`` values or another ``mask_type``."""
        logits = self.mask_type == "supermask"
        groups = [[(name, self.p[k].shape, gi == 0 or logits) for name, _, k in entries] for gi, entries in enumerate(self._adam_groups())]
        moments, step, hyper, extra = _import_adam(sd, groups, self.mask_type)
        host = {"w": (torch.zeros(self.m_w.numel()), torch.zeros(self.v_w.numel())),
                "s": (torch.zeros(self.m_s.numel()), torch.zeros(self.v_s.numel()))}
        for gi, entries in enumerate(self._adam_groups()):
            m, v = host["w" if gi == 0 else "s"]
            for name, offs, k in entries:
                if name in moments and (gi == 0 or logits):
                    n = self.p[k].numel()
                    m[offs[k]: offs[k] + n].copy_(moments[name][0].reshape(-1))
                    v[offs[k]: offs[k] + n].copy_(moments[name][1].reshape(-1))
        for (dm, dv), key in (((self.m_w, self.v_w), "w"), ((self.m_s, self.v_s), "s")):
            dm.copy_(host[key][0])
            dv.copy_(host[key][1])
        self.opt_step = step
        self._hyper.update(hyper)
        if extra is not None:
            self.step_id, self.seed = int(extra["step_id"]), int(extra["seed"])
            self.sparsity_target = extra.get("sparsity_target", self.sparsity_target)
        else:
            self.step_id = step
        self._wm_step = {}   # (operands cached for a step_id)


class ModuleTrainer:
    """``train_step`` for the configurations the fused engine does not lay out - ACORT weight sharing (``share_att_*`` /
    ``share_layer_*``, models/relation_transformer.py:80-89,162-176): the kernel-backed module tree under autograd (every
    forward / backward is a kernel, autograd accumulates the applications of a shared layer and draws a fresh Bernoulli mask per
    application like the reference), LanguageModelCriterion (utils/losses.py:32-43) + sparsity loss (pruning/prune.py:228-269),
    then clip_gradient + Adam for the two parameter groups (scripts/train_n_prune_transformer.py:67-82, utils/optim.py:116-126)
    as one ``sc_adam_clip`` launch per tensor.  It updates the module's own parameters (nothing to sync back)."""

    def __init__(self, model):
        self.model = model
        self.opt_step = 0
        self._mv = {}
        self._hyper = _adam_hyper(0.0, {})

    def train_step(self, att_feats, boxes, seqs, masks, att_masks=None, *, seq_per_img, lr, all_reduce=None, global_tokens=None,
                   mask_lr=100.0, clip=0.1, betas=(0.9, 0.98), eps=1e-9, mask_eps=1e-2, weight_decay=0.0, grad_scale=1.0,
                   sparsity_target=None, sparsity_weight=0.0, current_step=0, max_step=1):
        m = self.model
        dev = m._device()
        m.train()
        params = [(n, p) for n, p in m.named_parameters() if p.requires_grad]
        for _, p in params:
            p.grad = None
        seqs_d, masks_d = seqs.to(dev), masks.to(dev).float()
        assert seqs_d.shape[0] == att_feats.shape[0] * seq_per_img, (seqs_d.shape, att_feats.shape, seq_per_img)
        out = m(att_feats=att_feats.to(dev), boxes=boxes.to(dev), seqs=seqs_d, att_masks=None if att_masks is None else att_masks.to(dev))
        T = out.shape[1]
        target, w = seqs_d[:, 1: T + 1], masks_d[:, 1: T + 1]
        denom = w.sum() if global_tokens is None else global_tokens
        loss = -(out.gather(2, target.unsqueeze(2)).squeeze(2) * w).sum() / denom
        total = loss
        if getattr(m, "MASKED", False) and m.mask_type == "supermask" and sparsity_target is not None and sparsity_weight:
            total = total + m.compute_sparsity_loss(sparsity_target, sparsity_weight, current_step, max_step)
        total.backward()
        self._update(params, all_reduce, lr=lr, mask_lr=mask_lr, clip=clip, betas=betas, eps=eps, mask_eps=mask_eps,
                     weight_decay=weight_decay, grad_scale=grad_scale)
        return loss.detach()

    def _update(self, params, all_reduce, *, lr, mask_lr=100.0, clip=0.1, betas=(0.9, 0.98), eps=1e-9, mask_eps=1e-2, weight_decay=0.0,
                grad_scale=1.0):
        if all_reduce is not None:  # data parallel: sum the gradients of every rank (the loss is normalised by the global token count)
            flat = torch._utils._flatten_dense_tensors([p.grad for _, p in params])
            h = all_reduce(flat)
            if h is not None:
                h.wait()
            for (_, p), g in zip(params, torch._utils._unflatten_dense_tensors(flat, [p.grad for _, p in params])):
                p.grad.copy_(g)
        self.opt_step += 1
        self._hyper = _adam_hyper(lr, dict(mask_lr=mask_lr, betas=betas, eps=eps, mask_eps=mask_eps, weight_decay=weight_decay))
        with torch.no_grad():
            for n, p in params:
                is_logit = n.endswith("_pruning_mask")
                if n not in self._mv:
                    self._mv[n] = (torch.zeros_like(p, dtype=torch.float32).view(-1), torch.zeros_like(p, dtype=torch.float32).view(-1))
                mom, var = self._mv[n]
                g = p.grad.contiguous().view(-1)
                K.adam_clip(p.data.view(-1), g, mom, var, lr=mask_lr if is_logit else lr, betas=betas, eps=mask_eps if is_logit else eps,
                            weight_decay=0.0 if is_logit else weight_decay, clip=clip, grad_scale=grad_scale, step=self.opt_step)
                torch.autograd.graph.increment_version(p)  # (written through raw pointers: cached engines must notice)

    def scst_step(self, att_feats, boxes, att_masks=None, *, scorer, image_ids=None, opt=None, baseline="greedy", cider_weight=1.0,
                  bleu_weight=0.0, lr, all_reduce=None, **optim):
        """``OrtTrainer.scst_step`` for ACORT through the module tree (correctness path): greedy baseline in eval mode, rollout in
        train mode, CIDEr-D and sc_scst_targets on the device, RewardCriterion on the autograd teacher-forced log-probs, then the
        update of ``train_step``.  The train-mode rollout and the re-score draw their own supermask samples (module path)."""
        opt = dict(opt if opt is not None else {"beam_size": 5})
        S = scst_samples(opt, baseline, bleu_weight)
        m = self.model
        dev = m._device()
        c = m.cfg
        att_feats, boxes = att_feats.to(dev), boxes.to(dev)
        att_masks = None if att_masks is None else att_masks.to(dev)
        B, L = att_feats.shape[0], c.max_seq_length
        R = B * S
        bseq = None
        if baseline == "greedy":
            m.eval()
            bseq, _ = m(att_feats=att_feats, boxes=boxes, att_masks=att_masks, opt={"beam_size": 1}, mode="sample")
        m.train()
        seq, _ = m(att_feats=att_feats, boxes=boxes, att_masks=att_masks, opt=opt, mode="sample")
        seq = seq.reshape(R, L).to(torch.int32).contiguous()
        ids = (torch.arange(B, device=dev) if image_ids is None else torch.as_tensor(image_ids).to(dev)).to(torch.int32)
        score = scorer.score(seq, ids.repeat_interleave(S))
        bscore = scorer.score(bseq.reshape(B, L), ids) if bseq is not None else None
        i32, f32 = dict(dtype=torch.int32, device=dev), dict(dtype=torch.float32, device=dev)
        tokens, targets, tok_w, key_valid = (torch.empty(R * L, **i32), torch.empty(R * L, **i32), torch.empty(R * L, **f32),
                                             torch.empty(R * L, **f32))
        inv_norm, mask_sum, mean_reward = torch.empty(1, **f32), torch.empty(1, **f32), torch.empty(1, **f32)
        targ = dict(S=S, cider_weight=cider_weight, bos=c.bos_token_id, pad=c.pad_token_id, tokens=tokens, targets=targets, tok_w=tok_w,
                    key_valid=key_valid, inv_norm=inv_norm, mean_reward=mean_reward)
        K.scst_targets(seq, score, bscore, mask_sum=mask_sum, **targ)
        if all_reduce is not None:
            h = all_reduce(mask_sum)
            if h is not None:
                h.wait()
            K.scst_targets(seq, score, bscore, norm_in=mask_sum, **targ)
        params = [(n, p) for n, p in m.named_parameters() if p.requires_grad]
        for _, p in params:
            p.grad = None
        # teacher-forced log-probs of the sampled captions: input [BOS, s_0 .. s_{L-2}], target s (RewardCriterion)
        seqs = torch.cat([tokens.view(R, L).long(), seq[:, L - 1:].long()], 1)
        out = m(att_feats=att_feats, boxes=boxes, seqs=seqs, att_masks=att_masks)
        lp = out.gather(2, targets.view(R, L, 1).long()).squeeze(2)
        loss = -(lp * tok_w.view(R, L)).sum() * inv_norm[0]
        total = loss
        sp = {k: optim.pop(k) for k in ("sparsity_target", "sparsity_weight", "current_step", "max_step") if k in optim}
        if getattr(m, "MASKED", False) and m.mask_type == "supermask" and sp.get("sparsity_target") is not None and sp.get("sparsity_weight"):
            total = total + m.compute_sparsity_loss(sp["sparsity_target"], sp["sparsity_weight"], sp.get("current_step", 0),
                                                    sp.get("max_step", 1))
        total.backward()
        self._update(params, all_reduce, lr=lr, **optim)
        return loss.detach(), mean_reward, seq.view(B, S, L)

    def state_dict(self):
        return self.model.state_dict()

    # ---- resumable optimizer state (OrtTrainer.optimizer_state_dict) --------------------------------------------------------------
    def _adam_groups(self):
        """[[(name, parameter)]]: the trained parameters in ``named_parameters()`` order, weights, then (if any) mask logits."""
        params = [(n, p) for n, p in self.model.named_parameters() if p.requires_grad]
        logits = [(n, p) for n, p in params if n.endswith("_pruning_mask")]
        return [[(n, p) for n, p in params if not n.endswith("_pruning_mask")]] + ([logits] if logits else [])

    def _mask_type(self):
        return self.model.mask_type if getattr(self.model, "MASKED", False) else None

    @torch.no_grad()
    def optimizer_state_dict(self):
        """``OrtTrainer.optimizer_state_dict`` of the module's trained parameters: the moments of ``_mv`` in each parameter's shape
        (zeros before the first step), ``step`` = ``opt_step``.  The ``"trainer"`` key holds the mask type and the position of the
        process-wide Philox streams (``sampler._state`` seed, mask stream and dropout stream), so that the per-application
        Bernoulli masks and dropout continue where they stopped."""
        from .sampler import _state
        groups = []
        for entries in self._adam_groups():
            out = []
            for n, p in entries:
                m, v = self._mv.get(n, (torch.zeros(p.numel()), torch.zeros(p.numel())))
                out.append((n, (m.view(p.shape).cpu().clone(), v.view(p.shape).cpu().clone())))
            groups.append(out)
        trainer = {"mask_type": self._mask_type(), "seed": _state["seed"], "stream": _state["stream"], "drop": _state["drop"]}
        return _export_adam(groups, self._hyper, self.opt_step, trainer)

    @torch.no_grad()
    def load_optimizer_state_dict(self, sd):
        """Loads an ``optimizer_state_dict()`` (or a ``torch.optim.Adam`` state dict in that layout): the moments into ``_mv``,
        ``opt_step``, the hyper-parameters, and the sampler's stream position from the ``"trainer"`` key.  ValueError as for
        ``OrtTrainer.load_optimizer_state_dict``."""
        from .sampler import _state
        groups = self._adam_groups()
        moments, step, hyper, extra = _import_adam(sd, [[(n, p.shape, True) for n, p in entries] for entries in groups],
                                                   self._mask_type())
        for entries in groups:
            for n, p in entries:
                self._mv[n] = tuple(t.to(device=p.device, dtype=torch.float32).reshape(-1).clone() for t in moments[n])
        self.opt_step = step
        self._hyper.update(hyper)
        if extra is not None:
            _state.update(seed=int(extra["seed"]), stream=int(extra["stream"]), drop=int(extra["drop"]))

