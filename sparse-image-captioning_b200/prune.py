"""PruningMixin — drop-in for sparse_caption/pruning/prune.py (constants 17-42, mixin 46-476).

Mask enumeration, sparsity statistics, the supermask sparsity loss, dense / sparse state-dict export and the
one-shot / gradual magnitude / SNIP mask updates keep the reference's method names, arguments and results.
Hot items run in CUDA kernels (binarized-mask counting: sc_mask_count; weight pruning: sc_apply_mask); the mask
*schedulers* (run once, or every 1000 steps) are host-side torch code, out of the kernel scope (SURVEY.md 2.1 #3).
"""
import logging
import math
from argparse import ArgumentParser, _ArgumentGroup
from typing import Callable, Dict, Union

import torch

from . import kernels as K

logger = logging.getLogger(__name__)

MASK_FREEZE = "mask_freeze"
REGULAR = "supermask"
MAG_BLIND, MAG_UNIFORM, MAG_DIST = "mag_blind", "mag_uniform", "mag_dist"
MAG_GRAD_BLIND, MAG_GRAD_UNIFORM, MAG_GRAD_DIST = "mag_grad_blind", "mag_grad_uniform", "mag_grad_dist"
LOTTERY_MAG_BLIND, LOTTERY_MAG_UNIFORM, LOTTERY_MAG_DIST = "lottery_mag_blind", "lottery_mag_uniform", "lottery_mag_dist"
LOTTERY_MASK_FREEZE = "lottery_mask_freeze"
SNIP = "snip"

SUPER_MASKS = [REGULAR]
MAG_ANNEAL = [MAG_GRAD_BLIND, MAG_GRAD_UNIFORM]
MAG_HARD = [MAG_BLIND, MAG_UNIFORM, MAG_DIST]
LOTTERY = [LOTTERY_MAG_BLIND, LOTTERY_MAG_UNIFORM, LOTTERY_MAG_DIST, LOTTERY_MASK_FREEZE]
MAG_PRUNE_MASKS = MAG_HARD + MAG_ANNEAL + LOTTERY + [SNIP]
VALID_MASKS = SUPER_MASKS + MAG_PRUNE_MASKS + [MASK_FREEZE]

_BLIND = (MAG_BLIND, MAG_GRAD_BLIND, LOTTERY_MAG_BLIND)
_UNIFORM = (MAG_UNIFORM, MAG_GRAD_UNIFORM, LOTTERY_MAG_UNIFORM)
_DIST = (MAG_DIST, MAG_GRAD_DIST, LOTTERY_MAG_DIST)
_SUFFIX = "_pruning_mask"


def binarize(logits: torch.Tensor) -> torch.Tensor:
    """rint(sigmoid(S)) without gradient, bit-exact with the reference (== S > 1.5 * 2^-24)."""
    if logits.is_cuda:
        return K.apply_mask(torch.ones_like(logits), logits.detach().contiguous(), K.MASK_ROUND)
    return (logits.detach() > 1.5 * 2.0 ** -24).to(logits.dtype)


def densify_state_dict(state_dict):
    """utils/model_utils.py:110-118: sparse COO entries -> dense."""
    return {k: (v.to_dense() if torch.is_tensor(v) and v.is_sparse else v) for k, v in state_dict.items()}


def fold_masks(state_dict, mask_type):
    """state dict of a ``*_prune`` model -> dense-class state dict with every mask folded into its weight
    (what eval_model.py:64-77 obtains via state_dict_dense + key stripping).  Runs sc_apply_mask on CUDA tensors."""
    out = {}
    mode = K.MASK_ROUND if mask_type in SUPER_MASKS else K.MASK_RAW
    for k, v in state_dict.items():
        if k.endswith(_SUFFIX):
            continue
        m = state_dict.get(k + _SUFFIX)
        if m is None:
            out[k] = v
        elif v.is_cuda:
            out[k] = K.apply_mask(v.detach().float().contiguous(), m.detach().float().contiguous(), mode)
        else:
            out[k] = v * (binarize(m) if mode == K.MASK_ROUND else m)
    return out


def gradual_sparsity(sparsity_target, current_step, start_step, prune_steps, initial_sparsity=0.0, prune_frequency=1000):
    """The sparsity that update_masks_gradual prunes to at `current_step` (cubic schedule, prune.py:375-433), or None when
    no mask update is due at that step.  Shared by PruningMixin and trainer.OrtTrainer."""
    assert prune_frequency > 0, f"Pruning frequency must be greater than zero, saw `{prune_frequency}`"
    assert prune_steps > 0, f"Pruning steps must be greater than zero, saw `{prune_steps}`"
    end_step = start_step + prune_frequency * prune_steps
    in_range = current_step >= start_step and (current_step <= end_step or end_step < 0)
    if in_range and (current_step - start_step) % prune_frequency == 0:
        progress = min(1.0, max(0.0, (current_step - start_step) / (end_step - start_step)))
        return sparsity_target + (initial_sparsity - sparsity_target) * (1.0 - progress) ** 3
    return None


class _SparsityLossFn(torch.autograd.Function):
    """|target - sparsity| with the straight-through gradient of rounding_sigmoid: d nnz / dS = sigmoid'(S)."""

    @staticmethod
    def forward(ctx, target, total, *logits):
        if logits[0].is_cuda:
            nnz = K.mask_count([s.detach().contiguous() for s in logits]).to(torch.float32)[0]
        else:
            nnz = sum(binarize(s).sum() for s in logits)
        sparsity = 1.0 - nnz / total
        ctx.save_for_backward(*logits)
        ctx.sign = 1.0 if float(target - sparsity) >= 0 else -1.0  # d|t - s| / ds = -sign(t - s)
        ctx.total = total
        ctx.sparsity = sparsity
        return torch.abs(target - sparsity)

    @staticmethod
    def backward(ctx, grad):
        # d loss / d nnz = sign(target - sparsity) / total
        coeff = grad * (ctx.sign / ctx.total)
        outs = []
        for s in ctx.saved_tensors:
            p = torch.sigmoid(s)
            outs.append(coeff * p * (1 - p))
        return (None, None) + tuple(outs)


# noinspection PyAttributeOutsideInit
class PruningMixin:
    """Mixin to be used together with torch.nn.Module."""

    named_parameters: Callable
    state_dict: Callable
    load_state_dict: Callable

    def __init__(self, *, mask_type, mask_freeze_scope="", **kwargs):
        assert mask_type in VALID_MASKS, f"`mask_type` must be one of {VALID_MASKS}, saw `{mask_type}`"
        assert isinstance(mask_freeze_scope, str), f"`mask_freeze_scope` must be a str, saw `{type(mask_freeze_scope)}`"
        self.mask_type = mask_type
        scopes = [s for s in mask_freeze_scope.split(",") if s != ""]
        self.mask_freeze_scope = scopes if mask_freeze_scope != "" else None
        self.sparsity_target = 0.0
        super().__init__(**kwargs)

    # ---- enumeration -------------------------------------------------------------------------------
    @staticmethod
    def _pick(pairs, named):
        return [(n, p) if named else p for n, p in pairs]

    def all_pruning_masks(self, named=True):
        return self._pick(((n, p) for n, p in self.named_parameters() if n.endswith(_SUFFIX)), named)

    def all_weights(self, named=True):
        return self._pick(((n, p) for n, p in self.named_parameters() if not n.endswith(_SUFFIX)), named)

    def _weights_of(self, masks, named):
        wanted = {n[: -len(_SUFFIX)] for n, _ in masks}
        return self._pick(((n, p) for n, p in self.named_parameters() if n in wanted), named)

    def all_pruned_weights(self, named=True):
        return self._weights_of(self.all_pruning_masks(), named)

    def active_pruning_masks(self, named=True):
        masks = self.all_pruning_masks()
        if self.mask_freeze_scope is not None:
            masks = [(n, p) for n, p in masks if not any(n.startswith(s) for s in self.mask_freeze_scope)]
        return self._pick(masks, named)

    def active_pruned_weights(self, named=True):
        return self._weights_of(self.active_pruning_masks(), named)

    def trainable_pruning_masks(self, named=True):
        return self._pick(((n, p) for n, p in self.all_pruning_masks() if p.requires_grad), named)

    @property
    def total_mask_params(self):
        return sum(p.nelement() for p in self.all_pruning_masks(named=False))

    @property
    def total_weight_params(self):
        return sum(p.nelement() for p in self.all_weights(named=False))

    # ---- statistics --------------------------------------------------------------------------------
    @staticmethod
    def calculate_sparsities(tensor_list, count_nnz_fn):
        sizes = [t.nelement() for t in tensor_list]
        nnz = [count_nnz_fn(t) for t in tensor_list]
        per_tensor = [1.0 - (c / n) for c, n in zip(nnz, sizes)]
        total_nnz = sum(nnz)
        return 1.0 - (total_nnz / sum(sizes)), total_nnz, per_tensor

    def _binary_masks(self, masks):
        return [binarize(m) for m in masks] if self.mask_type in SUPER_MASKS else list(masks)

    @property
    def all_weight_sparsities(self):
        names, weights = zip(*self.all_pruned_weights(named=True))
        return self.calculate_sparsities(weights, lambda t: t.ne(0).float().sum()) + (names,)

    @property
    def all_mask_sparsities(self):
        names, masks = zip(*self.all_pruning_masks(named=True))
        return self.calculate_sparsities(self._binary_masks(masks), torch.sum) + (names,)

    @property
    def active_mask_sparsities(self):
        names, masks = zip(*self.active_pruning_masks(named=True))
        return self.calculate_sparsities(self._binary_masks(masks), torch.sum) + (names,)

    @property
    def all_mask_avg(self):
        return torch.cat([m.view(-1) for m in self.all_pruning_masks(named=False)]).mean()

    @property
    def active_mask_avg(self):
        return torch.cat([m.view(-1) for m in self.active_pruning_masks(named=False)]).mean()

    # ---- export ------------------------------------------------------------------------------------
    @torch.no_grad()
    def prune_weights(self):
        mode = K.MASK_ROUND if self.mask_type in SUPER_MASKS else K.MASK_RAW
        for w, m in zip(self.all_pruned_weights(named=False), self.all_pruning_masks(named=False)):
            if w.is_cuda:
                w.copy_(K.apply_mask(w.detach().contiguous(), m.detach().contiguous(), mode))
            else:
                w.mul_(binarize(m) if mode == K.MASK_ROUND else m)

    def state_dict_dense(self, destination=None, prefix="", keep_vars=False, discard_pruning_mask=False,
                         prune_weights=True, binarize_supermasks=False):
        if discard_pruning_mask and binarize_supermasks:
            raise ValueError("`discard_pruning_mask` and `binarize_supermasks` cannot be True at the same time.")
        if binarize_supermasks and self.mask_type not in SUPER_MASKS:
            raise ValueError(f"`binarize_supermasks` can only be True for mask_type in {SUPER_MASKS}.")
        if prune_weights:
            self.prune_weights()
        sd = self.state_dict(destination=destination, prefix=prefix, keep_vars=keep_vars)
        for name, _ in self.all_pruning_masks():
            key = prefix + name
            if discard_pruning_mask:
                del sd[key]
            elif binarize_supermasks:
                sd[key] = binarize(sd[key])
        return sd

    def state_dict_sparse(self, destination=None, prefix="", keep_vars=False, discard_pruning_mask=True,
                          prune_weights=True, binarize_supermasks=False):
        sd = self.state_dict_dense(destination=destination, prefix=prefix, keep_vars=keep_vars,
                                   discard_pruning_mask=discard_pruning_mask, prune_weights=prune_weights,
                                   binarize_supermasks=binarize_supermasks)
        pruned = {prefix + n for n, _ in self.all_pruned_weights(named=True)}
        return {k: (v.to_sparse() if torch.is_tensor(v) and k in pruned else v) for k, v in sd.items()}

    def load_sparse_state_dict(self, sparse_state_dict: Dict[str, torch.Tensor], strict: bool = True):
        self.load_state_dict(state_dict=densify_state_dict(sparse_state_dict), strict=strict)

    # ---- supermask sparsity loss (prune.py:228-269) ------------------------------------------------
    def compute_sparsity_loss(self, sparsity_target: float, weight: float, current_step: int, max_step: int):
        assert self.mask_type in SUPER_MASKS, f"Invalid mask type. Must be one of {SUPER_MASKS}"
        masks = self.active_pruning_masks(named=False)
        if len(masks) == 0:
            return 0.0
        total = float(sum(m.nelement() for m in masks))
        loss = _SparsityLossFn.apply(float(sparsity_target), total, *masks)
        anneal_rate = (1.0 + torch.cos(torch.tensor(min(1.0, current_step / max_step) * math.pi))) / 2
        scaled = loss * weight * (1.0 - anneal_rate.to(loss.device))
        self.sparsity_loss = {"loss": loss, "anneal_rate": anneal_rate, "loss_scaled": scaled}
        return scaled

    # ---- magnitude / SNIP mask updates (host-side, rare) -------------------------------------------
    @staticmethod
    def compute_mask(criterion, sparsity_target):
        assert isinstance(sparsity_target, float) and 0 <= sparsity_target < 1.0, \
            f"`sparsity_target` must be a float >= 0 and < 1, saw {sparsity_target}"
        n_prune = int(sparsity_target * criterion.nelement())
        assert 0 <= n_prune < criterion.nelement()
        mask = torch.ones_like(criterion)
        if n_prune > 0:
            mask.view(-1)[torch.topk(criterion.view(-1), k=n_prune, largest=False).indices] = 0
        return mask

    @torch.no_grad()
    def sparsity_check(self, warning_threshold: float = 0.999):
        _, _, sps, names = self.all_mask_sparsities
        high = [(n, float(s)) for n, s in zip(names, sps) if s > warning_threshold]
        if high:
            logger.warning(f"{type(self).__name__}: Pruning ({self.mask_type}): masks with sparsity > "
                           f"{warning_threshold}: " + "   ".join(f"{n} = {s:.5f}" for n, s in high))

    @torch.no_grad()
    def update_masks_once(self, sparsity_target: float):
        assert self.mask_type in MAG_PRUNE_MASKS, f"Invalid mask_type: {self.mask_type}. Must be one of {MAG_PRUNE_MASKS}"
        masks = self.active_pruning_masks(named=False)
        weights = self.active_pruned_weights(named=False)
        assert len(masks) == len(weights)

        def flat(ts):
            return torch.cat([t.reshape(-1) for t in ts])

        if self.mask_type == SNIP:
            assert all(m.grad is not None for m in masks)
            sal = flat([m.grad for m in masks])
            criteria = [sal / sal.sum()]
        elif self.mask_type in _DIST:
            criteria = [flat([torch.abs((w - w.mean()) / torch.std(w.reshape(-1), dim=0, unbiased=False)) for w in weights])]
        elif self.mask_type in _BLIND:
            criteria = [flat([w.abs() for w in weights])]
        elif self.mask_type in _UNIFORM:
            criteria = [w.abs() for w in weights]
        else:
            raise ValueError(f"Unknown `self.mask_type`: {self.mask_type}")
        new = [self.compute_mask(c, sparsity_target) for c in criteria]
        if len(new) == 1:
            new = torch.split(new[0], [m.nelement() for m in masks])
        assert len(new) == len(masks)
        for m, nm in zip(masks, new):
            m.view(-1).copy_(nm.reshape(-1))
        logger.info(f"{type(self).__name__}: Pruning ({self.mask_type}): Pruned to sparsity = `{sparsity_target:.5f}`")
        self.sparsity_target = sparsity_target
        self.sparsity_check()
        return True

    @torch.no_grad()
    def update_masks_gradual(self, sparsity_target: float, current_step: int, start_step: int, prune_steps: int,
                             initial_sparsity: float = 0.0, prune_frequency: int = 1000):
        """Cubic sparsity schedule of Zhu & Gupta (arXiv:1710.01878), prune.py:375-433."""
        assert self.mask_type in MAG_ANNEAL
        now = gradual_sparsity(sparsity_target, current_step, start_step, prune_steps, initial_sparsity, prune_frequency)
        if now is not None:
            self.update_masks_once(sparsity_target=now)
        return False  # the reference returns False on every path (prune.py:433)

    @staticmethod
    def add_argparse_args(parser: Union[_ArgumentGroup, ArgumentParser]):
        g = parser.add_argument_group("Pruning", "Arguments for weight pruning.")
        g.add_argument("--prune_type", type=str, default="", choices=VALID_MASKS, help="str: Type of pruning scheme.")
        g.add_argument("--prune_sparsity_target", type=float, default=0.8, help="float: Desired sparsity.")
        g.add_argument("--prune_mask_freeze_scope", type=str, default="", help="str: Scopes to freeze pruning masks.")
        g.add_argument("--prune_snip_grad_accum", type=int, default=1,
                       help="int: Number of batches of gradient accumulation for SNIP saliency computation.")
        g.add_argument("--prune_supermask_init", type=float, default=5.0, help="float: Init value of Supermask pruning masks.")
        g.add_argument("--prune_supermask_sparsity_weight", type=float, default=-1.0,
                       help="float: Weightage of Supermask sparsity loss.")
        g.add_argument("--prune_supermask_lr", type=float, default=1e2, help="float: Learning rate for Supermask.")
        g.add_argument("--prune_supermask_bypass_sigmoid_grad", action="store_true",
                       help="bool: If True, bypass sigmoid during gradient backprop (straight-through estimator).")
