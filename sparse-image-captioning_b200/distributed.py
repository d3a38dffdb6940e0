"""Data-parallel plumbing (one process per GPU, torch.distributed over NCCL / NVLink; gloo on CPU for tests).

The path shards by image (SURVEY.md section 8e): inference and SCST rollouts need no collective; SMP training needs one
exchange per step — a SUM all-reduce of the flat gradient buffers (weights AND mask logits), with every rank's loss
normalised by the GLOBAL token count so that the summed gradient equals the single-process gradient of the whole
batch (utils/losses.py:42 normalises by sum(mask)).  Value clipping happens after the exchange, inside the fused
Adam kernel, as in utils/optim.py:187-191.  All ranks must share the mask seed (sampler.set_mask_seed / OrtTrainer
seed): the reference draws ONE Bernoulli mask per layer per step for the whole batch (masked_layer.py:97).
"""
import torch
import torch.distributed as dist


def shard_range(n_items: int, rank: int, world: int):
    """Contiguous block partition of n_items (images) over ranks; the first n_items % world ranks get one extra."""
    base, extra = divmod(n_items, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def global_token_count(masks: torch.Tensor, T: int, group=None) -> torch.Tensor:
    """Sum over all ranks of the loss-mask entries masks[:, 1:T+1] (the denominator of LanguageModelCriterion)."""
    cnt = masks[:, 1: T + 1].float().sum().reshape(1).clone()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=group)
    return cnt


def make_all_reduce(group=None, async_op=False):
    """Callable for OrtTrainer.train_step(all_reduce=...): in-place SUM over ranks of one (slice of a) flat gradient
    buffer.  ``async_op``: return the work handle instead of waiting, so that the trainer can overlap the exchange of
    the buckets one backward phase finished with the next phase (OrtTrainer.grad_buckets); ``handle.wait()`` orders
    the current CUDA stream after the collective (NCCL) or blocks the host (gloo)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None

    def _ar(flat):
        work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
        return work if async_op else None

    return _ar


class ShardedExchange:
    """ZeRO-1 style exchange + update, bucket by bucket: reduce-scatter of a finished gradient range, the owner updates its
    1/world shard of the parameters (and keeps the only live copy of that shard's Adam moments), all-gather of the updated
    parameters.  Same bytes on the wire as the all-reduce it replaces, but the optimizer's HBM traffic (28 B per
    parameter) drops by the world size, and the whole chain of a bucket runs on a side stream underneath the next backward
    phase (SURVEY.md section 8e, "alternative if all-reduce does not hide").

    ``bucket(grad, param, a, b, update)``: grad / param are the flat fp32 buffers, [a, b) the finished range,
    ``update(lo, hi)`` applies the optimizer in place to param[lo:hi] from the rank-summed grad[lo:hi].  The range is cut
    into world equal shards plus a tail of < world elements that every rank updates redundantly (identical inputs ->
    identical results).  NCCL: everything is enqueued on ``self.stream``; gloo (CPU tests): blocking calls."""

    def __init__(self, group=None, device=None):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.nccl = dist.get_backend(group) == "nccl"
        self.stream = torch.cuda.Stream(device) if self.nccl else None
        self._tmp = None

    def _staging(self, n, like):
        if self._tmp is None or self._tmp.numel() < n or self._tmp.device != like.device:
            self._tmp = torch.empty(n, dtype=like.dtype, device=like.device)
        return self._tmp[:n]

    def shard(self, a, b):
        """(lo, hi, mid): this rank owns [lo, hi); [mid, b) is the redundantly updated tail."""
        n = (b - a) // self.world
        return a + self.rank * n, a + (self.rank + 1) * n, a + n * self.world

    def bucket(self, grad, param, a, b, update):
        lo, hi, mid = self.shard(a, b)
        n = hi - lo
        if self.nccl:
            cur = torch.cuda.current_stream(grad.device)
            self.stream.wait_stream(cur)  # the bucket's gradients were produced on the caller's stream
            with torch.cuda.stream(self.stream):
                self._bucket(grad, param, a, b, lo, hi, mid, n, update)
        else:
            self._bucket(grad, param, a, b, lo, hi, mid, n, update)

    def _bucket(self, grad, param, a, b, lo, hi, mid, n, update):
        if n > 0:
            if self.nccl:
                tmp = self._staging(n, grad)
                dist.reduce_scatter_tensor(tmp, grad[a:mid], op=dist.ReduceOp.SUM, group=self.group)
                grad[lo:hi].copy_(tmp)
            else:  # gloo has no reduce-scatter
                dist.all_reduce(grad[a:mid], op=dist.ReduceOp.SUM, group=self.group)
        if b > mid:
            dist.all_reduce(grad[mid:b], op=dist.ReduceOp.SUM, group=self.group)
        if n > 0:
            update(lo, hi)
        if b > mid:
            update(mid, b)
        self.gather(param, a, b)

    def gather(self, buf, a, b):
        """All-gather of ``buf[a, mid)`` in place from the owners of its shards (``shard(a, b)``); the tail ``[mid, b)`` is the same
        on every rank already.  The updated parameters of a bucket, or the optimizer state a rank keeps for its shards only."""
        lo, hi, mid = self.shard(a, b)
        if hi > lo:
            own = buf[lo:hi].clone()
            if self.nccl:
                dist.all_gather_into_tensor(buf[a:mid], own, group=self.group)
            else:
                parts = [torch.empty_like(own) for _ in range(self.world)]
                dist.all_gather(parts, own, group=self.group)
                buf[a:mid].copy_(torch.cat(parts))

    def finish(self):
        """Order the caller's stream after every bucket's chain."""
        if self.nccl:
            torch.cuda.current_stream(self.stream.device).wait_stream(self.stream)
