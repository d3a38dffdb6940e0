"""Launch sequence of the fused training step (OrtTrainer), recorded on the CPU: every kernel wrapper, raw ``lib.call`` and CUDA
stream / event operation is replaced by a recorder, so whole steps run on CPU tensors and leave a deterministic JSON trace of the
launches they would issue - each with its stream, tensors described by shape, dtype, stride, storage offset and storage ordinal
(the order in which the storage first appears), pointer-valued ints (descriptor tables, bit-63 seed pointers) mapped through the
same table.  A change to trainer.py that keeps the launch sequence (same kernels, order, arguments, buffers, Philox streams,
ring slots, side-stream forks and joins) keeps this output byte-identical.

    python scripts/train_launch_trace.py OUT.json
"""
import contextlib
import inspect
import json
import os
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle import ort_oracle as O
from sparse_caption_b200 import kernels as K, lib
from sparse_caption_b200.engine import ModelCfg
from sparse_caption_b200.trainer import OrtTrainer

TRACE = []
_storages = []     # (base, nbytes, tensor kept alive) in order of first appearance
_traced = [None]   # the trainer being traced: a pointer seen before its tensor is resolved through its tensors


def _ordinal(t):
    st = t.untyped_storage()
    base = st.data_ptr()
    for i, (b, _, _) in enumerate(_storages):
        if b == base:
            return i
    _storages.append((base, st.nbytes(), t))
    return len(_storages) - 1


def _lookup(p):
    for i, (b, n, _) in enumerate(_storages):
        if b <= p < b + n:
            return i, p - b
    for t in _collect(_traced[0]):
        st = t.untyped_storage()
        if st.nbytes() and st.data_ptr() <= p < st.data_ptr() + st.nbytes():
            return _ordinal(t), p - st.data_ptr()
    raise LookupError(f"pointer {p:#x} is in no tensor of the trainer")


class Ptr(int):
    """A pointer from lib.ptr: described through the storage table, never as its value."""


_tables = {}       # id -> (table, number of leading pointer columns) of the descriptor tables built by the run


def desc(a):
    if torch.is_tensor(a):
        d = ["T", list(a.shape), str(a.dtype).replace("torch.", ""), list(a.stride()), a.storage_offset(), _ordinal(a)]
        if a.dtype == torch.int64 and a.numel() <= 4096:   # descriptor tables: their buffers, extents and Philox streams
            n_ptr = _tables[id(a)][1] if id(a) in _tables else 0
            d.append([[["P", *_lookup(v)] if j < n_ptr and v else v for j, v in enumerate(row)] for row in a.view(a.shape[0], -1).tolist()])
        return d
    if isinstance(a, Ptr):
        return ["P", *_lookup(a)]
    if isinstance(a, int) and a >= 1 << 63:   # graph-mode Philox seed: a pointer with bit 63 set
        return ["S", *_lookup(a - (1 << 63))]
    if isinstance(a, (bool, int, float, str)) or a is None:
        return a
    if isinstance(a, (list, tuple)):
        return [desc(x) for x in a]
    if isinstance(a, (torch.dtype, torch.device)):
        return str(a)
    return type(a).__name__


# ---- streams and events ------------------------------------------------------------------------------------------------------
class Stream:
    count = 0

    def __init__(self, *a, **k):
        self.id, Stream.count = Stream.count, Stream.count + 1
        self.cuda_stream = self.id

    def wait_event(self, e):
        TRACE.append(["wait_event", self.id, e.id])

    def wait_stream(self, s):
        TRACE.append(["wait_stream", self.id, s.id])


class Event:
    count = 0

    def __init__(self, *a, **k):
        self.id, Event.count = Event.count, Event.count + 1

    def record(self, s=None):
        TRACE.append(["event.record", self.id, (s or _current[-1]).id])

    def synchronize(self):
        pass


_current = [Stream()]


@contextlib.contextmanager
def _on(s):
    _current.append(s)
    try:
        yield
    finally:
        _current.pop()


torch.cuda.Stream, torch.cuda.Event = Stream, Event
torch.cuda.current_stream = lambda *a: _current[-1]
torch.cuda.stream = _on
torch.Tensor.pin_memory = lambda self, *a: self

# ---- kernels ---------------------------------------------------------------------------------------------------------------
# run as they are: host-side descriptor tables, the PDL context, and wrappers that only forward to lib.call (recorded there)
KEEP = {"pad8", "mask_descriptors", "st_descriptors", "prune_descriptors", "_to_device", "mask_count", "pdl"}
_pdl = [7]


def _stub(name, f):
    sig = inspect.signature(f)

    def rec(*a, **kw):
        args = sig.bind(*a, **kw)
        args.apply_defaults()   # (an argument passed at its default value and one left out are the same launch)
        TRACE.append([name, _current[-1].id, [[k, desc(v)] for k, v in args.arguments.items()]])
        if name == "prune_stats":
            return torch.zeros(a[0].shape[0], 2, dtype=torch.float64)
        if name == "set_pdl":
            prev, _pdl[0] = _pdl[0], a[0]
            return prev
        return args.arguments.get("out")
    return rec


for _name, _f in list(vars(K).items()):
    if isinstance(_f, types.FunctionType) and _f.__module__ == K.__name__ and _name not in KEEP and not _name.startswith("__"):
        setattr(K, _name, _stub(_name, _f))
K._chk = lambda t, name: None


def _ptr(t):
    if t is None:
        return None
    _ordinal(t)
    return Ptr(t.data_ptr())


def _mask_descriptors(items, device, _build=K.mask_descriptors):
    table, tiles = _build(items, device)
    _tables[id(table)] = (table, 5)   # (w, s, u, out, outT pointers, then extents and the stream id)
    return table, tiles


K.mask_descriptors = _mask_descriptors


lib.ptr = _ptr
lib.call = lambda name, *a, meta=None: TRACE.append([name, _current[-1].id, desc(a)])
lib.stream = lambda: _current[-1].id
lib.load = lambda: types.SimpleNamespace(sc_adam_clip_st_chunk=lambda: 4096, sc_prune_chunk=lambda: 4096, sc_set_pdl=lambda m: 0)


# ---- cases -----------------------------------------------------------------------------------------------------------------
CFG = dict(d_model=512, dim_feedforward=1024, num_layers=3, num_heads=8, max_seq_length=9, att_feat_size=64, vocab_size=203)
SD = O.random_state_dict(O.Cfg(**CFG), seed=5, sparsity=0.0)
B, N, S, T = 6, 12, 2, 9
OPT = dict(sparsity_target=0.9, sparsity_weight=5.0, current_step=3, max_step=10)


def _batch(step, att_masks=False):
    g = torch.Generator().manual_seed(100 + step)
    seqs = torch.randint(4, CFG["vocab_size"], (B * S, T + 1), generator=g)
    masks = (torch.rand(B * S, T + 1, generator=g) < 0.8).float()
    am = (torch.rand(B, N, generator=g) < 0.7).float() if att_masks else None
    return torch.rand(B, N, CFG["att_feat_size"], generator=g), torch.rand(B, N, 4, generator=g), seqs, masks, am


def _trainer(mask_type="supermask", precision="bf16", attn16=False, overlap=False, **kw):
    kw = dict(dict(seed=11, dropout=0.1, drop_prob_src=0.3), **kw)
    tr = OrtTrainer(SD, ModelCfg(CFG), mask_type=mask_type, precision=precision, device="cpu", **kw)
    tr.fuse_attn_bwd, tr.overlap_opt = attn16, overlap
    return tr


def _collect(tr):
    seen, out = set(), []

    def walk(o):
        if torch.is_tensor(o):
            out.append(o)
        elif isinstance(o, dict):
            for v in o.values():
                walk(v)
        elif isinstance(o, (list, tuple)):
            for v in o:
                walk(v)
        elif hasattr(o, "__dict__") and type(o).__name__ == "TrainWs" and id(o) not in seen:
            seen.add(id(o))
            walk(vars(o))
    walk(vars(tr))
    return out


def _steps(tr, n=2, *, att_masks=False, **kw):
    for i in range(n):
        att, boxes, seqs, masks, am = _batch(i, att_masks)
        tr.train_step(att, boxes, seqs, masks, am, seq_per_img=S, lr=1e-3, **dict(OPT, **kw))


def _graph_steps(tr, n=2):
    for i in range(n):
        att, boxes, seqs, masks, _ = _batch(i)
        ws = tr._get_ws(B, N, S, T, False)
        tr.step_id += 1
        tr.load_batch(ws, att, boxes, seqs, masks)
        tr._upload_step(lr=1e-3, **OPT)
        tr._graph_body(ws, "all", dict(OPT, lr=1e-3))


def _all_reduce(t):
    TRACE.append(["all_reduce", desc(t)])


class _Exchange:
    def bucket(self, grad, param, a, b, update):
        TRACE.append(["exchange.bucket", desc(grad), desc(param), a, b])
        update(a, b)

    def finish(self):
        TRACE.append(["exchange.finish"])


def _snip(tr):
    att, boxes, seqs, masks, _ = _batch(0)
    tr.snip_saliency(att, boxes, seqs, masks, seq_per_img=S)
    tr.update_masks_once(0.5)
    tr.mask_sparsities()


def _materialize(tr):
    att, boxes, seqs, masks, _ = _batch(0)
    ws = tr._get_ws(B, N, S, T, False)
    tr.step_id += 1
    tr.load_batch(ws, att, boxes, seqs, masks)
    tr.forward(ws)
    tr.loss_and_backward(ws)
    tr.materialize_grads()
    tr.optimizer_step(lr=1e-3, **OPT)
    tr.training = False
    tr.forward(ws)


def _uniforms():
    g = torch.Generator().manual_seed(7)
    return {k: torch.rand(v.shape, generator=g) for k, v in SD.items() if k.endswith(".weight") and v.dim() == 2}


CASES = {}
for prec in ("bf16", "fp32"):
    for st in (True, False):
        for a16 in (False, True):
            CASES[f"{prec}-st{int(st)}-attn16{int(a16)}"] = (lambda p=prec, s=st, a=a16: _trainer(precision=p, fused_st=s, attn16=a), _steps)
CASES.update({
    "bf16-dense": (lambda: _trainer(mask_type=None), _steps),
    "fp32-dense": (lambda: _trainer(mask_type=None, precision="fp32"), _steps),
    "bf16-mag_blind": (lambda: _trainer(mask_type="mag_blind"), _steps),
    "bf16-att_masks": (lambda: _trainer(), lambda tr: _steps(tr, att_masks=True)),
    "fp32-uniforms": (lambda: _trainer(precision="fp32", uniforms=_uniforms()), _steps),
    "bf16-all_reduce": (lambda: _trainer(), lambda tr: _steps(tr, all_reduce=_all_reduce)),
    "bf16-all_reduce-attn16": (lambda: _trainer(attn16=True), lambda tr: _steps(tr, all_reduce=_all_reduce)),
    "bf16-exchange": (lambda: _trainer(fused_st=False), lambda tr: _steps(tr, exchange=_Exchange())),
    "fp32-exchange": (lambda: _trainer(precision="fp32", fused_st=False), lambda tr: _steps(tr, exchange=_Exchange())),
    "bf16-graph": (lambda: _trainer(use_graph=True), _graph_steps),
    "bf16-graph-overlap": (lambda: _trainer(use_graph=True, overlap=True), _graph_steps),
    "fp32-graph-st0": (lambda: _trainer(precision="fp32", use_graph=True, fused_st=False), _graph_steps),
    "bf16-snip": (lambda: _trainer(mask_type="snip"), _snip),
    "fp32-snip-st0": (lambda: _trainer(mask_type="snip", precision="fp32", fused_st=False), _snip),
    "bf16-mag_blind-update": (lambda: _trainer(mask_type="mag_blind"), lambda tr: (tr.update_masks_once(0.5), tr.mask_sparsities())),
    "bf16-supermask-sparsities": (lambda: _trainer(), lambda tr: tr.mask_sparsities()),
    "bf16-materialize-eval": (lambda: _trainer(), _materialize),
})


def main(path):
    out = {}
    for name, (make, run) in CASES.items():
        TRACE.clear()
        _storages.clear()
        _tables.clear()
        _pdl[0] = 7
        Stream.count, Event.count = 1, 0
        tr = _traced[0] = make()
        run(tr)
        TRACE.append(["state", tr.step_id, tr.opt_step, tr._seeds_dev.tolist(), tr._dyn_dev.tolist()])
        out[name] = list(TRACE)
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print(json.dumps({k: len(v) for k, v in out.items()}))


if __name__ == "__main__":
    main(sys.argv[1])
