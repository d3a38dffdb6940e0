"""Launch sequence of the fused training step (OrtTrainer) or of the inference engine (OrtEngine), recorded on the CPU: every
kernel wrapper, raw ``lib.call``, CUDA stream / event operation and CUDA graph capture / replay is replaced by a recorder, so whole
steps run on CPU tensors and leave a deterministic JSON trace of the launches they would issue - each with its stream, tensors
described by shape, dtype, stride, storage offset and storage ordinal (the order in which the storage first appears),
pointer-valued ints (descriptor tables, bit-63 seed pointers) mapped through the same table.  A change to trainer.py or engine.py
that keeps the launch sequence (same kernels, order, arguments, buffers, Philox streams, ring slots, side-stream forks and joins)
keeps this output byte-identical.

The engine cases also record the torch operations that do device work once the engine is built (state resets, output copies,
the bad-endings mask, token copies; allocations and views are left out) and start with a digest of every packed weight by slot
name, so a change in the order the weights are packed in does not show as a difference.

    python scripts/launch_trace.py trainer OUT.json
    python scripts/launch_trace.py engine OUT.json
"""
import contextlib
import hashlib
import inspect
import json
import os
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.utils._python_dispatch import TorchDispatchMode

from oracle import ort_oracle as O
from sparse_caption_b200 import kernels as K, lib
from sparse_caption_b200.engine import ModelCfg, OrtEngine
from sparse_caption_b200.trainer import OrtTrainer

TRACE = []
_storages = []     # (base, nbytes, tensor kept alive) in order of first appearance
_traced = [None]   # the trainer or engine being traced: a pointer seen before its tensor is resolved through its tensors
_owners = []       # the trainer that owns the memory of a traced rollout engine
_quiet = [0]       # > 0 while a recorder runs: its own torch operations are not part of the trace


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
    raise LookupError(f"pointer {p:#x} is in no tensor of the traced object")


class Ptr(int):
    """A pointer from lib.ptr: described through the storage table, never as its value."""


_tables = {}       # id -> (table, number of leading pointer columns) of the descriptor tables built by the run


def desc(a):
    if torch.is_tensor(a):
        d = ["T", list(a.shape), str(a.dtype).replace("torch.", ""), list(a.stride()), a.storage_offset(), _ordinal(a)]
        if a.dtype == torch.int64 and a.dim() and 0 < a.numel() <= 4096:   # descriptor tables: their buffers, extents and Philox streams
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
    if type(a).__name__ in STATES:   # search states and sparse weight packs: by the buffers they hold
        return [type(a).__name__, [[k, desc(v)] for k, v in sorted(vars(a).items())]]
    return type(a).__name__


STATES = {"BeamState", "GreedyState", "Tok", "CsrWeight", "SellWeight", "GsWeight"}


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
        with _recording():
            return record(*a, **kw)

    def record(*a, **kw):
        if name in PURE:
            return PURE[name](*a, **kw)
        args = sig.bind(*a, **kw)
        args.apply_defaults()   # (an argument passed at its default value and one left out are the same launch)
        TRACE.append([name, _current[-1].id, [[k, desc(v)] for k, v in args.arguments.items()]])
        if name == "cast_bf16" and args.arguments["out"] is None:   # (the allocating form: OrtEngine packs weights with it)
            return a[0].to(torch.bfloat16)
        if name == "prune_stats":
            return torch.zeros(a[0].shape[0], 2, dtype=torch.float64)
        if name == "set_pdl":
            prev, _pdl[0] = _pdl[0], a[0]
            return prev
        return args.arguments.get("out")
    return rec


@contextlib.contextmanager
def _recording():
    _quiet[0] += 1
    try:
        yield
    finally:
        _quiet[0] -= 1


# host-side sizes: answered without a trace entry
PURE = {"linear_topk_parts": K.linear_topk_parts, "beam_step_workspace_bytes": lambda B, beam: 64 * B * beam}

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


def _call(name, *a, meta=None):
    with _recording():
        TRACE.append([name, _current[-1].id, desc(a)])


lib.call = _call
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
        elif hasattr(o, "__dict__") and type(o).__name__ in WORKSPACES and id(o) not in seen:
            seen.add(id(o))
            walk(vars(o))
    for root in [tr] + _owners:
        walk(vars(root))
    return out


WORKSPACES = {"TrainWs", "OrtEngine", "EncWs", "DecWs", "DiverseWs", "StepWs", "BeamState", "GreedyState", "Tok"}


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


# ---- engine -----------------------------------------------------------------------------------------------------------------
class Graph:
    count = 0

    def __init__(self, *a, **k):
        self.id, Graph.count = Graph.count, Graph.count + 1

    def replay(self):
        TRACE.append(["graph.replay", self.id, _current[-1].id])


@contextlib.contextmanager
def _capture(g, *a, **k):
    TRACE.append(["graph.capture", g.id, _current[-1].id])
    yield
    TRACE.append(["graph.end", g.id])


class _TorchOps(TorchDispatchMode):
    """Records the torch operations that do device work; allocations (no tensor argument) and views are left out."""

    def __torch_dispatch__(self, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        out = func(*args, **kwargs)
        schema = func._schema
        tensors = [a for a in list(args) + list(kwargs.values()) if torch.is_tensor(a)
                   or (isinstance(a, (list, tuple)) and any(torch.is_tensor(x) for x in a))]
        view = not schema.is_mutable and all(r.alias_info is not None for r in schema.returns)
        if not _quiet[0] and tensors and not view:
            with _recording():
                TRACE.append([f"aten.{func.__name__}", _current[-1].id, desc(list(args)),
                              [[k, desc(v)] for k, v in sorted(kwargs.items())], desc(out)])
        return out


def _digest(t):
    if t is None:
        return None
    t = t.detach().contiguous()
    d = [list(t.shape), str(t.dtype).replace("torch.", "")]
    if _owners:   # a rollout engine's operands are written by the trainer's (stubbed) kernels: not their values
        return d
    return d + [hashlib.sha256(t.view(-1).view(torch.uint8).numpy().tobytes()).hexdigest()[:24]]


def _packed(v):
    """Digests of one packed weight: a linear's dense / folded / sparse operands, a LayerNorm's parameters, or a tensor."""
    if torch.is_tensor(v):
        return _digest(v)
    if isinstance(v, (int, tuple)):
        return v
    out = {}
    for k, x in sorted(vars(v).items()):
        if torch.is_tensor(x):
            out[k] = _digest(x)
        elif type(x).__name__ in STATES:
            out[k] = {kk: _digest(xx) if torch.is_tensor(xx) else str(xx) for kk, xx in sorted(vars(x).items())}
        elif isinstance(x, (int, float)) or x is None:
            out[k] = x
    return out


def _weights(eng):
    w = {name: _packed(getattr(eng, name)) for name in ("att_embed", "generator", "enc_norm", "dec_norm", "table", "pe",
                                                         "wg_w_all", "wg_b_all")}
    for stack in ("enc", "dec"):
        for u, e in getattr(eng, stack).items():
            for slot, v in sorted(e.items()):
                w[f"{stack}.{u}.{slot}"] = _packed(v)
    return w


ECFG = dict(CFG)
ACORT = dict(CFG, num_layers=4, share_att_encoder="kv", share_att_decoder="qk", share_layer_encoder=[0, 0, 1, 1],
             share_layer_decoder=[0, 1, 1, 0])
SDS = {}


def _sd(cfg, sparsity=0.0):
    key = (json.dumps(cfg, sort_keys=True), sparsity)
    if key not in SDS:
        SDS[key] = O.random_state_dict(O.Cfg(**cfg), seed=5, sparsity=sparsity)
    return SDS[key]


def _inputs(seed=0, b=B, masks=False):
    g = torch.Generator().manual_seed(200 + seed)
    am = None
    if masks:
        am = (torch.rand(b, N, generator=g) < 0.8).float()
        am[:, 0] = 1
    return torch.rand(b, N, CFG["att_feat_size"], generator=g), torch.rand(b, N, 4, generator=g), am


def _engine(cfg=ECFG, sparsity=0.0, **kw):
    return OrtEngine(_sd(cfg, sparsity), ModelCfg(cfg), device="cpu", **kw)


def _dec(*opts, masks=False, reps=2):
    """encode + decode per option dict, twice (the second call replays the captured graphs)."""
    def run(eng):
        for i in range(reps):
            att, boxes, am = _inputs(i, masks=masks)
            enc = eng.encode(att, boxes, am)
            for o in opts:
                eng.decode(enc, dict(o))
    return run


BEAM3, BEAM5, GREEDY = dict(beam_size=3), dict(beam_size=5), dict(beam_size=1)
BEAM_OPTS = dict(beam_size=3, temperature=0.7, decoding_constraint=1, bad_endings_ix=[7, 11, 5], penalized_col=1,
                 length_penalty="wu_0.9")
DIV2, DIV3 = dict(beam_size=4, group_size=2, diversity_lambda=0.5), dict(beam_size=6, group_size=3, diversity_lambda=0.3)
SAMPLE = dict(beam_size=0, num_random_sample=2, temperature=0.8)


def _uniform_sample(eng):
    att, boxes, _ = _inputs(0)
    enc = eng.encode(att, boxes)
    u = torch.rand(CFG["max_seq_length"], B * 2, generator=torch.Generator().manual_seed(3))
    eng.decode(enc, dict(SAMPLE, sample_uniforms=u))
    eng.decode(enc, dict(SAMPLE, sample_seed=17))


def _teacher_force(eng):
    att, boxes, am = _inputs(0, masks=True)
    enc = eng.encode(att, boxes, am)
    tokens = torch.randint(4, CFG["vocab_size"], (B * 2, CFG["max_seq_length"] - 1), generator=torch.Generator().manual_seed(4))
    eng.teacher_force(enc, tokens, beam=2)


def _logprobs_step(eng):
    g = torch.Generator().manual_seed(5)
    R, d = B * 3, CFG["d_model"]
    memory = torch.rand(B, N, d, generator=g)
    am = torch.ones(B, 1, N)
    am[:, :, -3:] = 0
    it = torch.full((B,), 2, dtype=torch.long)
    lp, caches = eng.logprobs_step(it, memory, am, None, 0)
    it = torch.randint(4, CFG["vocab_size"], (R,), generator=g)
    eng.logprobs_step(it, memory.repeat_interleave(3, 0), am.repeat_interleave(3, 0), caches, 1)


def _stepwise(opt):
    def run(eng):
        g = torch.Generator().manual_seed(6)
        V = CFG["vocab_size"]
        init_lp = torch.log_softmax(torch.rand(B, V, generator=g), -1)
        init_state = [torch.rand(1, B, 4, generator=g)]
        args = [torch.rand(B * opt["beam_size"], 5, generator=g), None]
        calls = [0]

        def get_logprobs_state(it, a, _none, state):
            calls[0] += 1
            lg = torch.rand(it.shape[0], V, generator=torch.Generator().manual_seed(calls[0]))
            return torch.log_softmax(lg, -1), [x + a.sum() * 0 for x in state]
        eng.beam_search_stepwise(init_state, init_lp, args, dict(opt), get_logprobs_state)
    return run


def _submit(eng):
    for i in range(2):
        att, boxes, _ = _inputs(i)
        for slot in (0, 1, 2):
            eng.submit(att, boxes, opt=[dict(BEAM3), dict(GREEDY), dict(SAMPLE)] if slot == 2 else dict(BEAM3), slot=slot)
        eng.wait()
        eng.wait(1, host=True)


def _prefetch(eng):
    for i in range(2):
        att, boxes, _ = _inputs(i)
        eng.submit(att, boxes, opt=dict(BEAM3), slot=1, prefetch=True)
        eng.wait(1)


def _ingest(eng):
    eng.zero_copy_ingest = 8
    for i in range(2):
        att, boxes, am = _inputs(i, masks=i == 1)
        eng.submit(att, boxes, am, opt=dict(BEAM3), slot=i)
    eng.wait()


def _rollout(precision="bf16"):
    tr = _trainer(precision=precision)
    _owners.append(tr)
    return tr.rollout_engine()


ECASES = {}
for prec in ("bf16", "fp32"):
    for fold in (False, True):
        for m in (False, True):
            ECASES[f"{prec}-fold{int(fold)}-masks{int(m)}"] = (
                lambda p=prec, f=fold: _engine(precision=p, ln_fold=f), _dec(GREEDY, BEAM3, BEAM5, DIV2, masks=m))
for be in ("csr", "sell", "auto"):
    ECASES[f"bf16-{be}"] = (lambda b=be: _engine(sparsity=0.997, sparse_backend=b), _dec(GREEDY, BEAM3, DIV2))
    ECASES[f"fp32-{be}"] = (lambda b=be: _engine(sparsity=0.997, sparse_backend=b, precision="fp32"), _dec(GREEDY, BEAM3))
ECASES.update({
    "bf16-auto-fold-ctas": (lambda: _engine(sparsity=0.997, sparse_backend="auto", ln_fold=True, dec_ctas=(48, 60)),
                            _dec(GREEDY, BEAM3, DIV2)),
    "bf16-fold-ctas-tiles": (lambda: _engine(ln_fold=True, dec_ctas=(48, 60), dec_tiles={"o": 3256}), _dec(GREEDY, BEAM3, DIV3)),
    "bf16-ctas-tiles": (lambda: _engine(dec_ctas=(40, 50), dec_tiles={"ff1": 3128}), _dec(GREEDY, BEAM5)),
    "bf16-nofuse": (lambda: _engine(fuse_topk=False), _dec(BEAM3, DIV2, DIV3)),
    "bf16-eager": (lambda: _engine(use_graphs=False), _dec(GREEDY, BEAM3, DIV2, SAMPLE)),
    "fp32-eager": (lambda: _engine(use_graphs=False, precision="fp32"), _dec(GREEDY, BEAM3, DIV3, SAMPLE)),
    "bf16-no_history": (lambda: _engine(no_history=True), _dec(GREEDY, BEAM3)),
    "bf16-acort": (lambda: _engine(ACORT), _dec(GREEDY, BEAM3, DIV2)),
    "bf16-acort-fold": (lambda: _engine(ACORT, ln_fold=True), _dec(GREEDY, BEAM5, masks=True)),
    "fp32-acort": (lambda: _engine(ACORT, precision="fp32"), _dec(GREEDY, BEAM3)),
    "bf16-beam-options": (lambda: _engine(), _dec(BEAM_OPTS, dict(BEAM_OPTS, length_penalty="avg_1.2", temperature=1.0),
                                                  dict(beam_size=3, length_penalty="avg_0.5"), dict(DIV3, **{k: v for k, v in BEAM_OPTS.items() if k != "beam_size"}))),
    "bf16-fold-beam-options": (lambda: _engine(ln_fold=True), _dec(BEAM_OPTS, dict(DIV2, bad_endings_ix=[5], penalized_col=1))),
    "fp32-beam-options": (lambda: _engine(precision="fp32"), _dec(BEAM_OPTS, dict(DIV2, length_penalty="wu_0.5", temperature=0.9))),
    "bf16-sample": (lambda: _engine(), _dec(SAMPLE, dict(SAMPLE, decoding_constraint=1))),
    "bf16-sample-uniforms": (lambda: _engine(), _uniform_sample),
    "bf16-teacher_force": (lambda: _engine(), _teacher_force),
    "fp32-fold-teacher_force": (lambda: _engine(precision="fp32", ln_fold=True), _teacher_force),
    "bf16-fold-teacher_force": (lambda: _engine(ln_fold=True), _teacher_force),
    "bf16-logprobs_step": (lambda: _engine(), _logprobs_step),
    "bf16-fold-logprobs_step": (lambda: _engine(ln_fold=True), _logprobs_step),
    "fp32-logprobs_step": (lambda: _engine(precision="fp32"), _logprobs_step),
    "bf16-stepwise-g1": (lambda: _engine(), _stepwise(dict(BEAM_OPTS, beam_size=3))),
    "bf16-stepwise-g2": (lambda: _engine(), _stepwise(dict(DIV2, bad_endings_ix=[5], length_penalty="avg_1.0"))),
    "bf16-stepwise-g3": (lambda: _engine(), _stepwise(dict(DIV3, temperature=0.5))),
    "bf16-submit": (lambda: _engine(), _submit),
    "bf16-prefetch": (lambda: _engine(), _prefetch),
    "bf16-ingest": (lambda: _engine(), _ingest),
    "bf16-rollout": (_rollout, _dec(BEAM3, GREEDY, DIV2, SAMPLE)),
    "fp32-rollout": (lambda: _rollout("fp32"), _dec(BEAM3, GREEDY)),
})


def _engine_stubs():
    torch.cuda.is_available = lambda: True
    torch.cuda.synchronize = lambda *a: None
    torch.cuda.CUDAGraph, torch.cuda.graph = Graph, _capture
    torch.Tensor.is_pinned = lambda self: True


def _reset():
    TRACE.clear()
    _storages.clear()
    _tables.clear()
    _owners.clear()
    _pdl[0] = 7
    Stream.count, Event.count, Graph.count = 1, 0, 0


def main(which, path):
    out = {}
    if which == "engine":
        _engine_stubs()
    for name, (make, run) in (CASES if which == "trainer" else ECASES).items():
        _reset()
        obj = _traced[0] = make()
        if which == "trainer":
            run(obj)
            TRACE.append(["state", obj.step_id, obj.opt_step, obj._seeds_dev.tolist(), obj._dyn_dev.tolist()])
        else:
            TRACE.clear()   # (weight packing: described by the digests below)
            TRACE.append(["weights", _weights(obj)])
            with _TorchOps():
                run(obj)
        out[name] = list(TRACE)
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print(json.dumps({k: len(v) for k, v in out.items()}))


if __name__ == "__main__":
    main(*sys.argv[1:3])
