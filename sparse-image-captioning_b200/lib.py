"""ctypes binding of the C ABI in include/sc_b200.h (built as csrc/libsc_b200.so).

The header is the single statement of the ABI: ``load()`` reads its declarations and derives every entry point's ctypes
argument and return types from them, and ``call()`` turns each Python argument into the ABI argument of the parameter it
fills, checking tensors against the header's conventions (device pointers, ``*_host`` pinned host pointers) on the way.

There is deliberately NO fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os
import re

import torch  # (also loads libcudart into the process before our library)

_HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(_HERE), "include", "sc_b200.h")
# SC_LIB_PATH: diagnostic override (same-box A/B of two builds of the library, scripts/); the product path is the in-tree build
LIB_PATH = os.environ.get("SC_LIB_PATH") or os.path.join(_HERE, "csrc", "libsc_b200.so")

F32, BF16 = 0, 1
MASK_NONE, MASK_ROUND, MASK_BERNOULLI, MASK_RAW, MASK_UNIFORM = 0, 1, 2, 3, 4

# parameter kinds: a value passed as is, a device pointer, a pinned host pointer (header name ending in _host), the stream
VALUE, DEVICE, HOST, STREAM = "value", "device", "host", "stream"
_VALUE_TYPES = {"int": C.c_int, "float": C.c_float, "double": C.c_double, "long": C.c_long, "size_t": C.c_size_t,
                "unsigned long long": C.c_ulonglong}
_RESTYPES = {"int": C.c_int, "const char *": C.c_char_p}


def parse_declarations(src):
    """Function declarations of a C header -> {name: (restype, [(parameter name, ctype, kind)])} for every ``sc_*`` function.
    Any pointer and ``sc_stream_t`` are ``c_void_p``; a type outside the map above is a RuntimeError, never a guess."""
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"^[ \t]*([A-Za-z_][\w \t*]*?)\s*\b(sc_\w+)\s*\(([^;{}]*)\)\s*;", src, flags=re.M):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        ret = " ".join(ret.replace("*", " * ").split())
        if ret not in _RESTYPES:
            raise RuntimeError(f"{name}: return type {ret!r} has no ctypes mapping")
        params = []
        for i, arg in enumerate([] if args in ("", "void") else args.split(",")):
            pm = re.fullmatch(r"(.*?)\s*\b(\w+)", arg.strip(), flags=re.S)
            pname, ptype = (pm.group(2), " ".join(re.sub(r"\bconst\b", " ", pm.group(1)).split())) if pm else (f"#{i}", arg)
            if "*" in ptype:
                params.append((pname, C.c_void_p, HOST if pname.endswith("_host") else DEVICE))
            elif ptype == "sc_stream_t":
                params.append((pname, C.c_void_p, STREAM))
            elif ptype in _VALUE_TYPES:
                params.append((pname, _VALUE_TYPES[ptype], VALUE))
            else:
                raise RuntimeError(f"{name}: parameter {pname} has type {ptype!r}, which has no ctypes mapping")
        out[name] = (_RESTYPES[ret], params)
    missed = set(re.findall(r"\b(sc_\w+)\s*\(", src)) - set(out)
    if missed:
        raise RuntimeError(f"declarations of {sorted(missed)} could not be parsed")
    return out


_lib = None
_params = {}   # name -> ([(parameter name, DEVICE | HOST | None)] without the trailing stream, whether the stream is appended)


def load():
    """Load the shared library (once) and bind every function the header declares.  Raises RuntimeError when the library has
    not been built or does not export a declared function."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"(or `make -C {os.path.dirname(LIB_PATH)}`).  There is no CPU/PyTorch fallback for this path.")
    with open(HEADER) as f:
        decl = parse_declarations(f.read())
    lib = C.CDLL(LIB_PATH)
    for name, (restype, params) in decl.items():
        if not hasattr(lib, name):
            raise RuntimeError(f"{name} is declared in {HEADER} but {LIB_PATH} does not export it")
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, [ctype for _, ctype, _ in params]
        stream = bool(params) and params[-1][2] == STREAM
        _params[name] = ([(p, kind if kind in (DEVICE, HOST) else None) for p, _, kind in params[:len(params) - stream]], stream)
    _lib = lib
    return lib


class Strided:
    """A row-strided view (e.g. ``q[:, d:]``) passed together with its leading dimension: ``call`` requires a unit inner stride
    of it instead of contiguity."""
    __slots__ = ("t",)

    def __init__(self, t):
        self.t = t


def _address(name, pname, kind, a, dev):
    """Address of tensor (or Strided view) ``a`` for pointer parameter ``pname`` of ``name``: a device pointer must be a CUDA
    tensor on the current device ``dev``, a host pointer a pinned CPU tensor; contiguous unless marked Strided.  Raises
    RuntimeError naming the parameter and what is wrong with it."""
    t = a.t if type(a) is Strided else a
    if kind is HOST:
        if t.is_cuda or not t.is_pinned():
            raise RuntimeError(f"{name}: {pname} must be a pinned CPU tensor, got a {'CUDA' if t.is_cuda else 'pageable CPU'} tensor")
    elif t.get_device() == dev:
        pass
    elif not t.is_cuda:
        raise RuntimeError(f"{name}: {pname} must be a CUDA tensor, got a {t.device.type} tensor: the B200 path has no CPU fallback")
    else:
        raise RuntimeError(f"{name}: {pname} is on cuda:{t.get_device()}, not on the current device cuda:{dev}: kernels launch on "
                           f"the current device, with no CPU fallback and no cross-device copy")
    if t is a:
        if not t.is_contiguous():
            raise RuntimeError(f"{name}: {pname} must be contiguous (strides {t.stride()})")
    elif t.stride(-1) != 1:
        raise RuntimeError(f"{name}: {pname} must have a unit inner stride (strides {t.stride()})")
    return t.data_ptr()


def address(t, name, pname):
    """Checked address of a tensor that a descriptor table of entry point ``name`` embeds (0 for None), as ``call`` checks
    pointer arguments."""
    if t is None:
        return 0
    return _address(name, pname, DEVICE, t, torch.cuda.current_device() if t.is_cuda else -2)


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


def _current():
    """(current device, the address of its current stream), read without building a torch.cuda.Stream; (-2, None) while CUDA is
    uninitialised, when no tensor can be a CUDA tensor."""
    if not torch.cuda.is_initialized():
        return -2, None
    dev = torch._C._cuda_getDevice()
    return dev, torch._C._cuda_getCurrentRawStream(dev)


def call(name, *args, meta=None):
    """Launch entry point ``name`` with ``args`` in the header's parameter order, the trailing stream left out: it is torch's
    current stream.  For a pointer parameter a tensor (or a Strided view) is checked and passed as its address and None as
    NULL; ints, including raw addresses, and floats pass unchanged.  Raises RuntimeError on a refused argument or a failed call."""
    global launch_count
    lib = _lib or load()
    try:
        params, has_stream = _params[name]
    except KeyError:
        raise RuntimeError(f"{name} is not declared in {HEADER}") from None
    if len(args) != len(params):
        raise TypeError(f"{name} takes {len(params)} arguments ({', '.join(p for p, _ in params)}), got {len(args)}")
    dev, stream = _current()
    # (the accepted device pointers are checked inline, _address() is the general case: this runs for every argument of every
    # eager launch)
    Tensor = torch.Tensor
    cargs = [a if kind is None or a is None or type(a) is int
             else a.data_ptr() if type(a) is Tensor and kind is DEVICE and a.get_device() == dev and a.is_contiguous()
             else a.t.data_ptr() if type(a) is Strided and kind is DEVICE and a.t.get_device() == dev and a.t.stride(-1) == 1
             else _address(name, p, kind, a, dev)
             for (p, kind), a in zip(params, args)]
    if has_stream:
        cargs.append(torch.cuda.current_stream().cuda_stream if stream is None else stream)
    if profile is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    rc = getattr(lib, name)(*cargs)
    if rc != 0:
        raise RuntimeError(f"{name} failed (status {rc}): {lib.sc_last_error().decode()}")
    if profile is not None:
        ev1.record()
        profile.append((name, meta, ev0, ev1))
    launch_count += 1
