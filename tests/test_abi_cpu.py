"""CPU tier: the C-ABI library builds/loads and exports every symbol include/sc_b200.h declares, and the ctypes types lib.py
derives from the header are the declared ones; no compute call is made (there is no GPU here)."""
import ctypes
import os

import pytest

from sparse_caption_b200 import lib


def _header_functions():
    with open(lib.HEADER) as f:
        return lib.parse_declarations(f.read())


def test_library_exports_every_declared_symbol():
    if not os.path.exists(lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    so = ctypes.CDLL(lib.LIB_PATH)
    decl = _header_functions()
    assert len(decl) >= 30
    for name in decl:
        assert hasattr(so, name), f"{name} declared in include/sc_b200.h but not exported"


def test_every_declaration_parses_into_known_ctypes_types():
    decl = _header_functions()
    known = {ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_long, ctypes.c_size_t, ctypes.c_ulonglong}
    for name, (restype, params) in decl.items():
        assert restype in (ctypes.c_int, ctypes.c_char_p), name
        assert all(ctype in known for _, ctype, _ in params), name
        assert len({p for p, _, _ in params}) == len(params), f"{name}: parameter names are not distinct"
        if name not in ("sc_last_error", "sc_version") and not name.endswith(("_chunk", "_parts", "_workspace_bytes", "_pdl")):
            assert params[-1][1:] == (ctypes.c_void_p, lib.STREAM), f"{name} does not end in its stream"
    assert decl["sc_last_error"] == (ctypes.c_char_p, []) and decl["sc_version"] == (ctypes.c_int, [])
    so = lib.load()
    for name, (restype, params) in decl.items():
        assert getattr(so, name).restype is restype and getattr(so, name).argtypes == [c for _, c, _ in params], name


def test_non_int_parameters_have_their_declared_types():
    """The positions an arity check cannot see: double, long, size_t, unsigned long long, and the pointer kinds."""
    decl = {name: {p: (ctype, kind) for p, ctype, kind in params} for name, (_, params) in _header_functions().items()}
    assert decl["sc_sparsity_coeff"]["total"] == (ctypes.c_double, lib.VALUE)
    assert decl["sc_ciderd_score"]["sigma"] == (ctypes.c_double, lib.VALUE)
    assert decl["sc_adam_clip_st"]["total_blocks"] == (ctypes.c_long, lib.VALUE)
    assert decl["sc_prune_select"]["total_blocks"] == (ctypes.c_long, lib.VALUE)
    assert decl["sc_cache_reorder"]["row_bytes"] == (ctypes.c_long, lib.VALUE)
    assert decl["sc_beam_step"]["workspace_bytes"] == (ctypes.c_size_t, lib.VALUE)
    assert decl["sc_linear_wgrad"]["workspace_bytes"] == (ctypes.c_size_t, lib.VALUE)
    assert decl["sc_apply_mask"]["n"] == (ctypes.c_size_t, lib.VALUE)
    for name, p in (("sc_linear", "seed"), ("sc_linear", "stream_id"), ("sc_linear_dropout", "drop_seed"), ("sc_sample_step", "seed"),
                    ("sc_adam_clip_st", "stream_base")):
        assert decl[name][p] == (ctypes.c_ulonglong, lib.VALUE), (name, p)
    assert decl["sc_linear"]["tile_n"] == (ctypes.c_int, lib.VALUE)
    assert decl["sc_linear_dropout"]["dropout_p"] == (ctypes.c_float, lib.VALUE)
    assert decl["sc_csr_spmm"]["col_idx"] == (ctypes.c_void_p, lib.DEVICE)
    assert decl["sc_bleu_stats"]["stats"] == (ctypes.c_void_p, lib.DEVICE)
    assert decl["sc_ingest_f32_bf16"]["pinned_host"] == (ctypes.c_void_p, lib.HOST)


@pytest.mark.parametrize("src,what", [
    ("int sc_x(int a, half b, sc_stream_t stream);", r"sc_x: parameter b has type 'half'"),
    ("int sc_x(int a, long long n);", r"sc_x: parameter n has type 'long long'"),
    ("int sc_x(unsigned n);", r"sc_x: parameter n has type 'unsigned'"),
    ("void sc_x(int a);", r"sc_x: return type 'void'"),
    ("int sc_x(int a,\n  int);", r"sc_x: parameter .* has type ''"),
])
def test_unknown_types_are_refused(src, what):
    with pytest.raises(RuntimeError, match=what):
        lib.parse_declarations("/* a comment: int sc_y(half h); */\n" + src)


def test_version_and_error_string():
    so = lib.load()
    assert so.sc_version() >= 100
    assert isinstance(so.sc_last_error(), bytes)


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(lib, "_lib", None)
    monkeypatch.setattr(lib, "LIB_PATH", "/nonexistent/libsc_b200.so")
    with pytest.raises(RuntimeError, match="no CPU/PyTorch fallback"):
        lib.load()
