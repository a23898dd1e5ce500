"""The C-ABI library loads, exports exactly what include/b200rnn.h declares, and its host-side logic
(descriptor validation, workspace sizing, error reporting) works without a GPU."""
import ctypes
import os
import re

import pytest

from conftest import ROOT
from b200rnn import _lib


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "b200rnn.h")).read()
    return sorted(set(re.findall(r"B200RNN_API\s+[\w\s\*]+?\b(b200rnn_\w+)\s*\(", text)))


def test_header_and_binding_agree():
    assert _declared_symbols() == sorted(_lib.SYMBOLS)


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in _declared_symbols():
        assert hasattr(lib, sym), sym
    assert _lib.load().b200rnn_version() == _lib.ABI_VERSION


def test_workspace_bytes_scale_with_the_problem():
    small = _lib.workspace_bytes(_lib.Desc(_lib.GRU, 8, 3, 256, 256, 2, 1, 1, 0.5, 0))
    big = _lib.workspace_bytes(_lib.Desc(_lib.GRU, 128, 120, 256, 256, 2, 1, 1, 0.5, 0))
    assert all(b > s > 0 for s, b in zip(small, big))
    # reserve holds, per layer: gates [T,B,3H] + hn [T,B,H]; plus layer-0 output raw and dropped [T,B,H]
    T, B, H = 120, 128, 256
    expect = 4 * T * B * (2 * 4 * H + 2 * H)
    assert expect <= big[0] <= expect * 1.01 + 4096
    # scratch: 18 [T,B,H] blocks (dG, dn*r, dy, dLN(x), hi/lo of dG, dn*r, X, h) + ~1.2 of GEMM partials and weights
    assert big[1] <= 20 * 4 * T * B * H
    lstm = _lib.workspace_bytes(_lib.Desc(_lib.LSTM, 64, 30, 1024, 256, 2, 2, 1, 0.0, 0))
    assert lstm[0] >= 4 * 30 * 64 * (2 * 2 * 5 * 256 + 2 * 256)


@pytest.mark.parametrize("desc,frag", [
    (_lib.Desc(7, 4, 4, 16, 128, 1, 1, 0, 0.0, 0), "mode"),
    (_lib.Desc(_lib.GRU, 4, 4, 16, 100, 1, 1, 0, 0.0, 0), "hidden_size"),
    (_lib.Desc(_lib.GRU, 4, 4, 16, 128, 1, 3, 0, 0.0, 0), "bad shape"),
    (_lib.Desc(_lib.LSTM, 4, 4, 0, 128, 1, 1, 0, 0.0, 0), "bad shape"),
    (_lib.Desc(_lib.LSTM, 4, 4, 16, 128, 1, 1, 0, 1.5, 0), "dropout_p"),
])
def test_invalid_descriptors_are_rejected_with_a_message(desc, frag):
    with pytest.raises(_lib.B200RNNError) as ei:
        _lib.workspace_bytes(desc)
    assert frag in str(ei.value)


def test_forward_rejects_null_pointers_before_touching_the_device():
    lib = _lib.load()
    d = _lib.Desc(_lib.GRU, 2, 2, 16, 128, 1, 1, 0, 0.0, 0)
    rc = lib.b200rnn_forward(ctypes.byref(d), None, 0, 0, None, None, 0, 0, None, None, None, None, 0, 0, None, None)
    assert rc == -1 and b"null pointer" in lib.b200rnn_last_error()


def _prototypes():
    """{name: [C parameter type strings]} parsed from include/b200rnn.h (comments stripped)."""
    text = open(os.path.join(ROOT, "include", "b200rnn.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    out = {}
    for m in re.finditer(r"B200RNN_API\s+[\w\s\*]+?\b(b200rnn_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        params = [p.strip() for p in m.group(2).replace("\n", " ").split(",")]
        out[m.group(1)] = [] if params in ([""], ["void"]) else params
    return out


def _kind_of_c(param: str) -> str:
    if "*" in param:
        return "ptr"
    for c_name, kind in (("uint64_t", "u64"), ("int64_t", "i64"), ("uint32_t", "u32"), ("size_t", "size"),
                         ("float", "f32"), ("int32_t", "i32"), ("int", "i32")):
        if re.search(rf"\b{c_name}\b", param):
            return kind
    raise AssertionError(f"unclassified C parameter: {param!r}")


def _kind_of_ctypes(t) -> str:
    if t is ctypes.c_void_p or t is ctypes.c_char_p or hasattr(t, "contents"):
        return "ptr"
    return {ctypes.c_uint64: "u64", ctypes.c_int64: "i64", ctypes.c_uint32: "u32", ctypes.c_size_t: "size",
            ctypes.c_float: "f32", ctypes.c_int: "i32", ctypes.c_int32: "i32"}[t]


def test_ctypes_argtypes_match_the_header_prototypes_parameter_by_parameter():
    """An argument added to the header but not to the binding (or bound with the wrong width) corrupts the call
    silently; compare every prototype with the ctypes signature."""
    lib = _lib.load()
    protos = _prototypes()
    assert sorted(protos) == sorted(_lib.SYMBOLS)
    for name, params in protos.items():
        argtypes = getattr(lib, name).argtypes
        assert argtypes is not None, f"{name}: no argtypes set"
        got = [_kind_of_ctypes(t) for t in argtypes]
        want = [_kind_of_c(p) for p in params]
        # size_t and u64 are the same register class on LP64; keep them distinct anyway, except where ctypes
        # aliases them (c_size_t is c_ulong is c_uint64 on this platform)
        norm = lambda ks: ["u64" if k == "size" else k for k in ks]  # noqa: E731
        assert norm(got) == norm(want), f"{name}: binding {got} vs header {want}"


def test_fuse_head_argument_block_matches_the_library():
    """The ctypes mirror of b200rnn_fuse_head_args must have the library's size; a stale binding is rejected with a
    message instead of corrupting the launch (checked before anything touches the device)."""
    lib = _lib.load()
    a = _lib.FuseHeadArgs(B=0, Ht=128, Ha=256)
    assert lib.b200rnn_fuse_head(ctypes.byref(a), None) == 0      # B == 0: accepted, nothing launched
    a.struct_bytes -= 8
    assert lib.b200rnn_fuse_head(ctypes.byref(a), None) == -1
    assert b"mismatched argument block" in lib.b200rnn_last_error()
    assert lib.b200rnn_comm_bytes() >= 2 * 8 * 768 * 4
    assert lib.b200rnn_fuse_head_scratch_floats(128, 128, 256, 0) == 128 * (8 + 384)
