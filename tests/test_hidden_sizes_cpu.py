"""Hidden sizes 64 and 512 next to 128 and 256, checked without a GPU: the descriptor accepts them, the workspace
layouts (reserve, scratch, weight cache) follow the same per-layer formulas at every width, other widths are still
rejected with a message naming the supported ones, and the recurrence kernels built for the new widths exist in the
library without local-memory traffic."""
import ctypes
import re
import shutil
import subprocess

import pytest

from b200rnn import _lib

SIZES = (64, 128, 256, 512)
NEW = (64, 512)


def _reserve_floats(G, T, B, H, L, D, p):
    """Per layer and direction: gates [T,B,G*H] + hn / c_t [T,B,H]; between layers the raw output [T,B,D*H] and,
    with dropout, the dropped copy."""
    per_layer = L * D * (G + 1) * H
    between = (L - 1) * D * H * (2 if p > 0 else 1)
    return T * B * (per_layer + between)


@pytest.mark.parametrize("H", SIZES)
@pytest.mark.parametrize("mode", [_lib.GRU, _lib.LSTM])
@pytest.mark.parametrize("D", [1, 2])
def test_workspace_follows_the_per_layer_formula(H, mode, D):
    G = 3 if mode == _lib.GRU else 4
    T, B, I, L, p = 120, 128, 256, 2, 0.5
    reserve, scratch = _lib.workspace_bytes(_lib.Desc(mode, B, T, I, H, L, D, 1, p, 0))
    expect = 4 * _reserve_floats(G, T, B, H, L, D, p)
    # 256-byte alignment of every block and a 256-byte header
    assert expect <= reserve <= expect * 1.01 + 4096, (H, mode, D, reserve, expect)
    # scratch: at least dG [T,B,G*H] per direction
    assert scratch >= 4 * T * B * D * G * H


@pytest.mark.parametrize("mode", [_lib.GRU, _lib.LSTM])
def test_reserve_is_linear_and_scratch_monotone_in_the_hidden_size(mode):
    """Every reserve block is a multiple of H at a fixed input width, so the reserve scales with H; the scratch grows
    with it (it also holds fixed-size GEMM partials)."""
    T, B, I = 30, 64, 1024
    ws = {H: _lib.workspace_bytes(_lib.Desc(mode, B, T, I, H, 2, 2, 1, 0.0, 0)) for H in SIZES}
    for H in SIZES:
        assert abs(ws[H][0] / ws[128][0] - H / 128) < 0.01, (H, ws[H][0], ws[128][0])
    assert all(ws[a][1] < ws[b][1] for a, b in zip(SIZES, SIZES[1:])), ws


@pytest.mark.parametrize("H", NEW)
@pytest.mark.parametrize("D", [1, 2])
def test_weight_cache_holds_the_split_of_every_input_weight(H, D):
    """b200rnn_wcache_bytes: hi + lo of weight_ih [G*H, I_l] per (layer, direction), I_0 = input, I_l = D*H."""
    lib = _lib.load()
    for mode, G in ((_lib.GRU, 3), (_lib.LSTM, 4)):
        I, L = 256, 2
        n = ctypes.c_size_t(0)
        d = _lib.Desc(mode, 8, 4, I, H, L, D, 0, 0.0, 0)
        assert lib.b200rnn_wcache_bytes(ctypes.byref(d), ctypes.byref(n)) == 0, lib.b200rnn_last_error()
        expect = 4 * 2 * D * G * H * (I + (L - 1) * D * H)
        assert expect <= n.value <= expect + 4 * 64 * (4 * L * D + 1), (mode, n.value, expect)


@pytest.mark.parametrize("H", [32, 96, 100, 192, 384, 1024])
def test_other_widths_are_rejected_naming_the_supported_ones(H):
    for mode in (_lib.GRU, _lib.LSTM):
        with pytest.raises(_lib.B200RNNError) as ei:
            _lib.workspace_bytes(_lib.Desc(mode, 4, 4, 16, H, 1, 1, 0, 0.0, 0))
        msg = str(ei.value)
        assert "hidden_size" in msg and "64, 128, 256 and 512" in msg, msg


cuobjdump = shutil.which("cuobjdump") or shutil.which("/usr/local/cuda/bin/cuobjdump")


@pytest.fixture(scope="module")
def recurrence_sass():
    if cuobjdump is None:
        pytest.skip("cuobjdump not available")
    txt = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    out, name = {}, None
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1) if re.search(r"rec_(fwd|bwd)_kernel", m.group(1)) else None
            if name:
                out[name] = []
        elif name is not None:
            m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
            if m:
                out[name].append(m.group(1))
    assert out, "no recurrence kernels in the library"
    return out


@pytest.mark.parametrize("H", NEW)
@pytest.mark.parametrize("mode", [_lib.GRU, _lib.LSTM])
@pytest.mark.parametrize("kind", ["fwd", "bwd"])
@pytest.mark.parametrize("vl", [0, 1])
def test_new_instantiations_exist_without_local_memory(recurrence_sass, H, mode, kind, vl):
    """Mangled names carry the template arguments <MODE, H, C, BS, KL, UPL, RG, VL[, PB]>: every mode x direction x
    lengths twin has at least one instantiation at the new width, and none of them spills to local memory."""
    pat = re.compile(rf"rec_{kind}_kernelILi{mode}ELi{H}E(?:Li\d+E){{5}}Lb{vl}E")
    hits = [n for n in recurrence_sass if pat.search(n)]
    assert hits, (kind, mode, H, vl)
    for n in hits:
        local = sorted({o for o in recurrence_sass[n] if o.startswith(("LDL", "STL"))})
        assert not local, (n, local)
