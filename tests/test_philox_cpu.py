"""The host copy of the library's dropout RNG (oracle/philox.py) and the masked-dropout oracle (oracle/masked.py).

The exact train-mode dropout tests (test_gpu_dropout_exact.py) rebuild every mask the kernels draw with this host
copy, so it is pinned here three ways: the Random123 known-answer vectors of Philox4x32-10, the library's own
``philox4x32_10`` (csrc/common.cuh) compiled as a host program, and the mask layout / threshold rules of the kernels.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import philox
from oracle.masked import MaskedRNN, masks_injected

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "icassp2022-depression_b200", "csrc")


def _words(seed, ctr_lo, ctr_hi):
    return [int(v) for v in philox.philox4x32_10(seed, ctr_lo, ctr_hi).reshape(-1)]


@pytest.mark.parametrize("key, ctr, want", [
    # Random123 kat_vectors, philox4x32 with 10 rounds: (k0, k1), (c0, c1, c2, c3) -> (x, y, z, w)
    ((0, 0), (0, 0, 0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF, 0xFFFFFFFF), (0xFFFFFFFF,) * 4, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0xA4093822, 0x299F31D0), (0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_matches_random123_known_answers(key, ctr, want):
    seed = key[1] << 32 | key[0]
    ctr_lo, ctr_hi = ctr[1] << 32 | ctr[0], ctr[3] << 32 | ctr[2]
    assert _words(seed, ctr_lo, ctr_hi) == list(want)


def test_philox_library_argument_order_vector():
    assert _words(0x1234567887654321, 5, 2) == [0xC501A859, 0x1AA3B008, 0x44F86293, 0x9DF427C9]


def test_philox_vectorised_equals_one_call_at_a_time():
    rng = np.random.default_rng(1)
    lo = rng.integers(0, 2**63, 64, dtype=np.uint64) * np.uint64(2) + np.uint64(1)   # full 64-bit range
    hi = rng.integers(0, 2**63, 64, dtype=np.uint64)
    batch = philox.philox4x32_10(0xDEADBEEFCAFEF00D, lo, hi)
    for i in range(64):
        assert _words(0xDEADBEEFCAFEF00D, int(lo[i]), int(hi[i])) == [int(v) for v in batch[i]]


def test_keep_mask_layout_is_counter_offset_plus_i_div_4_and_lane_i_mod_4():
    seed, offset, stream, p = 0x0123456789ABCDEF, 1000, 3, 0.5
    n = 37                                           # not a multiple of 4: the last counter is partly used
    m = philox.keep_mask(seed, offset, stream, n, p)
    thr = philox.threshold(p)
    for i in range(n):
        word = _words(seed, offset + i // 4, stream)[i % 4]
        assert m[i] == (word >= thr), i
    # a later offset is the same stream shifted by whole counters
    assert np.array_equal(philox.keep_mask(seed, offset + 2, stream, n - 8, p), m[8:])
    # the offset is a 64-bit counter: wrap-around is modular, as on the device
    w = philox.keep_mask(seed, 2**64 - 1, stream, 8, p)
    assert np.array_equal(w[4:], philox.keep_mask(seed, 0, stream, 4, p))


def test_streams_and_seeds_give_independent_masks():
    n, p = 1 << 16, 0.5
    a = philox.keep_mask(77, 0, 0, n, p)
    for other in (philox.keep_mask(77, 0, 1, n, p), philox.keep_mask(78, 0, 0, n, p),
                  philox.keep_mask(77, 1, 0, n, p)):
        agree = (a == other).mean()
        assert abs(agree - 0.5) < 5 * 0.5 / np.sqrt(n), agree   # independent Bernoulli(0.5): agreement ~ 1/2


def test_threshold_and_scale_edges():
    assert philox.threshold(0.0) == 0
    assert philox.threshold(1.0) == 0xFFFFFFFF          # fminf(2^32, 4294967295.f = 2^32), saturating cast
    assert philox.threshold(0.5) == 1 << 31
    assert philox.threshold(0.3) == int(np.float32(0.3) * np.float32(2.0**32))
    assert philox.scale(0.5) == np.float32(2.0)
    assert philox.scale(0.3) == np.float32(1.0) / np.float32(0.7)
    assert philox.scale(1.0) == 0.0
    assert philox.counters(1) == 1 and philox.counters(4) == 1 and philox.counters(5) == 2


def test_p0_keeps_everything_and_p1_keeps_nothing_after_scaling():
    n = 1 << 14
    assert philox.keep_mask(5, 9, 0, n, 0.0).all()
    assert np.array_equal(philox.dropout_factor(5, 9, 0, (n,), 0.0), np.ones(n, np.float32))
    assert not philox.dropout_factor(5, 9, 0, (n,), 1.0).any()


@pytest.mark.parametrize("p", [0.3, 0.5])
def test_keep_rate_within_5_sigma(p):
    n = 1_000_000
    rate = philox.keep_mask(0x9E3779B97F4A7C15, 123456789, 1, n, p).mean()
    sigma = np.sqrt(p * (1 - p) / n)
    assert abs(rate - (1 - p)) < 5 * sigma, (rate, sigma)


def test_numpy_philox_equals_the_library_source_compiled_for_the_host(tmp_path):
    """csrc/common.cuh's ``philox4x32_10`` (its host branch: the same rounds, 64-bit products for __umulhi) built
    with the nvcc the library build needs, on random (seed, counter, stream) triples."""
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc) and shutil.which(nvcc) is None:
        pytest.skip("nvcc not found")
    src = tmp_path / "philox_host.cu"
    src.write_text(
        '#include "common.cuh"\n'
        "#include <stdio.h>\n"
        "int main() {\n"
        "  unsigned long long s, lo, hi;\n"
        "  while (scanf(\"%llx %llx %llx\", &s, &lo, &hi) == 3) {\n"
        "    b200rnn::Philox4 r = b200rnn::philox4x32_10(s, lo, hi);\n"
        "    printf(\"%08x %08x %08x %08x\\n\", r.x, r.y, r.z, r.w);\n"
        "  }\n"
        "  return 0;\n"
        "}\n")
    exe = tmp_path / "philox_host"
    proc = subprocess.run([nvcc, "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)], capture_output=True,
                          text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr
    rng = np.random.default_rng(7)
    trip = rng.integers(0, 2**63, (256, 3), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, (256, 3),
                                                                                          dtype=np.uint64)
    trip[:8, 2] = np.arange(8, dtype=np.uint64)      # small stream ids, as the kernels use them
    inp = "".join(f"{int(a):x} {int(b):x} {int(c):x}\n" for a, b, c in trip)
    out = subprocess.run([str(exe)], input=inp, capture_output=True, text=True, timeout=60, check=True).stdout
    got = [[int(w, 16) for w in line.split()] for line in out.strip().splitlines()]
    assert len(got) == len(trip)
    for (s, lo, hi), g in zip(trip, got):
        assert _words(int(s), int(lo), int(hi)) == g


# ---- the masked oracle ---------------------------------------------------------------------------------------------

def _stack_case(kind, bidir, batch_first, L=3):
    torch.manual_seed(3)
    cls = torch.nn.LSTM if kind == "lstm" else torch.nn.GRU
    rnn = cls(5, 4, num_layers=L, dropout=0.5, batch_first=batch_first, bidirectional=bidir).double()
    return rnn


@pytest.mark.parametrize("kind, bidir, batch_first", [("gru", False, True), ("lstm", True, False)])
def test_masked_stack_with_all_ones_equals_stock_and_shares_parameters(kind, bidir, batch_first):
    rnn = _stack_case(kind, bidir, batch_first).eval()   # eval: stock applies no dropout
    T, B, D = 6, 3, 2 if bidir else 1
    x = torch.randn((B, T, 5) if batch_first else (T, B, 5), dtype=torch.float64)
    ones = [torch.ones(T, B, D * 4, dtype=torch.float64)] * 2
    y_r, s_r = rnn(x)
    y_m, s_m = MaskedRNN(rnn)(x, ones)
    assert torch.equal(y_r, y_m)
    for a, b in zip(s_r if kind == "lstm" else (s_r,), s_m if kind == "lstm" else (s_m,)):
        assert torch.equal(a, b)
    y_m.sum().backward()
    assert all(p.grad is not None and p.grad.abs().sum() > 0 for p in rnn.parameters())


def test_masked_stack_applies_each_factor_between_the_right_layers():
    rnn = _stack_case("gru", False, True).eval()
    T, B = 5, 2
    x = torch.randn(B, T, 5, dtype=torch.float64)
    f0 = torch.from_numpy(philox.dropout_factor(1, 0, 0, (T, B, 4), 0.5).astype(np.float64))
    f1 = torch.from_numpy(philox.dropout_factor(1, 0, 1, (T, B, 4), 0.5).astype(np.float64))
    y, h = MaskedRNN(rnn)(x, [f0, f1])
    # by hand: layer l's time-major output times f_l feeds layer l+1 (batch_first -> transpose the factor)
    st = MaskedRNN(rnn).layers
    y0, h0 = st[0](x)
    y1, h1 = st[1](y0 * f0.transpose(0, 1))
    y2, h2 = st[2](y1 * f1.transpose(0, 1))
    assert torch.equal(y, y2) and torch.equal(h, torch.cat([h0, h1, h2]))


def test_masked_stack_packed_input_masks_the_padded_layout():
    rnn = _stack_case("lstm", True, False, L=2).eval()
    T, B = 7, 4
    lens = torch.tensor([3, 7, 1, 5])
    x = torch.randn(T, B, 5, dtype=torch.float64)
    f = torch.from_numpy(philox.dropout_factor(9, 4, 0, (T, B, 8), 0.5).astype(np.float64))
    packed = torch.nn.utils.rnn.pack_padded_sequence(x, lens, enforce_sorted=False)
    y_p, (h_p, c_p) = MaskedRNN(rnn)(packed, [f])
    y_p, _ = torch.nn.utils.rnn.pad_packed_sequence(y_p)
    for b in range(B):   # each sequence alone, unpadded, with its slice of the mask
        n = int(lens[b])
        y_b, (h_b, c_b) = MaskedRNN(rnn)(x[:n, b:b + 1], [f[:n, b:b + 1]])
        assert torch.allclose(y_p[:n, b:b + 1], y_b, atol=1e-12)
        assert torch.allclose(h_p[:, b:b + 1], h_b, atol=1e-12) and torch.allclose(c_p[:, b:b + 1], c_b, atol=1e-12)


def test_masks_injected_reference_model_keeps_names_and_restores():
    from oracle import ref_models

    torch.manual_seed(0)
    cfg = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=8, hidden_dims=4)
    ref = ref_models.RefAudio(cfg).double().train()
    names = [n for n, _ in ref.named_parameters()]
    x = torch.randn(3, 5, 8, dtype=torch.float64)
    ones_h = torch.ones(3, 4, dtype=torch.float64)
    with masks_injected(ref, rnn={"lstm_net_audio": [torch.ones(5, 3, 4, dtype=torch.float64)]},
                        dropout={"fc_audio.0": ones_h, "fc_audio.3": ones_h}):
        a = ref(x)
        assert [n for n, _ in ref.named_parameters()] == names
    ref.eval()
    assert torch.allclose(a, ref(x), atol=1e-14)        # all-ones masks == no dropout
    assert "forward" not in vars(ref.lstm_net_audio) and "forward" not in vars(ref.fc_audio[0])
    with pytest.raises(TypeError):
        with masks_injected(ref, dropout={"fc_audio.1": ones_h}):
            pass
