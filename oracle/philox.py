"""ORACLE — host copy of the library's dropout RNG (numpy only), so that tests can rebuild every mask it draws.

Every dropout mask of the library comes from one counter-based generator, ``philox4x32_10`` of
``csrc/common.cuh`` (Random123's Philox4x32 with 10 rounds):

* one call ``philox4x32_10(seed, ctr_lo = offset + idx // 4, ctr_hi = stream_id)`` yields four uint32 words
  ``(x, y, z, w)``; element ``idx`` takes word ``idx % 4``;
* element ``idx`` is kept iff ``word >= thr`` with ``thr = (uint32)fminf(p * 2^32, 4294967295.f)`` computed in float32
  (``4294967295.f`` rounds to 2^32 and the device cast saturates to ``0xFFFFFFFF``), and a kept value is scaled by the
  float32 ``1 / (1 - p)`` (0 when p = 1);
* ``{seed, offset}`` is read from a device-resident ``int64[2]`` state before the draw, and the draw advances
  ``offset`` by the number of counters it may use.

The element index of each user:

* inter-layer RNN dropout (``b200rnn_forward_fused`` / ``_backward_fused``): element ``(t*B + b)*D*H + d*H + j`` of the
  dense time-major ``[T, B, D*H]`` output of layer ``l`` (batch in the caller's order, padded steps of a ragged batch
  included), stream ``l``. One draw per forward, of ``ceil(T*B*D*H / 4)`` counters, from the module's ``_rng_state``;
  the backward re-applies the mask of the forward whose reserve it is given.
* ``mlp_dropout`` (``b200rnn_mlp_dropout``): element ``b*n + j``; the input dropout on stream ``s``, the output
  dropout on stream ``s + 1``; ``{seed, offset}`` is the explicit header passed in.
* ``fuse_head`` (``b200rnn_fuse_head``): element ``b*Ht + j`` on streams 0 (``fc_out[0]``, attention context) and
  1 (``fc_out[3]``, text feature), ``b*Ha + j`` on streams 2 (``fc_audio[0]``, pooled audio) and 3 (``fc_audio[3]``,
  audio feature). One draw of ``ceil(B * max(Ht, Ha) / 4)`` counters per step from ``FusedFuseStep.rng_state``.
"""
from __future__ import annotations

import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_LO32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def philox4x32_10(seed, ctr_lo, ctr_hi) -> np.ndarray:
    """Philox4x32-10 in the argument order of ``csrc/common.cuh``: key ``(k0, k1) = (seed_lo, seed_hi)``, counter
    ``(c0, c1, c2, c3) = (ctr_lo_lo, ctr_lo_hi, ctr_hi_lo, ctr_hi_hi)``. ``ctr_lo`` / ``ctr_hi`` broadcast; returns
    uint32 ``[n, 4]`` (x, y, z, w)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    lo, hi = np.broadcast_arrays(np.asarray(ctr_lo, dtype=np.uint64).reshape(-1),
                                 np.asarray(ctr_hi, dtype=np.uint64).reshape(-1))
    c0, c1 = lo & _LO32, lo >> _S32
    c2, c3 = hi & _LO32, hi >> _S32
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _M0 * c0                       # < 2^64: exact in uint64
            p1 = _M1 * c2
            c0, c1, c2, c3 = ((p1 >> _S32) ^ c1 ^ k0, p1 & _LO32, (p0 >> _S32) ^ c3 ^ k1, p0 & _LO32)
            k0, k1 = (k0 + _W0) & _LO32, (k1 + _W1) & _LO32
    return np.stack([c0, c1, c2, c3], axis=1).astype(np.uint32)


def threshold(p: float) -> int:
    """``(uint32_t)fminf(p * 4294967296.0f, 4294967295.0f)`` as the kernels evaluate it (float32, saturating cast)."""
    t = np.float32(p) * np.float32(4294967296.0)
    t = min(t, np.float32(4294967295.0))     # the float32 constant is 2^32
    return 0xFFFFFFFF if float(t) >= 4294967296.0 else int(t)


def scale(p: float) -> np.float32:
    """The float32 factor a kept element is multiplied by: ``1 / (1 - p)``, and 0 for p = 1."""
    p = np.float32(p)
    return np.float32(1.0) / (np.float32(1.0) - p) if p < 1 else np.float32(0.0)


def keep_mask(seed, offset, stream_id, n: int, p: float) -> np.ndarray:
    """bool ``[n]``: element ``i`` is kept by the draw ``{seed, offset}`` on stream ``stream_id`` with probability
    ``p`` of being dropped (counter ``offset + i // 4``, word ``i % 4``)."""
    nq = (n + 3) // 4
    ctr = (np.uint64(int(offset) & 0xFFFFFFFFFFFFFFFF) + np.arange(nq, dtype=np.uint64))
    words = philox4x32_10(seed, ctr, np.uint64(stream_id)).reshape(-1)[:n]
    return words >= np.uint32(threshold(p))


def dropout_factor(seed, offset, stream_id, shape, p: float) -> np.ndarray:
    """float32 array of ``shape``: ``mask * scale(p)``, the factor the kernels multiply the row-major flattened
    tensor of that shape with."""
    n = int(np.prod(shape))
    return (keep_mask(seed, offset, stream_id, n, p).astype(np.float32) * scale(p)).reshape(shape)


def counters(n: int) -> int:
    """Counters one draw of ``n`` elements uses (the offset advance of the draw): ``ceil(n / 4)``."""
    return (int(n) + 3) // 4
