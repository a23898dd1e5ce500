"""ORACLE — the reference's models with train-mode dropout driven by GIVEN masks instead of torch's RNG.

``MaskedRNN`` restates a multi-layer stock ``nn.GRU`` / ``nn.LSTM`` layer by layer: one single-layer stock module per
layer, sharing the Parameter objects of the multi-layer module, with ``y_l * factor_l`` between layers (``factor`` =
keep mask times the dropout scale, see :mod:`oracle.philox`). This is exactly what stock does in train mode
(torch/nn/modules/rnn.py: dropout on every layer output but the last), with the Bernoulli draw replaced. Because the
Parameters are shared, autograd gradients and ``torch.optim`` steps land on the original module's parameters.

``masks_injected`` runs ``RefAudio`` / ``RefText`` / ``RefFusion`` (or any module tree) with such masks: the named
encoders go through ``MaskedRNN``, the named ``nn.Dropout`` modules multiply by a given factor. The model's parameter
names, ``state_dict`` and behaviour outside the ``with`` block are unchanged.
"""
from __future__ import annotations

import contextlib
from typing import Dict, Optional, Sequence

import numpy as np
import torch
from torch import nn
from torch.nn.modules import rnn as _stock
from torch.nn.utils import rnn as rnn_utils

from . import philox

_WEIGHTS = ("weight_ih", "weight_hh", "bias_ih", "bias_hh")


class MaskedRNN:
    """``(y, h_n)`` / ``(y, (h_n, c_n))`` of the stock multi-layer ``rnn`` with the inter-layer dropout given as
    ``factors[l]``, a ``[T, B, D*H]`` time-major tensor applied to the output of layer ``l`` (``l < num_layers - 1``).

    A ``PackedSequence`` input is padded between layers (batch in the caller's order, as
    ``pad_packed_sequence`` returns it and the kernels see it), multiplied, and re-packed.
    """

    def __init__(self, rnn: nn.Module):
        if not isinstance(rnn, (_stock.GRU, _stock.LSTM)):
            raise TypeError(f"expected a stock torch.nn.GRU / torch.nn.LSTM, got {type(rnn)}")
        self.rnn = rnn
        self.lstm = isinstance(rnn, _stock.LSTM)
        D = 2 if rnn.bidirectional else 1
        self.layers = []
        for l in range(rnn.num_layers):
            cls = _stock.LSTM if self.lstm else _stock.GRU
            in_l = rnn.input_size if l == 0 else D * rnn.hidden_size
            sub = cls(in_l, rnn.hidden_size, 1, batch_first=rnn.batch_first, bidirectional=rnn.bidirectional)
            for sfx in ("", "_reverse")[:D]:
                for w in _WEIGHTS:
                    setattr(sub, f"{w}_l0{sfx}", getattr(rnn, f"{w}_l{l}{sfx}"))   # the same Parameter object
            sub.train(rnn.training)
            self.layers.append(sub)

    def __call__(self, x, factors: Sequence[torch.Tensor], hx=None):
        if hx is not None:
            raise NotImplementedError("MaskedRNN starts from zero states, like every caller in the reference")
        L, bf = len(self.layers), self.rnn.batch_first
        if len(factors) != L - 1:
            raise ValueError(f"{L} layers need {L - 1} inter-layer masks, got {len(factors)}")
        packed = isinstance(x, rnn_utils.PackedSequence)
        hs, cs = [], []
        for l, sub in enumerate(self.layers):
            y, state = sub(x)
            h, c = state if self.lstm else (state, None)
            hs.append(h)
            cs.append(c)
            if l + 1 == L:
                break
            f = factors[l]
            if bf:
                f = f.transpose(0, 1)
            if packed:
                yp, lens = rnn_utils.pad_packed_sequence(y, batch_first=bf)
                x = rnn_utils.pack_padded_sequence(yp * f.to(yp.dtype), lens, batch_first=bf, enforce_sorted=False)
            else:
                x = y * f.to(y.dtype)
        h_n = torch.cat(hs, 0)
        if self.lstm:
            return y, (h_n, torch.cat(cs, 0))
        return y, h_n


def rnn_factors(state, T: int, B: int, DH: int, num_layers: int, p: float) -> list:
    """The inter-layer dropout factors one train-mode forward of a library RNN module draws from ``state`` =
    ``{seed, offset}`` (its ``_rng_state`` read before the call): layer ``l`` on stream ``l``, ``[T, B, D*H]`` each,
    float64."""
    seed, offset = (int(v) for v in state)
    return [torch.from_numpy(philox.dropout_factor(seed, offset, l, (T, B, DH), p).astype(np.float64))
            for l in range(num_layers - 1)]


def head_factors(state, B: int, Ht: int, Ha: int, p: float) -> Dict[str, torch.Tensor]:
    """The four dropout factors of one ``fuse_head`` step drawn from ``state`` = ``{seed, offset}``
    (``FusedFuseStep.rng_state`` read before the step), keyed by the ``fusion_net`` / ``RefFusion`` module they
    replace."""
    seed, offset = (int(v) for v in state)

    def f(stream, n):
        return torch.from_numpy(philox.dropout_factor(seed, offset, stream, (B, n), p).astype(np.float64))

    return {"fc_out.0": f(0, Ht), "fc_out.3": f(1, Ht), "fc_audio.0": f(2, Ha), "fc_audio.3": f(3, Ha)}


@contextlib.contextmanager
def masks_injected(model: nn.Module, rnn: Optional[Dict[str, Sequence[torch.Tensor]]] = None,
                   dropout: Optional[Dict[str, torch.Tensor]] = None):
    """Inside the block, ``model``'s submodule ``name`` of ``rnn`` (a stock multi-layer GRU / LSTM) runs as
    ``MaskedRNN`` with the given factors, and each ``nn.Dropout`` named in ``dropout`` multiplies its input by the
    given factor. Names are ``get_submodule`` paths (``"lstm_net"``, ``"fc_out.0"``)."""
    patched = []
    try:
        for name, factors in (rnn or {}).items():
            mod = model.get_submodule(name)
            stack = MaskedRNN(mod)
            mod.forward = lambda input, hx=None, _s=stack, _f=list(factors): _s(input, _f, hx)
            patched.append(mod)
        for name, factor in (dropout or {}).items():
            mod = model.get_submodule(name)
            if not isinstance(mod, nn.Dropout):
                raise TypeError(f"{name} is a {type(mod).__name__}, not nn.Dropout")
            mod.forward = lambda x, _f=factor: x * _f.to(x.dtype)
            patched.append(mod)
        yield model
    finally:
        for mod in patched:
            del mod.forward
