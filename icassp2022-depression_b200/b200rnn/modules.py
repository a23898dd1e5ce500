"""Drop-in ``nn.Module`` mirrors of ``torch.nn.GRU`` / ``torch.nn.LSTM`` backed by the sm_100a kernels.

They keep the constructor signature, parameter names / shapes / registration order
(``weight_ih_l{k}[_reverse]``, ``weight_hh_...``, ``bias_ih_...``, ``bias_hh_...``; torch rnn.py:171-216), the
default init U(-1/sqrt(H), 1/sqrt(H)) (rnn.py:308-311) and the ``forward`` return structure, so that

* ``state_dict`` round-trips with stock modules (fuse_net_whole.py:569-588 copies these keys by name),
* ``torch.save(model)`` pickles (audio_gru_whole.py:123-126),
* the reference model classes (audio_gru_whole.py:59-60, text_bilstm_whole.py:54-56,
  fuse_net_whole.py:266-268, 281-286) construct them unchanged once :func:`install` has rebound
  ``torch.nn.GRU`` / ``torch.nn.LSTM``.

``PackedSequence`` input is supported (per-sequence lengths in the kernels). Unused-by-the-reference features that
raise ``NotImplementedError``: proj_size, bias=False, non-None initial state, unbatched 2-D input.
"""
from __future__ import annotations

import math
import warnings
from typing import Callable, List, Optional

import torch
import torch.nn as nn

from . import _lib
from .functional import RNNConfig, prepare_weights, rnn_forward, rnn_forward_fused, rnn_ln_pool_sum

_TORCH_GRU = nn.GRU
_TORCH_LSTM = nn.LSTM
_module_counter = 0


class _B200RNNBase(nn.Module):
    _mode: int = -1
    _gates: int = 0

    def __init__(self, input_size: int, hidden_size: int, num_layers: int = 1, bias: bool = True,
                 batch_first: bool = False, dropout: float = 0.0, bidirectional: bool = False,
                 proj_size: int = 0, device=None, dtype=None) -> None:
        super().__init__()
        if not bias:
            raise NotImplementedError("b200rnn: bias=False is not used by the reference and not implemented")
        if proj_size != 0:
            raise NotImplementedError("b200rnn: proj_size is not used by the reference and not implemented")
        if dtype not in (None, torch.float32):
            raise NotImplementedError("b200rnn: float32 only")
        if not isinstance(dropout, (int, float)) or not 0 <= dropout <= 1 or isinstance(dropout, bool):
            raise ValueError("dropout should be a number in range [0, 1] representing the probability of an "
                             "element being zeroed")
        if dropout > 0 and num_layers == 1:
            warnings.warn("dropout option adds dropout after all but last recurrent layer, so non-zero dropout "
                          f"expects num_layers greater than 1, but got dropout={dropout} and num_layers={num_layers}")
        if hidden_size <= 0 or num_layers <= 0:
            raise ValueError("hidden_size and num_layers must be positive")
        self.input_size = input_size
        self.hidden_size = hidden_size
        self.num_layers = num_layers
        self.bias = bias
        self.batch_first = batch_first
        self.dropout = float(dropout)
        self.bidirectional = bidirectional
        self.proj_size = 0
        num_directions = 2 if bidirectional else 1
        gate_size = self._gates * hidden_size

        self._flat_weights_names: List[str] = []
        for layer in range(num_layers):
            for direction in range(num_directions):
                layer_input_size = input_size if layer == 0 else hidden_size * num_directions
                suffix = "_reverse" if direction == 1 else ""
                shapes = ((gate_size, layer_input_size), (gate_size, hidden_size), (gate_size,), (gate_size,))
                names = ("weight_ih_l{}{}", "weight_hh_l{}{}", "bias_ih_l{}{}", "bias_hh_l{}{}")
                for name, shape in zip(names, shapes):
                    pname = name.format(layer, suffix)
                    self.register_parameter(
                        pname, nn.Parameter(torch.empty(shape, dtype=torch.float32, device=device)))
                    self._flat_weights_names.append(pname)
        # device-resident Philox state {seed, offset} of the inter-layer dropout; advanced by the kernels so a
        # captured CUDA graph draws a new mask per replay. Not part of the state_dict.
        global _module_counter
        _module_counter += 1
        seed = (torch.initial_seed() * 0x9E3779B97F4A7C15 + _module_counter) & 0x7FFFFFFFFFFFFFFF
        self.register_buffer("_rng_state", torch.tensor([seed, 0], dtype=torch.int64, device=device),
                             persistent=False)
        # optional hook: callable(weights) -> list of gradient target tensors (see b200rnn.dp.GradBucket)
        self._grad_sink: Optional[Callable] = None
        self._wcache = None        # (key, tensor): TF32 split of the weight_ih matrices while they are frozen
        self.reset_parameters()

    # -- torch.nn.RNNBase API surface ---------------------------------------------------------------
    def reset_parameters(self) -> None:
        stdv = 1.0 / math.sqrt(self.hidden_size) if self.hidden_size > 0 else 0
        for weight in self.parameters():
            nn.init.uniform_(weight, -stdv, stdv)

    def flatten_parameters(self) -> None:  # cuDNN-ism; parameters are used in place here
        return None

    @property
    def _flat_weights(self) -> List[torch.Tensor]:
        return [getattr(self, n) for n in self._flat_weights_names]

    @property
    def all_weights(self) -> List[List[nn.Parameter]]:
        fw = self._flat_weights
        return [fw[i:i + 4] for i in range(0, len(fw), 4)]

    def extra_repr(self) -> str:
        s = "{input_size}, {hidden_size}"
        if self.num_layers != 1:
            s += ", num_layers={num_layers}"
        if self.batch_first is not False:
            s += ", batch_first={batch_first}"
        if self.dropout != 0:
            s += ", dropout={dropout}"
        if self.bidirectional is not False:
            s += ", bidirectional={bidirectional}"
        return s.format(**self.__dict__)

    def __setstate__(self, d):
        super().__setstate__(d)
        if "_grad_sink" not in self.__dict__:
            self._grad_sink = None
        self._wcache = None

    def __getstate__(self):
        d = self.__dict__.copy()
        d["_grad_sink"] = None  # closures over buckets are not picklable / not part of the model
        d["_wcache"] = None     # derived data
        return d

    def frozen_weight_cache(self):
        """TF32-split ``weight_ih`` cache for the no-grad fused forward, or None.

        Only while EVERY weight of the module is frozen (``requires_grad=False``, the fuse scripts' encoders:
        fuse_net_whole.py:590-593) - nothing this library launches updates such a tensor behind PyTorch's back. The
        cache is keyed on the parameters' storage addresses and version counters, so ``load_state_dict``, ``.to()`` or
        an in-place edit refresh it; trainable modules never use it (their weights change every step anyway)."""
        ws = self._flat_weights
        if any(w.requires_grad for w in ws) or not ws[0].is_cuda:
            self._wcache = None
            return None
        key = tuple((w.data_ptr(), w._version) for w in ws)
        if self._wcache is None or self._wcache[0] != key:
            if torch.cuda.is_current_stream_capturing():
                return None   # never (re)build under capture: a replay would not redo it
            self._wcache = (key, prepare_weights(ws, self._config()))
        return self._wcache[1]

    def _config(self) -> RNNConfig:
        return RNNConfig(mode=self._mode, input_size=self.input_size, hidden_size=self.hidden_size,
                         num_layers=self.num_layers, num_dirs=2 if self.bidirectional else 1,
                         dropout=self.dropout, training=self.training, batch_first=self.batch_first)

    def _run_packed(self, packed):
        """PackedSequence path (ragged DAIC-style sequences): pad, run with per-sequence lengths, re-pack exactly like
        torch (same batch_sizes / sorted_indices; h_n, c_n in the caller's original batch order)."""
        rnn_utils = nn.utils.rnn
        padded, lengths = rnn_utils.pad_packed_sequence(packed, batch_first=self.batch_first)
        out = rnn_forward(padded, self._flat_weights, self._config(), self._rng_state, self._grad_sink, lengths=lengths)
        y = out[0]
        bdim = 0 if self.batch_first else 1
        if packed.sorted_indices is not None:
            y = y.index_select(bdim, packed.sorted_indices)
            lens_sorted = lengths.index_select(0, packed.sorted_indices.cpu())
        else:
            lens_sorted = lengths
        repacked = rnn_utils.pack_padded_sequence(y, lens_sorted, batch_first=self.batch_first, enforce_sorted=True)
        y_packed = rnn_utils.PackedSequence(repacked.data, packed.batch_sizes, packed.sorted_indices,
                                            packed.unsorted_indices)
        return (y_packed, *out[1:])

    def _run(self, input, hx):
        if hx is not None:
            raise NotImplementedError("b200rnn: a non-None initial state is not implemented (the reference "
                                      "always starts from zeros, rnn.py:1432-1440)")
        if isinstance(input, nn.utils.rnn.PackedSequence):
            return self._run_packed(input)
        if input.dim() != 3:
            raise NotImplementedError("b200rnn: unbatched 2-D input is not implemented")
        return rnn_forward(input, self._flat_weights, self._config(), self._rng_state, self._grad_sink)

    def forward_ln_sum(self, input: torch.Tensor, ln: Optional[nn.LayerNorm] = None) -> torch.Tensor:
        """``self(ln(input))[0].sum(dim=time)`` — the audio branch of fuse_net_whole.py:360-362 / fuse_net.py:338-339.

        For widths the tensor-core projection takes, LayerNorm is folded into the layer-0 operand preparation and the
        time sum into the last layer's step loop. Without autograd (the reference's fuse scripts run it under
        ``torch.no_grad()``, fuse_net_whole.py:337) the normalised input and the [B,T,H] output never touch HBM; under
        autograd (audio_gru_whole.py:103-108 + loss.backward()) the same fusions run in both directions
        (``b200rnn_backward_fused``: LayerNorm backward, pooled-gradient broadcast inside the BPTT kernel). Otherwise
        the same value is computed unfused.
        """
        need_grad = torch.is_grad_enabled() and (input.requires_grad or any(p.requires_grad for p in self.parameters())
                                                 or (ln is not None and any(p.requires_grad for p in ln.parameters())))
        # the folded LayerNorm needs the tensor-core layer-0 projection, whose N = gates * hidden_size must be a
        # multiple of 128 (not so for a GRU with hidden_size 64)
        shape_ok = (input.is_cuda and input.dim() == 3 and
                    (ln is None or (self.input_size in (128, 256, 512, 1024) and ln.elementwise_affine and
                                    ln.bias is not None and (self._gates * self.hidden_size) % 128 == 0)))
        if need_grad and shape_ok and not isinstance(input, nn.utils.rnn.PackedSequence):
            # training graph: LayerNorm forward+backward folded around the layer-0 GEMMs, pooled gradient broadcast
            # inside the BPTT kernel (no [T,B,H] output gradient, no LN(x) autograd tensor)
            return rnn_ln_pool_sum(input, self._flat_weights, self._config(), self._rng_state, self._grad_sink,
                                   ln.weight if ln is not None else None, ln.bias if ln is not None else None,
                                   ln.eps if ln is not None else 1e-5)
        fusable = not need_grad and shape_ok
        if fusable:
            out = rnn_forward_fused(input, self._flat_weights, self._config(), self._rng_state,
                                    ln.weight if ln is not None else None, ln.bias if ln is not None else None,
                                    ln.eps if ln is not None else 1e-5, pool_sum=True,
                                    wcache=self.frozen_weight_cache())
            return out[0]
        seq = self(ln(input) if ln is not None else input)[0]
        return seq.sum(dim=1 if self.batch_first else 0)


class GRU(_B200RNNBase):
    """``torch.nn.GRU`` (gate order r,z,n; rnn.py:1221-1224) on hand-written sm_100a kernels."""

    _mode = _lib.GRU
    _gates = 3

    def forward(self, input, hx=None):
        y, h_n = self._run(input, hx)
        return y, h_n


class LSTM(_B200RNNBase):
    """``torch.nn.LSTM`` (gate order i,f,g,o; rnn.py:842-847) on hand-written sm_100a kernels."""

    _mode = _lib.LSTM
    _gates = 4

    def forward(self, input, hx=None):
        y, h_n, c_n = self._run(input, hx)
        return y, (h_n, c_n)


def install() -> None:
    """Rebind ``torch.nn.GRU`` / ``torch.nn.LSTM`` so unmodified reference code builds the B200 modules."""
    nn.GRU = GRU
    nn.LSTM = LSTM
    torch.nn.modules.GRU = GRU
    torch.nn.modules.LSTM = LSTM


def uninstall() -> None:
    nn.GRU = _TORCH_GRU
    nn.LSTM = _TORCH_LSTM
    torch.nn.modules.GRU = _TORCH_GRU
    torch.nn.modules.LSTM = _TORCH_LSTM


def from_torch(module: nn.Module) -> _B200RNNBase:
    """Build the B200 twin of a stock ``nn.GRU`` / ``nn.LSTM`` and copy its parameters."""
    if isinstance(module, _TORCH_GRU):
        cls = GRU
    elif isinstance(module, _TORCH_LSTM):
        cls = LSTM
    else:
        raise TypeError(f"expected torch.nn.GRU or torch.nn.LSTM, got {type(module)}")
    twin = cls(module.input_size, module.hidden_size, num_layers=module.num_layers, bias=module.bias,
               batch_first=module.batch_first, dropout=module.dropout, bidirectional=module.bidirectional,
               proj_size=getattr(module, "proj_size", 0))
    twin.load_state_dict(module.state_dict())
    twin.train(module.training)
    return twin
