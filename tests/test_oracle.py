"""CPU tests pinning the ORACLE: numpy restatement vs the executed dependency (torch.nn.GRU / nn.LSTM) and restated
model shells vs the golden fixtures recorded from the reference's own classes."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import params, ref_models
from oracle.rnn_numpy import NumpyRNN

FUSE_CFG = dict(text_embed_size=1024, text_hidden_dims=128, rnn_layers=2, dropout=0.3, num_classes=2,
                audio_hidden_dims=256, audio_embed_size=256)


def _close(summary: dict, tensor: torch.Tensor, rtol: float, what: str):
    got = params.summarize(tensor)
    assert set(got) == set(summary), what
    if "full" in summary:
        scale = max(np.abs(summary["full"]).max(), 1e-30)
        assert np.abs(got["full"] - summary["full"]).max() <= rtol * scale, what
        return
    scale = max(float(summary["absmax"][0]), 1e-30)
    assert np.abs(got["head"] - summary["head"]).max() <= rtol * scale, what
    assert np.abs(got["sample"] - summary["sample"]).max() <= rtol * scale, what
    assert abs(float(got["abssum"][0]) - float(summary["abssum"][0])) <= rtol * float(summary["abssum"][0]) + 1e-12, what


@pytest.mark.parametrize("kind,bi,L", [("gru", False, 2), ("gru", True, 1), ("lstm", True, 2), ("lstm", False, 1)])
def test_numpy_restatement_matches_torch(kind, bi, L):
    torch.manual_seed(0)
    I, H, B, T = 12, 16, 3, 7
    cls = torch.nn.GRU if kind == "gru" else torch.nn.LSTM
    ref = cls(I, H, num_layers=L, bidirectional=bi).double()
    x = torch.randn(T, B, I, dtype=torch.float64, requires_grad=True)
    out = ref(x)
    y = out[0]
    states = out[1] if isinstance(out[1], tuple) else (out[1],)
    orc = NumpyRNN(kind, [p.detach().numpy() for p in ref.parameters()], L, bi)
    res = orc.forward(x.detach().numpy())
    assert np.abs(res[0] - y.detach().numpy()).max() < 1e-12
    for a, b in zip(res[1:], states):
        assert np.abs(a - b.detach().numpy()).max() < 1e-12
    dy = torch.randn_like(y)
    dstates = [torch.randn_like(s) for s in states]
    (y * dy).sum().add(sum((s * d).sum() for s, d in zip(states, dstates))).backward()
    dx, dparams = orc.backward(dy.numpy(), dstates[0].numpy(), dstates[1].numpy() if len(dstates) > 1 else None)
    assert np.abs(dx - x.grad.numpy()).max() < 1e-11
    for p, g in zip(ref.parameters(), dparams):
        assert np.abs(g - p.grad.numpy()).max() < 1e-10


@pytest.mark.parametrize("kind,bi,L", [("gru", False, 2), ("gru", True, 2), ("lstm", True, 2), ("lstm", False, 1)])
def test_numpy_restatement_matches_torch_on_packed_ragged_batches(kind, bi, L):
    """PackedSequence semantics (the `lengths` argument the CUDA kernels take) against stock torch, fwd + bwd."""
    from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

    torch.manual_seed(1)
    I, H, B, T = 10, 12, 5, 9
    lengths = torch.tensor([9, 2, 5, 1, 7])
    cls = torch.nn.GRU if kind == "gru" else torch.nn.LSTM
    ref = cls(I, H, num_layers=L, bidirectional=bi).double()
    x = torch.randn(T, B, I, dtype=torch.float64, requires_grad=True)
    out = ref(pack_padded_sequence(x, lengths, enforce_sorted=False))
    y, _ = pad_packed_sequence(out[0], total_length=T)
    states = out[1] if isinstance(out[1], tuple) else (out[1],)
    orc = NumpyRNN(kind, [p.detach().numpy() for p in ref.parameters()], L, bi)
    res = orc.forward(x.detach().numpy(), lengths=lengths.numpy())
    assert np.abs(res[0] - y.detach().numpy()).max() < 1e-12
    for b in range(B):
        assert np.abs(res[0][int(lengths[b]):, b]).max(initial=0.0) == 0.0   # padded output rows are exactly 0
    for a, b in zip(res[1:], states):
        assert np.abs(a - b.detach().numpy()).max() < 1e-12
    dy = torch.randn_like(y)   # including garbage at padded positions: it must not reach any gradient
    dstates = [torch.randn_like(s) for s in states]
    (y * dy).sum().add(sum((s * d).sum() for s, d in zip(states, dstates))).backward()
    dx, dparams = orc.backward(dy.numpy(), dstates[0].numpy(), dstates[1].numpy() if len(dstates) > 1 else None)
    assert np.abs(dx - x.grad.numpy()).max() < 1e-11
    for b in range(B):
        assert np.abs(dx[int(lengths[b]):, b]).max(initial=0.0) == 0.0
    for p, g in zip(ref.parameters(), dparams):
        assert np.abs(g - p.grad.numpy()).max() < 1e-10


def _single(case, cls, regression):
    arrays, meta = load_golden(case)
    model = cls(meta["cfg"], regression=regression)
    params.fill_module(model)
    model.eval()
    x = params.inputs_for(case, meta["shape"]).requires_grad_(True)
    out = model(x)
    B = meta["shape"][0]
    if meta["loss"] == "ce":
        loss = torch.nn.CrossEntropyLoss()(out, params.labels_for(case, B))
    elif meta["loss"] == "l1":
        loss = torch.nn.L1Loss()(out, params.inputs_for(case + ":target", (B, 1)).abs() * 10)
    else:
        loss = torch.nn.SmoothL1Loss()(out, params.inputs_for(case + ":target", (B, 1)).abs() * 10)
    loss.backward()
    return arrays, model, x, out, loss


@pytest.mark.parametrize("case,cls,regression", [
    ("audio_clf_b3_t5", ref_models.RefAudio, False),
    ("text_clf_b3_t6", ref_models.RefText, False),
    ("audio_reg_b2_t3", ref_models.RefAudio, True),
    ("text_reg_b2_t3", ref_models.RefText, True),
    ("c1_text_b1_t32", ref_models.RefText, False),
])
def test_restated_models_reproduce_reference_goldens(case, cls, regression):
    arrays, model, x, out, loss = _single(case, cls, regression)
    assert np.abs(out.detach().numpy() - arrays["out"]).max() < 1e-6
    assert abs(loss.item() - float(arrays["loss"][0])) < 1e-6
    _close(arrays["dx"], x.grad, 1e-5, "dx")
    for n, p in model.named_parameters():
        key = "grad:" + n
        if key in arrays:
            _close(arrays[key], p.grad, 1e-5, key)
        else:
            assert p.grad is None or p.grad.abs().max() == 0, n


@pytest.mark.parametrize("case,regression", [("fuse_clf_b3_t3", False), ("fuse_reg_b3_t3", True)])
def test_restated_fusion_reproduces_reference_goldens(case, regression):
    arrays, meta = load_golden(case)
    cfg = dict(FUSE_CFG, num_classes=1 if regression else 2)
    model = ref_models.RefFusion(**cfg, regression=regression)
    params.fill_module(model)
    model.eval()
    B, T = meta["B"], meta["T"]
    audio = params.inputs_for(case + ":audio", (B, T, 256))
    text = params.inputs_for(case + ":text", (B, T, 1024))
    tf, af = model.pretrained_feature_tensors(audio, text)
    out = model(torch.cat((tf, af), dim=1))
    loss = ref_models.ref_fusion_loss(tf, af, arrays["target"], model)
    loss.backward()
    assert np.abs(tf.numpy() - arrays["text_feature"]).max() < 1e-6
    assert np.abs(af.numpy() - arrays["audio_feature"]).max() < 1e-5
    assert np.abs(out.detach().numpy() - arrays["out"]).max() < 1e-6
    assert abs(loss.item() - float(arrays["loss"][0])) < 1e-5
    _close(arrays["grad:fc_final.0.weight"], model.fc_final[0].weight.grad, 1e-5, "fc_final grad")
    # reference semantics: only fc_final.0.weight ever receives a gradient (fuse_net_whole.py:337, 590-593)
    assert [n for n, p in model.named_parameters() if p.grad is not None] == ["fc_final.0.weight"]


@pytest.mark.parametrize("case,kind", [("gru_boundary_b5_t24", "gru"), ("lstm_boundary_b5_t17", "lstm")])
def test_numpy_oracle_reproduces_reference_rnn_boundary(case, kind):
    """The float64 restatement against what the reference's own nn.GRU / nn.LSTM instance produced."""
    arrays, meta = load_golden(case)
    cls = ref_models.RefAudio if kind == "gru" else ref_models.RefText
    model = cls(meta["cfg"])
    params.fill_module(model)
    rnn = getattr(model, meta["attr"])
    x = params.inputs_for(case, meta["shape"])
    x_tm = x.permute(1, 0, 2).contiguous()
    orc = NumpyRNN(kind, [p.detach().numpy() for p in rnn.parameters()], rnn.num_layers, rnn.bidirectional)
    res = orc.forward(x_tm.numpy())
    y = torch.from_numpy(res[0])
    if not meta["time_major"]:
        y = y.permute(1, 0, 2).contiguous()
    _close(arrays["y"], y, 2e-6, "y")
    for i, s in enumerate(res[1:]):
        _close(arrays[f"state{i}"], torch.from_numpy(s), 2e-6, f"state{i}")
    w = params.inputs_for(case + ":w", y.shape)
    w_tm = w if meta["time_major"] else w.permute(1, 0, 2)
    whs = [params.inputs_for(case + f":wh{i}", s.shape).numpy() for i, s in enumerate(res[1:])]
    dx, dparams = orc.backward(w_tm.numpy(), whs[0], whs[1] if len(whs) > 1 else None)
    _close(arrays["dx"], torch.from_numpy(dx).permute(1, 0, 2).contiguous(), 1e-5, "dx")
    for (n, _), g in zip(rnn.named_parameters(), dparams):
        _close(arrays["grad:" + n], torch.from_numpy(g), 1e-5, n)


@pytest.mark.parametrize("key,name,cls,regression,shape", [
    ("audio_clf", "AudioBiLSTM", ref_models.RefAudio, False, (4, 6, 256)),
    ("text_clf", "TextBiLSTM", ref_models.RefText, False, (4, 6, 1024)),
    ("audio_reg", "AudioBiLSTM", ref_models.RefAudio, True, (4, 3, 256)),
    ("text_reg", "TextBiLSTM", ref_models.RefText, True, (4, 3, 1024)),
])
def test_ref_models_match_reference_live(key, name, cls, regression, shape):
    """The restated classes against the reference's own classes executed on the same weights and inputs (their
    parameter names and eval() outputs, with and without the head's final activation, recorded by
    oracle/make_golden.py)."""
    case = f"live_{key}_b{shape[0]}_t{shape[1]}"
    arrays, meta = load_golden(case)
    assert meta["cls"] == name and meta["shape"] == list(shape)
    mine = cls(meta["cfg"], regression=regression)
    assert [n for n, _ in mine.named_parameters()] == meta["names"]
    params.fill_module(mine)
    mine.eval()
    x = params.inputs_for(case, meta["shape"])
    with torch.no_grad():
        assert np.abs(mine(x).numpy() - arrays["out"]).max() <= 1e-6
        getattr(mine, meta["head"])[-1] = torch.nn.Identity()
        assert np.abs(mine(x).numpy() - arrays["pre_activation"]).max() <= 1e-6
