"""Host-side behaviour of the drop-in modules that needs no GPU: parameter naming / ordering, state-dict
interchange with stock torch.nn, pickling, install(), and loud failure on CPU tensors (no fallback)."""
import io
import pickle

import pytest
import torch
import torch.nn as nn

import b200rnn


@pytest.mark.parametrize("kind,kw", [
    ("GRU", dict(input_size=256, hidden_size=256, num_layers=2, dropout=0.5, batch_first=True)),
    ("LSTM", dict(input_size=1024, hidden_size=128, num_layers=2, dropout=0.5, bidirectional=True)),
])
def test_parameters_mirror_stock_modules(kind, kw):
    stock = getattr(b200rnn.modules, "_TORCH_" + kind)(**kw)
    mine = getattr(b200rnn, kind)(**kw)
    assert [(n, tuple(p.shape)) for n, p in stock.named_parameters()] == \
           [(n, tuple(p.shape)) for n, p in mine.named_parameters()]
    assert list(stock.state_dict().keys()) == list(mine.state_dict().keys())
    mine.load_state_dict(stock.state_dict())
    stock2 = getattr(b200rnn.modules, "_TORCH_" + kind)(**kw)
    stock2.load_state_dict(mine.state_dict())
    for a, b in zip(stock.parameters(), stock2.parameters()):
        assert torch.equal(a, b)
    assert repr(mine).startswith(kind + "(")
    bound = 1.0 / kw["hidden_size"] ** 0.5
    fresh = getattr(b200rnn, kind)(**kw)
    assert all(p.abs().max() <= bound for p in fresh.parameters())  # rnn.py:308-311 default init


def test_fuse_key_copy_pattern_works():
    """fuse_net_whole.py:569-588 copies the pretrained branches' tensors into fusion_net by key name."""
    cfg_a = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=256, hidden_dims=256, learning_rate=0)
    cfg_t = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=1024, hidden_dims=128, learning_rate=0,
                 bidirectional=True)
    audio, text = b200rnn.AudioBiLSTM(cfg_a), b200rnn.TextBiLSTM(cfg_t)
    fuse = b200rnn.fusion_net(1024, 128, 2, 0.3, 2, 256, 256)
    sd = fuse.state_dict()
    copied = 0
    for src in (text.state_dict(), audio.state_dict()):
        for k, v in src.items():
            if k in sd and sd[k].shape == v.shape:
                sd[k] = v
                copied += 1
    fuse.load_state_dict(sd, strict=False)
    assert copied >= 16 + 8 + 2
    assert torch.equal(fuse.lstm_net_audio.weight_hh_l1, audio.lstm_net_audio.weight_hh_l1)
    assert torch.equal(fuse.lstm_net.weight_ih_l0_reverse, text.lstm_net.weight_ih_l0_reverse)
    n_params = sum(p.numel() for p in fuse.parameters())
    assert n_params == 2614016  # SURVEY.md §3.3


def test_whole_module_pickle_roundtrip():
    """audio_gru_whole.py:123-126 saves with torch.save(model)."""
    m = b200rnn.AudioBiLSTM(dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=256, hidden_dims=256,
                                 learning_rate=0))
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    m2 = torch.load(buf, weights_only=False)
    assert isinstance(m2.lstm_net_audio, b200rnn.GRU)
    for a, b in zip(m.parameters(), m2.parameters()):
        assert torch.equal(a, b)
    assert pickle.loads(pickle.dumps(m.lstm_net_audio)).hidden_size == 256
    assert sum(p.numel() for p in m.parameters()) == 922114  # SURVEY.md §5


def test_install_rebinds_torch_nn():
    try:
        b200rnn.install()
        assert nn.GRU is b200rnn.GRU and nn.LSTM is b200rnn.LSTM
        m = nn.GRU(256, 256, num_layers=2, dropout=0.5, batch_first=True)
        assert isinstance(m, b200rnn.GRU)
    finally:
        b200rnn.uninstall()
    assert nn.GRU is b200rnn.modules._TORCH_GRU and nn.LSTM is b200rnn.modules._TORCH_LSTM


def test_cpu_tensors_fail_loudly_no_fallback():
    m = b200rnn.GRU(256, 256, num_layers=2, batch_first=True)
    with pytest.raises(b200rnn.B200RNNError, match="no CPU path"):
        m(torch.randn(2, 3, 256))


def test_unsupported_features_raise():
    with pytest.raises(NotImplementedError):
        b200rnn.GRU(8, 128, bias=False)
    with pytest.raises(NotImplementedError):
        b200rnn.LSTM(8, 128, proj_size=4)
    m = b200rnn.LSTM(8, 128)
    with pytest.raises(NotImplementedError):
        m(torch.randn(3, 2, 8), (torch.zeros(1, 2, 128), torch.zeros(1, 2, 128)))
    with pytest.raises(NotImplementedError):
        m(torch.randn(3, 8))
    with pytest.raises(ValueError):
        b200rnn.GRU(8, 128, dropout=1.5)


def test_reference_classes_build_on_the_dropin_when_installed():
    """After install(), model code that calls nn.GRU / nn.LSTM builds B200 modules. The restated reference classes
    (oracle/ref_models.py) are built that way and must come out as the reference's own ClassDefs did when they were
    built the same way (tests/golden/dropin_build.npz: recurrent module class, parameter names and shapes, and the
    parameters its init leaves at 0)."""
    from conftest import load_golden
    from oracle import make_golden as mg, ref_models

    _, meta = load_golden("dropin_build")
    try:
        b200rnn.install()
        model = ref_models.RefAudio(mg.AUDIO_CLF)
        assert isinstance(model.lstm_net_audio, b200rnn.GRU)
        model_t = ref_models.RefText(mg.TEXT_CLF)  # xavier init over the B200 LSTM (text_bilstm_whole.py:37-43)
        assert isinstance(model_t.lstm_net, b200rnn.LSTM)
        assert float(model_t.lstm_net.bias_ih_l0.detach().abs().max()) == 0.0
    finally:
        b200rnn.uninstall()
    for key, m in (("audio_clf", model), ("text_clf", model_t)):
        want = meta["built"][key]
        rnn = getattr(m, want["attr"])
        assert f"{type(rnn).__module__}.{type(rnn).__qualname__}" == want["rnn_class"], key
        assert [[n, list(p.shape)] for n, p in m.named_parameters()] == want["params"], key
        assert [n for n, p in m.named_parameters() if float(p.detach().abs().max()) == 0.0] == want["zero"], key


def test_fused_shell_entry_points_reject_host_tensors():
    """They hand raw pointers to CUDA kernels; a CPU tensor must raise before any launch."""
    from b200rnn import fused_head

    att = torch.nn.Sequential(torch.nn.Linear(8, 8), torch.nn.ReLU())
    with pytest.raises(b200rnn.B200RNNError, match="no CPU path"):
        fused_head.attention_pool(torch.randn(3, 2, 16), torch.randn(4, 2, 8), att)
    with pytest.raises(b200rnn.B200RNNError, match="no CPU path"):
        fused_head.mlp_dropout(torch.randn(2, 8), torch.nn.Linear(8, 8), 0.3, True, None, 0)
    model = b200rnn.fusion_net(text_embed_size=16, text_hidden_dims=128, rnn_layers=1, dropout=0.1, num_classes=2,
                               audio_hidden_dims=128, audio_embed_size=16)
    with pytest.raises(b200rnn.B200RNNError, match="no CPU path"):
        b200rnn.FusedFuseStep(model)
