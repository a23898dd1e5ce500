"""Train-mode dropout checked EXACTLY: every mask the kernels draw is rebuilt on the host and fed to the CPU oracle.

The library's dropout RNG is counter-based and documented (oracle/philox.py): before each call the {seed, offset} it
will use can be read from the device (``_rng_state`` of the RNN modules, ``FusedFuseStep.rng_state``, the explicit
header of ``mlp_dropout``). The tests read it, rebuild the masks with the host Philox, run the float64 oracle with those
masks injected (oracle/masked.py) and compare at the suite's usual tolerances: outputs and states <= 1e-5 abs, dx and
every parameter gradient <= 1e-4 of the tensor's largest entry, model-level values as in test_gpu_fuse_parity.py /
test_gpu_train_step.py. A stream id, counter layout, offset advance or forward/backward mask pairing that differs from
the documented one changes the masks and fails here, although it would keep the keep-rate statistics intact.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import philox
from oracle.masked import MaskedRNN, head_factors, masks_injected, rnn_factors

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OUT_TOL = 1e-5
GRAD_RTOL = 1e-4
HERE = os.path.dirname(os.path.abspath(__file__))


def _state(t):
    return [int(v) for v in t.detach().cpu().tolist()]


def _relmax(got, ref):
    got, ref = got.detach().cpu().double(), ref.detach().double()
    m = ref.abs().max().item()
    if m == 0.0:
        return got.abs().max().item()
    return (got - ref).abs().max().item() / m


def _make(kind, I, H, L, bi, bf, p, seed=0):
    import b200rnn

    torch.manual_seed(seed)
    cls = torch.nn.GRU if kind == "gru" else torch.nn.LSTM
    ref = cls(I, H, num_layers=L, bidirectional=bi, batch_first=bf, dropout=p)
    mine = b200rnn.from_torch(ref).to(DEV).train()
    return ref.double().train(), mine


def _states(out):
    s = out[1]
    return s if isinstance(s, tuple) else (s,)


def _advance(mine, T, B):
    D = 2 if mine.bidirectional else 1
    return philox.counters(T * B * D * mine.hidden_size)


def _forward_pair(ref, mine, x, seed=1, packed_lens=None):
    """One train-mode forward of both with the masks of mine's current {seed, offset}; returns the outputs, the leaf
    inputs and the random output weights of the scalar loss."""
    T, B = (x.shape[1], x.shape[0]) if mine.batch_first else (x.shape[0], x.shape[1])
    D = 2 if mine.bidirectional else 1
    st = _state(mine._rng_state)
    factors = rnn_factors(st, T, B, D * mine.hidden_size, mine.num_layers, mine.dropout)
    xr = x.double().requires_grad_(True)
    xm = x.to(DEV).requires_grad_(True)
    if packed_lens is not None:
        pk = torch.nn.utils.rnn.pack_padded_sequence
        out_r = MaskedRNN(ref)(pk(xr, packed_lens, batch_first=mine.batch_first, enforce_sorted=False), factors)
        out_m = mine(pk(xm, packed_lens, batch_first=mine.batch_first, enforce_sorted=False))
    else:
        out_r = MaskedRNN(ref)(xr, factors)
        out_m = mine(xm)
    assert _state(mine._rng_state) == [st[0], st[1] + _advance(mine, T, B)], "offset advance of one forward"
    return out_r, out_m, xr, xm


def _loss_pair(out_r, out_m, seed, packed):
    g = torch.Generator().manual_seed(seed)
    yr, ym = out_r[0], out_m[0]
    if packed:
        pad = torch.nn.utils.rnn.pad_packed_sequence
        yr, ym = pad(yr)[0], pad(ym)[0]
    w = torch.randn(yr.shape, generator=g, dtype=torch.float64)
    lr_, lm = (yr * w).sum(), (ym * w.to(DEV, torch.float32)).sum()
    for a, b in zip(_states(out_m), _states(out_r)):
        ws = torch.randn(b.shape, generator=g, dtype=torch.float64)
        lr_, lm = lr_ + (b * ws).sum(), lm + (a * ws.to(DEV, torch.float32)).sum()
    errs = {"y": (ym.detach().cpu().double() - yr.detach()).abs().max().item()}
    for i, (a, b) in enumerate(zip(_states(out_m), _states(out_r))):
        errs[f"state{i}"] = (a.detach().cpu().double() - b.detach()).abs().max().item()
    return lr_, lm, errs


def _grad_errs(ref, mine, xr, xm):
    errs = {"dx": _relmax(xm.grad, xr.grad)}
    for (n, pr), (_, pm) in zip(ref.named_parameters(), mine.named_parameters()):
        errs["d" + n] = _relmax(pm.grad, pr.grad)
        pr.grad, pm.grad = None, None
    return errs


def _assert_errs(errs, where):
    for k, v in errs.items():
        tol = OUT_TOL if (k == "y" or k.startswith("state")) else GRAD_RTOL
        assert v <= tol, f"{where}: {k} error {v:.3e} > {tol:.0e}  (all: {errs})"


def _check_case(kind, I, H, L, bi, bf, B, T, p, seed=0):
    ref, mine = _make(kind, I, H, L, bi, bf, p, seed)
    x = torch.randn((B, T, I) if bf else (T, B, I), generator=torch.Generator().manual_seed(seed + 100))
    out_r, out_m, xr, xm = _forward_pair(ref, mine, x)
    lr_, lm, errs = _loss_pair(out_r, out_m, seed + 200, False)
    lr_.backward()
    lm.backward()
    torch.cuda.synchronize()
    errs.update(_grad_errs(ref, mine, xr, xm))
    _assert_errs(errs, f"{kind} I={I} H={H} L={L} bi={bi} B={B} T={T} p={p}")
    return errs


RNN_CASES = {
    # id: kind, I, H, L, bi, batch_first, B, T, p
    "gru_c2_b64": ("gru", 256, 256, 2, False, True, 64, 120, 0.5),        # two-row GRU clusters
    "gru_c2_b128": ("gru", 256, 256, 2, False, True, 128, 120, 0.5),      # four-row GRU clusters
    "bilstm_c3": ("lstm", 1024, 256, 2, True, False, 64, 30, 0.5),
    "bilstm_h128_fuse_text": ("lstm", 1024, 128, 2, True, False, 32, 30, 0.3),
    "bigru_i37_ffma": ("gru", 37, 128, 2, True, False, 16, 20, 0.5),      # FFMA layer-0 projection
    "lstm_b13": ("lstm", 256, 128, 2, False, True, 13, 17, 0.5),
    "gru_t1": ("gru", 256, 256, 2, False, True, 8, 1, 0.5),
    "bilstm_l3": ("lstm", 64, 128, 3, True, False, 16, 12, 0.5),          # two dropouts: streams 0 and 1
    "gru_l3": ("gru", 256, 256, 3, False, True, 24, 16, 0.5),
    "gru_p1": ("gru", 256, 256, 2, False, True, 8, 10, 1.0),              # layer 1 sees zeros
}


@pytest.mark.parametrize("case", list(RNN_CASES))
def test_rnn_train_mode_forward_backward_matches_masked_oracle(case):
    _check_case(*RNN_CASES[case])


def test_eval_and_p0_do_not_advance_the_offset():
    _, mine = _make("gru", 256, 256, 2, False, True, 0.5)
    x = torch.randn(4, 6, 256, device=DEV)
    st = _state(mine._rng_state)
    with torch.no_grad():
        mine.eval()(x)
        assert _state(mine._rng_state) == st
        mine.train()
        mine.dropout = 0.0
        mine(x)
        assert _state(mine._rng_state) == st
        mine.dropout = 0.5
        mine(x)
    assert _state(mine._rng_state) == [st[0], st[1] + _advance(mine, 6, 4)]


def test_two_consecutive_forwards_use_successive_offsets():
    ref, mine = _make("lstm", 256, 128, 2, True, False, 0.5)
    g = torch.Generator().manual_seed(5)
    offsets = []
    for i in range(2):
        x = torch.randn(9, 12, 256, generator=g)
        offsets.append(_state(mine._rng_state)[1])
        out_r, out_m, xr, xm = _forward_pair(ref, mine, x)
        lr_, lm, errs = _loss_pair(out_r, out_m, 50 + i, False)
        lr_.backward()
        lm.backward()
        errs.update(_grad_errs(ref, mine, xr, xm))
        _assert_errs(errs, f"forward {i}")
    assert offsets[1] - offsets[0] == _advance(mine, 9, 12)


@pytest.mark.parametrize("kind", ["gru", "lstm"])
def test_backward_applies_the_mask_of_its_own_forward(kind):
    """y1 = m(x1); y2 = m(x2); backward of y1, then of y2: each backward reads the {seed, offset} its forward saved in
    the reserve, not the module's current state."""
    if kind == "gru":
        ref, mine = _make("gru", 256, 256, 2, False, True, 0.5)
        shape = (16, 20, 256)
    else:
        ref, mine = _make("lstm", 1024, 128, 2, True, False, 0.5)
        shape = (10, 16, 1024)
    g = torch.Generator().manual_seed(9)
    x1, x2 = torch.randn(*shape, generator=g), torch.randn(*shape, generator=g)
    f1 = _forward_pair(ref, mine, x1)
    f2 = _forward_pair(ref, mine, x2)
    for i, (out_r, out_m, xr, xm) in enumerate((f1, f2)):
        lr_, lm, errs = _loss_pair(out_r, out_m, 70 + i, False)
        lr_.backward()
        lm.backward()
        torch.cuda.synchronize()
        errs.update(_grad_errs(ref, mine, xr, xm))
        _assert_errs(errs, f"{kind} backward {i + 1}")


@pytest.mark.parametrize("kind", ["gru", "lstm"])
def test_packed_sequence_with_dropout_matches_masked_oracle(kind):
    if kind == "gru":
        ref, mine = _make("gru", 256, 256, 2, False, True, 0.5)
        B, T, I = 11, 23, 256
        x = torch.randn(B, T, I, generator=torch.Generator().manual_seed(3))
    else:
        ref, mine = _make("lstm", 1024, 128, 2, True, False, 0.5)
        B, T, I = 9, 14, 1024
        x = torch.randn(T, B, I, generator=torch.Generator().manual_seed(3))
    lens = torch.randint(1, T + 1, (B,), generator=torch.Generator().manual_seed(4))
    lens[3] = T                                     # the padded length the kernels see is the longest sequence
    out_r, out_m, xr, xm = _forward_pair(ref, mine, x, packed_lens=lens)
    lr_, lm, errs = _loss_pair(out_r, out_m, 90, True)
    lr_.backward()
    lm.backward()
    torch.cuda.synchronize()
    errs.update(_grad_errs(ref, mine, xr, xm))
    _assert_errs(errs, f"packed {kind}")


@pytest.mark.parametrize("kind", ["gru", "lstm"])
def test_fused_layernorm_rnn_time_sum_with_dropout(kind):
    """``forward_ln_sum`` (LayerNorm -> RNN -> sum over time, ``AudioBiLSTM.pooled``) with dropout 0.5: under autograd
    (``_LNRNNPoolFunction``: dx, LayerNorm weight and bias, every RNN weight) and under no_grad in train mode (the
    in-place ``dropout_split`` pass, nothing saved)."""
    if kind == "gru":
        ref, mine = _make("gru", 256, 256, 2, False, True, 0.5)
        B, T, I = 64, 120, 256
    else:
        ref, mine = _make("lstm", 1024, 128, 2, True, True, 0.5)
        B, T, I = 32, 30, 1024
    D = 2 if mine.bidirectional else 1
    torch.manual_seed(11)
    ln_r = torch.nn.LayerNorm(I).double()
    with torch.no_grad():
        ln_r.weight.uniform_(0.5, 1.5)
        ln_r.bias.uniform_(-0.2, 0.2)
    ln_m = torch.nn.LayerNorm(I).to(DEV)
    ln_m.load_state_dict(ln_r.state_dict())
    g = torch.Generator().manual_seed(12)
    x = torch.randn(B, T, I, generator=g)
    # ---- autograd ----
    st = _state(mine._rng_state)
    f = rnn_factors(st, T, B, D * mine.hidden_size, 2, 0.5)
    xr, xm = x.double().requires_grad_(True), x.to(DEV).requires_grad_(True)
    pr = MaskedRNN(ref)(ln_r(xr), f)[0].sum(1)
    pm = mine.forward_ln_sum(xm, ln_m)
    assert _state(mine._rng_state) == [st[0], st[1] + _advance(mine, T, B)]
    w = torch.randn(pr.shape, generator=g, dtype=torch.float64)
    (pr * w).sum().backward()
    (pm * w.to(DEV, torch.float32)).sum().backward()
    torch.cuda.synchronize()
    errs = {"y": (pm.detach().cpu().double() - pr.detach()).abs().max().item() / T}   # a sum of T outputs
    errs.update(_grad_errs(ref, mine, xr, xm))
    errs["dln.weight"] = _relmax(ln_m.weight.grad, ln_r.weight.grad)
    errs["dln.bias"] = _relmax(ln_m.bias.grad, ln_r.bias.grad)
    _assert_errs(errs, f"ln-rnn-sum {kind} autograd")
    # ---- no_grad, train mode ----
    x2 = torch.randn(B, T, I, generator=g)
    st = _state(mine._rng_state)
    f = rnn_factors(st, T, B, D * mine.hidden_size, 2, 0.5)
    with torch.no_grad():
        pr = MaskedRNN(ref)(ln_r(x2.double()), f)[0].sum(1)
        pm = mine.forward_ln_sum(x2.to(DEV), ln_m)
    assert _state(mine._rng_state) == [st[0], st[1] + _advance(mine, T, B)]
    err = (pm.cpu().double() - pr).abs().max().item() / T
    assert err <= OUT_TOL, (kind, "no_grad", err)


_CHILD = """
import sys
sys.path[:0] = {paths!r}
import torch
import test_gpu_dropout_exact as t
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    t._check_case(*t.RNN_CASES["gru_c2_b64"])
    torch.cuda.synchronize()
names = [e.name for e in prof.events()]
assert any("dropout_kernel" in n for n in names), "the forward without tensor cores must run dropout_kernel"
assert not any("dropout_split_kernel" in n for n in names), "B200RNN_NO_TC=1 must not run dropout_split_kernel"
print("child ok")
"""


def test_forward_without_tensor_cores_matches_masked_oracle():
    """With B200RNN_NO_TC=1 (read once per process, hence a child process) the forward applies the inter-layer
    dropout with ``dropout_kernel`` instead of ``dropout_split_kernel``: same masks, same results."""
    root = os.path.dirname(HERE)
    paths = [HERE, root, os.path.join(root, "icassp2022-depression_b200")]
    flags = [f for f, on in (("-s", sys.flags.no_user_site), ("-E", sys.flags.ignore_environment)) if on]
    env = dict(os.environ, B200RNN_NO_TC="1")
    proc = subprocess.run([sys.executable, *flags, "-B", "-c", _CHILD.format(paths=paths)], env=env,
                          capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0 and "child ok" in proc.stdout, proc.stdout[-3000:] + proc.stderr[-3000:]


@pytest.mark.parametrize("n", [128, 256])
def test_mlp_dropout_train_mode_matches_masked_oracle(n):
    from b200rnn import fused_head

    torch.manual_seed(n)
    B, p = 33, 0.3                                   # 33 rows: a partial batch tile
    lin = torch.nn.Linear(n, n).to(DEV)
    x = torch.randn(B, n, device=DEV)
    for seed, offset, stream in ((0x5DEECE66D, 0, 0), (0x123456789ABCDEF, 98765, 2)):
        hdr = torch.tensor([seed, offset], dtype=torch.int64, device=DEV)
        got = fused_head.mlp_dropout(x, lin, p, True, hdr, stream)
        f_in = torch.from_numpy(philox.dropout_factor(seed, offset, stream, (B, n), p).astype(np.float64))
        f_out = torch.from_numpy(philox.dropout_factor(seed, offset, stream + 1, (B, n), p).astype(np.float64))
        w, b = lin.weight.detach().cpu().double(), lin.bias.detach().cpu().double()
        want = torch.relu((x.cpu().double() * f_in) @ w.t() + b) * f_out
        torch.cuda.synchronize()
        assert (got.cpu().double() - want).abs().max().item() <= OUT_TOL, (n, stream)
        assert _state(hdr) == [seed, offset], "mlp_dropout reads its header, it does not advance it"


# ---- the benched fuse step, dropout 0.3 everywhere --------------------------------------------------------------------
FB, T_A, E_A, H_A, T_T, E_T, H_T = 128, 120, 256, 256, 30, 1024, 128
FUSE_P, FUSE_LR = 0.3, 8e-6


def _fuse_factors(mine, fused):
    return dict(
        rnn={"lstm_net": rnn_factors(_state(mine.lstm_net._rng_state), T_T, FB, 2 * H_T, 2, FUSE_P),
             "lstm_net_audio": rnn_factors(_state(mine.lstm_net_audio._rng_state), T_A, FB, H_A, 2, FUSE_P)},
        dropout=head_factors(_state(fused.rng_state), FB, H_T, H_A, FUSE_P))


@pytest.mark.parametrize("concurrent", [True, False], ids=["split_text_stage", "one_stream"])
@pytest.mark.parametrize("flavour", ["classification", "regression"])
def test_fused_fuse_step_train_mode_dropout_matches_masked_oracle(flavour, concurrent):
    """``FusedFuseStep`` at BASELINE configs[3] with dropout 0.3 in train mode - the step bench.py times - for three
    steps against ``RefFusion`` with all six masks injected: the text BiLSTM's and the audio GRU's inter-layer masks
    and the head's streams 0-3. Features (``features()``), output, loss and the Adam-updated ``fc_final.0.weight``."""
    import b200rnn
    from oracle import ref_models

    reg = flavour == "regression"
    args = dict(text_embed_size=E_T, text_hidden_dims=H_T, rnn_layers=2, dropout=FUSE_P, num_classes=1 if reg else 2,
                audio_hidden_dims=H_A, audio_embed_size=E_A, regression=reg)
    torch.manual_seed(0)
    ref = ref_models.RefFusion(**args)
    mine = b200rnn.fusion_net(**args)
    mine.load_state_dict(ref.state_dict())
    mine = mine.to(DEV).train()
    ref = ref.double().train()
    for m in (ref, mine):                            # fuse_net_whole.py:590-593
        for q in m.parameters():
            q.requires_grad = False
        m.fc_final[0].weight.requires_grad = True
    opt = torch.optim.Adam([ref.fc_final[0].weight], lr=FUSE_LR)
    fused = b200rnn.FusedFuseStep(mine, lr=FUSE_LR, concurrent_branches=concurrent)
    consume = philox.counters(FB * max(H_T, H_A))
    g = torch.Generator().manual_seed(4321)
    worst = {"feat": 0.0, "out": 0.0, "loss": 0.0, "w": 0.0}
    for _ in range(3):
        audio, text = torch.randn(FB, T_A, E_A, generator=g), torch.randn(FB, T_T, E_T, generator=g)
        y = torch.rand(FB, generator=g) * 3.0 if reg else torch.randint(0, 2, (FB,), generator=g)
        batch = b200rnn.FuseBatch(audio.to(DEV), text.to(DEV))
        # ---- features(): its own draw ----
        masks = _fuse_factors(mine, fused)
        h0 = _state(fused.rng_state)
        with masks_injected(ref, **masks):
            tf_r, af_r = ref.pretrained_feature_tensors(audio.double(), text.double())
        tf_m, af_m = fused.features(batch)
        assert _state(fused.rng_state) == [h0[0], h0[1] + consume]
        worst["feat"] = max(worst["feat"], (tf_m.cpu().double() - tf_r).abs().max().item(),
                            (af_m.cpu().double() - af_r).abs().max().item())
        # ---- the step: the next draw ----
        masks = _fuse_factors(mine, fused)
        h0, a0, t0 = _state(fused.rng_state), _state(mine.lstm_net_audio._rng_state), _state(mine.lstm_net._rng_state)
        opt.zero_grad()
        with masks_injected(ref, **masks):
            tf_r, af_r = ref.pretrained_feature_tensors(audio.double(), text.double())
        out_r = ref(torch.cat((tf_r, af_r), dim=1))
        loss_r = ref_models.ref_fusion_loss(tf_r, af_r, y.view(-1, 1) if reg else y, ref)
        loss_r.backward()
        opt.step()
        out_m, loss_m = fused(batch, y.to(DEV))
        torch.cuda.synchronize()
        assert _state(fused.rng_state) == [h0[0], h0[1] + consume], "head offset advance per step"
        assert _state(mine.lstm_net_audio._rng_state) == [a0[0], a0[1] + philox.counters(T_A * FB * H_A)]
        assert _state(mine.lstm_net._rng_state) == [t0[0], t0[1] + philox.counters(T_T * FB * 2 * H_T)]
        worst["out"] = max(worst["out"], (out_m.cpu().double() - out_r.detach()).abs().max().item())
        worst["loss"] = max(worst["loss"], abs(loss_m.item() - loss_r.item()) / max(1.0, abs(loss_r.item())))
        worst["w"] = max(worst["w"], (mine.fc_final[0].weight.detach().cpu().double()
                                      - ref.fc_final[0].weight.detach()).abs().max().item())
    print(flavour, concurrent, worst)
    assert worst["feat"] <= 1e-4 and worst["out"] <= 1e-4, worst
    assert worst["loss"] <= 1e-5, worst
    assert worst["w"] <= 1e-6, worst


# ---- graph-captured single-modality train steps, RNN dropout 0.5 ----------------------------------------------------

def _groups(model, wd):
    named = list(model.named_parameters())
    return [{"params": [p for n, p in named if "ln" not in n], "weight_decay": wd},
            {"params": [p for n, p in named if "ln" in n], "weight_decay": 0.0}]


@pytest.mark.parametrize("kind", ["audio", "text"])
def test_graph_captured_train_step_with_rnn_dropout_matches_masked_oracle(kind, lr=1e-3, wd=1e-2, steps=3):
    """``b200rnn.TrainStep`` (one CUDA graph: forward, fused softmax + CE, BPTT, AdamW) with the encoder's inter-layer
    dropout at the reference's 0.5, three replays against ``RefAudio`` / ``RefText`` with the same masks + AdamW, in
    the form of test_gpu_train_step.py. The masks are rebuilt from ``_rng_state`` read between replays: each replay
    draws a fresh mask on the device and its backward applies that same mask. The heads' own ``nn.Dropout`` modules
    draw from torch's RNG, which this library does not own, so their p is set to 0 on both sides."""
    import b200rnn
    from oracle import ref_models

    torch.manual_seed(0)
    if kind == "audio":   # BASELINE c2: B=64, T=120, 256-d, H=256
        cfg = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=256, hidden_dims=256)
        ref, mine = ref_models.RefAudio(cfg), b200rnn.AudioBiLSTM(cfg)
        shape, enc, D = (64, 120, 256), "lstm_net_audio", 1
    else:                 # BASELINE c3: B=64, T=30, 1024-d, H=256
        cfg = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=1024, hidden_dims=256, bidirectional=True)
        ref, mine = ref_models.RefText(cfg), b200rnn.TextBiLSTM(cfg)
        shape, enc, D = (64, 30, 1024), "lstm_net", 2
    mine.load_state_dict(ref.state_dict())
    mine = mine.to(DEV).train()
    ref = ref.double().train()
    for m in (ref, mine):
        for mod in m.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
    B, T = shape[0], shape[1]
    rnn_m = mine.get_submodule(enc)
    assert rnn_m.dropout == 0.5
    opt_r = torch.optim.AdamW(_groups(ref, wd), lr=lr)
    crit = torch.nn.CrossEntropyLoss()
    opt_m = b200rnn.FlatAdamW.like_reference(mine, lr=lr, weight_decay=wd)
    ts = b200rnn.TrainStep(mine, opt_m, shape, use_graph=True)
    ts.warmup_and_capture()
    p0 = {n: p.detach().clone() for n, p in ref.named_parameters()}
    g = torch.Generator().manual_seed(2468)
    worst_loss, grad_rel = 0.0, 0.0
    for s in range(steps):
        x = torch.randn(*shape, generator=g)
        y = torch.randint(0, 2, (B,), generator=g)
        st = _state(rnn_m._rng_state)
        xr = x.double().requires_grad_(True)
        opt_r.zero_grad()
        with masks_injected(ref, rnn={enc: rnn_factors(st, T, B, D * 256, 2, 0.5)}):
            out_r = ref(xr)
        loss_r = crit(out_r, y)
        loss_r.backward()
        if s == 0:
            g_ref = {n: p.grad.detach().clone() for n, p in ref.named_parameters() if p.grad is not None}
        opt_r.step()
        out_m, loss_m = ts.step(x.to(DEV), y.to(DEV))
        torch.cuda.synchronize()
        assert _state(rnn_m._rng_state) == [st[0], st[1] + philox.counters(T * B * D * 256)], "one draw per replay"
        worst_loss = max(worst_loss, abs(loss_m.item() - loss_r.item()))
        assert (out_m.cpu().double() - out_r.detach()).abs().max().item() < 1e-4, (kind, s)
        dx_rel = _relmax(ts.dx, xr.grad)
        assert dx_rel < 1e-4, (kind, s, "dx", dx_rel)
        if s == 0:
            for n, p in mine.named_parameters():
                if n in g_ref:
                    grad_rel = max(grad_rel, _relmax(p.grad, g_ref[n]))
    assert worst_loss <= 1e-5, (kind, worst_loss)
    assert grad_rel <= 1e-4, (kind, grad_rel)
    dev_all, moved = [], 0.0
    named_r = dict(ref.named_parameters())
    for n, p in mine.named_parameters():
        q = named_r[n].detach()
        if (q - p0[n]).abs().max().item() == 0.0:
            continue
        dev_all.append(((p.detach().cpu().double() - q).abs() / (lr * steps)).reshape(-1))
        moved = max(moved, (q - p0[n]).abs().max().item())
    dev_all = torch.cat(dev_all)
    assert moved > 0.5 * lr, "the oracle's parameters must have moved"
    q999 = torch.quantile(dev_all[torch.randperm(dev_all.numel())[:1_000_000]].float(), 0.999).item()
    assert q999 < 0.02, (kind, "99.9 % quantile of |dp| / (lr * steps)", q999)
    assert dev_all.max().item() <= 2.0 + 1e-3, (kind, dev_all.max().item())
