"""Hidden sizes 64 and 512 on the GPU, against stock torch.nn.GRU / nn.LSTM on the CPU.

H = 64 runs the H = 128 cluster layout at half the width (clusters of 2 CTAs); H = 512 runs 16-CTA clusters (the
non-portable maximum), and its LSTM backward streams one gate block of W_hh from L2 in every step. Covered here:
forward and backward of every layout (uni- / bidirectional, 1 and 2 layers, both batch layouts, odd batch, short
sequences) with h_n / c_n and their gradients, PackedSequence input (the per-length kernel twins), batches beyond one
wave (every new instantiation, the wide-batch fallbacks included, is launched), train-mode dropout with host-rebuilt
masks, the fused LayerNorm -> RNN -> time-sum entry point, bitwise determinism of the 16-CTA exchange, CUDA graph
capture, and one graph-captured TrainStep per model.

Tolerances are the suite's: outputs and states <= 1e-5 abs, gradients <= 1e-4 of the tensor's largest entry (pooled
time sums and model outputs <= 1e-4 abs, as in test_gpu_coverage.py / test_gpu_train_step.py).
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OUT_TOL = 1e-5
GRAD_RTOL = 1e-4


def _relmax(got, ref):
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    m = ref.abs().max().item()
    return (got - ref).abs().max().item() / m if m > 0 else got.abs().max().item()


def _make(kind, I, H, L=1, bi=False, bf=False, seed=0):
    import b200rnn

    torch.manual_seed(seed)
    cls = torch.nn.GRU if kind == "gru" else torch.nn.LSTM
    ref = cls(I, H, num_layers=L, bidirectional=bi, batch_first=bf)
    return ref, b200rnn.from_torch(ref).to(DEV)


def _states(out):
    return out[1] if isinstance(out[1], tuple) else (out[1],)


def _compare(ref, mine, x, lens=None, seed=1):
    """Forward + backward of both on the same input and loss weights (output and final states); returns the errors."""
    bf = mine.batch_first
    xr, xm = x.clone().requires_grad_(True), x.clone().to(DEV).requires_grad_(True)
    if lens is not None:
        pk = lambda t: torch.nn.utils.rnn.pack_padded_sequence(t, lens, batch_first=bf, enforce_sorted=False)  # noqa: E731
        out_r, out_m = ref(pk(xr)), mine(pk(xm))
        yr = torch.nn.utils.rnn.pad_packed_sequence(out_r[0], batch_first=bf)[0]
        ym = torch.nn.utils.rnn.pad_packed_sequence(out_m[0], batch_first=bf)[0]
    else:
        out_r, out_m = ref(xr), mine(xm)
        yr, ym = out_r[0], out_m[0]
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(yr.shape, generator=g)
    loss_r, loss_m = (yr * w).sum(), (ym * w.to(DEV)).sum()
    errs = {"y": (ym.detach().cpu() - yr.detach()).abs().max().item()}
    for i, (a, b) in enumerate(zip(_states(out_m), _states(out_r))):
        errs[f"state{i}"] = (a.detach().cpu() - b.detach()).abs().max().item()
        ws = torch.randn(b.shape, generator=g)
        loss_r, loss_m = loss_r + (b * ws).sum(), loss_m + (a * ws.to(DEV)).sum()
    loss_r.backward()
    loss_m.backward()
    torch.cuda.synchronize()
    errs["dx"] = _relmax(xm.grad, xr.grad)
    for (n, pr), (_, pm) in zip(ref.named_parameters(), mine.named_parameters()):
        errs["d" + n] = _relmax(pm.grad, pr.grad)
    return errs


def _assert(errs, where):
    for k, v in errs.items():
        tol = OUT_TOL if (k == "y" or k.startswith("state")) else GRAD_RTOL
        assert v <= tol, f"{where}: {k} error {v:.3e} > {tol:.0e} (all: {errs})"


@pytest.mark.parametrize("H", [64, 512])
@pytest.mark.parametrize("kind", ["gru", "lstm"])
@pytest.mark.parametrize("bi", [False, True])
@pytest.mark.parametrize("L", [1, 2])
@pytest.mark.parametrize("bf", [False, True])
def test_forward_backward_match_torch_cpu(H, kind, bi, L, bf):
    # I = 96: tensor-core layer-0 projection where G*H allows it; I = 40: the FFMA projection
    I, B, T = (96 if bf else 40), 7, 5
    ref, mine = _make(kind, I, H, L, bi, bf)
    x = torch.randn((B, T, I) if bf else (T, B, I), generator=torch.Generator().manual_seed(3))
    _assert(_compare(ref, mine, x), f"{kind} H={H} L={L} bi={bi} bf={bf}")


@pytest.mark.parametrize("H", [64, 512])
@pytest.mark.parametrize("kind", ["gru", "lstm"])
@pytest.mark.parametrize("bi", [False, True])
def test_packed_sequence_matches_torch_cpu(H, kind, bi):
    B, T, I = 9, 7, 64
    ref, mine = _make(kind, I, H, 2, bi, True, seed=2)
    lens = torch.tensor([7, 1, 4, 7, 2, 6, 3, 5, 7])
    x = torch.randn(B, T, I, generator=torch.Generator().manual_seed(4))
    _assert(_compare(ref, mine, x, lens=lens), f"packed {kind} H={H} bi={bi}")


@pytest.mark.parametrize("kind,H,B", [("gru", 64, 2100), ("lstm", 64, 2100), ("gru", 512, 130), ("lstm", 512, 130)])
@pytest.mark.parametrize("ragged", [False, True])
def test_batches_beyond_one_wave(kind, H, B, ragged):
    """H = 64: ceil(B / 4) two-CTA clusters exceed what the chip holds at once, so the 8-row fallback runs (in several
    waves). H = 512: a B200 holds at most 7 of the 16-CTA clusters at once, so 130 rows take several waves in every
    H = 512 kernel (2 to 8 batch rows per cluster)."""
    T, I = 3, 32
    ref, mine = _make(kind, I, H, 1, False, True, seed=5)
    x = torch.randn(B, T, I, generator=torch.Generator().manual_seed(6))
    lens = None
    if ragged:
        lens = torch.randint(1, T + 1, (B,), generator=torch.Generator().manual_seed(7))
        lens[0] = T
    _assert(_compare(ref, mine, x, lens=lens), f"{kind} H={H} B={B} ragged={ragged}")


DROPOUT_CASES = {
    "gru_h64": ("gru", 256, 64, 2, False, True, 13, 10, 0.5),
    "bilstm_h64": ("lstm", 64, 64, 2, True, False, 9, 8, 0.5),
    "bigru_h512": ("gru", 256, 512, 2, True, True, 7, 6, 0.5),
    "lstm_h512": ("lstm", 128, 512, 2, False, False, 5, 6, 0.5),
}


@pytest.mark.parametrize("case", list(DROPOUT_CASES))
def test_train_mode_dropout_matches_masked_oracle(case):
    """The masks are rebuilt with the host Philox (oracle/philox.py) and injected into the float64 oracle
    (oracle/masked.py), exactly as in test_gpu_dropout_exact.py."""
    from test_gpu_dropout_exact import _check_case

    _check_case(*DROPOUT_CASES[case])


@pytest.mark.parametrize("kind,H", [("gru", 64), ("lstm", 64), ("gru", 512), ("lstm", 512)])
def test_forward_ln_sum_with_and_without_autograd(kind, H):
    """LayerNorm -> RNN -> sum over time. Where the layer-0 projection takes the tensor cores (G*H a multiple of 128:
    all but the GRU at H = 64) LayerNorm is folded into it and the pooled gradient is broadcast inside the BPTT
    kernel; the GRU at H = 64 computes the same value unfused."""
    import b200rnn

    torch.manual_seed(8)
    B, T, I = 5, 6, 256
    cls = torch.nn.GRU if kind == "gru" else torch.nn.LSTM
    rnn_r, ln_r = cls(I, H, num_layers=2, batch_first=True), torch.nn.LayerNorm(I)
    with torch.no_grad():
        ln_r.weight.uniform_(0.5, 1.5)
        ln_r.bias.uniform_(-0.5, 0.5)
    rnn_m = b200rnn.from_torch(rnn_r).to(DEV)
    ln_m = torch.nn.LayerNorm(I).to(DEV)
    ln_m.load_state_dict(ln_r.state_dict())
    x = torch.randn(B, T, I)
    xr, xm = x.clone().requires_grad_(True), x.clone().to(DEV).requires_grad_(True)
    pr = rnn_r(ln_r(xr))[0].sum(dim=1)
    pm = rnn_m.forward_ln_sum(xm, ln_m)
    w = torch.randn_like(pr)
    (pr * w).sum().backward()
    (pm * w.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    assert (pm.detach().cpu() - pr.detach()).abs().max().item() < 1e-4
    assert _relmax(xm.grad, xr.grad) <= GRAD_RTOL
    assert _relmax(ln_m.weight.grad, ln_r.weight.grad) <= GRAD_RTOL
    assert _relmax(ln_m.bias.grad, ln_r.bias.grad) <= GRAD_RTOL
    for (n, pr_), (_, pm_) in zip(rnn_r.named_parameters(), rnn_m.named_parameters()):
        assert _relmax(pm_.grad, pr_.grad) <= GRAD_RTOL, n
    with torch.no_grad():
        assert (rnn_m.forward_ln_sum(xm.detach(), ln_m).cpu() - pr.detach()).abs().max().item() < 1e-4


def test_h512_is_bitwise_deterministic_over_repeated_runs():
    """The 16-CTA clusters exchange state through 15 peers per step; 10 repetitions of forward + backward (GRU and
    BiLSTM, two layers) must be bit-identical."""
    import b200rnn

    torch.manual_seed(9)
    for kind, B, T, I, bi in (("gru", 33, 24, 256, False), ("lstm", 17, 12, 256, True)):
        cls = b200rnn.GRU if kind == "gru" else b200rnn.LSTM
        m = cls(I, 512, num_layers=2, bidirectional=bi, batch_first=True).to(DEV)
        x = torch.randn(B, T, I, device=DEV, requires_grad=True)
        ref = None
        for _ in range(10):
            m.zero_grad()
            x.grad = None
            y = m(x)[0]
            y.square().sum().backward()
            got = [y.detach().clone(), x.grad.clone()] + [p.grad.clone() for p in m.parameters()]
            if ref is None:
                ref = got
            else:
                for a, b in zip(got, ref):
                    assert torch.equal(a, b), kind


@pytest.mark.parametrize("kind,H", [("gru", 64), ("lstm", 64), ("gru", 512), ("lstm", 512)])
def test_graph_capture_and_replay_of_forward_backward(kind, H):
    """One forward + backward captured into a CUDA graph and replayed on a new input gives what an eager run gives
    (the replay accumulates into zeroed gradients, the eager run writes fresh ones)."""
    import b200rnn

    torch.manual_seed(10)
    B, T, I = 6, 8, 64
    cls = b200rnn.GRU if kind == "gru" else b200rnn.LSTM
    m = cls(I, H, num_layers=2, bidirectional=True, batch_first=True).to(DEV)
    x = torch.randn(B, T, I, device=DEV, requires_grad=True)
    w = torch.randn(B, T, 2 * H, device=DEV)

    def step():
        (m(x)[0] * w).sum().backward()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()

    new_x = torch.randn(B, T, I, device=DEV)
    with torch.no_grad():
        x.copy_(new_x)
        x.grad.zero_()
        for p in m.parameters():
            p.grad.zero_()
    g.replay()
    torch.cuda.synchronize()
    got = [x.grad.clone()] + [p.grad.clone() for p in m.parameters()]

    xe = new_x.clone().requires_grad_(True)
    m.zero_grad()
    (m(xe)[0] * w).sum().backward()
    torch.cuda.synchronize()
    want = [xe.grad] + [p.grad for p in m.parameters()]
    for a, b in zip(got, want):
        assert _relmax(a, b) <= GRAD_RTOL, kind


def _groups(model, wd):
    named = list(model.named_parameters())
    return [{"params": [p for n, p in named if "ln" not in n], "weight_decay": wd},
            {"params": [p for n, p in named if "ln" in n], "weight_decay": 0.0}]


@pytest.mark.parametrize("kind", ["audio_h512", "text_h64"])
def test_train_step_at_other_hidden_dims_matches_cpu_oracle(kind):
    """b200rnn.TrainStep (one CUDA graph: forward, Softmax + CrossEntropy, backward, FlatAdamW), three steps, against
    the restated reference models + torch.optim.AdamW on the CPU - as test_gpu_train_step.py does at the benchmark's
    widths, here with the config's hidden_dims at 512 (audio GRU) and 64 (text BiLSTM)."""
    import b200rnn
    from oracle import ref_models

    lr, wd, steps = 1e-3, 1e-2, 3
    torch.manual_seed(0)
    if kind == "audio_h512":
        cfg = dict(num_classes=2, dropout=0.0, rnn_layers=2, embedding_size=256, hidden_dims=512)
        ref, mine = ref_models.RefAudio(cfg), b200rnn.AudioBiLSTM(cfg)
        shape = (24, 40, 256)
    else:
        cfg = dict(num_classes=2, dropout=0.0, rnn_layers=2, embedding_size=1024, hidden_dims=64, bidirectional=True)
        ref, mine = ref_models.RefText(cfg), b200rnn.TextBiLSTM(cfg)
        shape = (24, 30, 1024)
    mine.load_state_dict(ref.state_dict())
    mine = mine.to(DEV).train()
    ref.train()
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
        y = torch.randint(0, 2, (shape[0],), generator=g)
        xr = x.clone().requires_grad_(True)
        opt_r.zero_grad()
        out_r = ref(xr)
        loss_r = crit(out_r, y)
        loss_r.backward()
        if s == 0:
            g_ref = {n: p.grad.detach().clone() for n, p in ref.named_parameters() if p.grad is not None}
        opt_r.step()
        out_m, loss_m = ts.step(x.to(DEV), y.to(DEV))
        torch.cuda.synchronize()
        worst_loss = max(worst_loss, abs(loss_m.item() - loss_r.item()))
        assert (out_m.cpu() - out_r.detach()).abs().max().item() < 1e-4, (kind, s)
        assert _relmax(ts.dx, xr.grad) < 1e-4, (kind, s, "dx")
        if s == 0:
            gmax = max(v.abs().max().item() for v in g_ref.values())
            for n, p in mine.named_parameters():
                if n in g_ref:
                    grad_rel = max(grad_rel, (p.grad.cpu() - g_ref[n]).abs().max().item() / gmax)
    assert worst_loss <= 1e-5, (kind, worst_loss)
    assert grad_rel <= 1e-4, (kind, grad_rel)
    dev_all, moved = [], 0.0
    for n, p in mine.named_parameters():
        q = dict(ref.named_parameters())[n].detach()
        if (q - p0[n]).abs().max().item() == 0.0:
            continue
        dev_all.append(((p.detach().cpu() - q).abs() / (lr * steps)).reshape(-1))
        moved = max(moved, (q - p0[n]).abs().max().item())
    dev_all = torch.cat(dev_all)
    assert moved > 0.5 * lr
    q999 = torch.quantile(dev_all[torch.randperm(dev_all.numel())[:1_000_000]], 0.999).item()
    assert q999 < 0.02, (kind, q999)
    assert dev_all.max().item() <= 2.0 + 1e-3, (kind, dev_all.max().item())
