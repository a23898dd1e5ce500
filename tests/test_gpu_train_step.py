"""Assembled, graph-captured train steps of the single-modality scripts (SURVEY.md §8 a7 / f3) against the CPU oracle:
``b200rnn.TrainStep`` (zero_grad -> forward -> Softmax+CrossEntropy -> backward incl. dx -> FlatAdamW, one CUDA graph)
vs ``oracle.ref_models.RefAudio / RefText`` + ``nn.CrossEntropyLoss`` on the Softmax outputs + ``torch.optim.AdamW``
with the reference's parameter grouping (audio_gru_whole.py:161-201, 247-255, 307-308; text_bilstm_whole.py:154-193,
303-304), three consecutive steps at the BASELINE c2 / c3 sizes. Dropout is forced to 0 in train mode here, because
torch's dropout RNG cannot be reproduced. The same steps with the encoders' dropout at the reference's 0.5 are checked
with the library's own masks in test_gpu_dropout_exact.py.

Tolerances: loss <= 1e-5 abs per step; first-step gradients <= 1e-4 of the largest entry; parameters after three steps:
Adam's update is ~lr * sign(g) for |g| >> eps, so elements whose gradient is below the fp32 noise floor may move the
other way (deviation up to 2 lr per step) - the test bounds the bulk (99.9 % within 2 % of the distance travelled) and
the worst case (<= 2 lr per step).
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _groups(model, wd):
    named = list(model.named_parameters())
    return [{"params": [p for n, p in named if "ln" not in n], "weight_decay": wd},
            {"params": [p for n, p in named if "ln" in n], "weight_decay": 0.0}]


def _run(kind, lr=1e-3, wd=1e-2, steps=3, use_graph=True):
    import b200rnn
    from oracle import ref_models

    torch.manual_seed(0)
    if kind == "audio":   # BASELINE c2: B=64, T=120, 256-d, H=256
        cfg = dict(num_classes=2, dropout=0.0, rnn_layers=2, embedding_size=256, hidden_dims=256)
        ref, mine = ref_models.RefAudio(cfg), b200rnn.AudioBiLSTM(cfg)
        shape = (64, 120, 256)
    else:                 # BASELINE c3: B=64, T=30, 1024-d, H=256
        cfg = dict(num_classes=2, dropout=0.0, rnn_layers=2, embedding_size=1024, hidden_dims=256, bidirectional=True)
        ref, mine = ref_models.RefText(cfg), b200rnn.TextBiLSTM(cfg)
        shape = (64, 30, 1024)
    mine.load_state_dict(ref.state_dict())
    mine = mine.to(DEV).train()
    ref.train()
    opt_r = torch.optim.AdamW(_groups(ref, wd), lr=lr)
    crit = torch.nn.CrossEntropyLoss()
    opt_m = b200rnn.FlatAdamW.like_reference(mine, lr=lr, weight_decay=wd)
    ts = b200rnn.TrainStep(mine, opt_m, shape, use_graph=use_graph)
    ts.warmup_and_capture()
    p0 = {n: p.detach().clone() for n, p in ref.named_parameters()}
    g = torch.Generator().manual_seed(2468)
    worst_loss, grad_rel = 0.0, 0.0
    for s in range(steps):
        x = torch.randn(*shape, generator=g)
        y = torch.randint(0, 2, (shape[0],), generator=g)
        xr = x.clone().requires_grad_(True)            # Variable(..., requires_grad=True)
        opt_r.zero_grad()
        out_r = ref(xr)
        loss_r = crit(out_r, y)                         # CE on the Softmax outputs, as the reference does
        loss_r.backward()
        if s == 0:
            g_ref = {n: p.grad.detach().clone() for n, p in ref.named_parameters() if p.grad is not None}
        opt_r.step()
        out_m, loss_m = ts.step(x.to(DEV), y.to(DEV))
        torch.cuda.synchronize()
        worst_loss = max(worst_loss, abs(loss_m.item() - loss_r.item()))
        assert (out_m.cpu() - out_r.detach()).abs().max().item() < 1e-4, (kind, s)
        dx_rel = (ts.dx.cpu() - xr.grad).abs().max().item() / max(xr.grad.abs().max().item(), 1e-20)
        assert dx_rel < 1e-4, (kind, s, "dx", dx_rel)
        if s == 0:   # the optimiser has consumed the bucket but not cleared it: first-step gradients are still there
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
            continue                                   # parameter outside the graph (unused attention_layer etc.)
        dev_all.append(((p.detach().cpu() - q).abs() / (lr * steps)).reshape(-1))
        moved = max(moved, (q - p0[n]).abs().max().item())
    dev_all = torch.cat(dev_all)
    assert moved > 0.5 * lr, "the oracle's parameters must have moved"
    q999 = torch.quantile(dev_all[torch.randperm(dev_all.numel())[:1_000_000]], 0.999).item()
    assert q999 < 0.02, (kind, "99.9 % quantile of |dp| / (lr * steps)", q999)
    assert dev_all.max().item() <= 2.0 + 1e-3, (kind, dev_all.max().item())
    assert opt_m.step_count.item() == float(steps)
    return worst_loss, grad_rel, q999


def test_audio_gru_whole_train_step_matches_cpu_oracle_adamw_three_steps():
    print("audio c2:", _run("audio"))


def test_text_bilstm_whole_train_step_matches_cpu_oracle_adamw_three_steps():
    print("text c3:", _run("text"))


def test_train_step_eager_equals_graph():
    a = _run("audio", steps=2, use_graph=False)
    assert a[0] <= 1e-5


def test_softmax_cross_entropy_kernel_matches_torch_double_softmax():
    import b200rnn

    torch.manual_seed(4)
    for B, C in ((64, 2), (7, 5), (1, 2)):
        z = (torch.randn(B, C, device=DEV) * 3).requires_grad_(True)
        y = torch.randint(0, C, (B,), device=DEV)
        zr = z.detach().clone().requires_grad_(True)
        pr = torch.softmax(zr, dim=1)
        lr_ = torch.nn.functional.cross_entropy(pr, y)
        lr_.backward()
        p, l = b200rnn.softmax_cross_entropy(z, y)
        (l * 1.0).backward()
        assert (p - pr.detach()).abs().max().item() < 1e-6
        assert abs(l.item() - lr_.item()) < 1e-6
        assert (z.grad - zr.grad).abs().max().item() < 1e-7
    p, l = b200rnn.softmax_cross_entropy(torch.zeros(3, 2, device=DEV), torch.tensor([0, 5, 1], device=DEV))
    assert torch.isnan(l)
