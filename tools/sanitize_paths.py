#!/usr/bin/env python
"""Small shapes through every recurrence variant, for compute-sanitizer (memcheck / racecheck):
    compute-sanitizer --tool memcheck python tools/sanitize_paths.py
    compute-sanitizer --tool memcheck python tools/sanitize_paths.py rnn   # recurrence only
The GRU H=256 case runs at B = 9 (2-row clusters) and B = 80 (4-row clusters, above the 74-row cut).
"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "icassp2022-depression_b200"))
import torch, b200rnn
from torch.nn.utils.rnn import pack_padded_sequence
dev = torch.device("cuda:0")
torch.manual_seed(0)
for kind, I, H, L, bi, B in (("gru", 64, 256, 2, False, 9), ("lstm", 64, 128, 2, True, 9), ("gru", 32, 128, 1, True, 9),
                             ("lstm", 32, 256, 1, False, 9), ("gru", 64, 256, 2, False, 80)):
    cls = b200rnn.GRU if kind == "gru" else b200rnn.LSTM
    m = cls(I, H, num_layers=L, bidirectional=bi, batch_first=True, dropout=0.3 if L > 1 else 0.0).to(dev).train()
    T = 6
    x = torch.randn(B, T, I, device=dev, requires_grad=True)
    y = m(x)[0]
    y.sum().backward()
    lengths = torch.tensor([6, 1, 3, 6, 2, 5, 4, 6, 1] * 9)[:B]
    xp = pack_padded_sequence(x.detach().requires_grad_(True), lengths, batch_first=True, enforce_sorted=False)
    yp = m(xp)[0]
    yp.data.sum().backward()
    with torch.no_grad():
        m.eval()(x)
    torch.cuda.synchronize()
    print(kind, H, B, "ok", flush=True)
if sys.argv[1:] == ["rnn"]:
    sys.exit(0)
# round 2: the fused shells (LayerNorm prologue + pooled gradient under autograd, attention pooling fwd/bwd, Softmax+CE,
# MN-major wgrad GEMMs, the single-launch fuse head with Adam)
cfg = dict(num_classes=2, dropout=0.3, rnn_layers=2, embedding_size=256, hidden_dims=128)
am = b200rnn.AudioBiLSTM(cfg).to(dev).train()
xa = torch.randn(5, 7, 256, device=dev, requires_grad=True)
p, loss = b200rnn.softmax_cross_entropy(am.forward_logits(xa), torch.randint(0, 2, (5,), device=dev))
loss.backward()
tm = b200rnn.TextBiLSTM(dict(num_classes=2, dropout=0.3, rnn_layers=2, embedding_size=128, hidden_dims=128)).to(dev).train()
xt = torch.randn(5, 6, 128, device=dev, requires_grad=True)
tm(xt).sum().backward()
fm = b200rnn.fusion_net(128, 128, 2, 0.3, 2, 128, 128).to(dev).train()
for q in fm.parameters():
    q.requires_grad = False
fm.fc_final[0].weight.requires_grad = True
st = b200rnn.FusedFuseStep(fm, lr=1e-3)
for _ in range(2):
    st(b200rnn.FuseBatch(torch.randn(6, 5, 128, device=dev), torch.randn(6, 4, 128, device=dev)),
       torch.randint(0, 2, (6,), device=dev))
torch.cuda.synchronize()
print("sanitize_paths done")
