"""Parity of the BENCHED object at the BENCHED size: ``b200rnn.FusedFuseStep`` at BASELINE configs[3]
(B=128, audio [128,120,256], text [128,30,1024], H = 256 / 128) against the CPU oracle
(``oracle.ref_models.RefFusion`` + ``ref_fusion_loss`` + ``torch.optim.Adam``, i.e. stock torch.nn.GRU/LSTM — the
reference's own arithmetic, fuse_net_whole.py:421-465) for three consecutive train steps.

Tolerances (north_star: logits within 1e-4): features / logits <= 1e-4 abs, loss <= 1e-5 abs, the updated
``fc_final.0.weight`` <= 1e-6 abs, gradients of the all-trainable variant <= 1e-4 relative to the largest entry.
Torch's dropout RNG cannot be reproduced, so the comparison here runs (a) in ``eval()`` and (b) in ``train()`` with the
dropout probability forced to 0. (b) is NOT the code path bench.py times: with p = 0 the kernels skip the RNG setup,
the inter-layer dropout passes and the head's keep masks. The benched configuration, dropout 0.3 in train mode, is
checked against the oracle with the library's own masks in test_gpu_dropout_exact.py.
"""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, T_A, E_A, H_A, T_T, E_T, H_T = 128, 120, 256, 256, 30, 1024, 128
LR = 8e-6


def _args(p):
    return dict(text_embed_size=E_T, text_hidden_dims=H_T, rnn_layers=2, dropout=p, num_classes=2,
                audio_hidden_dims=H_A, audio_embed_size=E_A)


def _batches(n, seed=4321):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(B, T_A, E_A, generator=g), torch.randn(B, T_T, E_T, generator=g),
             torch.randint(0, 2, (B,), generator=g)) for _ in range(n)]


def _pair(p, train):
    import b200rnn
    from oracle import ref_models

    torch.manual_seed(0)
    ref = ref_models.RefFusion(**_args(p))
    for q in ref.parameters():                      # fuse_net_whole.py:590-593
        q.requires_grad = False
    ref.fc_final[0].weight.requires_grad = True
    mine = b200rnn.fusion_net(**_args(p))
    mine.load_state_dict(ref.state_dict())
    mine = mine.to(DEV)
    for q in mine.parameters():
        q.requires_grad = False
    mine.fc_final[0].weight.requires_grad = True
    ref.train(train)
    mine.train(train)
    return ref, mine


@pytest.mark.parametrize("mode", ["eval_p0.3", "train_p0"])
def test_fused_fuse_step_matches_cpu_oracle_for_three_steps_at_baseline_config3(mode):
    import b200rnn
    from oracle import ref_models

    train = mode == "train_p0"
    ref, mine = _pair(0.0 if train else 0.3, train)
    opt = torch.optim.Adam([ref.fc_final[0].weight], lr=LR)
    fused = b200rnn.FusedFuseStep(mine, lr=LR)
    worst = {"feat": 0.0, "logit": 0.0, "prob": 0.0, "loss": 0.0, "w": 0.0}
    for audio, text, y in _batches(3):
        # ---- oracle step (fuse_net_whole.py:421-465) ----
        opt.zero_grad()
        tf_r, af_r = ref.pretrained_feature_tensors(audio, text)
        cat_r = torch.cat((tf_r, af_r), dim=1)
        logits_r = cat_r @ ref.fc_final[0].weight.detach().t()
        probs_r = ref(cat_r)
        loss_r = ref_models.ref_fusion_loss(tf_r, af_r, y, ref)
        loss_r.backward()
        opt.step()
        # ---- fused CUDA step ----
        batch = b200rnn.FuseBatch(audio.to(DEV), text.to(DEV))
        w_before = mine.fc_final[0].weight.detach().clone()
        tf_m, af_m = fused.features(batch)
        logits_m = torch.cat((tf_m, af_m), dim=1) @ w_before.t()
        probs_m, loss_m = fused(batch, y.to(DEV))
        torch.cuda.synchronize()
        worst["feat"] = max(worst["feat"], (tf_m.cpu() - tf_r).abs().max().item(), (af_m.cpu() - af_r).abs().max().item())
        worst["logit"] = max(worst["logit"], (logits_m.cpu() - logits_r).abs().max().item())
        worst["prob"] = max(worst["prob"], (probs_m.cpu() - probs_r.detach()).abs().max().item())
        worst["loss"] = max(worst["loss"], abs(loss_m.item() - loss_r.item()))
        worst["w"] = max(worst["w"], (mine.fc_final[0].weight.detach().cpu() - ref.fc_final[0].weight.detach()).abs().max().item())
    print(mode, worst)
    assert worst["feat"] <= 1e-4 and worst["logit"] <= 1e-4 and worst["prob"] <= 1e-4, worst
    assert worst["loss"] <= 1e-5, worst
    assert worst["w"] <= 1e-6, worst


def test_all_grads_fuse_step_matches_cpu_oracle_at_baseline_config3():
    """The fine-tune variant (every parameter trainable, encoders inside autograd -> BPTT kernels, 10.46 MB bucket):
    loss and every parameter gradient against the CPU oracle at B=128, T=120/30, dropout 0 in train mode."""
    import b200rnn
    from oracle import ref_models

    torch.manual_seed(0)
    ref = ref_models.RefFusion(**_args(0.0)).train()
    mine = b200rnn.fusion_net(**_args(0.0))
    mine.load_state_dict(ref.state_dict())
    mine = mine.to(DEV).train()
    audio, text, y = _batches(1, seed=99)[0]

    out, (hid, _) = ref.lstm_net(text.permute(1, 0, 2))
    tf_r = ref.fc_out(ref_models._pool_with_attention(ref.attention_layer, out.permute(1, 0, 2), hid.permute(1, 0, 2)))
    af_r = ref.fc_audio(ref.lstm_net_audio(ref.ln(audio))[0].sum(1))
    loss_r = ref_models.ref_fusion_loss(tf_r, af_r, y, ref)
    loss_r.backward()

    crit = b200rnn.MyLoss(text_hidden_dims=H_T)
    a, t = audio.to(DEV), text.to(DEV)
    seq, (h_n, _) = mine.lstm_net(t.permute(1, 0, 2))
    tf_m = mine.fc_out(b200rnn.attention_pool(mine.attention_layer, seq.permute(1, 0, 2), h_n.permute(1, 0, 2)))
    af_m = mine.fc_audio(mine.lstm_net_audio(mine.ln(a))[0].sum(dim=1))
    loss_m = crit(tf_m, af_m, y.to(DEV), mine)
    loss_m.backward()
    torch.cuda.synchronize()
    assert abs(loss_m.item() - loss_r.item()) <= 1e-5
    ref_g = dict(ref.named_parameters())
    checked = 0
    for name, p in mine.named_parameters():
        gr = ref_g[name].grad
        if gr is None:
            assert p.grad is None or p.grad.abs().max().item() == 0.0, name
            continue
        rel = (p.grad.cpu() - gr).abs().max().item() / max(gr.abs().max().item(), 1e-12)
        assert rel <= 1e-4, (name, rel)
        checked += 1
    assert checked >= 30
