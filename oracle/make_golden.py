"""ORACLE tooling — generates tests/golden/*.npz from the REFERENCE's own classes.

    B200RNN_REFERENCE_ROOT=<reference>/DepressionCollected python oracle/make_golden.py   # writes tests/golden/

Each fixture is produced by executing the reference ``ClassDef``s (oracle/ast_loader.py) on CPU with torch
{torch_version}; weights and inputs are regenerated from names (oracle/params.py), so a fixture holds only small
arrays: inputs' tags/shapes, outputs, loss, input gradient and per-parameter gradient fingerprints.
All cases run in eval() (inter-layer / head dropout off): dropout RNG streams cannot be matched bit-for-bit,
SURVEY.md §8c.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ast_loader, params  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

AUDIO_CLF = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=256, batch_size=8, epochs=170,
                 learning_rate=6e-6, hidden_dims=256, bidirectional=False, cuda=False)     # audio_gru_whole.py:110-121
TEXT_CLF = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=1024, batch_size=4, epochs=150,
                learning_rate=1e-5, hidden_dims=128, bidirectional=True, cuda=False)       # text_bilstm_whole.py:247-258
AUDIO_REG = dict(num_classes=1, dropout=0.5, rnn_layers=2, embedding_size=256, batch_size=2, epochs=120,
                 learning_rate=1e-5, hidden_dims=256, bidirectional=False, cuda=False)     # audio_bilstm_perm.py:32-43
TEXT_REG = dict(num_classes=1, dropout=0.5, rnn_layers=2, embedding_size=1024, batch_size=2, epochs=110,
                learning_rate=1e-5, hidden_dims=128, bidirectional=True, cuda=False)       # text_bilstm_perm.py:24-35
FUSE = dict(num_classes=2, dropout=0.3, rnn_layers=2, audio_embed_size=256, text_embed_size=1024, batch_size=2,
            epochs=100, learning_rate=8e-6, audio_hidden_dims=256, text_hidden_dims=128, cuda=False)  # fuse_net_whole.py:398-411


def _save(name: str, arrays: dict, meta: dict) -> None:
    os.makedirs(OUT, exist_ok=True)
    flat = {}
    for k, v in arrays.items():
        if isinstance(v, dict):
            for kk, vv in v.items():
                flat[f"{k}::{kk}"] = vv
        else:
            flat[k] = np.asarray(v)
    flat["__meta__"] = np.frombuffer(json.dumps(meta).encode("utf-8"), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **flat)
    print(f"wrote {name}.npz  ({sum(np.asarray(v).nbytes for v in flat.values()) / 1024:.1f} KiB raw)")


def _grads(model: nn.Module) -> dict:
    out = {}
    for n, p in model.named_parameters():
        if p.grad is not None:
            out["grad:" + n] = params.summarize(p.grad)
    return out


def single_modal(case: str, key: str, cls_name: str, cfg: dict, shape, loss_kind: str) -> None:
    cls = ast_loader.load_classes(key, [cls_name])[cls_name]
    torch.manual_seed(0)
    model = cls(cfg)
    params.fill_module(model)
    model.eval()
    x = params.inputs_for(case, shape).requires_grad_(True)
    out = model(x)
    if loss_kind == "ce":       # CrossEntropyLoss applied on softmax outputs, audio_gru_whole.py:188,308
        tgt = params.labels_for(case, shape[0])
        loss = nn.CrossEntropyLoss()(out, tgt)
    elif loss_kind == "l1":     # audio_bilstm_perm.py:251
        tgt = params.inputs_for(case + ":target", (shape[0], 1)).abs() * 10
        loss = nn.L1Loss()(out, tgt)
    else:                       # SmoothL1, text_bilstm_perm.py:247
        tgt = params.inputs_for(case + ":target", (shape[0], 1)).abs() * 10
        loss = nn.SmoothL1Loss()(out, tgt)
    loss.backward()
    arrays = {"out": out.detach().numpy(), "loss": np.array([loss.item()]), "dx": params.summarize(x.grad)}
    arrays.update(_grads(model))
    _save(case, arrays, dict(case=case, ref=ast_loader.FILES[key], cls=cls_name, cfg=cfg, shape=list(shape),
                             loss=loss_kind, torch=torch.__version__))


def rnn_boundary(case: str, key: str, cls_name: str, cfg: dict, attr: str, shape, time_major: bool) -> None:
    """Pins the exact drop-in boundary: the reference model's own nn.GRU / nn.LSTM instance, longer sequences."""
    cls = ast_loader.load_classes(key, [cls_name])[cls_name]
    model = cls(cfg)
    params.fill_module(model)
    model.eval()
    rnn = getattr(model, attr)
    x = params.inputs_for(case, shape).requires_grad_(True)
    res = rnn(x.permute(1, 0, 2) if time_major else x)
    y = res[0]
    hs = res[1] if isinstance(res[1], tuple) else (res[1],)
    w = params.inputs_for(case + ":w", y.shape)
    wh = [params.inputs_for(case + f":wh{i}", h.shape) for i, h in enumerate(hs)]
    loss = (y * w).sum() + sum((h * k).sum() for h, k in zip(hs, wh))
    loss.backward()
    arrays = {"y": params.summarize(y), "dx": params.summarize(x.grad), "loss": np.array([loss.item()])}
    for i, h in enumerate(hs):
        arrays[f"state{i}"] = params.summarize(h)
    for n, p in rnn.named_parameters():
        arrays["grad:" + n] = params.summarize(p.grad)
    _save(case, arrays, dict(case=case, ref=ast_loader.FILES[key], cls=cls_name, cfg=cfg, attr=attr,
                             shape=list(shape), time_major=time_major, torch=torch.__version__))


def fuse(case: str, key: str, regression: bool, B: int, T: int) -> None:
    cfg = dict(FUSE)
    if regression:
        cfg["num_classes"] = 1
    loaded = ast_loader.load_classes(key, ["fusion_net", "MyLoss"], extra_globals={"config": cfg})
    model = loaded["fusion_net"](cfg["text_embed_size"], cfg["text_hidden_dims"], cfg["rnn_layers"], cfg["dropout"],
                                 cfg["num_classes"], cfg["audio_hidden_dims"], cfg["audio_embed_size"])
    params.fill_module(model)
    model.eval()
    audio = params.inputs_for(case + ":audio", (B, T, cfg["audio_embed_size"])).numpy()
    text = params.inputs_for(case + ":text", (B, T, cfg["text_embed_size"])).numpy()
    x = [[audio[i], text[i]] for i in range(B)]                      # fuse_net_whole.py:429-436
    if regression:
        y = (params.inputs_for(case + ":target", (B,)).abs() * 10).numpy().tolist()
    else:
        y = params.labels_for(case, B).numpy().tolist()
    text_feature, audio_feature = model.pretrained_feature(x)
    concat = torch.cat((text_feature, audio_feature), dim=1)          # fuse_net_whole.py:445
    out = model(concat)
    loss = loaded["MyLoss"]()(text_feature, audio_feature, y, model)
    loss.backward()
    arrays = {"text_feature": text_feature.numpy(), "audio_feature": audio_feature.numpy(),
              "out": out.detach().numpy(), "loss": np.array([loss.item()]), "target": np.asarray(y)}
    arrays.update(_grads(model))
    _save(case, arrays, dict(case=case, ref=ast_loader.FILES[key], cfg=cfg, B=B, T=T, regression=regression,
                             torch=torch.__version__))


def live_forward(case: str, key: str, cls_name: str, cfg: dict, shape, head: str) -> None:
    """The reference class's eval() forward and its parameter names, for checking the restated class against it.
    Also records the forward with the head's final activation removed: a regression head's ReLU maps every row of
    some of these cases to 0, which alone would pin nothing."""
    cls = ast_loader.load_classes(key, [cls_name])[cls_name]
    torch.manual_seed(0)
    model = cls(cfg)
    params.fill_module(model)
    model.eval()
    x = params.inputs_for(case, shape)
    with torch.no_grad():
        out = model(x)
        getattr(model, head)[-1] = nn.Identity()
        pre = model(x)
    _save(case, {"out": out.numpy(), "pre_activation": pre.numpy()},
          dict(case=case, ref=ast_loader.FILES[key], cls=cls_name, cfg=cfg, shape=list(shape), head=head,
               names=[n for n, _ in model.named_parameters()], torch=torch.__version__))


def dropin_build(case: str) -> None:
    """What the reference's classes construct once ``b200rnn.install()`` has rebound nn.GRU / nn.LSTM: the recurrent
    module's class, every parameter's name and shape, and which parameters the reference's own init leaves at 0."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                    "icassp2022-depression_b200"))
    import b200rnn

    built = {}
    try:
        b200rnn.install()
        for key, cls_name, cfg, attr in (("audio_clf", "AudioBiLSTM", AUDIO_CLF, "lstm_net_audio"),
                                         ("text_clf", "TextBiLSTM", TEXT_CLF, "lstm_net")):
            torch.manual_seed(0)
            model = ast_loader.load_classes(key, [cls_name])[cls_name](cfg)
            rnn = getattr(model, attr)
            built[key] = dict(
                ref=ast_loader.FILES[key], cls=cls_name, attr=attr,
                rnn_class=f"{type(rnn).__module__}.{type(rnn).__qualname__}",
                params=[[n, list(p.shape)] for n, p in model.named_parameters()],
                zero=[n for n, p in model.named_parameters() if float(p.detach().abs().max()) == 0.0])
    finally:
        b200rnn.uninstall()
    _save(case, {}, dict(case=case, built=built, torch=torch.__version__))


def main() -> None:
    if not ast_loader.available():
        raise SystemExit("reference tree not found; set B200RNN_REFERENCE_ROOT to its DepressionCollected directory")
    torch.set_num_threads(1)
    single_modal("audio_clf_b3_t5", "audio_clf", "AudioBiLSTM", AUDIO_CLF, (3, 5, 256), "ce")
    single_modal("text_clf_b3_t6", "text_clf", "TextBiLSTM", TEXT_CLF, (3, 6, 1024), "ce")
    single_modal("audio_reg_b2_t3", "audio_reg", "AudioBiLSTM", AUDIO_REG, (2, 3, 256), "l1")
    single_modal("text_reg_b2_t3", "text_reg", "TextBiLSTM", TEXT_REG, (2, 3, 1024), "smoothl1")
    # BASELINE.json configs[0]: text_bilstm_whole forward, batch=1, T=32, 1024-d, hidden=128
    single_modal("c1_text_b1_t32", "text_clf", "TextBiLSTM", TEXT_CLF, (1, 32, 1024), "ce")
    rnn_boundary("gru_boundary_b5_t24", "audio_clf", "AudioBiLSTM", AUDIO_CLF, "lstm_net_audio", (5, 24, 256), False)
    rnn_boundary("lstm_boundary_b5_t17", "text_clf", "TextBiLSTM", TEXT_CLF, "lstm_net", (5, 17, 1024), True)
    fuse("fuse_clf_b3_t3", "fuse_clf", False, 3, 3)
    fuse("fuse_reg_b3_t3", "fuse_reg", True, 3, 3)
    live_forward("live_audio_clf_b4_t6", "audio_clf", "AudioBiLSTM", AUDIO_CLF, (4, 6, 256), "fc_audio")
    live_forward("live_text_clf_b4_t6", "text_clf", "TextBiLSTM", TEXT_CLF, (4, 6, 1024), "fc_out")
    live_forward("live_audio_reg_b4_t3", "audio_reg", "AudioBiLSTM", AUDIO_REG, (4, 3, 256), "fc_audio")
    live_forward("live_text_reg_b4_t3", "text_reg", "TextBiLSTM", TEXT_REG, (4, 3, 1024), "fc_out")
    dropin_build("dropin_build")


if __name__ == "__main__":
    main()
