#!/usr/bin/env python
"""Recurrence and module times across hidden sizes, against cuDNN at the same shapes.

    python tools/hidden_sweep.py [--out FILE] [--iters N] [--warmup W]

Shapes: H in {64, 128, 256, 512} x B in {8, 64, 128} for
  * gru    : 2-layer GRU, input 256, T = 120 (the audio encoder of audio_gru_whole.py)
  * bilstm : 2-layer BiLSTM, input 1024, T = 30 (the text encoder of text_bilstm_whole.py)
Per shape, eager forward + backward of the whole module (loss = sum(y * w)):
  * rec_fwd_us / rec_bwd_us : mean duration of one recurrence launch (one layer, all directions), CUDA events recorded
    by the library around each launch (b200rnn_profile);
  * module_ms               : one forward + backward of the b200rnn module, CUDA events, profiling off;
  * cudnn_ms                : the same for torch.nn.GRU / nn.LSTM(...).cuda() (cuDNN).
One JSON line per shape (stdout, and appended to --out), each with the card name and power limit read at start.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "icassp2022-depression_b200"))
import b200rnn  # noqa: E402
from b200rnn import _lib  # noqa: E402

SHAPES = {"gru": dict(I=256, T=120, bi=False), "bilstm": dict(I=1024, T=30, bi=True)}


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    name, power, clk = [s.strip() for s in q.split(",")] if q.count(",") == 2 else (torch.cuda.get_device_name(0), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def time_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def run_shape(kind, H, B, iters, warmup):
    s = SHAPES[kind]
    I, T, bi = s["I"], s["T"], s["bi"]
    torch.manual_seed(0)
    dev = torch.device("cuda:0")
    ref = (torch.nn.GRU if kind == "gru" else torch.nn.LSTM)(I, H, num_layers=2, bidirectional=bi, batch_first=True)
    mine = b200rnn.from_torch(ref).to(dev).train()
    cudnn = ref.to(dev).train()
    x = torch.randn(B, T, I, device=dev, requires_grad=True)
    w = torch.randn(B, T, (2 if bi else 1) * H, device=dev)

    def step(m):
        def f():
            x.grad = None
            for p in m.parameters():
                p.grad = None
            (m(x)[0] * w).sum().backward()
        return f

    f_mine, f_ref = step(mine), step(cudnn)
    module_ms = time_ms(f_mine, iters, warmup)
    cudnn_ms = time_ms(f_ref, iters, warmup)
    _lib.profile(True)
    for _ in range(iters):
        f_mine()
    fwd_ms, nf = _lib.profile_read(_lib.PROF_REC_FWD)
    bwd_ms, nb = _lib.profile_read(_lib.PROF_REC_BWD)
    _lib.profile(False)
    # the same work again with profiling off, interleaved, to see the spread of the module timing
    module_ms2 = time_ms(f_mine, iters, 1)
    return {"kind": kind, "H": H, "B": B, "T": T, "I": I, "layers": 2, "bidirectional": bi,
            "rec_fwd_us": round(1e3 * fwd_ms / max(nf, 1), 2), "rec_bwd_us": round(1e3 * bwd_ms / max(nb, 1), 2),
            "rec_launches": [nf, nb], "module_ms": round(module_ms, 4), "module_ms_repeat": round(module_ms2, 4),
            "cudnn_ms": round(cudnn_ms, 4), "cudnn_enabled": torch.backends.cudnn.enabled}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--kinds", default="gru,bilstm")
    ap.add_argument("--sizes", default="64,128,256,512")
    ap.add_argument("--batches", default="8,64,128")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "hidden_sweep.py measures on a CUDA device"
    info = card()
    for kind in a.kinds.split(","):
        for H in [int(v) for v in a.sizes.split(",")]:
            for B in [int(v) for v in a.batches.split(",")]:
                row = dict(info, **run_shape(kind, H, B, a.iters, a.warmup))
                line = json.dumps(row)
                print(line, flush=True)
                if a.out:
                    with open(a.out, "a") as f:
                        f.write(line + "\n")


if __name__ == "__main__":
    main()
