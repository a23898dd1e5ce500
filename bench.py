#!/usr/bin/env python
"""bench.py — headline benchmark of the GRU/BiLSTM hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]  # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]  # reference CPU path (oracle port)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      # one rank per GPU, NCCL

Workload (config.workload): ONE fuse_net_whole train step, reference semantics (fuse_net_whole.py:421-465):
  pretrained_feature = audio GRU [B,120,256]->256 (2 layers) + text BiLSTM [B,30,1024]->128 (2 layers, bi) forward
  under no_grad with train-mode dropout, concat, fc_final forward, MyLoss two-head CE, backward (gradient reaches
  fc_final.0.weight only), one gradient all-reduce of the flat bucket, Adam step. B = 128 sequences per GPU
  (BASELINE.json configs[3]; configs[4] = the same at 8 ranks, global batch 1024). Synthetic N(0,1) features.

One JSON line on stdout (rank 0): metric/value = sequences/s with inputs resident in HBM (CUDA-graph replay, CUDA
events, max over ranks); e2e = same metric through the public API from pinned HOST buffers (H2D inside the timed
region, loss read back); roofline = dominant kernel (GRU forward recurrence) vs the measured HBM peak;
cpu_baseline = the oracle port of the reference on this box's host cores; extra = fwd+bwd ms/batch of the
BASELINE c2 / c3 module configs and the end-to-end fine-tune variant of the fuse step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "icassp2022-depression_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def usable_cores() -> int:
    """Host threads this process may really use: affinity mask, capped by the cgroup CPU quota if any."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


# The OpenMP pool must be sized BEFORE torch is imported: a plain `python bench.py` on the GPU box would otherwise
# start os.cpu_count() = 128 intra-op threads inside a 16-core cgroup quota; after the first parallel host copy they
# spin, the cgroup throttles the whole process and the launching thread with it (round-1 N=1 e2e: 1.21-1.36 ms/step
# against 0.90 with OMP_NUM_THREADS=1, profiles/README.md). torchrun sets OMP_NUM_THREADS=1 itself, which is why
# only the N=1 line showed it.
os.environ.setdefault("OMP_NUM_THREADS", str(usable_cores()))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "sequences/sec (fuse_net_whole train step)"
UNIT = "sequences/s"
B_PER_GPU = 128
T_AUDIO, E_AUDIO, H_AUDIO = 120, 256, 256
T_TEXT, E_TEXT, H_TEXT = 30, 1024, 128
FUSE_ARGS = dict(text_embed_size=E_TEXT, text_hidden_dims=H_TEXT, rnn_layers=2, dropout=0.3, num_classes=2,
                 audio_hidden_dims=H_AUDIO, audio_embed_size=E_AUDIO)   # fuse_net_whole.py:398-414
LR = 8e-6                                                               # fuse_net_whole.py:406, 416
N_ROTATE = 4  # distinct resident input batches; 4 x 31.5 MB of inputs + per-step intermediates > 126 MB L2


_REAL_STDOUT_FD = None


def _protect_stdout() -> None:
    """The contract is ONE JSON line on stdout; libraries (NCCL prints its version banner there) must not add to it.
    fd 1 is pointed at stderr for the life of the process; the JSON goes to the saved descriptor."""
    global _REAL_STDOUT_FD
    if _REAL_STDOUT_FD is None:
        sys.stdout.flush()
        _REAL_STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    fd = _REAL_STDOUT_FD if _REAL_STDOUT_FD is not None else 1
    os.write(fd, data)


def _log(msg: str) -> None:
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def _config(n_gpus: int) -> dict:
    return {
        "workload": ("fuse_net_whole train step, reference semantics (GRU[B,120,256]x2L + BiLSTM[B,30,1024,H128]x2L "
                     "forward under no_grad with train-mode dropout 0.3, fc_final fwd/bwd, MyLoss, Adam), "
                     "BASELINE.json configs[3]" + ("/[4]" if n_gpus > 1 else "")),
        "batch_per_gpu": B_PER_GPU,
        "global_batch": B_PER_GPU * n_gpus,
        "parallelism": f"dp{n_gpus}",
        "allreduce_bytes": 2 * (H_TEXT + H_AUDIO) * 4,
        "l2": f"inputs rotate over {N_ROTATE} resident batches (working set > 126 MB L2); no explicit flush",
    }


def _synthetic(B: int, seed: int):
    g = torch.Generator().manual_seed(seed)
    audio = torch.randn(B, T_AUDIO, E_AUDIO, generator=g)
    text = torch.randn(B, T_TEXT, E_TEXT, generator=g)
    labels = torch.randint(0, 2, (B,), generator=g)
    return audio, text, labels


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: oracle port of the reference on the host cores
# ------------------------------------------------------------------------------------------------
def _cpu_reference_steps(steps: int, warmup: int, with_list_conversion: bool = False, budget_s: float = 60.0):
    """Time the reference's CPU path for the same train step. Returns (seq/s, ms/step, cores, steps_done).

    Bounded: the step count is cut so that the whole call stays within ``budget_s`` seconds.
    """
    from oracle import ref_models

    cores = usable_cores()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = ref_models.RefFusion(**FUSE_ARGS)
    for p in model.parameters():                       # fuse_net_whole.py:590-593
        p.requires_grad = False
    model.fc_final[0].weight.requires_grad = True
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=LR)
    audio, text, labels = _synthetic(B_PER_GPU, 1234)
    pairs = [[audio[i].numpy(), text[i].numpy()] for i in range(B_PER_GPU)] if with_list_conversion else None

    def step():
        opt.zero_grad()
        if with_list_conversion:
            tf, af = model.pretrained_feature(pairs)
        else:
            tf, af = model.pretrained_feature_tensors(audio, text)
        out = model(torch.cat((tf, af), dim=1))
        loss = ref_models.ref_fusion_loss(tf, af, labels, model)
        loss.backward()
        opt.step()
        return out, loss

    tw = time.perf_counter()
    for _ in range(max(1, warmup)):
        step()
    per = (time.perf_counter() - tw) / max(1, warmup)
    steps = max(1, min(steps, int((budget_s - per * max(1, warmup)) / max(per, 1e-3))))
    _log(f"cpu reference: {cores} threads, warm-up step {per * 1e3:.0f} ms, timing {steps} steps"
         + (" (with list->tensor conversion)" if with_list_conversion else ""))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return B_PER_GPU * steps / dt, dt / steps * 1e3, cores, steps


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 40))
    warmup = max(1, min(args.warmup, 5))
    v, ms, cores, steps = _cpu_reference_steps(steps, warmup, budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": _config(args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{steps} full train steps of B={B_PER_GPU} (oracle/ref_models.RefFusion on stock "
                                   f"torch.nn.GRU/LSTM CPU, torch {torch.__version__}, {cores} threads, inputs already "
                                   "torch tensors; rank 0 only)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(line)


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


def _max_over_ranks(x: float, dev) -> float:
    if dist.is_initialized() and dist.get_world_size() > 1:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return x


def _barrier():
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _time_module_train(kind: str, dev, iters: int = 20, warmup: int = 5) -> dict:
    """fwd+bwd ms/batch of the BASELINE c2 / c3 model configs (full model step without optimizer)."""
    import b200rnn

    torch.manual_seed(0)
    if kind == "c2":   # audio_gru_whole train: B=64, T=120, 256-d, H=256
        cfg = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=256, hidden_dims=256, learning_rate=6e-6)
        model = b200rnn.AudioBiLSTM(cfg).to(dev).train()
        x = torch.randn(64, 120, 256, device=dev, requires_grad=True)
    else:              # text_bilstm_whole train: B=64, T=30, 1024-d, H=256
        cfg = dict(num_classes=2, dropout=0.5, rnn_layers=2, embedding_size=1024, hidden_dims=256, learning_rate=1e-5,
                   bidirectional=True)
        model = b200rnn.TextBiLSTM(cfg).to(dev).train()
        x = torch.randn(64, 30, 1024, device=dev, requires_grad=True)
    y = torch.randint(0, 2, (64,), device=dev)
    crit = torch.nn.CrossEntropyLoss()

    def step():
        loss = crit(model(x), y)
        loss.backward()

    # warm-up (allocates .grad buffers), then capture forward+backward into one CUDA graph; grads accumulate in
    # place across replays (zeroing them is an optimiser-side memset and is left out of "fwd+bwd")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    mode = "CUDA graph"
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step()
        run = g.replay
    except Exception as exc:
        _log(f"{kind}: graph capture of fwd+bwd failed ({type(exc).__name__}); timing eager launches")
        torch.cuda.synchronize()
        run, mode = step, "eager"
    for _ in range(warmup):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    res = {"fwd_bwd_ms_per_batch": ms, "sequences_per_s": 64 / ms * 1e3,
           "mode": mode + ", train mode (dropout on), dx computed, full model incl. loss"}
    del run
    # the whole train() body of the script (audio_gru_whole.py:161-201): zero_grad -> forward -> Softmax+CE ->
    # backward (dx too) -> AdamW with the reference's two parameter groups, one CUDA graph (b200rnn.TrainStep)
    try:
        lr = cfg["learning_rate"]
        opt = b200rnn.FlatAdamW.like_reference(model, lr=lr, weight_decay=1e-5)
        ts = b200rnn.TrainStep(model, opt, tuple(x.shape))
        ts.warmup_and_capture()
        xs, ys = x.detach(), y
        for _ in range(warmup):
            ts.step(xs, ys)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            ts.step(xs, ys)
        e1.record()
        torch.cuda.synchronize()
        ms2 = e0.elapsed_time(e1) / iters
        res["train_step_ms_per_batch"] = ms2
        res["train_step_sequences_per_s"] = 64 / ms2 * 1e3
        res["train_step_mode"] = ("b200rnn.TrainStep: zero_grad + fwd + fused Softmax/CrossEntropy + bwd + FlatAdamW "
                                  "(2 groups, wd 1e-5 / 0) in one CUDA graph; includes the input copy into the graph's "
                                  "static buffers; final loss %.6f" % float(ts.loss_value.item()))
    except Exception as exc:  # noqa: BLE001
        _log(f"{kind}: TrainStep timing failed: {type(exc).__name__}: {exc}")
        torch.cuda.synchronize()
    return res


def _parity_check(model, fused, dev) -> dict:
    """Checker leg (not timed, not shipped): the benched object at the benched size against the CPU oracle.

    ``FusedFuseStep.features`` + logits in ``eval()`` (dropout streams cannot match bit for bit in train mode) on one
    B=128 batch vs ``oracle.ref_models.RefFusion`` (stock torch.nn.GRU/LSTM on CPU = the reference's arithmetic,
    fuse_net_whole.py:336-374) with the same state_dict. tests/test_gpu_fuse_parity.py runs the full three-step
    version (loss, Adam update, train mode with p=0, all-grads variant).
    """
    from oracle import ref_models

    ref = ref_models.RefFusion(**FUSE_ARGS)
    ref.load_state_dict({k: v.detach().cpu() for k, v in model.state_dict().items()})
    ref.eval()
    audio, text, labels = _synthetic(B_PER_GPU, 4321)
    was_training = model.training
    model.eval()
    try:
        with torch.no_grad():
            tf_r, af_r = ref.pretrained_feature_tensors(audio, text)
            w = ref.fc_final[0].weight
            logits_r = torch.cat((tf_r, af_r), dim=1) @ w.t()
            loss_r = ref_models.ref_fusion_loss(tf_r, af_r, labels, ref)
            tf_m, af_m = fused.features(__import__("b200rnn").FuseBatch(audio.to(dev), text.to(dev)))
            torch.cuda.synchronize()
            tf_m, af_m = tf_m.cpu(), af_m.cpu()
            logits_m = torch.cat((tf_m, af_m), dim=1) @ w.t()
            loss_m = ref_models.ref_fusion_loss(tf_m, af_m, labels, ref)
    finally:
        model.train(was_training)
    out = {
        "against": "oracle.ref_models.RefFusion (stock torch.nn.GRU/LSTM, CPU), same weights, eval(), B=128 T=120/30",
        "features_max_abs": max((tf_m - tf_r).abs().max().item(), (af_m - af_r).abs().max().item()),
        "logits_max_abs": (logits_m - logits_r).abs().max().item(),
        "loss_abs": abs(loss_m.item() - loss_r.item()),
        "tolerance_logits": 1e-4,
    }
    out["ok"] = bool(out["logits_max_abs"] <= 1e-4 and out["features_max_abs"] <= 1e-4)
    return out


def _cudnn_comparator(dev, iters: int = 20, warmup: int = 5) -> dict:
    """Same-box yardstick (SURVEY.md 2.2): stock torch.nn.GRU / nn.LSTM on CUDA = cuDNN's RNN, same shapes as the
    encoders of the fuse step (and of BASELINE c2/c3), forward and forward+backward, CUDA-graph replay, next to this
    library's modules timed the same way. A library call - reported, not part of any headline number."""
    import b200rnn

    shapes = [("gru_fuse_B128_T120_I256_H256", "gru", 128, 120, 256, 256, False),
              ("bilstm_fuse_B128_T30_I1024_H128", "lstm", 128, 30, 1024, 128, True),
              ("gru_c2_B64_T120_I256_H256", "gru", 64, 120, 256, 256, False),
              ("bilstm_c3_B64_T30_I1024_H256", "lstm", 64, 30, 1024, 256, True)]
    out = {}

    def timed(fn):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        for _ in range(warmup):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        del g
        return e0.elapsed_time(e1) / iters

    for name, kind, B, T, I, H, bi in shapes:
        torch.manual_seed(0)
        cls = torch.nn.GRU if kind == "gru" else torch.nn.LSTM
        stock = cls(I, H, num_layers=2, bidirectional=bi, batch_first=True).to(dev)
        mine = b200rnn.from_torch(stock).to(dev)
        x = torch.randn(B, T, I, device=dev)
        xg = x.clone().requires_grad_(True)
        row = {}
        for label, mod in (("cudnn", stock), ("b200rnn", mine)):
            mod.eval()
            with torch.no_grad():
                row[label + "_fwd_ms"] = timed(lambda: mod(x))
            mod.train()   # dropout = 0: train mode only switches the saved-for-backward stores on

            def fb():
                y = mod(xg)[0]
                y.sum().backward()

            try:
                row[label + "_fwd_bwd_ms"] = timed(fb)
            except Exception as exc:  # noqa: BLE001
                row[label + "_fwd_bwd_ms"] = None
                _log(f"cudnn comparator {name} {label} fwd+bwd failed: {type(exc).__name__}: {exc}")
                torch.cuda.synchronize()
        out[name] = row
    out["note"] = ("stock torch.nn.GRU/LSTM(...).cuda() (cuDNN RNN, fp32, TF32 off by torch default) vs b200rnn modules; "
                   "2 layers, batch_first, CUDA-graph replay, dropout 0; fwd = eval no_grad, fwd_bwd = y.sum().backward()")
    return out


def run_ours(args) -> None:
    import b200rnn
    from b200rnn import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this implementation has no CPU path (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.set_num_threads(1)   # the timed loops are launch loops: no intra-op pool spinning beside them (see top)
    # pin the rank to the CPUs / memory of its GPU's NUMA node before any pinned buffer exists (8 ranks on a 2-socket box:
    # 0.813 -> 0.773 ms/step device-resident, 0.877 -> 0.808 ms/step end-to-end)
    numa = b200rnn.bind_host_thread_to_gpu_numa_node(dev)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    n_gpus = world
    K, W = args.steps, max(args.warmup, 3)

    # ---- model (reference construction + freezing, fuse_net_whole.py:413-416, 590-593) --------------------
    torch.manual_seed(0)
    model = b200rnn.fusion_net(**FUSE_ARGS).to(dev)
    for p in model.parameters():
        p.requires_grad = False
    model.fc_final[0].weight.requires_grad = True
    b200rnn.broadcast_parameters(model)
    model.train()
    criterion = b200rnn.MyLoss(text_hidden_dims=H_TEXT)
    fused, bucket = None, None
    if args.generic_head:   # PyTorch shells around the encoders: attention, MLP heads, MyLoss, autograd, torch Adam
        bucket = b200rnn.GradBucket(model)
        opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=LR, capturable=True)
    else:                   # the same step on the library's fused head kernel (b200rnn.FusedFuseStep): the gradient
        #                     exchange across ranks happens inside that kernel over NVLink peer stores ("peer") or,
        #                     with --exchange nccl, as a separate ncclAllReduce + Adam launch
        fused = b200rnn.FusedFuseStep(model, lr=LR, exchange=args.exchange, concurrent_branches=not args.one_stream,
                                      allow_fallback=True)   # no CUDA IPC peer mapping -> ncclAllReduce, all ranks together
        _log(f"rank {rank}: gradient exchange = {fused.exchange}; numa binding {numa}")

    # ---- synthetic shards: rank r owns its own 128 sequences of the global batch (weak scaling) -------
    host = [_synthetic(B_PER_GPU, 1234 + 100 * rank + i) for i in range(N_ROTATE)]
    dev_in = [(a.to(dev), t.to(dev), y.to(dev)) for a, t, y in host]
    loss_buf = torch.zeros((), device=dev)

    def train_step(audio, text, labels, loss_out=None):
        loss_out = loss_buf if loss_out is None else loss_out
        if fused is not None:
            out, loss = fused(b200rnn.FuseBatch(audio, text), labels)   # includes the gradient exchange and Adam
            loss_out.copy_(loss)
            return out
        bucket.zero()
        tf, af = model.pretrained_feature(b200rnn.FuseBatch(audio, text))
        out = model(torch.cat((tf, af), dim=1))
        loss = criterion(tf, af, labels, model)
        loss.backward()
        bucket.allreduce()
        opt.step()
        loss_out.copy_(loss.detach())
        return out

    _log(f"rank {rank}/{world}: model built, host cores usable {usable_cores()} (os.cpu_count {os.cpu_count()})")
    parity = None
    if rank == 0 and fused is not None and not args.no_parity:
        parity = _parity_check(model, fused, dev)
        _log("parity vs CPU oracle: " + json.dumps(parity))
    _barrier()
    # ---- eager warm-up (also counts this library's launches per step) -------------------------------
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        train_step(*dev_in[0])
        c0 = _lib.launch_count()
        train_step(*dev_in[1])
        launches_per_step = _lib.launch_count() - c0
        train_step(*dev_in[2])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()

    # ---- capture one CUDA graph per resident input batch ---------------------------------------------
    graphs, graph_outs, use_graph = [], [], not args.no_graph
    if use_graph:
        try:
            pool = None
            for i in range(N_ROTATE):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    graph_outs.append(train_step(*dev_in[i]))
                pool = g.pool()
                graphs.append(g)
        except Exception as exc:  # e.g. NCCL capture unsupported: fall back to eager launches
            if rank == 0:
                print(f"[bench] CUDA-graph capture failed ({type(exc).__name__}: {exc}); running eager", file=sys.stderr)
            use_graph, graphs, graph_outs = False, [], []
            torch.cuda.synchronize()

    def run_step(i: int):
        """One train step; returns the model output tensor the step wrote (a graph's static output when replayed)."""
        if use_graph:
            graphs[i % N_ROTATE].replay()
            return graph_outs[i % N_ROTATE]
        return train_step(*dev_in[i % N_ROTATE])

    _log(f"graphs captured: {use_graph}; launches/step {launches_per_step}")
    # ---- (A) device-resident throughput: W warm-up + exactly K timed steps ----------------------------
    for i in range(W):
        run_step(i)
    sampler = ClockSampler(local_rank)
    _barrier()
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _barrier()
    e0.record()
    for i in range(K):
        out = run_step(W + i)
    e1.record()
    _barrier()
    ms_total = _max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # before the e2e leg below trains the model further
        _dump_outputs(args.dump_outputs, {"out": out, "loss": loss_buf})
    ms_per_step = ms_total / K
    value = B_PER_GPU * n_gpus * K / (ms_total * 1e-3)

    _log(f"device-resident: {ms_per_step:.3f} ms/step, {value:.0f} seq/s")
    # ---- (B) end-to-end through the public API from pinned host buffers ------------------------------
    # double-buffered: H2D of step i+1 (copy stream) overlaps the compute of step i; the loss is read back
    # into pinned memory every step.
    stagers = [b200rnn.PinnedStager((B_PER_GPU, T_AUDIO, E_AUDIO), (B_PER_GPU, T_TEXT, E_TEXT), dev) for _ in range(2)]
    lab_dev = [torch.empty(B_PER_GPU, dtype=torch.int64, device=dev) for _ in range(2)]
    lab_host = [torch.empty(B_PER_GPU, dtype=torch.int64).pin_memory() for _ in range(N_ROTATE)]
    pinned = []
    for i in range(N_ROTATE):
        a = torch.empty(B_PER_GPU, T_AUDIO, E_AUDIO).pin_memory().copy_(host[i][0])
        t = torch.empty(B_PER_GPU, T_TEXT, E_TEXT).pin_memory().copy_(host[i][1])
        lab_host[i].copy_(host[i][2])
        pinned.append((a, t))
    loss_host = torch.zeros(max(K, 1) + W + 4).pin_memory()
    loss_slot = [torch.zeros((), device=dev) for _ in range(2)]   # per staging slot: read back on the copy stream
    e2e_graphs = []
    if use_graph:
        try:
            pool = graphs[0].pool()
            for s in range(2):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    train_step(stagers[s].d_audio, stagers[s].d_text, lab_dev[s], loss_slot[s])
                e2e_graphs.append(g)
        except Exception:
            e2e_graphs = []
    copy_stream = torch.cuda.Stream()
    main = torch.cuda.current_stream()
    in_ready = [torch.cuda.Event() for _ in range(2)]
    in_free = [torch.cuda.Event() for _ in range(2)]

    # Preferred form of the same pipeline: ONE graph per step that contains the step on staging slot s AND, as a parallel
    # branch, the pinned-host -> device copy of the NEXT step's inputs into the other slot, and the loss read-back at its
    # end. No per-step cross-stream events on the launching stream (they cost ~30 us of inter-graph gap per step); the
    # copies are still made every step, from pinned host memory, inside the timed region.
    pf_graphs = []
    loss_pin = [torch.zeros(1).pin_memory() for _ in range(N_ROTATE)]
    if use_graph and N_ROTATE % 2 == 0:
        try:
            pool = graphs[0].pool()
            for k in range(N_ROTATE):
                s, ns, nk = k % 2, (k + 1) % 2, (k + 1) % N_ROTATE
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    cur = torch.cuda.current_stream()
                    copy_stream.wait_stream(cur)
                    with torch.cuda.stream(copy_stream):
                        stagers[ns].d_audio.copy_(pinned[nk][0], non_blocking=True)
                        stagers[ns].d_text.copy_(pinned[nk][1], non_blocking=True)
                        lab_dev[ns].copy_(lab_host[nk], non_blocking=True)
                    train_step(stagers[s].d_audio, stagers[s].d_text, lab_dev[s], loss_slot[s])
                    loss_pin[k].copy_(loss_slot[s].reshape(1), non_blocking=True)
                    cur.wait_stream(copy_stream)
                pf_graphs.append(g)
        except Exception as exc:  # noqa: BLE001
            _log(f"e2e: prefetch-in-graph capture failed ({type(exc).__name__}: {exc}); using the event pipeline")
            pf_graphs = []
            torch.cuda.synchronize()

    def e2e_issue_copy(i: int):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(in_free[s])
            if i >= 2:   # the loss of the step that last used this slot (step i-2): device -> pinned host, every step
                loss_host[i - 2:i - 1].copy_(loss_slot[s].reshape(1), non_blocking=True)
            a, t = pinned[i % N_ROTATE]
            stagers[s].d_audio.copy_(a, non_blocking=True)
            stagers[s].d_text.copy_(t, non_blocking=True)
            lab_dev[s].copy_(lab_host[i % N_ROTATE], non_blocking=True)
            in_ready[s].record(copy_stream)

    def e2e_compute(i: int):
        s = i % 2
        main.wait_event(in_ready[s])
        if e2e_graphs:
            e2e_graphs[s].replay()
        else:
            train_step(stagers[s].d_audio, stagers[s].d_text, lab_dev[s], loss_slot[s])
        in_free[s].record(main)

    for s in range(2):
        in_free[s].record(main)
    total = W + K
    _barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if pf_graphs:
        e2e_issue_copy(0)                       # inputs of step 0; every later step's inputs arrive by the graphs
        main.wait_stream(copy_stream)
        for i in range(W):
            pf_graphs[i % N_ROTATE].replay()
        _barrier()
        f0.record()
        for i in range(W, total):
            pf_graphs[i % N_ROTATE].replay()
        f1.record()
        _barrier()
        loss_host[total - 1] = loss_pin[(total - 1) % N_ROTATE][0]
    else:
        # warm-up part (untimed), pipeline primed one copy ahead
        e2e_issue_copy(0)
        for i in range(W):
            e2e_issue_copy(i + 1)
            e2e_compute(i)
        _barrier()
        f0.record()
        for i in range(W, total):
            if i + 1 < total:
                e2e_issue_copy(i + 1)
            e2e_compute(i)
        # the last two losses are still on the device: read them back inside the timed region as well
        with torch.cuda.stream(copy_stream):
            for i in (total - 2, total - 1):
                if i >= 0:
                    copy_stream.wait_event(in_free[i % 2])
                    loss_host[i:i + 1].copy_(loss_slot[i % 2].reshape(1), non_blocking=True)
        main.wait_stream(copy_stream)
        f1.record()
        _barrier()
    # the H2D of the first timed step was issued before f0; charge it by adding one exposed copy time below
    e2e_ms = _max_over_ranks(f0.elapsed_time(f1), dev)
    h2d_bytes = stagers[0].h2d_bytes + B_PER_GPU * 8
    tcp0, tcp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tcp0.record()
    e2e_issue_copy(0)
    main.wait_stream(copy_stream)
    tcp1.record()
    torch.cuda.synchronize()
    one_copy_ms = tcp0.elapsed_time(tcp1)
    e2e_ms_total = e2e_ms + _max_over_ranks(one_copy_ms, dev)
    e2e_value = B_PER_GPU * n_gpus * K / (e2e_ms_total * 1e-3)
    final_loss = float(loss_host[total - 1])

    _log(f"e2e: {e2e_ms_total / K:.3f} ms/step, {e2e_value:.0f} seq/s (one H2D alone {one_copy_ms:.3f} ms)")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": _config(n_gpus),
        "cuda_graph": bool(use_graph),
        "shells": "fused head kernel (b200rnn.FusedFuseStep)" if fused is not None else "PyTorch ops",
        "encoder_branches": ("two streams (audio high priority)" if (fused is not None and fused.concurrent_branches)
                             else "one stream"),
        "numa_binding": numa,
        "grad_exchange": (fused.exchange if fused is not None else ("nccl" if world > 1 else "none")),
        "gpu_launches": int(launches_per_step * K),
        "gpu_launches_per_step": int(launches_per_step),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms_total / K, "h2d_ms_alone": one_copy_ms,
                "how": ("one CUDA graph per step = the step on staging slot s + (parallel branch) the pinned-host -> device "
                        "copy of the next step's inputs into the other slot + the loss read-back to pinned memory; "
                        if pf_graphs else
                        "pinned host -> device copies double-buffered on a copy stream with events, graph replay of the "
                        "step, every step's loss copied back to pinned memory on the copy stream; ") +
                       "first copy of the timed region added unoverlapped",
                "final_loss": final_loss},
    }

    finetune = None
    if not args.quick:   # every rank: the fine-tune variant all-reduces its 10.46 MB gradient bucket
        try:
            finetune = _finetune_variant(dev, world)
            _log(f"fine-tune variant: {finetune['ms_per_step']:.3f} ms/step")
        except Exception as exc:  # noqa: BLE001
            _log(f"fine-tune variant failed: {type(exc).__name__}: {exc}")
            finetune = {"error": f"{type(exc).__name__}: {exc}"}
    if rank == 0:
        line["clocks"] = clocks
        line["parity"] = parity
        # ---- roofline of the dominant kernel: forward GRU recurrence (2 launches per step) --------------
        hbm_peak, peak_src = _peaks()
        x_a = dev_in[0][0]
        with torch.no_grad():
            for _ in range(3):
                model.lstm_net_audio(x_a)
            torch.cuda.synchronize()
            _lib.profile(True)
            reps = 10
            for i in range(reps):
                model.lstm_net_audio(dev_in[i % N_ROTATE][0])
            torch.cuda.synchronize()
            rec_ms, rec_n = _lib.profile_read(_lib.PROF_REC_FWD)
            gemm_ms, gemm_n = _lib.profile_read(_lib.PROF_GEMM)
            _lib.profile(False)
        B, T, I, H = B_PER_GPU, T_AUDIO, E_AUDIO, H_AUDIO
        p_layer = 3 * H * I + 3 * H * H + 6 * H
        alg_bytes = 4 * (B * T * I + p_layer + B * T * H)      # SURVEY.md §8(d): read layer input, params once, write output
        alg_flops = 2 * B * T * 3 * H * H                       # recurrent contraction of this launch
        t_launch = rec_ms / max(rec_n, 1) * 1e-3
        achieved = alg_bytes / t_launch / 1e9
        traffic = None   # dram bytes per launch from the committed ncu --set full capture of this kernel
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as fh:
                traffic = json.load(fh)["r02_ncu_rec_fwd.csv"]["dram_bytes_per_launch"]
        except Exception:
            pass
        line["roofline"] = {
            "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
            "traffic": traffic, "traffic_source": "profiles/r02_ncu_rec_fwd.csv (one ncu --set full capture of this kernel, "
                                                  "cold L2: includes the x-projection read that is an L2 hit in the real "
                                                  "step; a constant from that capture, not measured by this run)",
            "peak_source": peak_src,
            "kernel": "rec_fwd_kernel<GRU,H=256> (persistent cluster recurrence, one launch per layer)",
            "launch_ms": t_launch * 1e3, "launches_timed": rec_n,
            "algorithmic_bytes_per_launch": alg_bytes,
            "share_of_step": 2 * t_launch * 1e3 / ms_per_step,
            "note": "the recurrence is FFMA/shared-memory bound, not HBM bound (SURVEY.md §7): see ffma",
            "ffma": {"achieved_tflops": alg_flops / t_launch / 1e12, "peak_tflops": 74.5,
                     "frac": alg_flops / t_launch / 1e12 / 74.5,
                     "peak_source": "148 SMs x 128 FMA x 2 x 1.965 GHz (nominal fp32)"},
            "gemm_ms_per_launch": gemm_ms / max(gemm_n, 1),
        }
        # ---- secondary module configs (fwd+bwd ms/batch) and the end-to-end fine-tune variant -----------
        _log(f"roofline pass: rec launch {t_launch * 1e3:.3f} ms x{rec_n}")
        extra = {}
        if finetune is not None:
            extra["c4_finetune_all_grads_B128_per_gpu"] = finetune
        # rank-0-only block: nothing in here may contain a collective
        if not args.quick and world == 1:
            extra["c2_audio_gru_whole_train_B64_T120"] = _time_module_train("c2", dev)
            extra["c3_text_bilstm_whole_train_B64_T30_H256"] = _time_module_train("c3", dev)
            extra["cudnn_comparator"] = _cudnn_comparator(dev)
        line["extra"] = extra
        _log("extras done: " + json.dumps(extra)[:400])
        # ---- CPU baseline on this box's host cores (bounded sample) -----------------------------------
        if n_gpus == 1 and not args.no_cpu_baseline:
            v, ms, cores, nst = _cpu_reference_steps(steps=8, warmup=1, budget_s=30.0)
            v2, ms2, _, _ = _cpu_reference_steps(steps=2, warmup=1, with_list_conversion=True, budget_s=30.0)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{nst} train steps of B={B_PER_GPU} after 1 warm-up ({ms:.0f} ms/step) with the oracle port "
                          f"(oracle/ref_models.py on stock torch.nn CPU kernels, {cores} threads); with the reference's "
                          f"list->tensor conversion (fuse_net_whole.py:343) it is {v2:.1f} seq/s ({ms2:.0f} ms/step)"}
        _emit(line)
    pf_graphs.clear()
    _teardown(graphs, e2e_graphs, world, fused)


def _dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write what the last timed step returned to its caller as ``out_dir/<name>.npy`` in float32, so that two builds
    run with the same arguments (hence the same seeded inputs and weights) can be compared output for output."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    _log(f"outputs of the last timed step written to {out_dir}: {sorted(arrays)}")


def _teardown(graphs, e2e_graphs, world: int, fused=None) -> None:
    """Normal interpreter exit (the driver's exit hook records which .so files this process loaded).

    Round 1 left with os._exit(0) because a 2-rank run once hung in destroy_process_group while captured graphs still
    held NCCL kernels. Order that avoids it: drop the graphs, synchronise, barrier, destroy the group. A watchdog thread
    covers the residual risk without hiding the process from exit hooks: if the teardown has not finished after 30 s it
    runs the registered atexit functions itself and only then leaves hard.
    """
    import atexit
    import threading

    done = threading.Event()

    def watchdog():
        if not done.wait(30.0):
            _log("teardown watchdog: destroy_process_group did not return in 30 s; running exit hooks, leaving hard")
            try:
                atexit._run_exitfuncs()
            finally:
                os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    graphs.clear()
    e2e_graphs.clear()
    torch.cuda.synchronize()
    if fused is not None:
        fused.close()          # flush a deferred update, unmap the peer exchange buffers (barrier inside)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    done.set()
    sys.stdout.flush()
    sys.stderr.flush()


def _finetune_variant(dev, world: int, iters: int = 20, warmup: int = 5) -> dict:
    """fuse step with every parameter trainable and the encoders inside autograd (SURVEY.md §3.3 (b)): BiLSTM + GRU
    forward and BPTT kernels, ONE all-reduce of the 10.46 MB gradient bucket, Adam - one CUDA graph
    (b200rnn.FuseFineTuneStep). Entered by EVERY rank (it contains a collective); time = max over ranks."""
    import b200rnn

    torch.manual_seed(0)
    model = b200rnn.fusion_net(**FUSE_ARGS).to(dev).train()
    b200rnn.broadcast_parameters(model)
    opt = b200rnn.FlatAdamW([{"params": list(model.parameters()), "weight_decay": 0.0}], lr=LR, model=model)
    step = b200rnn.FuseFineTuneStep(model, opt, B_PER_GPU, T_AUDIO, T_TEXT)
    rank = int(os.environ.get("RANK", "0"))
    audio, text, labels = [t.to(dev) for t in _synthetic(B_PER_GPU, 99 + rank)]
    mode = "CUDA graph"
    try:
        step.warmup_and_capture()
    except Exception as exc:  # noqa: BLE001
        _log(f"fine-tune variant: graph capture failed ({type(exc).__name__}: {exc}); eager")
        torch.cuda.synchronize()
        step.use_graph, mode = False, "eager"
    for _ in range(warmup):
        step.step(audio, text, labels)
    _barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step.step(audio, text, labels)
    e1.record()
    _barrier()
    ms = _max_over_ranks(e0.elapsed_time(e1), dev) / iters
    out = {"ms_per_step": ms, "sequences_per_s": B_PER_GPU * world / ms * 1e3, "n_gpus": world,
           "grad_bucket_bytes": opt.nbytes, "allreduce": "one ncclAllReduce over the flat bucket" if world > 1 else "none",
           "final_loss": float(step.loss_value.item()),
           "mode": mode + "; RNN fwd+bwd through the BPTT kernels, all 2,614,016 parameters trainable, FlatAdamW (Adam)"}
    step.graph = None
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly (no CUDA graph)")
    ap.add_argument("--generic-head", action="store_true",
                    help="run the dense shells / loss / Adam as PyTorch ops instead of the fused shell kernels")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the pre-timing parity check against the CPU oracle")
    ap.add_argument("--quick", action="store_true", help="skip the secondary module timings")
    ap.add_argument("--one-stream", action="store_true",
                    help="serialise the audio and text encoder branches on one stream (default: the audio branch runs "
                         "on a second, high-priority stream = parallel branches of the CUDA graph)")
    ap.add_argument("--exchange", choices=["auto", "peer", "peer_async", "nccl", "none"], default="peer_async",
                    help="data-parallel gradient exchange of the fused step: in-kernel NVLink peer stores (peer: wait at "
                         "the end of the step; peer_async: send now, sum + Adam at the start of the next step beside "
                         "the encoders, flushed after the last step) or NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0: model output [B,2] and "
                         "loss) as DIR/out.npy and DIR/loss.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    _protect_stdout()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args)
        return
    if args.gpus != world and world == 1 and args.gpus > 1:
        raise SystemExit(f"--gpus {args.gpus} needs a torchrun launch with {args.gpus} ranks (WORLD_SIZE=1 here)")
    run_ours(args)


if __name__ == "__main__":
    main()
