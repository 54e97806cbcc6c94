"""The denoiser stage's two training paths on the workload of scripts/bench_denoiser.py, one process.

    python scripts/bench_denoiser_autograd.py [--reps 7] [--warmup 2] [--out profiles/r07_bench_denoiser_autograd.json]

Batch: 32 clips x 10 s at 32 kHz with 2 s RIRs -> on_after_batch_transfer -> 512 instances per side (2.01 s, bf16),
alpha = 0.25, random-init weights (student and teacher), global_step 5000.  Four calls, alternated in every repetition
after a warm-up of each, CUDA events around each call, medians over --reps:
  forward_backward    the fused forward + hand-written backward into the flat gradient buffer (no optimizer)
  autograd_fwd_bwd    zero_grad, Denoiser.forward in grad mode, loss.backward()
  train_step          the fused step: forward, backward, clip + AdamW kernel
  stock_step          the Lightning-style step: training_step, loss.backward(), clip_grad_norm_(1.0), torch.optim.AdamW
                      and the LambdaLR of configure_optimizers, zero_grad
Per call: peak allocated memory above the resident state and libwavjepa_b200 launches, each from one extra call that
follows a call of its own kind; the device time of wj_mse_pair / wj_mse_pair_bwd from one profiled autograd call on its
own, with the bytes each must move.  The card's name, power limit and maximum SM clock are read in the same call
(nvidia-smi)."""
import argparse
import json
import os
import subprocess
import sys

os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import wavjepa_b200 as w  # noqa: E402
from wavjepa_b200 import _lib  # noqa: E402
from wavjepa_b200.denoiser import Denoiser  # noqa: E402

SPEC = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def build(dev):
    torch.manual_seed(0)
    m = Denoiser(feature_extractor=w.ConvFeatureExtractor(conv_layers_spec=SPEC, in_channels=1),
                 transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                 transformer_encoder_cfg=w.TransformerEncoderCFG.create(), nr_samples_per_audio=16, alpha=0.25)
    teacher = w.JEPA(feature_extractor=w.ConvFeatureExtractor(conv_layers_spec=SPEC, in_channels=1),
                     transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
                     transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                     transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
                     transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384), process_audio_seconds=2.01)
    m._set_teacher({"state_dict": teacher.state_dict()})
    m.to(dev)
    m.global_step = 5000
    return m


def batch(dev):
    B, T32, R, S = 32, 320000, 64000, 2
    g = torch.Generator(device=dev).manual_seed(0)
    audio = torch.rand(B, T32, device=dev, generator=g) * 2 - 1
    rir = torch.randn(B, 2, R, device=dev, generator=g) * torch.exp(-torch.arange(R, device=dev) / 8000.0) * 0.05
    noise = torch.randn(B, T32, device=dev, generator=g) * 0.3
    nrirs = torch.randn(B, S, 2, R, device=dev, generator=g) * torch.exp(-torch.arange(R, device=dev) / 8000.0) * 0.05
    return (audio, rir, noise, torch.full((B,), T32 // 2, device=dev), torch.full((B,), 1000, device=dev), nrirs,
            torch.full((B,), 10.0, device=dev))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join("profiles", "r07_bench_denoiser_autograd.json"))
    args = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    m = build(dev)
    gen16, clean16 = m.on_after_batch_transfer(batch(dev), 0)
    N = gen16.shape[0]
    conf = m.configure_optimizers()
    opt, sched = conf["optimizer"], conf["lr_scheduler"]["scheduler"]
    params = [p for p in m.parameters() if p.requires_grad]
    # the stock path resumed at the fused path's step: the scheduler's position (its lr) and AdamW's step count
    for p in params:
        opt.state[p] = dict(step=torch.tensor(5000.0), exp_avg=torch.zeros_like(p), exp_avg_sq=torch.zeros_like(p))
    sched.last_epoch = 5000
    for grp in opt.param_groups:
        grp["lr"] = m.lr_at(5000)

    def autograd_fwd_bwd():
        m.zero_grad(set_to_none=True)
        m(gen16, clean16)["loss"].backward()

    def stock_step():
        out = m.training_step((gen16, clean16), 0)
        out["loss"].backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        sched.step()
        opt.zero_grad(set_to_none=True)

    calls = {
        "forward_backward": lambda: m.forward_backward(gen16, clean16),
        "autograd_fwd_bwd": autograd_fwd_bwd,
        "train_step": lambda: m.train_step(gen16, clean16),
        "stock_step": stock_step,
    }
    for _ in range(args.warmup):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    for _ in range(args.reps):
        for k, fn in calls.items():
            times[k].append(event_ms(fn))
    rows = {}
    for k, fn in calls.items():
        fn()      # the counted call follows one of its own kind (the stock step's weight refresh is then its own)
        m.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        n0 = _lib.kernel_launches()
        fn()
        torch.cuda.synchronize()
        ms = float(np.median(times[k]))
        rows[k] = {"ms_median": round(ms, 2), "ms_all": [round(t, 2) for t in times[k]],
                   "instances_per_s": round(N / (ms / 1e3), 1),
                   "peak_allocated_above_resident_gib": round((torch.cuda.max_memory_allocated() - base) / 2**30, 2),
                   "library_launches": int(_lib.kernel_launches() - n0)}
        print(k, json.dumps(rows[k]), flush=True)
    m.zero_grad(set_to_none=True)
    with _lib.KernelProfile() as kp:
        autograd_fwd_bwd()
    prof = kp.summary()
    M = N * m.total_patches * m.encoder_embedding_dim
    loss_kernels = {}
    # bytes the kernels must move: mse_pair reads both feature halves and the targets; its backward also writes
    # the gradient of both halves
    for name, nbytes in (("wj_mse_pair", 12 * M), ("wj_mse_pair_bwd", 20 * M)):
        c, t = prof.get(name, (0, 0.0))
        loss_kernels[name] = {"calls": c, "ms": round(t, 4), "bytes": nbytes,
                              "gb_per_s": round(nbytes / (t / 1e3) / 1e9, 1) if t else None}
    out = {
        "gpu": gpu_info(),
        "workload": f"denoiser stage: 32 clips x 10 s @ 32 kHz -> {N} instances per side (clean + generated) of 2.01 s, "
                    "alpha 0.25, random-init student and teacher, global_step 5000; calls alternated in one process, "
                    "CUDA events, medians",
        "calls": rows,
        "autograd_minus_fused_ms": round(rows["autograd_fwd_bwd"]["ms_median"] - rows["forward_backward"]["ms_median"], 2),
        "stock_minus_fused_step_ms": round(rows["stock_step"]["ms_median"] - rows["train_step"]["ms_median"], 2),
        "loss_kernels_in_one_profiled_autograd_call": loss_kernels,
    }
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
