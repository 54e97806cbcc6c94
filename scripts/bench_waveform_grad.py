"""A perceptual-loss training step through a frozen encoder: the waveform gradient of `JEPA.get_audio_representation`.

    python scripts/bench_waveform_grad.py [--batch 256] [--w2v2-batch 128] [--steps 5] [--warmup 2] [--out FILE]

Workload (DESIGN.md 2.3): WavJEPA-base with every parameter frozen; in front of it a trainable residual enhancer
x + nn.Conv1d(1, 1, 33, padding=16)(x), small so that the encoder dominates.  One step: features(clean) under no_grad,
features(enhancer(noisy)), MSE between them, backward (through the whole encoder down to conv block 0's data gradient),
torch.optim.AdamW on the enhancer.  Geometries as scripts/bench_finetune.py: base (B = --batch x 2.01 s dense) and the
wav2vec2 extractor (B = --w2v2-batch x 4.02 s).

Rows per geometry, in one process:
  frozen             the step above (data-gradient-only backward);
  encoder_trainable  the same step with every encoder parameter requires_grad=True (its weight gradients are computed
                     and dropped, the optimizer still steps the enhancer only): the weight-gradient work the frozen
                     backward avoids;
  baseline           the oracle restatement (oracle/jepa_oracle.py local_features + run_stack), frozen, eager under
                     bf16 autocast on the same GPU.
Per row: ms/step (CUDA events, median of --steps after --warmup), instances/s, peak allocated memory.  For the two
native rows, from one separately profiled step: GEMM FLOPs counted from the GEMM launch shapes and the GEMM kernels' own
time, and the time of conv block 0's data-gradient entry point (wj_conv0_gn_gelu_bwd_dx: its two passes over dY and the
overlap-add)."""
import argparse
import json
import os
import subprocess
import sys

os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import wavjepa_b200 as w  # noqa: E402
from wavjepa_b200 import _lib, hear  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

GEMM_ENTRY_POINTS = ("wj_gemm_bf16", "wj_gemm_wgrad_bf16", "wj_gemm_dgrad_bf16")
CONV0_DX = "wj_conv0_gn_gelu_bwd_dx"


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def build(cfg: jo.Cfg, seconds: float, dev):
    ex = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=1)
    m = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
               transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
               process_audio_seconds=seconds)
    m.load_state_dict(jo.make_state_dict(cfg, seed=3), strict=True)
    return m.to(dev).requires_grad_(False)


def enhancer(dev):
    torch.manual_seed(0)
    e = torch.nn.Conv1d(1, 1, 33, padding=16)
    torch.nn.init.normal_(e.weight, std=1e-3)
    torch.nn.init.zeros_(e.bias)
    return e.to(dev)


def make_step(features, enh, clean, noisy, after_backward=None):
    opt = torch.optim.AdamW(enh.parameters(), lr=1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.no_grad():
            target = features(clean)
        loss = F.mse_loss(features(noisy + enh(noisy)), target)
        loss.backward()
        if after_backward is not None:
            after_backward()
        opt.step()
        return loss
    return step


def timed(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    times = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return times, torch.cuda.max_memory_allocated()


def profile(step):
    with _lib.KernelProfile() as kp:
        step()
    torch.cuda.synchronize()
    g_ms = flops = c_ms = 0.0
    n_conv0 = 0
    for name, e0, e1, meta, _ in kp.records:
        if name in GEMM_ENTRY_POINTS:
            g_ms += e0.elapsed_time(e1)
            flops += meta[0]
        elif name == CONV0_DX:
            c_ms += e0.elapsed_time(e1)
            n_conv0 += 1
    return flops, g_ms, c_ms, n_conv0


def row_of(times, peak, B):
    ms = float(np.median(times))
    return {"ms_per_step": round(ms, 2), "ms_all": [round(t, 2) for t in times],
            "instances_per_s": round(B / (ms / 1e3), 1), "peak_allocated_gib": round(peak / 2**30, 2)}


def run_geometry(name, cfg, seconds, B, args, dev):
    g = torch.Generator().manual_seed(1)
    clean = (torch.randn(B, 1, cfg.target_length, generator=g) * 0.3).to(dev)
    noisy = clean + 0.1 * torch.randn(B, 1, cfg.target_length, generator=g).to(dev)
    rows = {}
    model = build(cfg, seconds, dev)
    for variant in ("frozen", "encoder_trainable"):
        model.requires_grad_(variant == "encoder_trainable")
        step = make_step(model.get_audio_representation, enhancer(dev), clean, noisy,
                         after_backward=lambda: model.zero_grad(set_to_none=True))
        times, peak = timed(step, args.steps, args.warmup)
        row = row_of(times, peak, B)
        flops, g_ms, c_ms, n_c = profile(step)
        ms = row["ms_per_step"]
        row.update({"gemm_tflop_per_step": round(flops / 1e12, 2),
                    "gemm_kernel_ms": round(g_ms, 2),
                    "gemm_tflop_s_over_gemm_kernel_time": round(flops / 1e9 / g_ms, 1) if g_ms else None,
                    "gemm_tflop_s_over_step_time": round(flops / 1e9 / ms, 1),
                    "conv0_dx_ms": round(c_ms, 3), "conv0_dx_calls": n_c})
        rows[variant] = row
        print(name, variant, json.dumps(row), flush=True)
        del step
        torch.cuda.empty_cache()
    del model
    torch.cuda.empty_cache()
    sd = {k: v.to(dev) for k, v in jo.make_state_dict(cfg, seed=3).items()}

    def eager_features(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return jo.run_stack(jo.local_features(x, sd, cfg), sd, "encoder", cfg.layers, cfg.nhead, None).float()

    bstep = make_step(eager_features, enhancer(dev), clean, noisy)
    btimes, bpeak = timed(bstep, args.baseline_steps, 1)
    rows["baseline"] = {"impl": "oracle restatement (oracle/jepa_oracle.py local_features + run_stack) on CUDA, "
                                "frozen, eager, bf16 autocast", **row_of(btimes, bpeak, B)}
    rows["speedup_vs_baseline"] = round(rows["baseline"]["ms_per_step"] / rows["frozen"]["ms_per_step"], 2)
    rows["encoder_trainable_over_frozen"] = round(rows["encoder_trainable"]["ms_per_step"] /
                                                  rows["frozen"]["ms_per_step"], 2)
    print(name, "baseline", json.dumps(rows["baseline"]), flush=True)
    del bstep, sd
    torch.cuda.empty_cache()
    return {"batch": B, "seconds": seconds, "tokens_per_step": B * cfg.total_patches, "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--w2v2-batch", type=int, default=128)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--baseline-steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    out = {
        "workload": "perceptual-loss step: frozen WavJEPA-base, residual Conv1d(1, 1, 33) enhancer in front; "
                    "features(clean) under no_grad, MSE to features(enhancer(noisy)), backward to the enhancer, "
                    "torch.optim.AdamW on the enhancer; synthetic weights (oracle make_state_dict, seed 3) and seeded "
                    "Gaussian audio, inputs resident in HBM",
        "gpu": gpu_info(),
        "base_2.01s": run_geometry("base", jo.Cfg(), 2.01, args.batch, args, dev),
        "w2v2_4.02s": run_geometry("w2v2", jo.Cfg(spec=hear.W2V2_SPEC, seconds=4.02), 4.02, args.w2v2_batch, args, dev),
    }
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
