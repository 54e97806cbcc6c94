"""Whole-clip training steps through the HEAR / HF entry points in training mode (DESIGN.md 2.5).

    python scripts/bench_hear_finetune.py [--batch 32] [--seconds 10] [--steps 10] [--warmup 3] [--out FILE]

Workload: B = --batch clips of --seconds s (16 kHz, seeded uniform noise, resident in HBM), WavJEPA-base with synthetic
weights (oracle make_state_dict, seed 3), 2.01 s chunks (10 s -> 5 chunks, the last one padded).  Rows, in one process:
  hf_finetune     `hf.WavJEPAModel` after .train(): model(input_values) -> scene embedding (mean over frames) ->
                  nn.Linear(768, 10) -> cross-entropy -> backward -> torch.optim.AdamW over the encoder's feature path and
                  the head;
  waveform_grad   the same clips through the frozen model (every parameter requires_grad=False) with the audio
                  requiring grad: scene embedding -> MSE to a fixed target -> backward to the waveform -> one signed
                  gradient step on the audio (input saliency / adversarial-style optimisation of the clip);
  baseline        the fine-tuning step of hf_finetune through the oracle restatement of the HEAR runtime
                  (oracle/jepa_oracle.py hear_timestamp_embeddings: per-clip loudness, chunk loop, fp32 parameters), eager
                  under bf16 autocast on the same GPU.
Per row: ms/step (CUDA events, median of --steps after --warmup), clips/s, peak allocated memory.  From one separately
profiled waveform_grad step (hf_finetune's audio needs no gradient, so its backward stops at the chunks): time and
algorithmic bytes of the two preprocessing backward kernels (wj_crop_norm_bwd, wj_clip_gain_bwd) and of the chunk
forward (wj_crop_norm), as GB/s."""
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

from wavjepa_b200 import _lib, hf  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

PATH = ("extract_audio.", "feature_norms.", "post_extraction_mapper.", "encoder.")
KERNELS = ("wj_crop_norm", "wj_crop_norm_bwd", "wj_clip_gain_bwd")
N_CLASSES = 10


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


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


def row_of(times, peak, B):
    ms = float(np.median(times))
    return {"ms_per_step": round(ms, 2), "ms_all": [round(t, 2) for t in times],
            "clips_per_s": round(B / (ms / 1e3), 1), "peak_allocated_gib": round(peak / 2**30, 2)}


def kernel_rows(step):
    with _lib.KernelProfile() as kp:
        step()
    out = {}
    for name, (calls, ms, nbytes) in kp.hbm_summary().items():
        if name in KERNELS:
            out[name] = {"calls": calls, "ms": round(ms, 4), "algorithmic_MB": round(nbytes / 1e6, 2),
                         "GB_per_s": round(nbytes / 1e6 / ms, 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--baseline-steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    B, L = args.batch, int(args.seconds * 16000)
    g = torch.Generator().manual_seed(1)
    audio = (torch.rand(B, L, generator=g) * 2 - 1).to(dev)
    labels = torch.randint(0, N_CLASSES, (B,), generator=g).to(dev)
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    rows = {}

    # ---- hf_finetune
    model = hf.WavJEPAModel.from_pretrained({"state_dict": sd}).to(dev).train()
    torch.manual_seed(0)
    head = torch.nn.Linear(768, N_CLASSES).to(dev)
    params = [p for n, p in model.runtime.model.named_parameters() if n.startswith(PATH)]
    opt = torch.optim.AdamW([{"params": params, "lr": 1e-5}, {"params": list(head.parameters()), "lr": 1e-3}])

    def finetune_step():
        opt.zero_grad(set_to_none=True)
        emb, _ = model(audio)
        loss = F.cross_entropy(head(emb.mean(dim=1)), labels)
        loss.backward()
        opt.step()
        return loss
    times, peak = timed(finetune_step, args.steps, args.warmup)
    rows["hf_finetune"] = row_of(times, peak, B)
    print("hf_finetune", json.dumps(rows["hf_finetune"]), flush=True)

    # ---- waveform_grad (frozen model)
    model.requires_grad_(False)
    target = torch.randn(B, 768, generator=g).to(dev)
    x = audio.clone().requires_grad_(True)

    def waveform_step():
        x.grad = None
        emb, _ = model(x)
        loss = F.mse_loss(emb.mean(dim=1), target)
        loss.backward()
        with torch.no_grad():
            x.sub_(1e-4 * x.grad.sign())
        return loss
    times, peak = timed(waveform_step, args.steps, args.warmup)
    rows["waveform_grad"] = row_of(times, peak, B)
    kernels = kernel_rows(waveform_step)   # the audio gradient runs the preprocessing backward
    print("waveform_grad", json.dumps(rows["waveform_grad"]), flush=True)
    del model, opt, x
    torch.cuda.empty_cache()

    # ---- baseline: the oracle's HEAR computation, eager, bf16 autocast
    leaves = {}
    ref_sd = {}
    for k, v in sd.items():
        if id(v) not in leaves:
            leaves[id(v)] = v.to(dev).requires_grad_(k.startswith(PATH))
        ref_sd[k] = leaves[id(v)]
    real_stack = jo.run_stack
    jo.run_stack = lambda x_, sd_, prefix, n, nhead, m, **kw: real_stack(x_, sd_, prefix, n, nhead,
                                                                         None if m is None else m.to(x_.device), **kw)
    torch.manual_seed(0)
    bhead = torch.nn.Linear(768, N_CLASSES).to(dev)
    bopt = torch.optim.AdamW([{"params": [v for k, v in ref_sd.items() if k.startswith(PATH)], "lr": 1e-5},
                              {"params": list(bhead.parameters()), "lr": 1e-3}])

    def baseline_step():
        bopt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            emb, _ = jo.hear_timestamp_embeddings(audio, ref_sd, cfg)
            loss = F.cross_entropy(bhead(emb.float().mean(dim=1)), labels)
        loss.backward()
        bopt.step()
        return loss
    btimes, bpeak = timed(baseline_step, args.baseline_steps, 1)
    jo.run_stack = real_stack
    rows["baseline"] = {"impl": "oracle restatement of the HEAR runtime (oracle/jepa_oracle.py hear_timestamp_embeddings) "
                                "on CUDA, eager, bf16 autocast, same head / loss / AdamW", **row_of(btimes, bpeak, B)}
    rows["finetune_speedup_vs_baseline"] = round(rows["baseline"]["ms_per_step"] / rows["hf_finetune"]["ms_per_step"], 2)
    print("baseline", json.dumps(rows["baseline"]), flush=True)

    out = {
        "workload": f"whole-clip steps: {B} clips x {args.seconds:g} s through hf.WavJEPAModel in training mode "
                    "(WavJEPA-base, synthetic weights, 2.01 s chunks, 200 tokens each); scene embedding -> "
                    f"Linear(768, {N_CLASSES}) -> cross-entropy -> backward -> AdamW, and the frozen-model waveform "
                    "gradient step; inputs resident in HBM",
        "gpu": gpu_info(),
        "batch": B, "seconds": args.seconds, "chunks_per_clip": L // 32159 + 1,
        "rows": rows,
        "preprocessing_kernels": kernels,
    }
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
