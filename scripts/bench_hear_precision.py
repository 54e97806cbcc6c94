"""HEAR feature extraction in both inference precisions (JEPA.inference_precision "bf16" / "tf32"), one process, same
weights, configs[3] geometry (256 clips x 10 s through get_timestamp_embeddings); bench.py stays on configs[1].

    python scripts/bench_hear_precision.py [--reps 3] [--out FILE]

After a warm-up of both modes the calls alternate bf16 / tf32 (CUDA events around each call, input resident in HBM).
A separate profiled tf32 call attributes time to the tf32 GEMMs (wj_gemm_tf32, FLOPs from their shapes) for their
achieved rate against the 1,125 TFLOP/s dense TF32 data-sheet figure.  Parity: each mode's relative L2 against the CPU
oracle (the reference's fp32 computation) on a 2-clip subset."""
import argparse
import json
import os
import subprocess
import sys

os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from wavjepa_b200 import _lib, hear  # noqa: E402
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

TF32_PEAK = 1125.0   # TFLOP/s, dense TF32, one B200 (HGX B200 data sheet / 16)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--clips", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    _lib.require_device()
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    rt = hear.load_model({"state_dict": sd})
    model = rt.model
    audio = oi.hear_inputs(args.clips, 160000, seed=7).to(dev)

    def call(mode):
        model.inference_precision = mode
        return rt.get_timestamp_embeddings(audio)[0]

    for mode in ("bf16", "tf32", "bf16", "tf32"):
        call(mode)
    torch.cuda.synchronize()
    times = {"bf16": [], "tf32": []}
    for _ in range(args.reps):
        for mode in ("bf16", "tf32"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call(mode)
            e1.record()
            torch.cuda.synchronize()
            times[mode].append(e0.elapsed_time(e1))
    with _lib.KernelProfile() as kp:
        call("tf32")
    torch.cuda.synchronize()
    g_ms = g_flops = 0.0
    fam = {}
    for name, e0, e1, meta, _ in kp.records:
        ms = e0.elapsed_time(e1)
        fam[name] = fam.get(name, 0.0) + ms
        if name == "wj_gemm_tf32":
            g_ms += ms
            g_flops += meta[0]
    # parity on a 2-clip subset against the CPU oracle
    torch.set_num_threads(os.cpu_count())
    sub = audio[:2].cpu()
    with torch.no_grad():
        ref, _ = jo.hear_timestamp_embeddings(sub, sd, jo.Cfg())
    parity = {}
    for mode in ("bf16", "tf32"):
        model.inference_precision = mode
        e = rt.get_timestamp_embeddings(sub.to(dev))[0].double().cpu().numpy()
        parity[mode] = float(np.linalg.norm(e - ref.double().numpy()) / np.linalg.norm(ref.double().numpy()))
    out = {
        "workload": f"configs[3] geometry: HEAR get_timestamp_embeddings, {args.clips} clips x 10 s "
                    f"(random-init WavJEPA-base weights, seeded uniform noise), input resident in HBM",
        "gpu": gpu_info(),
        "modes": {m: {"ms_per_call": round(float(np.median(t)), 2), "ms_all": [round(v, 2) for v in t],
                      "clips_per_s": round(args.clips / (float(np.median(t)) / 1e3), 1),
                      "rel_l2_vs_cpu_oracle_2_clips": parity[m]} for m, t in times.items()},
        "tf32_gemms": {"ms": round(g_ms, 2), "tflop": round(g_flops / 1e12, 2),
                       "achieved_tflop_s": round(g_flops / 1e9 / g_ms, 1) if g_ms else None,
                       "share_of_1125_tflop_s_datasheet": round(g_flops / 1e9 / g_ms / TF32_PEAK, 3) if g_ms else None},
        "tf32_profiled_call_ms_by_entry_point": {k: round(v, 2) for k, v in sorted(fam.items(), key=lambda kv: -kv[1])},
    }
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
