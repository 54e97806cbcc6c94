"""Per-layer hidden states (JEPA.get_hidden_states) on the workloads users run them in, one process.

    python scripts/bench_hidden_states.py [--clips 256] [--batch 256] [--reps 3] [--steps 5] [--warmup 2] [--out FILE]

(a) HEAR, configs[3] geometry (256 clips x 10 s through get_timestamp_embeddings): the final features (layer=None)
    against hidden state 6 and hidden state 12 (hear.load_model(..., layer=k)), one runtime per option over the same
    weights, calls alternated after a warm-up of each; CUDA events around every call, input resident in HBM.
(b) The base fine-tuning step of scripts/bench_finetune.py (B dense 2.01 s windows, full and extractor-frozen) with two
    heads: the final features -> mean over tokens -> nn.Linear(768, 50), and a SUPERB-style head, the softmax-weighted
    sum of all 13 hidden states -> mean -> the same Linear, its layer weights trained by the same torch.optim.AdamW.
    Per head: ms/step (median of --steps after --warmup), peak allocated memory of a step, and the summed device time of
    the wj_add_rows_f32 launches (the gradient injections) in one profiled step, run on its own after the timed steps.
The card's name, power limit and maximum SM clock are read in the same call (nvidia-smi)."""
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
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

N_CLASSES = 50
PATH = ("extract_audio.", "feature_norms.", "post_extraction_mapper.", "encoder.")
HEAR_LAYERS = (None, 6, 12)


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


def bench_hear(args, dev):
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    rts = {k: hear.load_model({"state_dict": sd}, layer=k) for k in HEAR_LAYERS}
    audio = oi.hear_inputs(args.clips, 160000, seed=7).to(dev)
    for _ in range(2):
        for k in HEAR_LAYERS:
            rts[k].get_timestamp_embeddings(audio)
    torch.cuda.synchronize()
    times = {k: [] for k in HEAR_LAYERS}
    for _ in range(args.reps):
        for k in HEAR_LAYERS:
            times[k].append(event_ms(lambda: rts[k].get_timestamp_embeddings(audio)))
    out = {}
    for k, t in times.items():
        ms = float(np.median(t))
        out["final_features" if k is None else f"layer_{k}"] = {
            "ms_per_call": round(ms, 2), "ms_all": [round(v, 2) for v in t],
            "clips_per_s": round(args.clips / (ms / 1e3), 1)}
    return out


def build(cfg: jo.Cfg, variant: str, dev):
    ex = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=1)
    m = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
               transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384), process_audio_seconds=2.01)
    m.load_state_dict(jo.make_state_dict(cfg, seed=3), strict=True)
    m.to(dev)
    if variant != "full":
        m.extract_audio.requires_grad_(False)
    return m


def make_step(model, head, audio, labels, superb):
    params = [p for n, p in model.named_parameters() if n.startswith(PATH) and p.requires_grad]
    mix = torch.nn.Parameter(torch.zeros(model._enc_stack.n_layers + 1, device=audio.device))
    opt = torch.optim.AdamW(params + list(head.parameters()) + ([mix] if superb else []), lr=1e-5)

    def step():
        opt.zero_grad(set_to_none=True)
        if superb:
            hs = model.get_hidden_states(audio)
            x = sum(wk * h for wk, h in zip(torch.softmax(mix, 0), hs))
        else:
            x = model.get_audio_representation(audio)
        loss = F.cross_entropy(head(x.mean(dim=1)), labels)
        loss.backward()
        opt.step()
        return loss
    return step


def bench_finetune(args, dev):
    cfg = jo.Cfg()
    B = args.batch
    g = torch.Generator().manual_seed(1)
    audio = torch.randn(B, 1, cfg.target_length, generator=g).to(dev).bfloat16()
    labels = torch.randint(0, N_CLASSES, (B,), generator=g).to(dev)
    out = {}
    for variant in ("full", "extractor_frozen"):
        rows = {}
        for head_kind in ("final_features_mean_linear", "superb_weighted_sum_13_mean_linear"):
            torch.manual_seed(0)
            head = torch.nn.Linear(cfg.d_model, N_CLASSES).to(dev)
            model = build(cfg, variant, dev)
            step = make_step(model, head, audio, labels, head_kind.startswith("superb"))
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            times = [event_ms(step) for _ in range(args.steps)]
            peak = torch.cuda.max_memory_allocated()
            with _lib.KernelProfile() as kp:
                step()
            add = kp.summary().get("wj_add_rows_f32", (0, 0.0))
            ms = float(np.median(times))
            rows[head_kind] = {"ms_per_step": round(ms, 2), "ms_all": [round(t, 2) for t in times],
                               "instances_per_s": round(B / (ms / 1e3), 1),
                               "peak_allocated_gib": round(peak / 2**30, 2),
                               "add_rows_launches_in_profiled_step": add[0],
                               "add_rows_ms_in_profiled_step": round(add[1], 3)}
            print(variant, head_kind, json.dumps(rows[head_kind]), flush=True)
            del model, step, head
            torch.cuda.empty_cache()
        out[variant] = rows
    return {"batch": B, "seconds": 2.01, "variants": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=256)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    out = {
        "gpu": gpu_info(),
        "hear_workload": f"configs[3] geometry: HEAR get_timestamp_embeddings, {args.clips} clips x 10 s (random-init "
                         "WavJEPA-base weights, seeded uniform noise), input resident in HBM; layer=None / 6 / 12",
        "hear": bench_hear(args, dev),
        "finetune_workload": "scripts/bench_finetune.py base step (dense 2.01 s windows, synthetic weights seed 3, "
                             "seeded Gaussian audio): head on the final features vs a SUPERB softmax-weighted sum of "
                             "all 13 hidden states, torch.optim.AdamW",
        "finetune": bench_finetune(args, dev),
    }
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
