"""One fine-tuning step through `JEPA.get_audio_representation`, against a torch-eager bf16-autocast step in the same process.

    python scripts/bench_finetune.py [--batch 256] [--w2v2-batch 128] [--steps 5] [--warmup 2] [--out FILE]

Workload (DESIGN.md 2.2): features of B dense 2.01 s windows (WavJEPA-base, 200 tokens each) -> mean over tokens ->
nn.Linear(768, 50) -> cross-entropy -> backward -> torch.optim.AdamW over the trainable parameters and the head; also the
wav2vec2-extractor geometry (4.02 s windows, B = --w2v2-batch).  Variants: full fine-tune, extractor frozen, and
everything below encoder layer 6 frozen (extractor, feature norm, mapper, layers 0-5: with the mapper trainable the
gradient would still have to pass through the lower layers).  Per variant: ms/step (CUDA events, median of --steps after
--warmup), instances/s, peak allocated memory of a step, and the GEMM rate from FLOPs counted from the GEMM shapes of
one profiled step (over the GEMM kernels' own time, and over the step time).

Baseline: the same step in eager PyTorch under bf16 autocast on the same GPU -- the executed reference when it is staged
(oracle/ref_loader.py) and its get_audio_representation carries a graph, otherwise the oracle restatement
(oracle/jepa_oracle.py: local_features + run_stack) moved to CUDA.  The output names which one ran."""
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

N_CLASSES = 50
PATH = ("extract_audio.", "feature_norms.", "post_extraction_mapper.", "encoder.")
GEMM_ENTRY_POINTS = ("wj_gemm_bf16", "wj_gemm_wgrad_bf16", "wj_gemm_dgrad_bf16")
VARIANTS = ("full", "extractor_frozen", "below_layer_6_frozen")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def build(cfg: jo.Cfg, seconds: float, variant: str, dev):
    ex = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=1)
    m = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
               transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
               process_audio_seconds=seconds)
    m.load_state_dict(jo.make_state_dict(cfg, seed=3), strict=True)
    m.to(dev)
    if variant != "full":
        m.extract_audio.requires_grad_(False)
    if variant == "below_layer_6_frozen":
        for mod in (m.feature_norms, m.post_extraction_mapper, *m.encoder.layers[:6]):
            mod.requires_grad_(False)
    return m


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


def native_step(model, head, audio, labels):
    params = [p for n, p in model.named_parameters() if n.startswith(PATH) and p.requires_grad]
    opt = torch.optim.AdamW(params + list(head.parameters()), lr=1e-5)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = F.cross_entropy(head(model.get_audio_representation(audio).mean(dim=1)), labels)
        loss.backward()
        opt.step()
        return loss
    return step


def eager_step(cfg: jo.Cfg, seconds: float, variant: str, head, audio, labels, dev):
    """(step, label): the same step in eager PyTorch under bf16 autocast."""
    from oracle import ref_loader
    if ref_loader.find_reference() is not None:
        ref = ref_loader.load_reference()
        ext = ref.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=1)
        model = ref.JEPA(feature_extractor=ext, transformer_encoder_cfg=ref.TransformerEncoderCFG.create(),
                         transformer_encoder_layers_cfg=ref.TransformerLayerCFG.create(),
                         transformer_decoder_cfg=ref.TransformerEncoderCFG.create(),
                         transformer_decoder_layers_cfg=ref.TransformerLayerCFG.create(d_model=384),
                         process_audio_seconds=seconds, compile_modules=False).to(dev)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            probe = model.get_audio_representation(audio[:2], None)
        if probe.requires_grad:
            if variant != "full":
                model.extract_audio.requires_grad_(False)
            if variant == "below_layer_6_frozen":
                for mod in (model.feature_norms, model.post_extraction_mapper, *model.encoder.layers[:6]):
                    mod.requires_grad_(False)
            params = [p for n, p in model.named_parameters() if n.startswith(PATH) and p.requires_grad]
            opt = torch.optim.AdamW(params + list(head.parameters()), lr=1e-5)

            def step():
                opt.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    feats = model.get_audio_representation(audio, None)
                    loss = F.cross_entropy(head(feats.float().mean(dim=1)), labels)
                loss.backward()
                opt.step()
                return loss
            return step, "executed reference (labhamlet/wavjepa JEPA.get_audio_representation), eager, bf16 autocast"
        del model
    sd = {k: v.to(dev) for k, v in jo.make_state_dict(cfg, seed=3).items()}
    frozen = ("extract_audio.",) if variant != "full" else ()
    if variant == "below_layer_6_frozen":
        frozen += ("feature_norms.", "post_extraction_mapper.") + tuple(f"encoder.layers.{i}." for i in range(6))
    for k, v in sd.items():
        v.requires_grad_(k.startswith(PATH) and not k.startswith(frozen))
    params = [v for v in sd.values() if v.requires_grad]
    opt = torch.optim.AdamW(params + list(head.parameters()), lr=1e-5)
    x = audio.float()

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            feats = jo.run_stack(jo.local_features(x, sd, cfg), sd, "encoder", cfg.layers, cfg.nhead, None)
            loss = F.cross_entropy(head(feats.float().mean(dim=1)), labels)
        loss.backward()
        opt.step()
        return loss
    return step, "oracle restatement (oracle/jepa_oracle.py local_features + run_stack) on CUDA, eager, bf16 autocast"


def gemm_profile(step):
    with _lib.KernelProfile() as kp:
        step()
    torch.cuda.synchronize()
    ms = flops = 0.0
    for name, e0, e1, meta, _ in kp.records:
        if name in GEMM_ENTRY_POINTS:
            ms += e0.elapsed_time(e1)
            flops += meta[0]
    return flops, ms


def run_geometry(name, cfg, seconds, B, args, dev, with_baseline):
    g = torch.Generator().manual_seed(1)
    audio = torch.randn(B, 1, cfg.target_length, generator=g).to(dev).bfloat16()
    labels = torch.randint(0, N_CLASSES, (B,), generator=g).to(dev)
    rows = {}
    for variant in VARIANTS:
        torch.manual_seed(0)
        head = torch.nn.Linear(cfg.d_model, N_CLASSES).to(dev)
        model = build(cfg, seconds, variant, dev)
        step = native_step(model, head, audio, labels)
        times, peak = timed(step, args.steps, args.warmup)
        flops, g_ms = gemm_profile(step)
        ms = float(np.median(times))
        row = {"ms_per_step": round(ms, 2), "ms_all": [round(t, 2) for t in times],
               "instances_per_s": round(B / (ms / 1e3), 1), "peak_allocated_gib": round(peak / 2**30, 2),
               "gemm_tflop_per_step": round(flops / 1e12, 2),
               "gemm_tflop_s_over_gemm_kernel_time": round(flops / 1e9 / g_ms, 1) if g_ms else None,
               "gemm_tflop_s_over_step_time": round(flops / 1e9 / ms, 1)}
        del model, step
        torch.cuda.empty_cache()
        if with_baseline:
            torch.manual_seed(0)
            head = torch.nn.Linear(cfg.d_model, N_CLASSES).to(dev)
            bstep, label = eager_step(cfg, seconds, variant, head, audio, labels, dev)
            btimes, bpeak = timed(bstep, args.baseline_steps, 1)
            bms = float(np.median(btimes))
            row["baseline"] = {"impl": label, "ms_per_step": round(bms, 2), "ms_all": [round(t, 2) for t in btimes],
                               "instances_per_s": round(B / (bms / 1e3), 1), "peak_allocated_gib": round(bpeak / 2**30, 2),
                               "gemm_tflop_s_over_step_time": round(flops / 1e9 / bms, 1)}
            row["speedup_vs_baseline"] = round(bms / ms, 2)
            del bstep
            torch.cuda.empty_cache()
        rows[variant] = row
        print(name, variant, json.dumps(row), flush=True)
    return {"batch": B, "seconds": seconds, "tokens_per_step": B * cfg.total_patches, "variants": rows}


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
        "workload": "fine-tuning step: get_audio_representation (dense windows) -> mean over tokens -> "
                    f"nn.Linear(768, {N_CLASSES}) -> cross-entropy -> backward -> torch.optim.AdamW; synthetic weights "
                    "(oracle make_state_dict, seed 3) and seeded Gaussian audio, input resident in HBM",
        "gpu": gpu_info(),
        "base_2.01s": run_geometry("base", jo.Cfg(), 2.01, args.batch, args, dev, True),
        "w2v2_4.02s": run_geometry("w2v2", jo.Cfg(spec=hear.W2V2_SPEC, seconds=4.02), 4.02, args.w2v2_batch, args, dev,
                                   True),
    }
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
