#!/usr/bin/env python
"""WavJEPA-base pre-training throughput on B200 (BASELINE.json: "train 2s-instances/s at 1/2/4/8 B200").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config train|hear|nat]    # our arm (N>1: under torchrun)
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]              # the reference's own CPU path

--config train (default, BASELINE.json configs[1]/[2]): one step = one full SSL pre-training step: 64 clips x 8 random
crops of 2.01 s (512 instances / GPU) of synthetic 16 kHz noise, random-init WavJEPA-base weights: GPU mask generation
(AudioSet masker) -> crop + normalise -> conv encoder -> student on visible tokens -> predictor -> EMA-teacher targets ->
masked latent MSE -> hand-written backward (bucketed NCCL all-reduce overlapped when N > 1) -> global-norm clip + AdamW
with the EMA teacher update folded in.  Nothing is skipped.
--config nat (configs[4]): the same step for WavJEPA-Nat (binaural, per-channel extractors, 400 tokens / instance).
--config hear (configs[3]): HEAR `get_timestamp_embeddings` on 256 clips x 10 s (replicas only when N > 1).

`value`  : instances/s (clips/s for hear) with the step's input already resident in HBM (CUDA events, max over ranks).
`e2e`    : the same step driven from pinned HOST buffers (H2D of the batch and a D2H read of the result -- the loss, or
           the embeddings for hear -- inside the timed region, wall clock between device synchronisations, max over ranks).
`roofline`: the dominant kernel (the tcgen05 GEMM / implicit-GEMM-conv kernel, all its launches of one step):
           executed GEMM FLOPs / summed CUDA-event durations, against the measured bf16 peak; `traffic` = DRAM bytes per
           launch from the committed ncu capture next to the algorithmic A + W + output bytes counted live.
`hbm_kernels`: every HBM-bound kernel family of the step: algorithmic bytes, ms, GB/s, fraction of the measured HBM peak.
`cpu_baseline` / `--impl reference`: the EXECUTED, unmodified reference (oracle/ref_bench.py over baseline/_ref or
           /root/reference) on the host cores, BASELINE.json configs[0] (2 clips x 8 crops); the oracle port only if no
           reference checkout travelled.  `gpu_torch_baseline`: the same reference step on this GPU under torch eager +
           bf16 autocast (what a user of the reference gets on this box today), outside the timed region.

--dump-outputs DIR: after the timed steps, writes what the last timed step handed its caller as DIR/<name>.npy, so that
two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.  train / nat:
loss (float64), and of the model state the step updated -- params (trained parameters), teacher (EMA teacher encoder),
adam_exp_avg, adam_exp_avg_sq -- each a fixed seeded sample of 2^21 elements in optimizer_state_dict() name order.
hear: embeddings (the same kind of sample) and timestamps.  float32 unless noted; about 32 MiB in all.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

# activations of consecutive steps differ in size (mask-dependent token counts): let the caching allocator grow its
# segments in place instead of cudaMalloc-ing new ones in the middle of a timed step
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "WavJEPA-base train 2s-instances/s at 1/2/4/8 B200; tensor-pipe % of peak"
UNIT = "instances/s"
CLIPS, CROPS, CLIP_LEN = 64, 8, 160000
SPEC = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)]
MASKER = dict(target_masks_per_context=4, context_mask_prob=0.65, context_mask_length=10, target_prob=0.25,
              target_length=10, ratio_cutoff=0.1)   # configs/masker/AudioSet.yaml
HEAR_CLIPS = 256
DUMP_SAMPLE = 1 << 21         # elements kept of each output larger than this (--dump-outputs)
HBM_WRITE_PEAK_GBS = 3906.0   # measured: torch memset / fill of 1 GiB on this pool's B200 (scripts/bw_probe.py)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def load_traffic():
    """Per-kernel DRAM bytes per launch from the committed ncu capture of one step of this build
    (scripts/kernel_traffic.py -> profiles/r02_kernel_traffic.json); None when absent."""
    p = os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")
    return json.load(open(p)) if os.path.exists(p) else None


def dump_outputs(out_dir, outputs):
    """Writes each tensor of `outputs` as out_dir/<name>.npy (float64 stays float64, anything else becomes float32).
    A tensor of more than DUMP_SAMPLE elements is reduced to the elements at DUMP_SAMPLE fixed positions of its
    flattened form (seed 0, ascending): the same positions for every run and build with the same output size."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), size=DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        t = t.cpu().double() if t.dtype == torch.float64 else t.cpu().float()
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def _train_outputs(model, loss):
    """The last training step's loss and the model state it updated, for --dump-outputs."""
    import torch

    opt = model.optimizer_state_dict()
    params = dict(model.named_parameters())
    names = opt["param_names"]
    return {"loss": loss.double(),
            "params": torch.cat([params[n].detach().reshape(-1) for n in names]),
            "teacher": torch.cat([p.detach().reshape(-1) for p in model.teacher_encoder.parameters()]),
            "adam_exp_avg": torch.cat([opt["state"][n]["exp_avg"].reshape(-1) for n in names]),
            "adam_exp_avg_sq": torch.cat([opt["state"][n]["exp_avg_sq"].reshape(-1) for n in names])}


# ===================================================================================================== FLOP model
def conv_macs(spec, length, cin=1):
    macs, L, first = 0, length, 0
    for i, (dim, k, s) in enumerate(spec):
        L = (L - k) // s + 1
        m = L * dim * cin * k
        if i == 0:
            first = m
        macs += m
        cin = dim
    return macs, first


def stack_macs(n, d, layers=12):
    return layers * (n * 12 * d * d + 2 * n * n * d)


def algorithmic_flops(n_c, n_v, n_t, B, T=200, D=768, Dp=384, n_cnn=1):
    """SURVEY.md 8(d): useful (mask-exact) FLOPs of one training step; masked-out work earns no credit."""
    conv, conv0 = conv_macs(SPEC, 32159)
    conv, conv0 = conv * B * n_cnn, conv0 * B * n_cnn
    mapper = B * T * 512 * D
    student = sum(stack_macs(int(n), D) for n in n_c)
    teacher = B * stack_macs(T, D)
    predictor = sum(stack_macs(int(n), Dp) for n in n_v)
    d2e = int(sum(n_t)) * Dp * D
    e2d = int(sum(n_c)) * D * Dp
    return 2.0 * (3 * (conv + mapper + student + e2d + predictor + d2e) - conv0 + teacher)


# ===================================================================================================== clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


# ===================================================================================================== our arm
def build_model(device, nat: bool = False):
    import torch
    import wavjepa_b200 as w

    torch.manual_seed(0)
    if nat:   # WavJEPA-Nat: one CNN per channel, channel-major tokens (audio_channel_feature_extractor.py:40-179)
        ex = w.ConvChannelFeatureExtractor(conv_layers_spec=SPEC, in_channels=2, share_weights_over_channels=False)
    else:
        ex = w.ConvFeatureExtractor(conv_layers_spec=SPEC, in_channels=1)
    model = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                   transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
                   lr=4e-4, adam_betas=(0.9, 0.98), adam_weight_decay=0.04, process_audio_seconds=2.01,
                   nr_samples_per_audio=CROPS, average_top_k_layers=8)   # configs/trainer/default_trainer.yaml
    return model.to(device)


def _dist_env(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for N > 1 launch with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N")
    return world, rank, local


def _hbm_kernels(kp, peaks, traffic):
    """One entry per HBM-bound kernel family of the profiled step: algorithmic bytes (declared by wavjepa_b200/ops.py
    from the tensor shapes of each call), CUDA-event time, GB/s and the fraction of the measured HBM copy peak."""
    names = {"wj_conv0_gn_gelu_fwd": "conv0+GroupNorm+GELU fwd", "wj_conv0_gn_gelu_bwd": "conv0+GroupNorm+GELU bwd",
             "wj_add_layernorm_fwd": "residual add + LayerNorm fwd", "wj_add_layernorm_bwd": "residual add + LayerNorm bwd",
             "wj_layernorm_fwd": "LayerNorm fwd (feature/final norms)", "wj_layernorm_bwd": "LayerNorm bwd (feature/final norms)",
             "wj_target_accum": "teacher-target instance norm + layer mean",
             "wj_target_combine": "teacher-target instance norm + layer mean (all top-K layers, one pass)", "wj_masked_mse": "masked latent MSE fwd+bwd",
             "wj_adamw_ema_step": "clip + AdamW + EMA teacher", "wj_adamw_step": "clip + AdamW", "wj_ema_update": "EMA teacher",
             "wj_sumsq": "gradient norm", "wj_colsum": "bias-gradient column sums", "wj_crop_norm": "crop + normalise"}
    out = []
    for name, (calls, ms, nb) in sorted(kp.hbm_summary().items(), key=lambda kv: -kv[1][1]):
        if name not in names or ms <= 0:
            continue
        gbs = nb / (ms * 1e-3) / 1e9
        e = {"kernel": name[3:], "what": names[name], "calls": calls, "ms": round(ms, 3),
             "algorithmic_bytes": int(nb), "gbs": round(gbs, 1), "frac": round(gbs / peaks["hbm"], 4)}
        if name == "wj_conv0_gn_gelu_fwd":
            # 99 % of this kernel's bytes are WRITES: a write-only stream tops out at 3.9 TB/s on this pool (memset /
            # fill, scripts/bw_probe.py), not at the 6.5 TB/s of the read+write copy that `hbm_peak_gbs` measures
            e["frac_of_write_peak"] = round(gbs / HBM_WRITE_PEAK_GBS, 4)
            e["write_peak_gbs"] = HBM_WRITE_PEAK_GBS
        # (the ncu launch list cannot tell the stand-alone wj_colsum calls from the colsum launches made inside
        # wj_attn_varlen_bwd_bias, so no traffic figure is attached to that family)
        if traffic is not None and name != "wj_colsum" and name[3:] in traffic.get("by_entry", {}):
            t = traffic["by_entry"][name[3:]]
            e["traffic"] = t["dram_bytes_per_step"]
            e["traffic_over_algorithmic"] = round(t["dram_bytes_per_step"] / max(nb, 1), 3)
        out.append(e)
    return out


def run_native(args):
    import torch
    import torch.distributed as dist
    import wavjepa_b200 as w
    from wavjepa_b200 import _lib
    from wavjepa_b200.dist import BucketedAllReduce

    world, rank, local = _dist_env(args)
    nat = args.config == "nat"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_device()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.deterministic:
        from wavjepa_b200 import ops as _ops
        _ops.set_deterministic(True, (512 if nat else 256) << 20)
    model = build_model(dev, nat=nat)
    model.reserve_workspace((130 if nat else 80) << 30)   # setup: the activation pool of a 512-instance step exists up front
    model.global_step = 1000          # lr(0) == 0 (warm-up from 0): start inside the warm-up so AdamW moves weights
    if world > 1:
        # (WJ_BUCKET_MB: measurement override of the gradient bucket size)
        bucket_mb = int(os.environ.get("WJ_BUCKET_MB", "0"))
        model.attach_data_parallel(BucketedAllReduce(bucket_bytes=bucket_mb << 20) if bucket_mb else BucketedAllReduce())
    C_in = 2 if nat else 1
    masker = w.TimeInverseBlockMasker(**MASKER, channel_based_masking=nat, seed=1234, row0=rank * (1 << 24), device=dev)
    B = CLIPS * CROPS
    T = model.total_patches
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    n_pool = 3
    host_clips = [torch.randn(CLIPS, C_in, CLIP_LEN, generator=torch.Generator().manual_seed(100 * rank + i)).pin_memory()
                  for i in range(n_pool)]
    dev_clips = [c.to(dev) for c in host_clips]
    stage = torch.empty(CLIPS, C_in, CLIP_LEN, device=dev)
    last_mi = {}

    def step(clips):
        ctx, tgt, vis = masker(batch_size=B, n_times=T, in_channels=C_in)
        starts = torch.randint(0, CLIP_LEN - model.target_length + 1, (CLIPS, CROPS), device=dev, generator=gen)
        x16, _, _, _ = model.on_after_batch_transfer((clips, ctx.view(CLIPS, CROPS, T), tgt.view(CLIPS, CROPS, 4, T),
                                                      vis.view(CLIPS, CROPS, 4, T)), 0, starts=starts)
        loss = model.train_step(x16, ctx, tgt, vis)
        last_mi["mi"] = model._last_mi
        return loss

    def note(msg):
        if os.environ.get("WJ_BENCH_VERBOSE"):
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---------------------------------------------------------------- device-resident arm (`value`)
    note("model built")
    for i in range(args.warmup):
        step(dev_clips[i % n_pool])
        note(f"warm-up step {i} issued")
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    k0 = _lib.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss = None
    for i in range(args.steps):
        loss = step(dev_clips[i % n_pool])
    e1.record()
    barrier()
    launches = _lib.kernel_launches() - k0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, _train_outputs(model, loss))
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total / 1e3)
    final_loss = loss.item()
    note(f"timed region done: {ms_step:.1f} ms/step")

    # ---------------------------------------------------------------- end-to-end arm (`e2e`): host clips in, loss out
    def e2e_step(i):
        stage.copy_(host_clips[i % n_pool], non_blocking=True)
        return step(stage).item()

    for i in range(2):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * B * args.steps / e2e_s
    note("e2e region done")
    h2d = CLIPS * C_in * CLIP_LEN * 4
    d2h = 4 + 8 * 4   # loss scalar + the mask totals read by the host to size the packed buffers

    # ---------------------------------------------------------------- DP consistency (N > 1): replicas bit-identical?
    dp_check = None
    if world > 1:
        cs = torch.stack([model._flat_p.double().sum(), model._flat_t.double().sum(),
                          model._flat_p.view(torch.int32).long().sum().double()])
        lo, hi = cs.clone(), cs.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dp_check = {"param_checksum_max_minus_min": float((hi - lo).abs().max().item()),
                    "what": "fp64 sum of student parameters, of EMA-teacher parameters and integer sum of the parameter "
                            "bit patterns after all timed steps: max - min over ranks (0 = replicas bit-identical)"}
        if dp_check["param_checksum_max_minus_min"] != 0.0:
            # name what differs: per-tensor bit-pattern sums of parameters, Adam moments and the last all-reduced gradient
            names = list(model._train_names)
            per = torch.stack([torch.stack([model._view(buf, n_).view(torch.int32).long().sum() for n_ in names])
                               for buf in (model._flat_p, model._adam_m, model._adam_v, model._flat_g)])
            allr = [torch.empty_like(per) for _ in range(world)]
            dist.all_gather(allr, per)
            A = torch.stack(allr)                                # [world, 4, n_tensors]
            diff = (A != A[0]).any(0)
            dp_check["components_max_minus_min"] = [float(v) for v in (hi - lo).abs().tolist()]
            for k, lab in enumerate(("params", "adam_m", "adam_v", "last_grads")):
                idx = torch.nonzero(diff[k]).flatten().tolist()
                dp_check[f"{lab}_tensors_differ"] = len(idx)
                dp_check[f"{lab}_first"] = [names[i] for i in idx[:6]]
            dp_check["ranks_differing_from_rank0"] = [r for r in range(world) if bool((A[r] != A[0]).any())]

    # ---------------------------------------------------------------- per-kernel attribution (outside the timed region)
    # every rank runs this extra step (its gradient all-reduce is a collective); only rank 0 brackets its launches
    kp = None
    if rank == 0:
        with _lib.KernelProfile() as kp:
            step(dev_clips[0])
    else:
        step(dev_clips[0])
    barrier()

    out = None
    if rank == 0:
        peaks = load_peaks()
        traffic = load_traffic()
        summ = kp.summary()
        gemm_names = ("wj_gemm_bf16", "wj_gemm_dgrad_bf16", "wj_gemm_wgrad_bf16")
        g_calls = sum(summ[n][0] for n in gemm_names if n in summ)
        g_ms = sum(summ[n][1] for n in gemm_names if n in summ)
        g_flops = sum(m[0] for (n, _, _, m, _) in kp.records if n in gemm_names and m)
        g_bytes = sum(nb for (n, _, _, _, nb) in kp.records if n in gemm_names and nb)
        fam_ms = {n[3:]: round(t, 3) for n, (c, t) in sorted(summ.items(), key=lambda kv: -kv[1][1])}
        fam_calls = {n[3:]: c for n, (c, t) in summ.items()}
        prof_total = sum(t for (_, t) in summ.values())
        achieved = g_flops / (g_ms * 1e-3) / 1e12
        mi = last_mi["mi"]
        f_alg = algorithmic_flops(mi.n_c.tolist(), mi.n_v.tolist(), mi.n_t.tolist(), B, T=T, n_cnn=C_in)
        roofline = {"bound": "tensor", "kernel": "gemm_kernel<BN,MODE> (tcgen05.mma + TMA; Linear fwd/dgrad/wgrad and "
                    "implicit-GEMM Conv1d)", "achieved": round(achieved, 1), "peak": peaks["bf16_sustained"],
                    "unit": "TFLOP/s", "frac": round(achieved / peaks["bf16_sustained"], 4),
                    "peak_source": peaks["source"] + ", sustained figure (kernel timed inside a long step)",
                    "launches_per_step": g_calls, "avg_launch_ms": round(g_ms / max(g_calls, 1), 4),
                    "flops_per_step": g_flops, "share_of_step": round(g_ms / prof_total, 4), "traffic": None,
                    "algorithmic_bytes_per_launch": round(g_bytes / max(g_calls, 1), 1),
                    "algorithmic_bytes_note": "A + W + every output / residual / saved-factor operand of each GEMM launch, "
                                              "counted from the call arguments of this very step"}
        if traffic is not None and "gemm" in traffic and not nat:
            t = traffic["gemm"]
            roofline["traffic"] = t["dram_bytes_per_launch_avg"]
            roofline["traffic_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum per GEMM launch, ncu over the %d GEMM "
                                        "launches of one step of this build (%s)" % (t["launches"], traffic.get("source", "")))
        out = {"metric": METRIC if not nat else "WavJEPA-Nat (binaural) train 2s-instances/s", "value": round(value, 1),
               "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": {"workload": ("configs[4]: WavJEPA-Nat binaural SSL pre-training step, 64 clips x 8 crops of 2.01 s x 2 "
                                       "channels (512 instances/GPU, 400 tokens each), per-channel extractors, random-init "
                                       "weights, AudioSet masker with channel-based masking, AdamW+EMA included") if nat else
                                      ("configs[1]: WavJEPA-base SSL pre-training step, 64 clips x 8 crops of 2.01 s "
                                       "(512 instances/GPU), random-init weights, AudioSet masker, AdamW+EMA included"),
                          "instances_per_gpu": B, "global_instances": world * B, "tokens_per_instance": T,
                          "parallelism": f"dp{world}", **({"deterministic": True} if args.deterministic else {}),
                          "l2": "no explicit flush: every step streams > 30 GB of activations (>> 126 MB L2) and "
                                "rotates 3 different 41 MB clip batches"},
               "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_s / args.steps * 1e3, 3)},
               "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
               "hbm_kernels": _hbm_kernels(kp, peaks, traffic),
               "hbm_peak_gbs": peaks["hbm"],
               "step_tensor": {"alg_flops_per_step": f_alg, "alg_tflops": round(f_alg / (ms_step * 1e-3) / 1e12, 1),
                               "frac_of_peak": round(f_alg / (ms_step * 1e-3) / 1e12 / peaks["bf16_sustained"], 4),
                               "note": "useful mask-exact FLOPs (SURVEY.md 8d) / whole step time incl. optimizer"},
               "kernel_ms_per_step": fam_ms, "kernel_calls_per_step": fam_calls, "loss": final_loss,
               "host_cpus": os.cpu_count()}
        if dp_check is not None:
            out["dp_check"] = dp_check
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        if world == 1 and not nat:
            # the reference arms run AFTER our model is gone from the device (the dense reference needs the memory)
            import gc
            del model, dev_clips, stage, kp, step, e2e_step, masker
            last_mi.clear()
            gc.collect()
            torch.cuda.empty_cache()
            if not args.no_cpu_baseline:
                out["cpu_baseline"] = cpu_baseline(budget_s=25.0)
            if not args.no_gpu_baseline:
                out["gpu_torch_baseline"] = gpu_torch_baseline(ours=value)
        print(json.dumps(out), flush=True)


# ===================================================================================================== HEAR (configs[3])
def run_hear(args):
    """configs[3]: HEAR/HF feature extraction, 256 clips x 10 s (160000 samples) per GPU -> [256, 996, 768] + timestamps.
    Replicas only (SURVEY.md 8e): at N > 1 every rank embeds its own 256 clips, no collective on the data path."""
    import torch
    import torch.distributed as dist
    import wavjepa_b200 as w
    from wavjepa_b200 import _lib, hear

    world, rank, local = _dist_env(args)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_device()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    init = w.JEPA(feature_extractor=w.ConvFeatureExtractor(conv_layers_spec=hear.BASE_SPEC, in_channels=1),
                  transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
                  transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                  transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
                  transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384), process_audio_seconds=2.01)
    model = hear.load_model({"state_dict": init.state_dict()})     # random-init weights (no network for checkpoints)
    n, L = HEAR_CLIPS, CLIP_LEN
    host = [(torch.rand(n, L, generator=torch.Generator().manual_seed(7 + 10 * rank + i)) * 2 - 1).pin_memory() for i in range(2)]
    devb = [h.to(dev) for h in host]
    stage = torch.empty(n, L, device=dev)
    emb_host = torch.empty(n, 996, 768).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    for i in range(args.warmup):
        hear.get_timestamp_embeddings(devb[i % 2], model)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    k0 = _lib.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        emb, ts = hear.get_timestamp_embeddings(devb[i % 2], model)
    e1.record()
    barrier()
    launches = _lib.kernel_launches() - k0
    clocks = sampler.stop() if sampler else None
    assert tuple(emb.shape) == (n, 996, 768) and tuple(ts.shape) == (n, 996) and bool(torch.isfinite(emb).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"embeddings": emb, "timestamps": ts})
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / args.steps
    value = world * n * args.steps / (ms_total / 1e3)

    def e2e_step(i):
        stage.copy_(host[i % 2], non_blocking=True)
        e, _ = hear.get_timestamp_embeddings(stage, model)
        emb_host.copy_(e, non_blocking=True)
        torch.cuda.synchronize()

    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    kp = None
    if rank == 0:
        with _lib.KernelProfile() as kp:
            hear.get_timestamp_embeddings(devb[0], model)
    barrier()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = load_peaks()
    summ = kp.summary()
    gemm_names = ("wj_gemm_bf16", "wj_gemm_dgrad_bf16", "wj_gemm_wgrad_bf16")
    g_calls = sum(summ[x][0] for x in gemm_names if x in summ)
    g_ms = sum(summ[x][1] for x in gemm_names if x in summ)
    g_flops = sum(m[0] for (x, _, _, m, _) in kp.records if x in gemm_names and m)
    g_bytes = sum(nb for (x, _, _, _, nb) in kp.records if x in gemm_names and nb)
    prof_total = sum(t for (_, t) in summ.values())
    achieved = g_flops / (g_ms * 1e-3) / 1e12
    dense = 45.35e9 * 5 * n   # SURVEY.md 8d: 45.35 GFLOP per 2.01 s chunk, 5 chunks per 10 s clip
    out = {"metric": "WavJEPA-base HEAR feature extraction, 10 s clips/s (configs[3])", "value": round(value, 1),
           "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16", "data": "synthetic",
           "config": {"workload": "configs[3]: HEAR get_timestamp_embeddings (hear_configs/WavJEPA.py), 256 clips x 10 s "
                                  "(160000 samples, U(-1,1)) per GPU -> [256, 996, 768] fp32 + timestamps; random-init weights; "
                                  "replicas only at N > 1",
                      "clips_per_gpu": n, "parallelism": f"replicas{world}",
                      "l2": "two alternating 164 MB input batches; each call streams > 10 GB of activations"},
           "e2e": {"value": round(world * n * args.steps / e2e_s, 1), "unit": "clips/s", "h2d_bytes_per_step": n * L * 4,
                   "d2h_bytes_per_step": n * 996 * 768 * 4, "ms_per_step": round(e2e_s / args.steps * 1e3, 3)},
           "gpu_launches": int(launches), "clocks": clocks,
           "roofline": {"bound": "tensor", "kernel": "gemm_kernel<BN,MODE> (tcgen05.mma + TMA)", "achieved": round(achieved, 1),
                        "peak": peaks["bf16_sustained"], "unit": "TFLOP/s", "frac": round(achieved / peaks["bf16_sustained"], 4),
                        "peak_source": peaks["source"] + ", sustained figure", "launches_per_step": g_calls,
                        "avg_launch_ms": round(g_ms / max(g_calls, 1), 4), "flops_per_step": g_flops,
                        "share_of_step": round(g_ms / prof_total, 4), "traffic": None,
                        "algorithmic_bytes_per_launch": round(g_bytes / max(g_calls, 1), 1)},
           "hbm_kernels": _hbm_kernels(kp, peaks, None), "hbm_peak_gbs": peaks["hbm"],
           "step_tensor": {"alg_flops_per_step": dense, "alg_tflops": round(dense / (ms_step * 1e-3) / 1e12, 1),
                           "frac_of_peak": round(dense / (ms_step * 1e-3) / 1e12 / peaks["bf16_sustained"], 4),
                           "note": "dense inference FLOPs (SURVEY.md 8d) / whole call time"},
           "kernel_ms_per_step": {x[3:]: round(t, 3) for x, (c, t) in sorted(summ.items(), key=lambda kv: -kv[1][1])},
           "host_cpus": os.cpu_count()}
    if world == 1 and not args.no_cpu_baseline:
        from oracle import ref_bench
        if ref_bench.available():
            torch.set_num_threads(os.cpu_count() or 1)
            r = ref_bench.time_hear(2, CLIP_LEN)
            out["cpu_baseline"] = {"value": round(r["clips_per_s"], 3), "unit": "clips/s", "cores": torch.get_num_threads(),
                                   "kind": "reference", "sample": "the executed reference's RuntimeJEPA.get_timestamp_embeddings "
                                   f"(fp32 torch CPU) on 2 clips x 10 s: {r['s']:.2f} s"}
    print(json.dumps(out), flush=True)


# ===================================================================================================== reference arms
def _oracle_port_step(n_inst):
    """Fallback when no reference checkout is present: the op-for-op oracle restatement of the same training step."""
    import torch
    from oracle import inputs as oi
    from oracle import jepa_oracle as jo

    torch.set_num_threads(os.cpu_count() or 1)
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=0)
    names = [k for k in sd if not k.startswith(("teacher_encoder.", "pos_encoding"))]
    params = [sd[k].requires_grad_(True) for k in names]
    opt = torch.optim.AdamW(params, lr=4e-4 * 1000 / 100000, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.04)
    inp = oi.training_inputs(cfg, max(1, n_inst // CROPS), CROPS, seed=1234, masker="audioset")

    def step():
        opt.zero_grad(set_to_none=True)
        out = jo.forward(inp["audio"], inp["ctx_masks"], inp["target_indices"], inp["ctx_and_target_masks"], sd, cfg)
        out["loss"].backward()
        with torch.no_grad():
            jo.ema_update(sd, step=1000)
        torch.nn.utils.clip_grad_norm_(params, 5.0)
        opt.step()
        return out["loss"].item()

    return step


def _reference_cpu_step(n_clips):
    """-> (step, instances per step, kind, description): the executed reference when a checkout is reachable."""
    import torch
    from oracle import ref_bench

    torch.set_num_threads(os.cpu_count() or 1)
    if ref_bench.available():
        step, n_inst = ref_bench.train_step_fn("cpu", n_clips)
        return step, n_inst, "reference", ("the UNMODIFIED reference (labhamlet/wavjepa, imported from %s through "
                                           "oracle/ref_loader.py): on_after_batch_transfer + training_step (forward, EMA) + "
                                           "backward + clip_grad_norm_(5) + AdamW + LR schedule, fp32 torch CPU, dense tokens"
                                           % os.path.relpath(ref_bench.ref_loader.find_reference(), ROOT))
    return _oracle_port_step(n_clips * CROPS), n_clips * CROPS, "port", \
        "oracle port of the training step (no reference checkout on this machine), fp32 torch CPU, dense tokens"


def cpu_baseline(budget_s: float):
    """BASELINE.json configs[0] on the host cores: 2 clips x 8 crops through the executed reference, bounded sample."""
    import torch

    step, n_inst, kind, what = _reference_cpu_step(2)
    t0 = time.perf_counter()
    step()                                    # warm-up (also sizes the sample)
    t1 = time.perf_counter() - t0
    reps = max(1, min(3, int(budget_s / max(t1, 1e-3)) - 1))
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = (time.perf_counter() - t0) / reps
    out = {"value": round(n_inst / dt, 3), "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
           "sample": f"{reps} x one training step of configs[0] (2 clips x 8 crops of 2.01 s = {n_inst} instances): {what}; "
                     f"{dt:.2f} s/step"}
    if kind == "reference":
        from oracle import ref_bench
        try:
            torch.set_num_threads(1)
            m = ref_bench.time_masks(128)
            torch.set_num_threads(os.cpu_count() or 1)
            out["masks_rows_per_s_1thread"] = {k: round(v, 1) for k, v in m.items()}
        except Exception as e:   # the training-step number stands on its own
            out["masks_rows_per_s_1thread"] = {"error": str(e)[:200]}
    return out


def gpu_torch_baseline(ours: float):
    """The same-box bar BASELINE.md 4 promises: the unmodified reference's training step on THIS GPU under torch eager +
    bf16 autocast (its `bf16-mixed` trainer precision), 64 clips x 8 crops (halved on OOM), in a fresh process."""
    from oracle import ref_bench

    if not ref_bench.available():
        return {"unavailable": "no reference checkout on this machine (baseline/_ref not staged)"}
    cmd = [sys.executable, "-m", "oracle.ref_bench", "--device", "cuda", "--clips", str(CLIPS), "--steps", "3", "--warmup", "2"]
    try:
        r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=420)
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
        d = json.loads(line)
        tr = d["train"]
        if "error" in tr:
            return {"unavailable": tr["error"]}
        return {"value": round(tr["instances_per_s"], 1), "unit": UNIT, "ms_per_step": round(tr["s_per_step"] * 1e3, 1),
                "instances_per_step": tr["instances_per_step"], "peak_mem_gib": round(tr.get("peak_mem_gib", 0.0), 1),
                "torch": d.get("torch"), "ours_over_this": round(ours / tr["instances_per_s"], 2),
                "what": "the unmodified reference (dense tokens, nn.TransformerEncoder / SDPA / cuDNN through torch eager, "
                        "bf16 autocast, torch.optim.AdamW, per-parameter EMA loop) running the same training step on this "
                        "GPU; reported beside the timed region, not inside it"}
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the training step, all host threads, on
    BASELINE.json configs[0] (the reference's CPU-runnable case: 2 clips x 8 crops), shrunk only if K + W steps would
    not fit in a few minutes."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch

    n_clips = 2
    step, n_inst, kind, what = _reference_cpu_step(n_clips)
    t0 = time.perf_counter()
    step()
    t_first = time.perf_counter() - t0
    if t_first * (args.steps + args.warmup) > 300 and n_clips > 1:   # keep the whole run within a few minutes
        n_clips = 1
        step, n_inst, kind, what = _reference_cpu_step(n_clips)
    for _ in range(max(0, args.warmup - 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = n_inst * args.steps / dt
    sample = f"each step = one training step on {n_clips} clip(s) x {CROPS} crops of 2.01 s ({n_inst} instances): {what}"
    out = {"impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 1),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "configs[0]/[1] training step on a bounded CPU sample: " + sample,
                      "instances_per_step": n_inst},
           "cpu_baseline": {"value": round(v, 3), "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                            "sample": sample},
           "e2e": {"value": round(v, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "host_cpus": os.cpu_count()}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="train", choices=["train", "hear", "nat"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--deterministic", action="store_true",
                    help="time the step with bit-reproducible reductions (ops.set_deterministic); not the default bench line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this implementation's timed step (--impl native)")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "hear":
        run_hear(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
