"""End-to-end parity on the B200: the wavjepa_b200 module API (JEPA / maskers / HEAR runtime, all compute through
libwavjepa_b200.so) against (1) the golden fixtures produced by the executed reference (tests/golden/*.npz) and
(2) the CPU oracle run live on the same seeded inputs.

Tolerances (SURVEY.md 8d, north_star): masks bit-exact; features / targets / predictions rel-L2 <= 1e-2; loss rel
<= 1e-3; one-step gradients rel-L2 <= 2e-2 per parameter tensor (bf16 operands, fp32 accumulation -- the reference's
own bf16-autocast run sits at 5e-3..9e-3 against its fp32 run)."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import wavjepa_b200 as w  # noqa: E402
from wavjepa_b200 import _lib, hear, ops  # noqa: E402
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402
from oracle import masks_oracle as mo  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
DEV = "cuda"

FEAT_TOL = 1e-2
LOSS_TOL = 1e-3
GRAD_TOL = 2e-2


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


def build_model(cfg: jo.Cfg, sd=None, **kw):
    if cfg.per_channel:
        ex = w.ConvChannelFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=cfg.in_channels,
                                           share_weights_over_channels=False)
    else:
        ex = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=cfg.in_channels)
    m = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
               transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
               process_audio_seconds=2.01, nr_samples_per_audio=8, average_top_k_layers=cfg.top_k, lr=4e-4,
               adam_weight_decay=0.04, **kw)
    if sd is not None:
        m.load_state_dict({k: v.detach() for k, v in sd.items()}, strict=True)
    return m.to(DEV)


@pytest.fixture(autouse=True, scope="module")
def _device():
    _lib.require_device()
    torch.manual_seed(0)


CASES = [
    ("train_c1", dict(), 4, 1234, "audioset"),
    ("train_speech", dict(), 2, 4321, "librispeech"),
    ("train_nat", dict(in_channels=2, per_channel=True), 2, 55, "audioset"),
]


def _gpu_masks(cfg, B, seed, masker):
    if masker == "audioset":
        mk = w.TimeInverseBlockMasker(target_masks_per_context=4, context_mask_prob=0.65, context_mask_length=10,
                                      target_prob=0.25, target_length=10, ratio_cutoff=0.1,
                                      channel_based_masking=cfg.per_channel, seed=seed, row0=0)
    else:
        mk = w.SpeechMasker(target_masks_per_context=4, target_prob=0.1, target_length=10, ratio_cutoff=0.5,
                            min_context_len=5, seed=seed, row0=0)
    out = mk(batch_size=B, n_times=cfg.total_patches, in_channels=cfg.in_channels if cfg.per_channel else 1)
    mk.check()
    return out


@pytest.mark.parametrize("name,cfgkw,crops,seed,masker", CASES)
def test_train_step_matches_reference_goldens(name, cfgkw, crops, seed, masker):
    cfg = jo.Cfg(**cfgkw)
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    meta = json.load(open(os.path.join(GOLD, f"{name}.json")))
    sd = jo.make_state_dict(cfg, seed=3)
    model = build_model(cfg, sd)
    inp = oi.training_inputs(cfg, 1, crops, seed=seed, masker=masker)
    B = inp["audio"].shape[0]
    # ---- masks: the CUDA masker reproduces the oracle's (= the reference's, tests/test_oracle_cpu.py) bit for bit
    c_m, t_m, v_m = _gpu_masks(cfg, B, seed, masker)
    assert torch.equal(c_m.cpu(), inp["ctx_masks"])
    assert torch.equal(t_m.cpu(), inp["target_indices"])
    assert torch.equal(v_m.cpu(), inp["ctx_and_target_masks"])
    # ---- crop + normalise kernel == the host-side restatement (bf16 output)
    clips = inp["clips"].to(DEV)
    model.nr_samples_per_audio = crops
    x16, c2, t2, v2 = model.on_after_batch_transfer(
        (clips, c_m[None], t_m[None], v_m[None]), 0, starts=inp["starts"].to(DEV))
    assert rel(x16.float().cpu().numpy(), inp["audio"].numpy()) < 2e-3
    # ---- forward (the same bf16 audio the reference saw)
    audio = inp["audio"].to(DEV).bfloat16()
    out = model(audio, c_m, t_m, v_m)
    loss = out["loss"]
    assert abs(loss.item() - float(g["loss"])) / float(g["loss"]) < LOSS_TOL
    G, T = t_m.shape[1], t_m.shape[2]
    preds_t = out["preds"].view(B, G, T, -1)[t_m]
    for k, t in (("local_features", out["local_features"]), ("contextual_features", out["contextual_features"]),
                 ("targets", out["targets"]), ("preds_at_targets", preds_t)):
        assert list(t.shape) == meta[k]["shape"], k
        assert rel(oi.subsample(t.cpu()), g[k]) < FEAT_TOL, (k, rel(oi.subsample(t.cpu()), g[k]))
    # ---- backward through the autograd bridge: per-parameter gradients
    loss.backward()
    params = dict(model.named_parameters())
    worst = 0.0
    for n_, ref_norm in meta["grad_norms"].items():
        gr = params[n_].grad
        assert gr is not None, n_
        e = abs(float(gr.norm()) - ref_norm) / (ref_norm + 1e-12)
        worst = max(worst, e)
        assert e < GRAD_TOL, (n_, e)
    for k in g.files:
        if k.startswith("grad::"):
            e = rel(oi.subsample(params[k[6:]].grad.cpu()), g[k])
            assert e < GRAD_TOL, (k, e)
    # ---- EMA with the pre-step student (decay 0.999 at step 0)
    model._step_teacher()
    tw = dict(model.teacher_encoder.named_parameters())["layers.3.linear1.weight"]
    assert np.allclose(oi.subsample(tw.cpu()), g["teacher_after_ema::layers.3.linear1.weight"], rtol=0, atol=1e-9)


def test_forward_matches_live_oracle_on_fresh_inputs():
    """Same comparison against the oracle executed here (inputs that are not in the fixtures)."""
    torch.set_num_threads(os.cpu_count())
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=11)
    inp = oi.training_inputs(cfg, 1, 3, seed=777, masker="audioset", row0=40)
    with torch.no_grad():
        ref = jo.forward(inp["audio"], inp["ctx_masks"], inp["target_indices"], inp["ctx_and_target_masks"], sd, cfg)
    model = build_model(cfg, sd)
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, seed=777, row0=40)
    c_m, t_m, v_m = mk(batch_size=3, n_times=200, in_channels=1)
    assert torch.equal(c_m.cpu(), inp["ctx_masks"]) and torch.equal(t_m.cpu(), inp["target_indices"])
    with torch.no_grad():
        out = model(inp["audio"].to(DEV).bfloat16(), c_m, t_m, v_m)
    assert abs(out["loss"].item() - ref["loss"].item()) / ref["loss"].item() < LOSS_TOL
    assert rel(out["local_features"].cpu().numpy(), ref["local_features"].numpy()) < FEAT_TOL
    assert rel(out["targets"].cpu().numpy(), ref["targets"].numpy()) < FEAT_TOL
    assert rel(out["contextual_features"].float().cpu().numpy(), ref["contextual_features"].numpy()) < FEAT_TOL
    ti = inp["target_indices"]
    B, G, T = ti.shape
    ours = out["preds"].view(B, G, T, -1)[t_m].float().cpu().numpy()
    theirs = ref["preds"].view(B, G, T, -1)[ti].numpy()
    assert rel(ours, theirs) < FEAT_TOL


def test_train_step_run_to_run_difference_is_summation_order_only():
    """Two identical models stepped on the same clips and masks: no atomics touch an activation gradient (the predictor
    context gradient is a fixed-order gather, the conv-0 reduction runs in fp64), so parameter gradients differ only by
    the order of fp32 atomic sums in their own final reductions (measured 5e-7; round 1: 4e-3 on the conv-0 weight)."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=5)
    inp = oi.training_inputs(cfg, 2, 4, seed=33, masker="audioset")
    a, b = build_model(cfg, sd), build_model(cfg, sd)
    a.global_step = b.global_step = 50000
    audio = inp["audio"].to(DEV).bfloat16()
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    la, lb = a.train_step(audio, c_m, t_m, v_m), b.train_step(audio, c_m, t_m, v_m)
    assert abs(la.item() - lb.item()) < 1e-6
    for n_ in a._train_names:
        ga, gb = a._view(a._flat_g, n_).double(), b._view(b._flat_g, n_).double()
        assert (ga - gb).norm().item() <= 1e-5 * gb.norm().item() + 1e-12, n_


def test_host_known_padding_pattern_equals_the_device_mask_path():
    """get_audio_representation(host_mask=...) (the HEAR chunk geometry, known on the host, repeating per clip) builds its
    packed index without a device read-back and must give exactly what the padding_mask path gives."""
    cfg = jo.Cfg()
    m = build_model(cfg, jo.make_state_dict(cfg, seed=5))
    T = m.total_patches
    P, reps = 5, 3
    pat = torch.zeros(P, T, dtype=torch.bool)
    pat[3, 150:] = True                       # a partly padded chunk
    pat[4, :] = True                          # a chunk that lies entirely in the padding
    pat[1, 20:40] = True                      # (not prefix-shaped: the index is general)
    audio = torch.randn(P * reps, 1, m.target_length, device=DEV).bfloat16()
    a = m.get_audio_representation(audio, pat.repeat(reps, 1).to(DEV))
    b = m.get_audio_representation(audio, None, host_mask=pat.numpy())
    assert torch.equal(a, b)
    b2 = m.get_audio_representation(audio, None, host_mask=pat.numpy())     # cached index
    assert torch.equal(a, b2)
    with pytest.raises(ValueError):
        m.get_audio_representation(audio[:7], None, host_mask=pat.numpy())


def test_deterministic_mode_is_bit_reproducible():
    """ops.set_deterministic(True): every reduction that ends in floating-point atomics takes the workspace + fixed-order
    path instead, so two identical models stepped on the same inputs end with bit-identical gradients, parameters, EMA
    teacher and loss -- and agree with the default mode up to summation order."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=5)
    inp = oi.training_inputs(cfg, 2, 4, seed=35, masker="audioset")
    audio = inp["audio"].to(DEV).bfloat16()
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    ref = build_model(cfg, sd)
    ref.global_step = 50000
    l_ref = ref.train_step(audio, c_m, t_m, v_m)
    ops.set_deterministic(True, 128 << 20)
    try:
        a, b = build_model(cfg, sd), build_model(cfg, sd)
        a.global_step = b.global_step = 50000
        for _ in range(2):     # two steps: the second starts from the first's (identical) update
            la, lb = a.train_step(audio, c_m, t_m, v_m), b.train_step(audio, c_m, t_m, v_m)
            assert la.item() == lb.item()
            assert torch.equal(a._flat_g, b._flat_g)
            assert torch.equal(a._flat_p, b._flat_p) and torch.equal(a._flat_t, b._flat_t)
    finally:
        ops.set_deterministic(False)
    a2 = build_model(cfg, sd)
    a2.global_step = 50000
    ops.set_deterministic(True, 128 << 20)
    try:
        l2 = a2.train_step(audio, c_m, t_m, v_m)
    finally:
        ops.set_deterministic(False)
    assert abs(l2.item() - l_ref.item()) < 1e-6
    for n_ in ref._train_names:
        g1, g2 = ref._view(ref._flat_g, n_).double(), a2._view(a2._flat_g, n_).double()
        # (the attention in_proj bias gradient is taken from the stored bf16 dqkv in this mode, from dO for the value
        # third in the default one: equal up to bf16 rounding of the summands, 4e-5)
        tol = 2e-4 if n_.endswith("in_proj_bias") else 1e-5
        assert (g1 - g2).norm().item() <= tol * g1.norm().item() + 1e-12, n_


def test_fused_train_step_equals_bridge_plus_torch_adamw():
    """train_step (hand-written backward + fused clip/AdamW/EMA) against the reference-style loop on a twin model
    (train.py:177-178, wavjepa/jepa.py:215-228, :330-331):
      (1) its gradients == the autograd-bridge gradients of forward().backward() (the same hand-written backward behind
          autograd: equal up to the order of the fp32 atomic sums in the parameter-gradient reductions);
      (2) its parameter update == clip_grad_norm_ + torch.optim.AdamW applied to those same gradients (tight);
      (3) the teacher moved by the EMA of the PRE-step student."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=5)
    inp = oi.training_inputs(cfg, 1, 4, seed=31, masker="audioset")
    a = build_model(cfg, sd)
    b = build_model(cfg, sd)
    a.global_step = b.global_step = 50000          # lr(0) == 0 would hide the optimizer (warm-up from 0)
    lr = b.lr_at(50000)
    audio = inp["audio"].to(DEV).bfloat16()
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    loss_a = a.train_step(audio, c_m, t_m, v_m)
    grads_a = {n: a._view(a._flat_g, n).clone() for n in a._train_names}
    out = b(audio, c_m, t_m, v_m)
    out["loss"].backward()
    assert abs(loss_a.item() - out["loss"].item()) < 1e-6
    pb = dict(b.named_parameters())
    for n_, g in grads_a.items():
        assert rel(g.cpu().numpy(), pb[n_].grad.cpu().numpy()) < GRAD_TOL, n_
    # (2) the reference optimizer step on model b, fed with model a's gradients
    trainables = [p for p in b.parameters() if p.requires_grad]
    for n_, g in grads_a.items():
        pb[n_].grad = g.clone()
    opt = torch.optim.AdamW(trainables, lr=lr, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.04)
    for p_ in trainables:   # the optimizer has taken 50000 steps (all with zero moments here): same bias correction
        opt.state[p_] = dict(step=torch.tensor(50000.0), exp_avg=torch.zeros_like(p_), exp_avg_sq=torch.zeros_like(p_))
    b._step_teacher()
    torch.nn.utils.clip_grad_norm_(trainables, 5.0)
    opt.step()
    pa = dict(a.named_parameters())
    for n_ in pa:
        d = (pa[n_].detach() - pb[n_].detach()).abs().max().item()
        scale = pb[n_].detach().abs().max().item() + 1e-12
        assert d <= 2e-6 * scale + 1e-3 * lr, (n_, d)
    # weights moved, teacher moved
    moved = (pa["encoder.layers.0.linear1.weight"].detach().cpu() - sd["encoder.layers.0.linear1.weight"]).abs().max()
    assert moved > 0
    assert a.global_step == 50001


def test_instances_are_independent_at_scale():
    """Size-independent property at a larger batch: every instance's local features / targets are unaffected by the
    other instances in the batch (no batch statistics anywhere, SURVEY.md 8e), and the loss of the batch equals the
    target-count-weighted mean of the per-half losses."""
    cfg = jo.Cfg()
    model = build_model(cfg, jo.make_state_dict(cfg, seed=2))
    B = 48
    g = torch.Generator().manual_seed(5)
    audio = torch.randn(B, 1, cfg.target_length, generator=g).to(DEV).bfloat16()
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, seed=9, row0=0)
    c_m, t_m, v_m = mk(batch_size=B, n_times=200, in_channels=1)
    with torch.no_grad():
        full = model(audio, c_m, t_m, v_m)
        h = B // 2
        lo = model(audio[:h], c_m[:h], t_m[:h], v_m[:h])
        hi = model(audio[h:], c_m[h:], t_m[h:], v_m[h:])
    assert torch.equal(full["local_features"][:h], lo["local_features"])
    assert torch.equal(full["targets"][h:], hi["targets"])
    n_lo, n_hi = t_m[:h].sum().item(), t_m[h:].sum().item()
    mix = (lo["loss"].item() * n_lo + hi["loss"].item() * n_hi) / (n_lo + n_hi)
    assert abs(full["loss"].item() - mix) / mix < 1e-5


@pytest.mark.parametrize("tag,n", [("3s", 48000), ("exact", 64318), ("10s", 160000)])
def test_hear_entry_points_match_reference_goldens(tag, n):
    g = np.load(os.path.join(GOLD, "hear.npz"))
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    model = hear.load_model({"state_dict": {k.replace("encoder.", "encoder._orig_mod.", 1) if k.startswith("encoder.")
                                            else k: v for k, v in sd.items()}})
    assert model.sample_rate == 16000 and model.scene_embedding_size == 768 and model.timestamp_embedding_size == 768
    assert model.unit_frames == 32159 and model.output_steps == 200
    audio = oi.hear_inputs(2, n, seed=11).to(DEV)
    emb, ts = hear.get_timestamp_embeddings(audio, model)
    assert list(emb.shape) == g[f"{tag}_shape"].tolist() and emb.dtype == torch.float32
    assert rel(oi.subsample(emb.cpu()), g[f"{tag}_emb"]) < FEAT_TOL
    assert abs(float(emb.norm()) - float(g[f"{tag}_l2"])) / float(g[f"{tag}_l2"]) < FEAT_TOL
    assert ts.shape == emb.shape[:2]
    assert np.allclose(ts[0].numpy(), g[f"{tag}_ts"], rtol=1e-6, atol=1e-4)
    if tag == "3s":
        scene = hear.get_scene_embeddings(audio, model)
        assert rel(scene.cpu().numpy(), g["3s_scene"]) < FEAT_TOL


def test_hear_against_live_oracle_with_silent_clip():
    """Edge cases of hear_api/feature_helper.py:5-13 and runtime.py:107-116: an all-zero clip (rms == 0 -> no gain,
    zero std chunks) next to a normal one, 1 s long (a single padded chunk)."""
    torch.set_num_threads(os.cpu_count())
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    audio = oi.hear_inputs(2, 16000, seed=3)
    audio[1] = 0
    with torch.no_grad():
        ref_emb, ref_ts = jo.hear_timestamp_embeddings(audio, sd, cfg)
    model = hear.load_model({"state_dict": sd})
    emb, ts = model(audio.to(DEV))
    assert emb.shape == ref_emb.shape == (2, 100, 768)
    assert rel(emb[0].cpu().numpy(), ref_emb[0].numpy()) < FEAT_TOL
    assert rel(emb[1].cpu().numpy(), ref_emb[1].numpy()) < FEAT_TOL
    assert torch.allclose(ts, ref_ts)


# ------------------------------------------------------------------------------------------------- 8(f)-3 interop rows
def test_arch_wrapper_matches_reference_goldens():
    from wavjepa_b200.arch import WavJEPAModelWrapper

    g = np.load(os.path.join(GOLD, "interop.npz"))
    cfg = jo.Cfg()
    model = build_model(cfg, jo.make_state_dict(cfg, seed=3))
    wrap = WavJEPAModelWrapper(model, DEV, None)
    assert wrap.get_sampling_rate() == 16000 and wrap.get_classification_embedding_size() == 768
    for tag, n in (("a", 40000), ("b", 64318)):
        v = wrap.get_embeddings(oi.hear_inputs(1, n, seed=21)[0])
        assert v.shape == (768,)
        assert rel(v.cpu().numpy(), g[f"arch_{tag}"]) < FEAT_TOL, tag
    with pytest.raises(TypeError):
        wrap.get_sequence_embeddings(torch.zeros(16000))


def test_w2v2_extractor_hear_model_matches_reference_goldens():
    g = np.load(os.path.join(GOLD, "interop.npz"))
    cfg2 = jo.Cfg(spec=hear.W2V2_SPEC, seconds=4.02)
    model = hear.load_model_w2v2({"state_dict": jo.make_state_dict(cfg2, seed=3)})
    assert model.unit_frames == 64319 and model.output_steps == 200
    emb, ts = model.get_timestamp_embeddings(oi.hear_inputs(2, 100000, seed=12).to(DEV))
    assert list(emb.shape) == g["w2v2_shape"].tolist()
    assert rel(oi.subsample(emb.cpu()), g["w2v2_emb"]) < FEAT_TOL
    assert np.allclose(ts[0].numpy(), g["w2v2_ts"], rtol=1e-6, atol=1e-4)


def test_large_model_forward_matches_reference_goldens():
    g = np.load(os.path.join(GOLD, "interop.npz"))
    cfgL = jo.Cfg(d_model=1024, nhead=16, layers=24)
    ex = w.ConvFeatureExtractor(conv_layers_spec=cfgL.spec, in_channels=1)
    model = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                   transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
                   process_audio_seconds=2.01, nr_samples_per_audio=8, average_top_k_layers=8, size="large")
    assert model.encoder_embedding_dim == 1024 and len(model.encoder.layers) == 24
    model.load_state_dict(jo.make_state_dict(cfgL, seed=3), strict=True)
    model.to(DEV)
    inp = oi.training_inputs(cfgL, 1, 2, seed=77, masker="audioset")
    with torch.no_grad():
        out = model(inp["audio"].to(DEV).bfloat16(), inp["ctx_masks"].to(DEV), inp["target_indices"].to(DEV),
                    inp["ctx_and_target_masks"].to(DEV))
    assert abs(out["loss"].item() - float(g["large_loss"])) / float(g["large_loss"]) < LOSS_TOL
    assert rel(oi.subsample(out["local_features"].cpu()), g["large_local"]) < FEAT_TOL
    assert rel(oi.subsample(out["targets"].cpu()), g["large_targets"]) < 1.5 * FEAT_TOL   # 24 layers of bf16 operands


def test_checkpoint_round_trip(tmp_path):
    """Lightning-style checkpoint with torch.compile's `_orig_mod` infix (hear_api/runtime.py:63-77) -> load_model(path);
    and our state_dict written back has the reference's names."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=9)
    ck = {"state_dict": {(k.replace("extract_audio.", "extract_audio._orig_mod.", 1) if k.startswith("extract_audio.")
                          else k.replace("decoder.", "decoder._orig_mod.", 1) if k.startswith("decoder.") else k): v
                         for k, v in sd.items()}, "global_step": 123}
    path = str(tmp_path / "step=123.ckpt")
    torch.save(ck, path)
    rt = hear.load_model(path)
    back = rt.model.state_dict()
    assert list(back.keys()) == list(sd.keys())
    for k in ("extract_audio.cnn.3.0.weight", "decoder.layers.4.linear1.bias", "teacher_encoder.layers.7.norm2.weight",
              "pos_encoding_decoder", "mask_token"):
        assert torch.equal(back[k].cpu(), sd[k]), k


# ------------------------------------------------------------------------------------------------- 8(f)-2 input pipeline
def test_gpu_input_pipeline_matches_reference_preprocessing():
    """Resample (Kaiser sinc) -> -14 dBFS RMS -> pad / crop to 10 s on the GPU == the data module's CPU path
    (WebAudioDataModule.py:43-61, dataset_functions.py:92-114) restated with the reference's own resampler."""
    pytest.importorskip("torchaudio")
    from wavjepa_b200.preprocess import GpuAudioPipeline

    g = torch.Generator().manual_seed(3)
    cases = [(48000, 5.0, 1), (44100, 12.3, 2), (16000, 10.0, 1), (22050, 3.7, 1), (32000, 10.0, 1), (8000, 2.0, 1),
             (16000, 11.0, 1), (44100, 0.05, 1)]
    waves, srs = [], []
    for sr_, dur, ch in cases:
        n = int(sr_ * dur)
        wv = torch.randn(ch, n, generator=g) * 0.1 if ch > 1 else torch.randn(n, generator=g) * 0.1
        waves.append(wv)
        srs.append(sr_)
    waves.append(torch.zeros(30000))          # silent clip: rms == 0 -> untouched
    srs.append(48000)
    pipe = GpuAudioPipeline(sr=16000, seconds=10, device=DEV)
    clips = pipe(waves, srs)
    assert clips.shape == (len(waves), 1, 160000) and clips.dtype == torch.float32
    for i, (wv, sr_) in enumerate(zip(waves, srs)):
        ref = jo.data_pre_process(wv, sr_)
        got = clips[i].cpu()
        scale = ref.abs().max().item() + 1e-12
        assert (got - ref).abs().max().item() <= 2e-5 * scale + 1e-7, (i, sr_, (got - ref).abs().max().item(), scale)
    assert clips[-1].abs().max().item() == 0.0
    # feeds the training hook directly
    model = build_model(jo.Cfg(), jo.make_state_dict(jo.Cfg(), seed=3))
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, seed=1, row0=0)
    n = clips.shape[0]
    c_m, t_m, v_m = mk(batch_size=n * 8, n_times=200, in_channels=1)
    x16, *_ = model.on_after_batch_transfer((clips, c_m.view(n, 8, -1), t_m.view(n, 8, 4, -1), v_m.view(n, 8, 4, -1)), 0)
    assert x16.shape == (n * 8, 1, 32159) and torch.isfinite(x16.float()).all()


# ------------------------------------------------------------------------------------------------- denoiser stage
def _denoiser(alpha, nr=2):
    from wavjepa_b200.denoiser import Denoiser
    cfg = jo.Cfg()
    ext = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=1)
    m = Denoiser(feature_extractor=ext, transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                 transformer_encoder_cfg=w.TransformerEncoderCFG.create(), resample_sr=16000,
                 process_audio_seconds=2.01, nr_samples_per_audio=nr, size="base", alpha=alpha)
    sd_s = jo.make_state_dict(cfg, seed=11)
    own = {k: v for k, v in sd_s.items() if k in m.state_dict()}
    m.load_state_dict(own, strict=True)
    m._set_teacher({"state_dict": jo.make_state_dict(cfg, seed=12)})
    return m.to(DEV)


def test_denoiser_stage_matches_reference_goldens():
    """SURVEY.md 8(f)-4: scene generation + resampling + crops, Denoiser.forward losses and every parameter gradient
    against the fixtures of the executed reference (fp32 CPU); bf16 kernels -> the tolerances of the JEPA step."""
    g = np.load(os.path.join(GOLD, "denoiser.npz"))
    meta = json.load(open(os.path.join(GOLD, "denoiser.json")))
    m = _denoiser(meta["alpha"])
    batch = oi.denoiser_batch()
    starts, perm = torch.from_numpy(g["starts"]), torch.from_numpy(g["perm"])
    gen16, clean16 = m.on_after_batch_transfer(tuple(t.to(DEV) for t in batch), 0, starts=starts, perm=perm)
    assert gen16.dtype == torch.bfloat16 and tuple(gen16.shape) == (4, 1, 32159)
    assert rel(oi.subsample(gen16.float().cpu()), g["gen"]) < 3e-3
    assert rel(oi.subsample(clean16.float().cpu()), g["clean"]) < 3e-3
    assert abs(float(gen16.float().norm()) - float(g["gen_l2"])) / float(g["gen_l2"]) < 1e-3
    # the reference's own inputs (restated on the host, pinned in tests/test_oracle_cpu.py) for the model comparison
    gen_o, clean_o = jo.denoiser_batch(batch, starts, perm)
    out, grads = m.forward_backward(gen_o.bfloat16().to(DEV), clean_o.bfloat16().to(DEV))
    for k, gk in (("loss", "loss"), ("loss_clean", "loss_clean"), ("loss_denoise_dereverb", "loss_dd")):
        assert abs(out[k].item() - float(g[gk])) / float(g[gk]) < 2e-3, (k, out[k].item(), float(g[gk]))
    out_f = m(gen_o.bfloat16().to(DEV), clean_o.bfloat16().to(DEV))
    assert abs(out_f["loss"].item() - out["loss"].item()) < 1e-5
    for n_, ref_norm in meta["grad_norms"].items():
        e = abs(float(grads[n_].norm()) - ref_norm) / (ref_norm + 1e-12)
        assert e < GRAD_TOL, (n_, e)
    for k in g.files:
        if k.startswith("grad:"):
            e = rel(oi.subsample(grads[k[5:]].cpu()), g[k])
            assert e < GRAD_TOL, (k, e)


def test_denoiser_train_step_learns():
    m = _denoiser(0.25, nr=4)
    m.global_step = 5000                      # past the warm-up: lr = 1e-4
    g = torch.Generator().manual_seed(0)
    clean = torch.randn(8, 1, 32159, generator=g).bfloat16().to(DEV)
    gen = (clean.float() + 0.3 * torch.randn(8, 1, 32159, generator=g).to(DEV)).bfloat16()
    before = {n: p.detach().clone() for n, p in m.named_parameters() if p.requires_grad}
    teacher_before = m.teacher.encoder.layers[0].linear1.weight.detach().clone()
    losses = [m.train_step(gen, clean)["loss"].item() for _ in range(6)]
    assert losses[-1] < losses[0], losses
    assert m.global_step == 5006
    moved = [n for n, p in m.named_parameters() if p.requires_grad and not torch.equal(p.detach(), before[n])]
    assert "encoder.layers.0.linear1.weight" in moved and "extract_audio.cnn.0.0.weight" in moved
    assert torch.equal(m.teacher.encoder.layers[0].linear1.weight, teacher_before)      # frozen


def test_generate_scene_cases():
    """The four branches of generate_scene (generate_scenes_batch.py:148-188) and the 32 -> 16 kHz resampler."""
    import torchaudio
    from wavjepa_b200 import denoiser as dn
    audio, source_rir, noise, noise_len, noise_start, noise_rirs, snr = oi.denoiser_batch(B=3, T32=40000, rir_len=1500, seed=9)
    dev = lambda t: t.to(DEV)
    # RIR and noise: pinned by the golden test above; here against the live oracle on a different batch
    full = dn.generate_scene(dev(source_rir), dev(noise_rirs), dev(audio), dev(noise), dev(noise_len), dev(noise_start), dev(snr))
    assert rel(full.cpu().numpy(), jo.generate_scene(source_rir, noise_rirs, audio, noise, noise_len, noise_start, snr).numpy()) < 1e-5
    # RIR only
    only_rir = dn.generate_scene(dev(source_rir), None, dev(audio), [None], None, None, None)
    assert tuple(only_rir.shape) == (3, 1, 40000)
    assert rel(only_rir.cpu().numpy(), jo.scene_convolve_with_rir(audio, source_rir[:, [0]]).numpy()) < 1e-5
    # noise only (raw source + scaled noise)
    only_noise = dn.generate_scene([None], None, dev(audio), dev(noise), dev(noise_len), dev(noise_start), dev(snr))
    ref = jo.scene_add_noise(audio[:, None], noise[:, None], snr, noise_start, noise_len)
    assert rel(only_noise.cpu().numpy(), ref.numpy()) < 1e-6
    # neither: the source passes through
    assert dn.generate_scene([None], None, dev(audio), [None], None, None, None) is not None
    assert torch.equal(dn.generate_scene([None], None, dev(audio), [None], None, None, None).cpu(), audio)
    # resample == torchaudio with the reference's arguments (wavjepa/denoiser.py:29-41)
    r = dn.resample(dev(audio).unsqueeze(1), 16000, 32000)
    t = torchaudio.functional.resample(audio.unsqueeze(1), 32000, 16000, lowpass_filter_width=64, rolloff=0.9475937167399596,
                                       resampling_method="sinc_interp_kaiser", beta=14.769656459379492)
    assert tuple(r.shape) == tuple(t.shape) and rel(r.cpu().numpy(), t.numpy()) < 1e-5


# ------------------------------------------------------------------------------------------------- round-2 additions
GRAD_CASES = [("audioset", dict(), 3, 2024), ("librispeech", dict(), 2, 77), ("audioset", dict(in_channels=2, per_channel=True), 2, 5)]


@pytest.mark.parametrize("masker,cfgkw,crops,seed", GRAD_CASES)
def test_every_parameter_gradient_elementwise_against_live_oracle(masker, cfgkw, crops, seed):
    """Direction, not only norm: the FULL gradient tensor of EVERY trainable parameter (rel-L2 over all elements) against
    the fp32 CPU oracle (itself pinned to the executed reference by tests/golden) on inputs that are not in the fixtures.
    The key third of in_proj_bias has an exactly-zero true gradient (softmax is invariant to a constant key shift); both
    sides only hold rounding noise there, so it is compared as part of the whole bias tensor."""
    torch.set_num_threads(os.cpu_count())
    cfg = jo.Cfg(**cfgkw)
    sd = jo.make_state_dict(cfg, seed=seed)
    inp = oi.training_inputs(cfg, 1, crops, seed=seed, masker=masker)
    ref_sd = {k: v.clone().requires_grad_(not k.startswith(("teacher_encoder.", "pos_encoding"))) for k, v in sd.items()}
    ref = jo.forward(inp["audio"], inp["ctx_masks"], inp["target_indices"], inp["ctx_and_target_masks"], ref_sd, cfg)
    ref["loss"].backward()
    model = build_model(cfg, sd)
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    out = model(inp["audio"].to(DEV).bfloat16(), c_m, t_m, v_m)
    assert abs(out["loss"].item() - ref["loss"].item()) / ref["loss"].item() < LOSS_TOL
    out["loss"].backward()
    worst, n_checked = ("", 0.0), 0
    for n_, p_ in model.named_parameters():
        if not p_.requires_grad:
            continue
        g_ref = ref_sd[n_].grad
        assert g_ref is not None and p_.grad is not None, n_
        e = rel(p_.grad.cpu().numpy(), g_ref.numpy())
        worst = max(worst, (n_, e), key=lambda t: t[1])
        n_checked += 1
        assert e < GRAD_TOL, (n_, e)
    assert n_checked >= 300, n_checked
    print(f"worst per-tensor gradient rel-L2: {worst}")


def test_parity_at_b512_on_sampled_instances():
    """BASELINE.json configs[1] size (512 instances): instances are independent, so the features / targets / predictions
    of a few instances of the full batch must equal the oracle run on just those instances."""
    torch.set_num_threads(os.cpu_count())
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=8)
    B = 512
    g = torch.Generator().manual_seed(123)
    audio = torch.randn(B, 1, cfg.target_length, generator=g).bfloat16()
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, seed=4, row0=0)
    c_m, t_m, v_m = mk(batch_size=B, n_times=200, in_channels=1)
    model = build_model(cfg, sd)
    with torch.no_grad():
        out = model(audio.to(DEV), c_m, t_m, v_m)
    pick = [0, 137, 300, 511]
    with torch.no_grad():
        ref = jo.forward(audio[pick].float(), c_m[pick].cpu(), t_m[pick].cpu(), v_m[pick].cpu(), sd, cfg)
    assert rel(out["local_features"][pick].cpu().numpy(), ref["local_features"].numpy()) < FEAT_TOL
    assert rel(out["targets"][pick].cpu().numpy(), ref["targets"].numpy()) < FEAT_TOL
    G, T = t_m.shape[1], t_m.shape[2]
    ours = out["preds"].view(B, G, T, -1)[pick][t_m[pick]].float().cpu().numpy()
    theirs = ref["preds"].view(len(pick), G, T, -1)[t_m[pick].cpu()].numpy()
    assert rel(ours, theirs) < FEAT_TOL
    assert torch.isfinite(out["loss"]).item()


def test_optimizer_state_round_trip():
    """ADVICE r1: a fused-path run must be resumable.  checkpoint() after two steps -> load_checkpoint() into a fresh
    model -> the third step matches the uninterrupted run (same LR / EMA schedule position, same Adam moments)."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=21)
    inp = oi.training_inputs(cfg, 1, 2, seed=9, masker="audioset")
    audio = inp["audio"].to(DEV).bfloat16()
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    a = build_model(cfg, sd)
    a.global_step = 60000
    for _ in range(2):
        a.train_step(audio, c_m, t_m, v_m)
    ck = a.checkpoint()
    assert ck["global_step"] == 60002 and len(ck["optimizer_states"][0]["state"]) == len(a._train_names)
    b = build_model(cfg, None)
    b.load_checkpoint(ck)
    assert b.global_step == 60002
    assert torch.equal(b._adam_m, a._adam_m) and torch.equal(b._adam_v, a._adam_v)
    # .to() of an already-initialised model keeps the moments (they used to be dropped with the flat buffers)
    m_before = b._adam_m.clone()
    b.to("cpu")
    b.to(DEV)
    b._ensure_ready()
    assert b._adam_m is not None and torch.equal(b._adam_m, m_before)
    la = a.train_step(audio, c_m, t_m, v_m)
    lb = b.train_step(audio, c_m, t_m, v_m)
    assert abs(la.item() - lb.item()) < 1e-5
    pa, pb = dict(a.named_parameters()), dict(b.named_parameters())
    for n_ in pa:   # (fp32 atomics in two backward kernels make two runs differ by rounding noise, not more)
        d = (pa[n_].detach() - pb[n_].detach()).abs().max().item()
        assert d <= 1e-5 * (pa[n_].detach().abs().max().item() + 1e-12) + 1e-8, (n_, d)
    ta, tb = dict(a.teacher_encoder.named_parameters()), dict(b.teacher_encoder.named_parameters())
    for n_ in ta:
        assert torch.allclose(ta[n_], tb[n_], rtol=0, atol=1e-7), n_
    # a restart WITHOUT the optimizer state is visibly different (this is what the API prevents)
    c = build_model(cfg, {k: v for k, v in ck["state_dict"].items()})
    assert c.global_step == 0 and c.lr_at(c.global_step) == 0.0


def test_stock_optimizer_path_advances_global_step():
    """ADVICE r1: forward() + loss.backward() + configure_optimizers(): without a Lightning trainer the optimizer's step
    hook advances global_step, so the EMA decay anneals (wavjepa/jepa.py:186-191)."""
    cfg = jo.Cfg()
    model = build_model(cfg, jo.make_state_dict(cfg, seed=1))
    inp = oi.training_inputs(cfg, 1, 2, seed=3, masker="audioset")
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    opt = model.configure_optimizers()["optimizer"]
    d0 = model._get_ema_decay()
    for _ in range(2):
        out = model.training_step((inp["audio"].to(DEV).bfloat16(), c_m, t_m, v_m), 0)
        out["loss"].backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
    assert model.global_step == 2 and model._get_ema_decay() > d0


def test_denoiser_default_clip_is_the_reference_trainers():
    """ADVICE r1: the reference trains the denoiser stage with gradient_clip_val=1.0 (denoise.py:125-126).  The fused
    step == clip_grad_norm_(1.0) + torch.optim.AdamW on the same gradients."""
    m = _denoiser(0.25, nr=2)
    assert m._core.grad_clip == 1.0
    m.global_step = 5000
    g = torch.Generator().manual_seed(3)
    clean = torch.randn(4, 1, 32159, generator=g).bfloat16().to(DEV)
    gen = (clean.float() + 0.5 * torch.randn(4, 1, 32159, generator=g).to(DEV)).bfloat16()
    before = {n: p.detach().clone() for n, p in m.named_parameters() if p.requires_grad and not n.startswith("teacher.")}
    _, grads = m.forward_backward(gen, clean)
    grads = {n: gr.clone() for n, gr in grads.items()}
    total = torch.sqrt(sum((gr.double() ** 2).sum() for gr in grads.values())).item()
    assert total > 1.0, "the test needs a gradient norm above the clip value"
    twins = {n: torch.nn.Parameter(before[n].clone()) for n in grads}
    for n, gr in grads.items():
        twins[n].grad = gr.clone()
    opt = torch.optim.AdamW(list(twins.values()), lr=m.lr_at(5000), betas=m.hparams.adam_betas, eps=m.hparams.adam_eps,
                            weight_decay=m.hparams.adam_weight_decay)
    for p_ in twins.values():
        opt.state[p_] = dict(step=torch.tensor(5000.0), exp_avg=torch.zeros_like(p_), exp_avg_sq=torch.zeros_like(p_))
    torch.nn.utils.clip_grad_norm_(list(twins.values()), 1.0)
    opt.step()
    m.train_step(gen, clean)
    now = dict(m.named_parameters())
    for n in grads:   # (the second backward differs from the first by atomics noise only)
        d = (now[n].detach() - twins[n].detach()).abs().max().item()
        assert d <= 1e-2 * m.lr_at(5000) + 2e-6 * twins[n].detach().abs().max().item(), (n, d)


def test_shared_conv_weights_are_announced_once_final():
    """ADVICE r1: with share_weights_over_channels=True both channel passes add into the same conv gradients; a bucket
    must not be announced (and all-reduced) before the last pass.  A recording reducer checks that nothing changes in
    flat[offset:] after ready(offset).  The denoiser's backward announces its buckets the same way."""
    cfg = jo.Cfg(in_channels=2, per_channel=True)
    ex = w.ConvChannelFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=2, share_weights_over_channels=True)
    model = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                   transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
                   process_audio_seconds=2.01, nr_samples_per_audio=2, average_top_k_layers=8).to(DEV)
    model.global_step = 1000

    class Recorder:
        world_size = 1

        def __init__(self):
            self.flat, self.log = None, []

        def begin(self, flat):
            self.flat, self.log = flat, []

        def ready(self, offset):
            self.log.append((offset, self.flat[offset:].double().sum().item(), self.flat[offset:].abs().double().sum().item()))

        def finish(self):
            pass

    rec = Recorder()
    model.attach_data_parallel(rec, sync=False)
    g = torch.Generator().manual_seed(1)
    audio = torch.randn(2, 2, cfg.target_length, generator=g).bfloat16().to(DEV)
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, channel_based_masking=True, seed=2, row0=0)
    c_m, t_m, v_m = mk(batch_size=2, n_times=400, in_channels=2)
    model.train_step(audio, c_m, t_m, v_m)
    den = _denoiser(0.25, nr=2)
    den_rec = Recorder()
    den.attach_data_parallel(den_rec, sync=False)
    clean = torch.randn(4, 1, 32159, generator=g).bfloat16().to(DEV)
    gen = (clean.float() + 0.5 * torch.randn(4, 1, 32159, generator=g).to(DEV)).bfloat16()
    den.forward_backward(gen, clean)
    for r, flat in ((rec, model._flat_g), (den_rec, den._core._flat_g)):
        assert len(r.log) > 20
        offs = [o for o, _, _ in r.log]
        assert offs == sorted(offs, reverse=True), "ready() offsets must move from the end of the buffer to its start"
        for off, s1, s2 in r.log:
            assert flat[off:].double().sum().item() == s1 and flat[off:].abs().double().sum().item() == s2, off


@pytest.mark.parametrize("kind", ["mono", "w2v2", "nat", "nat_shared"])
def test_standalone_extractor_forward_equals_the_models_conv_output(kind):
    """`extract_audio(x)` is, bit for bit, the conv output the model computes from its flat buffers for the same audio
    (w2v2 at 4.02 s: a 401-row input to its last block), and after a fused train_step, which updates the parameters in
    place without bumping their versions, it reads the updated weights."""
    spec, seconds = (hear.W2V2_SPEC, 4.02) if kind == "w2v2" else (hear.BASE_SPEC, 2.01)
    if kind.startswith("nat"):
        ex = w.ConvChannelFeatureExtractor(conv_layers_spec=spec, in_channels=2,
                                           share_weights_over_channels=kind == "nat_shared")
    else:
        ex = w.ConvFeatureExtractor(conv_layers_spec=spec, in_channels=1)
    model = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                   transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
                   transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
                   process_audio_seconds=seconds, nr_samples_per_audio=2, average_top_k_layers=8).to(DEV)
    model.global_step = 50000   # an lr at which one step moves the bf16 working weights
    Cin, T = ex.in_channels, model.total_patches
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, Cin, model.target_length, generator=g).bfloat16().to(DEV)
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, channel_based_masking=Cin == 2, seed=6, row0=0)
    masks = mk(batch_size=2, n_times=T, in_channels=Cin)

    def model_conv_output():
        _, (_, f2, _, _) = model._local_features(x, save=False)
        return f2.view(2, T, -1)

    model.train_step(x, *masks)   # builds the flat buffers: the parameters keep their storage from here on
    before = model.extract_audio(x)
    assert before.shape == (2, T, ex.embedding_dim) and before.dtype == torch.bfloat16
    assert torch.equal(before, model_conv_output())
    model.train_step(x, *masks)
    after = model.extract_audio(x)
    assert not torch.equal(after, before)
    assert torch.equal(after, model_conv_output())


def test_hear_nat_runtime_matches_reference_goldens():
    """VERDICT r1 missing 5: the binaural HEAR runtime (hear_api/runtime_natjepa.py: channel fix-up, joint normalisation,
    channel-major mask, channel mean) against fixtures made by EXECUTING the reference's get_timestamp_embeddings
    (tests/golden/make_golden.py::golden_hear_nat) and against the live oracle on fresh inputs."""
    torch.set_num_threads(os.cpu_count())
    g = np.load(os.path.join(GOLD, "hear_nat.npz"))
    cfg = jo.Cfg(in_channels=2, per_channel=True)
    sd = jo.make_state_dict(cfg, seed=3)
    model = hear.load_model_nat({"state_dict": sd})
    assert model.output_steps == 200 and model.unit_frames == 32159 and model.embedding_size == 768
    gen = torch.Generator().manual_seed(17)
    stereo = torch.rand(2, 2, 48000, generator=gen) * 2 - 1
    emb, ts = hear.get_timestamp_embeddings(stereo.to(DEV), model)
    assert list(emb.shape) == list(g["stereo_shape"]) and np.allclose(ts[0].cpu().numpy(), g["stereo_ts"], rtol=1e-6)
    assert rel(oi.subsample(emb.cpu()), g["stereo_emb"]) < FEAT_TOL
    assert abs(float(emb.norm()) - float(g["stereo_l2"])) / float(g["stereo_l2"]) < 2e-3
    scene = hear.get_scene_embeddings(stereo.to(DEV), model)
    assert rel(scene.cpu().numpy(), g["stereo_scene"]) < FEAT_TOL
    mono = oi.hear_inputs(2, 40000, seed=19)
    emb, ts = model.get_timestamp_embeddings(mono.to(DEV))       # mono input is duplicated onto both channels
    assert list(emb.shape) == list(g["mono_shape"]) and rel(oi.subsample(emb.cpu()), g["mono_emb"]) < FEAT_TOL
    # live oracle, exact multiple of the unit (a whole extra padded chunk) and a 4-channel clip
    four = torch.rand(1, 4, 64318, generator=gen) * 2 - 1
    with torch.no_grad():
        ref, rts = jo.hear_nat_timestamp_embeddings(four, sd, cfg)
    emb, ts = model.get_timestamp_embeddings(four.to(DEV))
    assert tuple(emb.shape) == tuple(ref.shape) == (1, 400, 768)
    assert rel(emb.cpu().numpy(), ref.numpy()) < FEAT_TOL and np.allclose(ts.cpu().numpy(), rts.numpy(), rtol=1e-6)
    with pytest.raises(_lib.WavJepaLibError):
        hear.RuntimeJEPA(in_channels=2, weights={"state_dict": sd}, is_spectrogram=False, process_seconds=2.01,
                         extractor=w.ConvChannelFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=2), model_size="base", sr=16000)


def test_hf_call_shape(tmp_path):
    """VERDICT r1 missing 3 / SURVEY H5: AutoFeatureExtractor / AutoModel call shape of README.md:72-108 and
    hear_configs/WavJEPA_huggingface.py (values = the HEAR runtime's, which the goldens pin)."""
    from wavjepa_b200 import hf
    g = np.load(os.path.join(GOLD, "hear.npz"))
    cfg = jo.Cfg()
    path = os.path.join(tmp_path, "ckpt.pt")
    torch.save({"state_dict": {k.replace("encoder.", "encoder._orig_mod.", 1) if k.startswith("encoder.") else k: v
                               for k, v in jo.make_state_dict(cfg, seed=3).items()}}, path)
    model = hf.WavJEPAModel.from_pretrained(path, trust_remote_code=True).to(DEV)
    ext = hf.WavJEPAFeatureExtractor.from_pretrained("labhamlet/wavjepa-base", trust_remote_code=True)
    audio = oi.hear_inputs(2, 160000, seed=11)
    feats = ext(audio.to(DEV), return_tensors="pt")["input_values"]
    emb, ts = model(feats)
    assert tuple(emb.shape) == (2, 996, 768) and tuple(ts.shape) == (2, 996)
    assert rel(oi.subsample(emb.cpu()), g["10s_emb"]) < FEAT_TOL and np.allclose(ts[0].cpu().numpy(), g["10s_ts"], rtol=1e-6)
    m2 = hf.load_model(path)
    assert m2.sample_rate == 16000
    e2, _ = hf.get_timestamp_embeddings([audio[0], audio[1, :150000]], m2)   # ragged list -> zero-padded batch
    assert tuple(e2.shape) == (2, 996, 768)
    assert tuple(hf.get_scene_embeddings(audio.to(DEV), m2).shape) == (2, 768)
    # the Nat pair: [B, 2, L] in, same call
    nat_sd = jo.make_state_dict(jo.Cfg(in_channels=2, per_channel=True), seed=3)
    nat = hf.WavJEPAModel.from_pretrained({"state_dict": nat_sd})
    assert isinstance(nat.runtime, hear.RuntimeNatJEPA)
    emb, ts = nat(hf.WavJEPAFeatureExtractor.from_pretrained("labhamlet/wavjepa-nat-base")(torch.zeros(1, 2, 48000))["input_values"])
    assert tuple(emb.shape) == (1, 299, 768)


def test_gpu_batch_assembler_tuple_contract():
    """VERDICT r1 missing 8: the 4-tuple of WebAudioDataModule._retrieve_sample + .batched (WebAudioDataModule.py:43-74)
    assembled on the device: audio == the CPU preprocessing of the data module, masks == the seeded masker's."""
    import torchaudio
    from wavjepa_b200.data import GpuBatchAssembler
    g = torch.Generator().manual_seed(3)
    samples = [(torch.randn(2, 44100 * 3, generator=g) * 0.1, 44100), (torch.randn(16000 * 12, generator=g) * 0.3, 16000),
               (torch.randn(48000 * 5, generator=g) * 0.05, 48000)]
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, seed=11, row0=5, device=DEV)
    asm = GpuBatchAssembler(mk, nr_samples_per_audio=8, nr_time_points=200, in_channels=1, device=DEV)
    audio, c_m, t_m, v_m = asm(samples)
    assert tuple(audio.shape) == (3, 1, 160000) and tuple(c_m.shape) == (3, 8, 200) and tuple(t_m.shape) == (3, 8, 4, 200)
    for i, (wv, sr) in enumerate(samples):
        ref = jo.data_pre_process(wv, sr)[0]
        assert rel(audio[i, 0].cpu().numpy(), ref.numpy()) < 1e-4, i
    rc, rt, rv, _ = mo.time_inverse_masks(11, 5, 24, 200)
    assert np.array_equal(c_m.reshape(24, 200).cpu().numpy(), rc) and np.array_equal(v_m.reshape(24, 4, 200).cpu().numpy(), rv)
    # the tuple feeds the training hook unchanged
    model = build_model(jo.Cfg(), jo.make_state_dict(jo.Cfg(), seed=3))
    x16, c2, t2, v2 = model.on_after_batch_transfer((audio, c_m, t_m, v_m), 0)
    assert tuple(x16.shape) == (24, 1, 32159) and tuple(c2.shape) == (24, 200) and tuple(t2.shape) == (24, 4, 200)
    model.shuffle_crops = True      # reference behaviour: audio rows permuted, masks untouched (jepa.py:314-316)
    x16s, c3, _, _ = model.on_after_batch_transfer((audio, c_m, t_m, v_m), 0)
    assert torch.equal(c3, c2) and x16s.shape == x16.shape
