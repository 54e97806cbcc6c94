"""The reference-precision (TF32) inference mode on the B200: its kernels against plain fp32 restatements in torch, the
HEAR / Nat / w2v2 / ARCH entry points against the reference's fp32 goldens and the live CPU oracle, and its contract
(opt-in, the default bf16 path unchanged, training unaffected).

Tolerances: kernels against an fp64 product of the same pre-rounded operands 2e-5 (summation order only); outputs rounded
to tf32 against the reference rounded the same way 1e-4; end to end 2e-3 relative L2 per returned tensor, and at most
0.35 x the distance of the bf16 path on the same input."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import wavjepa_b200 as w  # noqa: E402
from wavjepa_b200 import _lib, hear, ops  # noqa: E402
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
DEV = "cuda"

FP32_TOL = 2e-5
ROUNDED_TOL = 1e-4
E2E_TOL = 2e-3
GAIN = 0.35


def rel(a, b):
    a = np.asarray(torch.as_tensor(a).double().cpu() if torch.is_tensor(a) else a, dtype=np.float64)
    b = np.asarray(torch.as_tensor(b).double().cpu() if torch.is_tensor(b) else b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


def tf32r(x: torch.Tensor) -> torch.Tensor:
    """Round to nearest tf32, ties away from zero (cvt.rna.tf32.f32)."""
    b = x.float().contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def low_bits_zero(x: torch.Tensor) -> bool:
    return bool(((x.contiguous().view(torch.int32) & 0x1FFF) == 0).all())


@pytest.fixture(autouse=True, scope="module")
def _device():
    _lib.require_device()
    torch.manual_seed(0)


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, device=DEV, generator=g) * scale


# ------------------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("M,N,K,epi", [
    (1000, 2304, 768, "bias_bf16"),          # in_proj -> qkv (M not a multiple of 128)
    (1024, 3072, 768, "bias_gelu_round"),    # linear1 + exact GELU (operand of linear2)
    (777, 768, 3072, "bias_f32"),            # linear2
    (640, 768, 512, "bias_resid"),           # post_extraction_mapper + positional table
    (300, 640, 256, "plain_round"),          # N % 256 != 0: 128-column tiles
])
def test_gemm_tf32_linear(M, N, K, epi):
    a = tf32r(_rand(M, K, seed=1))
    wt = tf32r(_rand(N, K, scale=K ** -0.5, seed=2))
    bias = _rand(N, scale=0.1, seed=3)
    ref = a.double() @ wt.double().T
    kw = {}
    if epi != "plain_round":
        kw["bias"] = bias
        ref = ref + bias.double()
    if epi == "bias_resid":
        T = 160
        pos = _rand(T, N, seed=4)
        kw.update(resid=pos, resid_mod=T)
        ref = ref + pos.double().repeat(M // T + 1, 1)[:M]
    if epi == "bias_gelu_round":
        kw["act"] = ops.ACT_GELU_ERF
        ref = F.gelu(ref)
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16 if epi == "bias_bf16" else torch.float32)
    ops.gemm_tf32(ops.plain_operand(a), wt, M, 1, out, round_out=epi.endswith("round"), **kw)
    if epi == "bias_bf16":
        assert rel(out, ref) < 4e-3                                   # bf16 resolution
        assert rel(out, ref.to(torch.bfloat16)) < 3e-4
    elif epi.endswith("round"):
        assert low_bits_zero(out)
        assert rel(out, tf32r(ref)) < ROUNDED_TOL
        assert rel(out, ref) < 1e-3
    else:
        assert rel(out, ref) < FP32_TOL


@pytest.mark.parametrize("k,L_in", [(3, 200), (3, 201), (2, 100), (2, 101)])
def test_gemm_tf32_conv(k, L_in):
    """Conv1d(512, 512, k, stride 2) + exact GELU as an implicit GEMM over channels-last fp32 activations, at even input
    lengths (pair view) and odd ones (inference only: the w2v2 spec)."""
    B, C = 3, 512
    x = tf32r(_rand(B, L_in, C, seed=5))
    wk = tf32r(_rand(C, k * C, scale=(k * C) ** -0.5, seed=6))   # tap-major [O, k*C]
    L_out = (L_in - k) // 2 + 1
    g = torch.empty(B, L_out, C, device=DEV)
    a_op = ops.conv_operand(x, k) if L_in % 2 == 0 else \
        ops.make_operand(x, k * C, L_out, B, row_stride=2 * C, batch_stride=L_in * C)
    ops.gemm_tf32(a_op, wk, L_out, B, g.view(-1, C), act=ops.ACT_GELU_ERF, round_out=True)
    win = x.double().unfold(1, k, 2)[:, :L_out]                     # [B, L_out, C, k]
    ref = F.gelu(win.permute(0, 1, 3, 2).reshape(B, L_out, k * C) @ wk.double().T)
    assert low_bits_zero(g)
    assert rel(g, tf32r(ref)) < ROUNDED_TOL


@pytest.mark.parametrize("Cin", [1, 2])
def test_conv0_fp32(Cin):
    B, C, L = 2, 512, 16003
    x = _rand(B, Cin, L, seed=7)
    w0 = _rand(C, Cin, 10, scale=0.3, seed=8)
    gw, gb = 1 + _rand(C, scale=0.1, seed=9), _rand(C, scale=0.1, seed=10)
    L0 = (L - 10) // 5 + 1
    out = torch.empty(B, L0, C, device=DEV)
    mom, st = ops.conv0_workspaces(B, Cin, C, DEV)
    ops.conv0_fwd_f32(x, w0, gw, gb, out, mom, st)
    h = F.conv1d(x.double(), w0.double(), stride=5)
    ref = F.gelu(F.group_norm(h, C, gw.double(), gb.double(), eps=1e-5)).transpose(1, 2)
    assert low_bits_zero(out)
    assert rel(out, tf32r(ref)) < ROUNDED_TOL


def test_attention_fp32_output():
    """bf16 Q/K/V (and P) on the tensor cores, O in fp32: sequence lengths over the 128 / 256 / 512-key kernels."""
    D, H = 768, 12
    for lens in ([77, 128, 5], [200, 129, 256], [400, 257, 512, 31]):
        cu_l = [0]
        for n in lens:
            cu_l.append(cu_l[-1] + n)
        cu = torch.tensor(cu_l, device=DEV, dtype=torch.int32)
        qkv = _rand(cu_l[-1], 3 * D, seed=len(lens)).to(torch.bfloat16)
        out = torch.empty(cu_l[-1], D, device=DEV)
        ops.attn_fwd_f32(qkv, cu, len(lens), max(lens), D, H, out)
        ref = torch.empty(cu_l[-1], D, device=DEV, dtype=torch.float64)
        for s in range(len(lens)):
            q, kk, v = qkv[cu_l[s]:cu_l[s + 1]].double().view(-1, 3, H, D // H).unbind(1)
            p = torch.softmax(torch.einsum("qhd,khd->hqk", q, kk) / (D // H) ** 0.5, dim=-1)
            ref[cu_l[s]:cu_l[s + 1]] = torch.einsum("hqk,khd->qhd", p, v).reshape(-1, D)
        assert low_bits_zero(out)
        assert rel(out, ref) < 6e-3, lens                         # bf16 P: the existing attention tolerance
        bf = torch.empty(cu_l[-1], D, device=DEV, dtype=torch.bfloat16)
        ops.attn_fwd(qkv, cu, len(lens), max(lens), D, H, bf)
        assert rel(out, bf) < 4e-3, lens                            # the same computation, stored wider
    with pytest.raises(_lib.WavJepaLibError):                      # head dim 32 is not built: refused, no fallback
        ops.attn_fwd_f32(qkv, cu, len(lens), max(lens), 384, 12, torch.empty(cu_l[-1], 384, device=DEV))


def test_add_layernorm_fp32_addend():
    M, D = 1001, 768
    x, a = _rand(M, D, seed=11), _rand(M, D, scale=0.5, seed=12)
    g, b = 1 + _rand(D, scale=0.1, seed=13), _rand(D, scale=0.1, seed=14)
    o32, op = torch.empty(M, D, device=DEV), torch.empty(M, D, device=DEV)
    ops.add_layernorm_fwd_f32(x, a, g, b, 1e-6, o32, op)
    ref = F.layer_norm(x.double() + a.double(), (D,), g.double(), b.double(), eps=1e-6)
    assert rel(o32, ref) < FP32_TOL
    assert low_bits_zero(op) and rel(op, tf32r(ref)) < ROUNDED_TOL
    ops.add_layernorm_fwd_f32(x, None, g, b, 1e-6, None, op)
    assert rel(op, tf32r(F.layer_norm(x.double(), (D,), g.double(), b.double(), eps=1e-6))) < ROUNDED_TOL


# ------------------------------------------------------------------------------------------------------------ end to end
def _hear_sd(cfg):
    sd = jo.make_state_dict(cfg, seed=3)
    return {k.replace("encoder.", "encoder._orig_mod.", 1) if k.startswith("encoder.") else k: v for k, v in sd.items()}


@pytest.fixture(scope="module")
def hear_models():
    sd = _hear_sd(jo.Cfg())
    return hear.load_model({"state_dict": sd}), hear.load_model({"state_dict": sd}, precision="tf32")


@pytest.mark.parametrize("tag,n", [("3s", 48000), ("exact", 64318), ("10s", 160000)])
def test_hear_tf32_matches_reference_goldens(hear_models, tag, n):
    g = np.load(os.path.join(GOLD, "hear.npz"))
    m16, m32 = hear_models
    audio = oi.hear_inputs(2, n, seed=11).to(DEV)
    emb, ts = hear.get_timestamp_embeddings(audio, m32)
    assert list(emb.shape) == g[f"{tag}_shape"].tolist() and emb.dtype == torch.float32
    d32 = rel(oi.subsample(emb.cpu()), g[f"{tag}_emb"])
    d16 = rel(oi.subsample(hear.get_timestamp_embeddings(audio, m16)[0].cpu()), g[f"{tag}_emb"])
    assert d32 < E2E_TOL and d32 < GAIN * d16, (d32, d16)
    assert np.allclose(ts[0].numpy(), g[f"{tag}_ts"], rtol=1e-6, atol=1e-4)
    if tag == "3s":
        scene = hear.get_scene_embeddings(audio, m32)
        assert rel(scene.cpu().numpy(), g["3s_scene"]) < E2E_TOL


def _live(hear_models, audio):
    m16, m32 = hear_models
    with torch.no_grad():
        ref, ref_ts = jo.hear_timestamp_embeddings(audio, jo.make_state_dict(jo.Cfg(), seed=3), jo.Cfg())
    e32, ts = m32(audio.to(DEV))
    e16, _ = m16(audio.to(DEV))
    assert e32.shape == ref.shape and torch.allclose(ts, ref_ts)
    return e32.cpu(), e16.cpu(), ref


def test_hear_tf32_against_live_oracle_with_silent_clip(hear_models):
    torch.set_num_threads(os.cpu_count())
    audio = oi.hear_inputs(2, 16000, seed=3)
    audio[1] = 0
    e32, e16, ref = _live(hear_models, audio)
    d32, d16 = rel(e32[0], ref[0]), rel(e16[0], ref[0])
    assert d32 < E2E_TOL and d32 < GAIN * d16, (d32, d16)
    assert rel(e32[1], ref[1]) < E2E_TOL       # the silent clip: both paths see the same constant chunk


def test_hear_tf32_against_live_oracle_on_structured_audio(hear_models):
    """A non-white input at a realistic level: a seeded harmonic tone, a silent gap and a noise burst."""
    torch.set_num_threads(os.cpu_count())
    gen = torch.Generator().manual_seed(29)
    t = torch.arange(56000) / 16000.0
    f0 = 180.0 + 40.0 * torch.rand(2, 1, generator=gen)
    tone = sum(0.3 / h * torch.sin(2 * np.pi * h * f0 * t + torch.rand(2, 1, generator=gen) * 6.28) for h in range(1, 6))
    audio = tone * 0.2
    audio[:, 20000:28000] = 0
    audio[:, 40000:46000] += 0.3 * torch.randn(2, 6000, generator=gen)
    e32, e16, ref = _live(hear_models, audio)
    d32, d16 = rel(e32, ref), rel(e16, ref)
    assert d32 < E2E_TOL and d32 < GAIN * d16, (d32, d16)


def test_hear_nat_tf32_matches_reference_goldens():
    g = np.load(os.path.join(GOLD, "hear_nat.npz"))
    cfg = jo.Cfg(in_channels=2, per_channel=True)
    sd = jo.make_state_dict(cfg, seed=3)
    m32 = hear.load_model_nat({"state_dict": sd}, precision="tf32")
    m16 = hear.load_model_nat({"state_dict": sd})
    stereo = (torch.rand(2, 2, 48000, generator=torch.Generator().manual_seed(17)) * 2 - 1).to(DEV)
    e32, ts = hear.get_timestamp_embeddings(stereo, m32)
    assert list(e32.shape) == list(g["stereo_shape"]) and np.allclose(ts[0].cpu().numpy(), g["stereo_ts"], rtol=1e-6)
    d32 = rel(oi.subsample(e32.cpu()), g["stereo_emb"])
    d16 = rel(oi.subsample(hear.get_timestamp_embeddings(stereo, m16)[0].cpu()), g["stereo_emb"])
    assert d32 < E2E_TOL and d32 < GAIN * d16, (d32, d16)
    assert rel(hear.get_scene_embeddings(stereo, m32).cpu(), g["stereo_scene"]) < E2E_TOL
    mono = oi.hear_inputs(2, 40000, seed=19).to(DEV)
    assert rel(oi.subsample(m32.get_timestamp_embeddings(mono)[0].cpu()), g["mono_emb"]) < E2E_TOL


def test_w2v2_and_arch_tf32_match_reference_goldens():
    from wavjepa_b200.arch import WavJEPAModelWrapper

    g = np.load(os.path.join(GOLD, "interop.npz"))
    cfg2 = jo.Cfg(spec=hear.W2V2_SPEC, seconds=4.02)
    sd2 = jo.make_state_dict(cfg2, seed=3)
    audio = oi.hear_inputs(2, 100000, seed=12).to(DEV)
    e32, ts = hear.load_model_w2v2({"state_dict": sd2}, precision="tf32").get_timestamp_embeddings(audio)
    e16, _ = hear.load_model_w2v2({"state_dict": sd2}).get_timestamp_embeddings(audio)
    assert list(e32.shape) == g["w2v2_shape"].tolist()
    d32, d16 = rel(oi.subsample(e32.cpu()), g["w2v2_emb"]), rel(oi.subsample(e16.cpu()), g["w2v2_emb"])
    assert d32 < E2E_TOL and d32 < GAIN * d16, (d32, d16)
    # ARCH: the wrapper uses whatever the model it is given is set to
    rt = hear.load_model({"state_dict": jo.make_state_dict(jo.Cfg(), seed=3)})
    wrap = WavJEPAModelWrapper(rt.model, DEV, None)
    for tag, n in (("a", 40000), ("b", 64318)):
        clip = oi.hear_inputs(1, n, seed=21)[0]
        rt.model.inference_precision = "bf16"
        d16 = rel(wrap.get_embeddings(clip).cpu(), g[f"arch_{tag}"])
        rt.model.inference_precision = "tf32"
        d32 = rel(wrap.get_embeddings(clip).cpu(), g[f"arch_{tag}"])
        assert d32 < E2E_TOL and d32 < GAIN * d16, (tag, d32, d16)


# ------------------------------------------------------------------------------------------------------------ contract
def test_precision_contract():
    cfg = jo.Cfg()
    sd = _hear_sd(cfg)
    audio = oi.hear_inputs(2, 40000, seed=5).to(DEV)
    e_default, _ = hear.load_model({"state_dict": sd})(audio)
    e_bf16, _ = hear.load_model({"state_dict": sd}, precision="bf16")(audio)
    assert torch.equal(e_default, e_bf16)
    with pytest.raises(ValueError):
        hear.load_model({"state_dict": sd}, precision="fp16")
    rt = hear.load_model({"state_dict": sd}, precision="tf32")
    with pytest.raises(ValueError):
        rt.model.inference_precision = "fp32"
    assert rt.model.inference_precision == "tf32"
    # load_state_dict with new weights invalidates the tf32 working copy
    e_old, _ = rt(audio)
    rt.model.load_state_dict(jo.make_state_dict(cfg, seed=4), strict=False)
    e_new, _ = rt(audio)
    fresh, _ = hear.load_model({"state_dict": jo.make_state_dict(cfg, seed=4)}, precision="tf32")(audio)
    assert not torch.equal(e_old, e_new) and torch.equal(e_new, fresh)


def test_training_forward_ignores_inference_precision():
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=11)
    inp = oi.training_inputs(cfg, 1, 2, seed=777, masker="audioset", row0=40)
    mk = w.TimeInverseBlockMasker(4, 0.65, 10, 0.25, 10, 0.1, seed=777, row0=40)
    c_m, t_m, v_m = mk(batch_size=2, n_times=200, in_channels=1)
    ex = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=cfg.in_channels)
    m = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
               transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384), process_audio_seconds=2.01)
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV)
    audio = inp["audio"].to(DEV).bfloat16()
    ops.set_deterministic(True)
    try:
        with torch.no_grad():
            l16 = m(audio, c_m, t_m, v_m)["loss"].clone()
            m.inference_precision = "tf32"
            m.get_audio_representation(audio.float())          # builds the tf32 working copy
            l32 = m(audio, c_m, t_m, v_m)["loss"].clone()
    finally:
        ops.set_deterministic(False)
    assert torch.equal(l16, l32)
