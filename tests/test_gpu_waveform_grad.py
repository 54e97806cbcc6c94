"""Backpropagation of `JEPA.get_audio_representation` to the input waveform on the B200: conv block 0's data-gradient
kernel against an fp64 restatement, the model's `audio.grad` against torch autograd through the fp32 CPU oracle (frozen
and trainable), the contract (bit-identical features, device and dtype of the gradient, limits), the data-gradient-only
backward of frozen parts, and a perceptual-loss training loop.

Tolerances are the project's: the conv-0 kernel rel-L2 < 4e-3 (tests/test_gpu_kernels.py), every gradient rel-L2 <= 2e-2
against the fp32 oracle (bf16 operands, fp32 accumulation).  Calibration: the reference itself, run under bf16 CPU
autocast, puts its `audio.grad` at rel-L2 1.41e-2 (mono base), 1.53e-2 (w2v2 4.02 s) and 1.41e-2 (Nat per-channel) from
its own fp32 `audio.grad` (B = 2, the inputs of `_case`, seed 7): the waveform gradient is the noisiest gradient of the
model in bf16, and 2e-2 is the bound kept for it."""
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import wavjepa_b200 as w  # noqa: E402
from wavjepa_b200 import _lib, hear, jepa, ops  # noqa: E402
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

DEV = "cuda"
GRAD_TOL = 2e-2
BF16_TOL = 4e-3
PATH = ("extract_audio.", "feature_norms.", "post_extraction_mapper.", "encoder.")


def rel(a, b):
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(autouse=True, scope="module")
def _device():
    _lib.require_device()
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())


@pytest.fixture
def deterministic():
    ops.set_deterministic(True)
    yield
    ops.set_deterministic(False)


# ------------------------------------------------------------------------------------------------ conv-0 kernel
def _conv0_problem(B, Cin, L, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    C = 512
    x = torch.randn(B, Cin, L, device=DEV, generator=g).bfloat16()
    wt = torch.randn(C, Cin, 10, device=DEV, generator=g) * (2.0 / (Cin * 10)) ** 0.5
    gamma = 1.0 + 0.1 * torch.randn(C, device=DEV, generator=g)
    beta = 0.1 * torch.randn(C, device=DEV, generator=g)
    L0 = (L - 10) // 5 + 1
    out = torch.empty(B, L0, C, device=DEV, dtype=torch.bfloat16)
    mom, stats = ops.conv0_workspaces(B, Cin, C, DEV)
    ops.conv0_fwd(x, wt, gamma, beta, out, mom, stats)
    dy = torch.randn(B, L0, C, device=DEV, generator=g).bfloat16()
    return x, wt, gamma, beta, mom, stats, dy


def _conv0_dx(x, wt, gamma, beta, mom, stats, dy, weights=False, workspace=None):
    dx = torch.full(x.shape, float("nan"), device=DEV)
    wg = (torch.zeros_like(wt), torch.zeros(wt.shape[0], device=DEV), torch.zeros(wt.shape[0], device=DEV)) if weights \
        else (None, None, None)
    ops.conv0_bwd_dx(x, wt, gamma, beta, mom, stats, dy, dx, *wg, workspace=workspace)
    return dx, wg


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("L", [1237, 32159, 64319])
@pytest.mark.parametrize("Cin", [1, 2])
def test_conv0_dx_matches_fp64(Cin, L, B):
    x, wt, gamma, beta, mom, stats, dy = _conv0_problem(B, Cin, L, seed=Cin * 7 + B)
    C = wt.shape[0]
    # the restatement of test_conv0_gn_gelu_fwd_bwd in fp64: bf16 weights, bf16-rounded conv output (straight-through)
    xr = x.double().requires_grad_(True)
    h = F.conv1d(xr, wt.bfloat16().double(), stride=5)
    hq = h + (h.float().bfloat16().double() - h).detach()
    y = F.gelu(F.group_norm(hq, C, gamma.double(), beta.double(), 1e-5))
    ref, = torch.autograd.grad(y, xr, dy.double().transpose(1, 2))
    dx, _ = _conv0_dx(x, wt, gamma, beta, mom, stats, dy)
    e = rel(dx, ref)
    assert e < BF16_TOL, e
    L0 = (L - 10) // 5 + 1
    covered = 5 * (L0 - 1) + 10
    assert covered <= L
    assert torch.equal(dx[..., covered:], torch.zeros_like(dx[..., covered:]))   # after the last window: exactly 0
    assert torch.isfinite(dx).all()
    # default mode: no atomics on the path to dx, bit-identical run to run
    dx2, _ = _conv0_dx(x, wt, gamma, beta, mom, stats, dy)
    assert torch.equal(dx, dx2)
    # the optional weight gradients are those of the existing backward; dx does not depend on requesting them
    ops.set_deterministic(True)
    try:
        dw, dg, db = torch.zeros_like(wt), torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
        red = torch.empty(B, 2 + Cin * 10, C, device=DEV, dtype=torch.float64)
        ops.conv0_bwd(x, wt, gamma, beta, mom, stats, dy, red, dw, dg, db)
        runs = []
        for fill in (0xFF, 0xFF, 0x7F):   # NaN-poisoned twice, then huge finite values
            ops._det_ws.fill_(fill)
            ws = ops.conv0_bwd_dx_workspace(B, Cin, L, C, DEV).fill_(fill)
            runs.append(_conv0_dx(x, wt, gamma, beta, mom, stats, dy, weights=True, workspace=ws))
    finally:
        ops.set_deterministic(False)
    for dxr, (dw2, dg2, db2) in runs:
        assert torch.equal(dxr, dx)
        assert torch.equal(dw2, dw) and torch.equal(dg2, dg) and torch.equal(db2, db)


def test_conv0_dx_refuses_partial_weight_outputs():
    x, wt, gamma, beta, mom, stats, dy = _conv0_problem(1, 1, 1237)
    dx = torch.empty(x.shape, device=DEV)
    with pytest.raises(_lib.WavJepaLibError):
        ops.conv0_bwd_dx(x, wt, gamma, beta, mom, stats, dy, dx, torch.zeros_like(wt), None, None)


# ------------------------------------------------------------------------------------------------ model vs oracle
def build(cfg: jo.Cfg, sd, seconds=2.01, size="base", share=False):
    if cfg.per_channel:
        ex = w.ConvChannelFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=cfg.in_channels,
                                           share_weights_over_channels=share)
    else:
        ex = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=cfg.in_channels)
    m = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
               transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
               process_audio_seconds=seconds, nr_samples_per_audio=8, average_top_k_layers=cfg.top_k, size=size)
    if share:
        sd = {k: v for k, v in sd.items() if not k.startswith("extract_audio.cnns.1.")}
    m.load_state_dict({k: v.detach() for k, v in sd.items()}, strict=True)
    return m.to(DEV)


def hear_mask(T=200):
    """Padding pattern of one 10 s clip in 2.01 s chunks (hear.embed_chunks)."""
    pad, n_chunks, cut_off, total_steps = hear.hear_geometry(160000, 32159, 16000, T)
    mask = torch.zeros(max(total_steps, n_chunks * T), dtype=torch.bool)
    mask[cut_off:total_steps] = True
    return mask[:n_chunks * T].reshape(n_chunks, T)


def ragged_mask(B, T, lengths):
    m = torch.zeros(B, T, dtype=torch.bool)
    for b, n in enumerate(lengths):
        m[b, n:] = True
    return m


# name -> (cfg kwargs, seconds, size, shared extractor, batch, mask kind): the geometries of test_gpu_finetune.py and a
# two-channel mono extractor
CASES = {
    "mono_dense": (dict(), 2.01, "base", False, 2, None),
    "padding_mask_ragged": (dict(), 2.01, "base", False, 3, "ragged"),
    "host_mask_hear_10s": (dict(), 2.01, "base", False, 5, "hear"),
    "nat_per_channel": (dict(in_channels=2, per_channel=True), 2.01, "base", False, 2, None),
    "nat_shared": (dict(in_channels=2, per_channel=True), 2.01, "base", True, 2, None),
    "w2v2_4s": (dict(spec=hear.W2V2_SPEC, seconds=4.02), 4.02, "base", False, 2, None),
    "large": (dict(d_model=1024, nhead=16, layers=24), 2.01, "large", False, 2, None),
    "mono_cin2": (dict(in_channels=2), 2.01, "base", False, 2, None),
}


def _case(name, seed=7):
    cfgkw, seconds, size, share, B, mask = CASES[name]
    cfg = jo.Cfg(**cfgkw)
    sd = jo.make_state_dict(cfg, seed=seed)
    if share:   # one CNN for both channels: the oracle reads the same leaf tensors for channel 1
        for k in list(sd):
            if k.startswith("extract_audio.cnns.1."):
                sd[k] = sd["extract_audio.cnns.0." + k[len("extract_audio.cnns.1."):]]
    g = torch.Generator().manual_seed(seed)
    audio = (torch.randn(B, cfg.in_channels, cfg.target_length, generator=g) * 0.5).bfloat16().float()
    T = cfg.total_patches
    hidden = None
    if mask == "ragged":
        hidden = ragged_mask(B, T, [T, 137, 61])
    elif mask == "hear":
        hidden = hear_mask(T)
        assert hidden.shape[0] == B and hidden.any() and not hidden.all()
    proj = torch.randn(B, T, cfg.d_model, generator=g)
    if hidden is not None:
        proj = proj * (~hidden)[..., None]          # the loss reads the visible rows only
    return cfg, sd, seconds, size, share, audio, hidden, mask, proj


def _oracle(cfg, sd, audio, hidden, proj):
    """fp32 CPU autograd: (audio.grad, {name: param grad})."""
    leaves, ref_sd = {}, {}
    for k, v in sd.items():
        if id(v) not in leaves:
            leaves[id(v)] = v.clone().requires_grad_(k.startswith(PATH))
        ref_sd[k] = leaves[id(v)]
    a = audio.clone().requires_grad_(True)
    feats = jo.run_stack(jo.local_features(a, ref_sd, cfg), ref_sd, "encoder", cfg.layers, cfg.nhead, hidden)
    (feats * proj).sum().backward()
    return a.grad, {k: v.grad for k, v in ref_sd.items() if k.startswith(PATH)}


def _features(model, audio, hidden, mask):
    if mask == "hear":
        return model.get_audio_representation(audio, None, host_mask=hidden.numpy())
    return model.get_audio_representation(audio, None if hidden is None else hidden.to(DEV))


@pytest.mark.parametrize("name", list(CASES))
def test_waveform_gradient_matches_the_oracle(name):
    cfg, sd, seconds, size, share, audio, hidden, mask, proj = _case(name)
    ref_dx, ref_g = _oracle(cfg, sd, audio, hidden, proj)
    model = build(cfg, sd, seconds, size, share)
    with torch.no_grad():
        f0 = _features(model, audio.to(DEV), hidden, mask)
    # ---- frozen model: the waveform gradient only
    model.requires_grad_(False)
    a = audio.to(DEV).requires_grad_(True)
    feats = _features(model, a, hidden, mask)
    assert feats.grad_fn is not None and torch.equal(feats.detach(), f0)
    (feats * proj.to(DEV)).sum().backward()
    e_frozen = rel(a.grad, ref_dx)
    assert e_frozen <= GRAD_TOL, e_frozen
    assert all(p.grad is None for p in model.parameters())
    if mask == "hear":
        # samples whose every window feeds only padded tokens: their gradient comes through block 0's GroupNorm alone
        hop, rf = 1, 1
        for (_, k, s) in reversed(cfg.spec):
            rf, hop = (rf - 1) * s + k, hop * s
        vis = (~hidden).sum(1)
        part = vis < hidden.shape[1]
        assert part.any()
        region = torch.zeros_like(audio, dtype=torch.bool)
        for b in torch.nonzero(part).flatten().tolist():
            region[b, :, (int(vis[b]) - 1) * hop + rf:] = True
        assert region.any()
        assert ref_dx[region].abs().max() > 0
        e_pad = rel(a.grad[region.to(DEV)], ref_dx[region])
        assert e_pad <= GRAD_TOL, e_pad
    # ---- trainable path and the waveform in one backward
    for n_, p_ in model.named_parameters():
        p_.requires_grad_(n_.startswith(PATH))
    a2 = audio.to(DEV).requires_grad_(True)
    feats = _features(model, a2, hidden, mask)
    assert torch.equal(feats.detach(), f0)
    (feats * proj.to(DEV)).sum().backward()
    e_train = rel(a2.grad, ref_dx)
    assert e_train <= GRAD_TOL, e_train
    worst = ("", 0.0)
    for n_, p_ in model.named_parameters():
        if not n_.startswith(PATH):
            assert p_.grad is None, n_
            continue
        e = rel(p_.grad, ref_g[n_])
        worst = max(worst, (n_, e), key=lambda t: t[1])
        assert e < GRAD_TOL, (n_, e)
    print(f"{name}: audio.grad rel-L2 frozen {e_frozen:.2e}, trainable {e_train:.2e}; worst parameter {worst}")


# ------------------------------------------------------------------------------------------------ contract
def test_contract_device_dtype_and_inference_path_saves_nothing(monkeypatch):
    cfg = jo.Cfg()
    model = build(cfg, jo.make_state_dict(cfg, seed=9))
    model.requires_grad_(False)
    g = torch.Generator().manual_seed(9)
    base = (torch.randn(2, 1, cfg.target_length, generator=g) * 0.5)
    proj = torch.randn(2, cfg.total_patches, cfg.d_model, generator=g).to(DEV)
    with torch.no_grad():
        f0 = model.get_audio_representation(base.to(DEV))
    # audio not requiring grad, frozen model: the inference path -- not through _FeatureBridge, no graph, and no
    # saving kernels: no encoder or conv activations kept, no LayerNorm statistics requested
    calls, saves = [], []
    real_bridge = jepa._FeatureBridge.apply
    monkeypatch.setattr(jepa._FeatureBridge, "apply", lambda *a_, **k_: calls.append(1) or real_bridge(*a_, **k_))
    real_stack, real_conv, real_ln = model._enc_stack.forward, jepa.conv_stack_forward, ops.layernorm_fwd
    monkeypatch.setattr(model._enc_stack, "forward", lambda *a_, **k_: saves.append(a_[6]) or real_stack(*a_, **k_))
    monkeypatch.setattr(jepa, "conv_stack_forward", lambda *a_, **k_: saves.append(a_[6]) or real_conv(*a_, **k_))
    monkeypatch.setattr(ops, "layernorm_fwd", lambda *a_, **k_: saves.append(a_[6] is not None) or real_ln(*a_, **k_))
    f = model.get_audio_representation(base.to(DEV))
    assert f.grad_fn is None and not f.requires_grad and not calls
    assert len(saves) == 4 and not any(saves)   # conv stack, feature norm, encoder, final norm
    assert torch.equal(f, f0)
    saves.clear()
    grads = {}
    for dev in ("cpu", DEV):
        for dt in (torch.float32, torch.bfloat16):
            a = base.to(device=dev, dtype=dt).detach().clone().requires_grad_(True)
            feats = model.get_audio_representation(a)
            if dt == torch.float32:
                assert torch.equal(feats.detach(), f0)
            loss = (feats * proj).sum()
            loss.backward(retain_graph=True)
            assert a.grad.device == a.device and a.grad.dtype == dt and a.grad.shape == a.shape
            grads[(dev, dt)] = a.grad.float().cpu()
            with pytest.raises(RuntimeError, match="already backpropagated"):
                loss.backward()
    assert calls and all(saves[:4])   # the waveform-gradient calls ran the saving forward
    # every input dtype / device reads the same bf16 waveform: one gradient, returned in each caller's dtype
    assert torch.equal(grads[("cpu", torch.float32)], grads[(DEV, torch.float32)])
    assert torch.equal(grads[(DEV, torch.bfloat16)], grads[(DEV, torch.float32)].bfloat16().float())
    # tf32 stays forward-only
    model.inference_precision = "tf32"
    t = model.get_audio_representation(base.to(DEV).requires_grad_(True))
    assert t.grad_fn is None and not t.requires_grad


def test_product_surfaces_stay_inference_only_with_a_waveform_requiring_grad(tmp_path):
    from wavjepa_b200 import hf
    from wavjepa_b200.arch import WavJEPAModelWrapper
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    rt = hear.load_model({"state_dict": sd})
    audio = oi.hear_inputs(2, 48000, seed=11).to(DEV).requires_grad_(True)
    emb, _ = hear.get_timestamp_embeddings(audio, rt)
    assert not emb.requires_grad
    assert not hear.get_scene_embeddings(audio, rt).requires_grad
    path = os.path.join(tmp_path, "ckpt.pt")
    torch.save({"state_dict": sd}, path)
    model = hf.WavJEPAModel.from_pretrained(path).to(DEV)
    feats = hf.WavJEPAFeatureExtractor.from_pretrained("labhamlet/wavjepa-base")(audio.detach(), return_tensors="pt")
    e2, _ = model(feats["input_values"].requires_grad_(True))
    assert not e2.requires_grad
    wrap = WavJEPAModelWrapper(build(cfg, sd), DEV, None)
    assert not wrap.get_embeddings(oi.hear_inputs(1, 40000, seed=21)[0].requires_grad_(True)).requires_grad


# ------------------------------------------------------------------------------------------------ frozen parts
def _spy(monkeypatch):
    calls = {"gemm_wgrad": 0, "colsum": 0, "conv0_bwd": 0, "conv0_bwd_dx_weights": 0}
    for name in ("gemm_wgrad", "colsum", "conv0_bwd"):
        real = getattr(ops, name)

        def counted(*a, _real=real, _name=name, **k):
            calls[_name] += 1
            return _real(*a, **k)
        monkeypatch.setattr(ops, name, counted)
    real_dx = ops.conv0_bwd_dx

    def dx_counted(*a, **k):
        if (len(a) > 8 and a[8] is not None) or k.get("dw") is not None:
            calls["conv0_bwd_dx_weights"] += 1
        return real_dx(*a, **k)
    monkeypatch.setattr(ops, "conv0_bwd_dx", dx_counted)
    return calls


def test_frozen_parts_do_no_weight_work(deterministic, monkeypatch):
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=4)
    g = torch.Generator().manual_seed(4)
    B = 4
    audio = (torch.randn(B, 1, cfg.target_length, generator=g) * 0.5).to(DEV)
    proj = torch.randn(B, cfg.total_patches, cfg.d_model, generator=g).to(DEV)
    model = build(cfg, sd)

    def step(audio_grad):
        a = audio.clone().requires_grad_(audio_grad)
        (model.get_audio_representation(a) * proj).sum().backward()
        grads = {n: None if p.grad is None else p.grad.clone() for n, p in model.named_parameters() if n.startswith(PATH)}
        model.zero_grad(set_to_none=True)
        return (a.grad.clone() if audio_grad else None), grads

    dx_full, g_full = step(True)                     # everything trainable (also the warm-up)
    calls = _spy(monkeypatch)
    model.requires_grad_(False)
    dx_frozen, g_frozen = step(True)
    assert calls == {"gemm_wgrad": 0, "colsum": 0, "conv0_bwd": 0, "conv0_bwd_dx_weights": 0}, calls
    assert all(v is None for v in g_frozen.values())
    assert torch.equal(dx_frozen, dx_full)           # the data-gradient chain is the same bits without weight work
    # only the extractor trains (audio not requiring grad): no encoder-layer or mapper weight gradient
    model.extract_audio.requires_grad_(True)
    _, g_ex = step(False)
    assert calls["gemm_wgrad"] == len(cfg.spec) - 1 and calls["colsum"] == 0 and calls["conv0_bwd"] == 1, calls
    model.encoder.requires_grad_(True)
    _, g_ex_enc = step(False)
    for n_, gr in g_ex.items():
        if n_.startswith("extract_audio."):
            assert torch.equal(gr, g_ex_enc[n_]) and torch.equal(gr, g_full[n_]), n_
        else:
            assert gr is None, n_
    # the extractor and the waveform: block 0 takes its weight gradients from the data-gradient entry point
    model.encoder.requires_grad_(False)
    for k in calls:
        calls[k] = 0
    dx_ex, g_ex_dx = step(True)
    assert calls["conv0_bwd_dx_weights"] == 1 and calls["conv0_bwd"] == 0
    assert calls["gemm_wgrad"] == len(cfg.spec) - 1, calls
    assert torch.equal(dx_ex, dx_full)
    for n_, gr in g_ex_dx.items():
        if n_.startswith("extract_audio."):
            assert torch.equal(gr, g_full[n_]), n_


# ------------------------------------------------------------------------------------------------ perceptual loss
def _enhancer():
    torch.manual_seed(5)
    enh = torch.nn.Conv1d(1, 1, 33, padding=16)
    torch.nn.init.normal_(enh.weight, std=1e-3)
    torch.nn.init.zeros_(enh.bias)
    return enh


def test_enhancer_trains_through_the_frozen_encoder():
    """The perceptual-loss recipe of scripts/bench_waveform_grad.py: a residual Conv1d enhancer in front of the frozen
    encoder, MSE between features(enhancer(noisy)) and features(clean), torch.optim.AdamW on the enhancer.

    The enhancer's weight gradient projects the waveform gradient onto 33 shifted copies of the input, which amplifies
    bf16 noise: the reference itself under bf16 CPU autocast is 2.9e-2 from its fp32 weight gradient on these inputs,
    above the 2e-2 model tolerance.  So the first-step weight gradient is held to the reference's own bf16 distance,
    measured live.  The bias gradient is zero in exact arithmetic (a constant offset is removed by block 0's GroupNorm;
    fp32 gives ~6e-10): it is checked to be negligible against the weight gradient, not in relative terms."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=13)
    g = torch.Generator().manual_seed(13)
    B = 4
    clean = torch.randn(B, 1, cfg.target_length, generator=g) * 0.3
    noisy = clean + 0.1 * torch.randn(B, 1, cfg.target_length, generator=g)
    # first-step gradient of the enhancer against the oracle
    enh_ref = _enhancer()
    with torch.no_grad():
        tgt_ref = jo.run_stack(jo.local_features(clean, sd, cfg), sd, "encoder", cfg.layers, cfg.nhead, None)
    x = noisy + enh_ref(noisy)
    F.mse_loss(jo.run_stack(jo.local_features(x, sd, cfg), sd, "encoder", cfg.layers, cfg.nhead, None), tgt_ref).backward()
    enh_bf = _enhancer()
    with torch.autocast("cpu", dtype=torch.bfloat16):
        with torch.no_grad():
            tgt_bf = jo.run_stack(jo.local_features(clean, sd, cfg), sd, "encoder", cfg.layers, cfg.nhead, None).float()
        f_bf = jo.run_stack(jo.local_features(noisy + enh_bf(noisy).float(), sd, cfg), sd, "encoder", cfg.layers,
                            cfg.nhead, None).float()
    F.mse_loss(f_bf, tgt_bf).backward()
    e_ref_bf16 = rel(enh_bf.weight.grad, enh_ref.weight.grad)
    model = build(cfg, sd)
    model.requires_grad_(False)
    enh = _enhancer().to(DEV)
    opt = torch.optim.AdamW(enh.parameters(), lr=2e-3)
    c_d, n_d = clean.to(DEV), noisy.to(DEV)
    with torch.no_grad():
        tgt = model.get_audio_representation(c_d)
    losses = []
    for it in range(20):
        opt.zero_grad(set_to_none=True)
        loss = F.mse_loss(model.get_audio_representation(n_d + enh(n_d)), tgt)
        loss.backward()
        if it == 0:
            e_w = rel(enh.weight.grad, enh_ref.weight.grad)
            assert e_w <= e_ref_bf16, (e_w, e_ref_bf16)
            b_ratio = float(enh.bias.grad.abs().max() / enh.weight.grad.norm())
            assert b_ratio < 1e-2, b_ratio
        opt.step()
        losses.append(loss.item())
    assert all(p.grad is None for p in model.parameters())
    assert losses[-1] < losses[0], losses
    print(f"enhancer: first-step weight gradient rel-L2 {e_w:.2e} (reference under bf16 autocast {e_ref_bf16:.2e}), "
          f"|bias grad| / |weight grad| {b_ratio:.1e}; loss {losses[0]:.4e} -> {losses[-1]:.4e}")
