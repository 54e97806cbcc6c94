"""Whole-clip fine-tuning and waveform gradients through the HEAR runtimes and `hf.WavJEPAModel` in training mode
(DESIGN.md 2.5) on the B200: the backward kernels of the chunk normalisation and the loudness gain against fp64 torch
autograd, the end-to-end gradients against torch autograd through the fp32 CPU oracle's HEAR computation, and the
opt-in contract (eval mode and no_grad launch exactly the inference kernels, tf32 forward-only, frozen models compute
data gradients only, one backward per graph, deterministic mode, a stock optimizer on the HF stand-in).

Tolerances are the project's (tests/test_gpu_model.py): embeddings rel-L2 <= 1e-2, every parameter gradient tensor and
the waveform gradient rel-L2 <= 2e-2 against the fp32 oracle (bf16 operands, fp32 accumulation)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from wavjepa_b200 import _lib, hear, hf, ops  # noqa: E402
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

DEV = "cuda"
UNIT = 32159
FEAT_TOL = 1e-2
GRAD_TOL = 2e-2
KERNEL_TOL = 1e-5
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


# ------------------------------------------------------------------------------------------------ fp64 references
def ref_gain(x):
    """hear_api/feature_helper.py:5-13 per clip over the whole (C, L) clip, fp64: [B, C, L] -> [B] (1 when rms == 0)."""
    out = []
    for a in x:
        rms = torch.sqrt(torch.mean(a ** 2))
        out.append(torch.ones((), dtype=x.dtype) if rms == 0 else 10 ** ((-14.0 - 20 * torch.log10(rms)) / 20))
    return torch.stack(out)


def ref_chunks(a, g, unit=UNIT):
    """hear_api/runtime.py:12-16,107-137: g * a zero-padded to whole units (a full extra unit on an exact multiple),
    each unit normalised by its mean and unbiased std over (C, unit) jointly -> [B * n_chunks, C, unit].  g: [B], or
    [B, n_chunks] (one gain per chunk: its gradient is each chunk's share of the clip gain's).  Where the std is 0 every
    z - mean is 0; torch's std backward is NaN there, so its gradient term is dropped (std detached)."""
    B, C, L = a.shape
    n = L // unit + 1
    g = g[:, None].expand(B, n) if g.dim() == 1 else g
    ap = F.pad(a, (0, n * unit - L))
    out = []
    for b in range(B):
        for i in range(n):
            ch = ap[b, :, i * unit:(i + 1) * unit] * g[b, i]
            sd = ch.std()
            if float(sd.detach()) == 0.0:
                sd = sd.detach()
            out.append((ch - ch.mean()) / (sd + 1e-5))
    return torch.stack(out)


def clips(B, C, L, seed, silent=()):
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(B, C, L, generator=g) * 2 - 1) * torch.linspace(0.2, 1.0, B)[:, None, None]
    for b in silent:
        x[b] = 0
    return x


# name -> (B, C, L, silent clips)
KERNEL_CASES = {
    "ragged_mono": (2, 1, 70000, ()),
    "exact_multiple": (2, 1, 2 * UNIT, ()),
    "stereo_joint": (2, 2, 50000, ()),
    "short_with_silent_clip": (3, 1, 16000, (1,)),
}


@pytest.mark.parametrize("name", list(KERNEL_CASES))
def test_chunk_norm_backward_matches_fp64(name):
    B, C, L, silent = KERNEL_CASES[name]
    x = clips(B, C, L, seed=3, silent=silent)
    n = L // UNIT + 1
    g = torch.Generator().manual_seed(4)
    dy = torch.randn(B * n, C, UNIT, generator=g)
    gain = ops.clip_gain(x.to(DEV).contiguous())
    # fp64 autograd of the chunk normalisation with respect to the audio and each chunk's gain
    a64 = x.double().requires_grad_(True)
    g64 = gain.cpu().double()[:, None].repeat(1, n).requires_grad_(True)
    y64 = ref_chunks(a64, g64)
    (y64 * dy.double()).sum().backward()
    ref_part = g64.grad
    # the kernels: forward output, then the backward
    y = torch.empty(B * n, C, UNIT, device=DEV)
    starts = (torch.arange(n, device=DEV, dtype=torch.int32) * UNIT).repeat(B)
    ops.crop_norm(x.to(DEV).contiguous(), starts, n, UNIT, None, y, gain=gain)
    assert rel(y, y64.detach()) < KERNEL_TOL
    da, part = ops.crop_norm_bwd(x.to(DEV).contiguous(), gain, dy.to(DEV), UNIT)
    assert torch.isfinite(da).all() and torch.isfinite(part).all()
    e_da = max(rel(da[b], a64.grad[b]) for b in range(B))   # per clip: a silent clip's gradient is ~1e5 larger
    assert e_da < KERNEL_TOL, e_da
    e_g = rel(part, ref_part)
    assert e_g < 1e-4, (e_g, part, ref_part)
    for b in silent:   # std 0 in every chunk of a silent clip: dz = (dy - mean dy) / 1e-5, no gain term
        assert (part[b] == 0).all()
    if L % UNIT == 0:
        # the all-padding chunk holds no sample: its gradient reaches nothing
        assert (part[:, -1] == 0).all()
        dy2 = dy.clone().view(B, n, C, UNIT)
        dy2[:, -1] = torch.randn(B, C, UNIT, generator=g)
        da2, part2 = ops.crop_norm_bwd(x.to(DEV).contiguous(), gain, dy2.view(B * n, C, UNIT).to(DEV), UNIT)
        assert torch.equal(da2, da) and torch.equal(part2, part)
    # bit-identical from run to run
    da_b, part_b = ops.crop_norm_bwd(x.to(DEV).contiguous(), gain, dy.to(DEV), UNIT)
    assert torch.equal(da_b, da) and torch.equal(part_b, part)
    print(f"{name}: da rel-L2 {e_da:.2e}, dgain rel-L2 {e_g:.2e}")


@pytest.mark.parametrize("C", [1, 2, 4])
def test_clip_gain_backward_matches_fp64(C):
    B, L, parts = 3, 50000, 2
    x = clips(B, C, L, seed=5, silent=(2,))
    g = torch.Generator().manual_seed(6)
    dpart = torch.randn(B, parts, generator=g)
    x64 = x.double().requires_grad_(True)
    gain64 = ref_gain(x64)
    (gain64 * dpart.double().sum(1)).sum().backward()
    xd = x.to(DEV).contiguous()
    gain = ops.clip_gain(xd)
    assert rel(gain, gain64.detach()) < 1e-5
    dx = ops.clip_gain_bwd(xd, gain, dpart.to(DEV))
    e = rel(dx, x64.grad)
    assert e < KERNEL_TOL, e
    assert (dx[2] == 0).all()                    # rms == 0: the gain is the constant 1
    assert torch.equal(ops.clip_gain_bwd(xd, gain, dpart.to(DEV)), dx)


def test_chunk_norm_backward_refuses_other_geometries():
    """Only the HEAR chunking (crop j at j * unit, L // unit + 1 crops) has a backward; the pre-training crops of
    on_after_batch_transfer (16 crops of 2.01 s at random starts of 10 s clips) stay forward-only."""
    x = clips(2, 1, 160000, seed=7).to(DEV).contiguous()
    gain = ops.clip_gain(x)
    for crops in (16, 4, 6):
        with pytest.raises(_lib.WavJepaLibError, match="HEAR chunking"):
            ops.crop_norm_bwd(x, gain, torch.zeros(2 * crops, 1, UNIT, device=DEV), UNIT)
    ops.crop_norm_bwd(x, gain, torch.zeros(2 * 5, 1, UNIT, device=DEV), UNIT)


# ------------------------------------------------------------------------------------------------ runtime preprocessing
def ref_mix(x, nat):
    """feature_helper.py:53-81: mono runtime: stereo averaged, first of four channels; Nat: mono duplicated, first of
    four duplicated, stereo kept."""
    C = x.shape[1]
    if nat:
        return x if C == 2 else torch.cat([x[:, :1], x[:, :1]], dim=1)
    return x.mean(dim=1, keepdim=True) if C == 2 else x[:, :1]


@pytest.fixture(scope="module")
def runtimes():
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    sd_nat = jo.make_state_dict(jo.Cfg(in_channels=2, per_channel=True), seed=3)
    return {False: hear.load_model({"state_dict": sd}), True: hear.load_model_nat({"state_dict": sd_nat})}


@pytest.mark.parametrize("nat", [False, True])
@pytest.mark.parametrize("C", [1, 2, 4])
def test_runtime_preprocessing_gradient_matches_fp64(runtimes, nat, C):
    """to_feature's gain, down-mix / channel fix-up and the chunk normalisation: the audio gradient of the kernels'
    graph against fp64 autograd of the reference's preprocessing (a 2nd clip silent)."""
    rt = runtimes[nat]
    B, L = 2, 40000
    x = clips(B, C, L, seed=8 + C, silent=(1,))
    x64 = x.double().requires_grad_(True)
    y64 = ref_chunks(ref_mix(x64, nat), ref_gain(x64))
    dy = torch.randn(y64.shape, generator=torch.Generator().manual_seed(9))
    (y64 * dy.double()).sum().backward()
    xd = x.to(DEV).requires_grad_(True)
    a, gain = rt.to_feature(xd, graph=True)
    y = hear._ChunkNorm.apply(a, gain, rt.unit_frames)
    assert y.shape == y64.shape and rel(y.detach(), y64.detach()) < KERNEL_TOL
    (y * dy.to(DEV)).sum().backward()
    for b in range(B):   # per clip: the silent clip's gradient (dy - mean dy) / 1e-5 is orders of magnitude larger
        e = rel(xd.grad[b], x64.grad[b])
        assert e < KERNEL_TOL, (b, e)


# ------------------------------------------------------------------------------------------------ end to end
# name -> (cfg kwargs, loader, loader kwargs, layer, scene)
E2E = {
    "mono": (dict(), hear.load_model, dict(), None, False),
    "w2v2_4s": (dict(spec=hear.W2V2_SPEC, seconds=4.02), hear.load_model_w2v2, dict(), None, False),
    "nat_per_channel": (dict(in_channels=2, per_channel=True), hear.load_model_nat, dict(), None, False),
    "nat_shared": (dict(in_channels=2, per_channel=True), hear.load_model_nat,
                   dict(share_weights_over_channels=True), None, False),
    "mono_layer5": (dict(), hear.load_model, dict(), 5, False),
    "mono_scene": (dict(), hear.load_model, dict(), None, True),
}


def _e2e_case(name, seed=7):
    cfgkw, loader, lkw, layer, scene = E2E[name]
    cfg = jo.Cfg(**cfgkw)
    sd = jo.make_state_dict(cfg, seed=seed)
    if lkw.get("share_weights_over_channels"):   # one CNN for both channels: the oracle reads the same leaves
        for k in list(sd):
            if k.startswith("extract_audio.cnns.1."):
                sd[k] = sd["extract_audio.cnns.0." + k[len("extract_audio.cnns.1."):]]
    L = 70000 if name == "w2v2_4s" else 40000
    audio = oi.hear_inputs(2, L, seed=seed + 1)
    if cfg.per_channel:   # a stereo clip: the two channels differ
        audio = torch.stack([audio, oi.hear_inputs(2, L, seed=seed + 2)], dim=1)
    return cfg, sd, loader, lkw, layer, scene, audio


def _oracle(cfg, sd, audio, layer, scene, proj, monkeypatch):
    leaves, ref_sd = {}, {}
    for k, v in sd.items():
        if id(v) not in leaves:
            leaves[id(v)] = v.clone().requires_grad_(k.startswith(PATH))
        ref_sd[k] = leaves[id(v)]
    if layer is not None:   # the oracle's HEAR computation reading hidden state `layer` (no final norm)
        real_stack = jo.run_stack
        monkeypatch.setattr(jo, "run_stack", lambda x, sd_, prefix, n, nhead, m, **kw:
                            real_stack(x, sd_, prefix, layer, nhead, m, final_norm=False))
    a = audio.clone().requires_grad_(True)
    emb, _ = (jo.hear_nat_timestamp_embeddings if cfg.per_channel else jo.hear_timestamp_embeddings)(a, ref_sd, cfg)
    monkeypatch.undo()
    out = emb.mean(dim=1) if scene else emb
    (out * proj).sum().backward()
    return out.detach(), a.grad, {k: v.grad for k, v in ref_sd.items() if k.startswith(PATH)}


@pytest.mark.parametrize("name", list(E2E))
def test_whole_clip_gradients_match_the_oracle(name, monkeypatch):
    cfg, sd, loader, lkw, layer, scene, audio = _e2e_case(name)
    rt = loader({"state_dict": sd}, layer=layer, **lkw)
    assert not rt.training
    ad = audio.to(DEV)
    call = rt.get_scene_embeddings if scene else (lambda x: rt.get_timestamp_embeddings(x)[0])
    ref_eval = call(ad)                                   # eval mode: no graph
    assert ref_eval.grad_fn is None
    rt.train()
    a = ad.clone().requires_grad_(True)
    out = call(a)
    assert out.grad_fn is not None
    assert torch.equal(out.detach(), ref_eval)           # training mode changes no bit of the embeddings
    proj = torch.randn(out.shape, generator=torch.Generator().manual_seed(11))
    ref_out, ref_da, ref_g = _oracle(cfg, sd, audio, layer, scene, proj, monkeypatch)
    e_emb = rel(out.detach(), ref_out)
    assert e_emb <= FEAT_TOL, e_emb
    (out * proj.to(DEV)).sum().backward()
    e_audio = rel(a.grad, ref_da)
    assert a.grad.dtype == torch.float32 and e_audio <= GRAD_TOL, e_audio
    worst, n_checked = ("", 0.0), 0
    for n_, p_ in rt.model.named_parameters():
        ref = ref_g.get(n_)
        if ref is None:   # off the path (or above hidden state `layer`): no gradient
            assert p_.grad is None, n_
            continue
        assert p_.grad is not None, n_
        e = rel(p_.grad, ref)
        worst = max(worst, (n_, e), key=lambda t: t[1])
        n_checked += 1
        assert e < GRAD_TOL, (n_, e)
    n_layers = cfg.layers if layer is None else layer
    assert n_checked >= 12 * n_layers + 4 + len(cfg.spec), n_checked
    print(f"{name}: emb rel-L2 {e_emb:.2e}, audio.grad {e_audio:.2e}, worst parameter {worst} over {n_checked}")


# ------------------------------------------------------------------------------------------------ contract
def _launches(fn):
    with _lib.KernelProfile() as kp:
        out = fn()
    torch.cuda.synchronize()
    return [r[0] for r in kp.records], out


def test_eval_mode_and_no_grad_launch_the_inference_kernels():
    """The kernels of the eval-mode call in no_grad mode (loudness gain, bf16 chunks, the inference forward) are what a
    call launches in eval mode whatever requires grad, and in training mode under no_grad."""
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    rt = hear.load_model({"state_dict": sd})
    audio = oi.hear_inputs(2, 48000, seed=11).to(DEV)
    with torch.no_grad():
        rt.get_timestamp_embeddings(audio)   # first call: working weight copies
        base, e0 = _launches(lambda: rt.get_timestamp_embeddings(audio)[0])
    assert base[:2] == ["wj_clip_gain", "wj_crop_norm"]
    assert not any("bwd" in k or "wgrad" in k for k in base)
    # eval mode in grad mode with a trainable model and audio requiring grad
    seq, e1 = _launches(lambda: rt.get_timestamp_embeddings(audio.clone().requires_grad_(True))[0])
    assert seq == base and e1.grad_fn is None and torch.equal(e1, e0)
    # training mode under no_grad
    rt.train()
    with torch.no_grad():
        seq, e2 = _launches(lambda: rt.get_timestamp_embeddings(audio.clone().requires_grad_(True))[0])
    assert seq == base and torch.equal(e2, e0)
    # training mode in grad mode builds the graph
    e3 = rt.get_timestamp_embeddings(audio.clone().requires_grad_(True))[0]
    assert e3.grad_fn is not None and torch.equal(e3.detach(), e0)


def test_tf32_stays_forward_only_in_training_mode():
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    rt = hear.load_model({"state_dict": sd}, precision="tf32").train()
    a = oi.hear_inputs(2, 40000, seed=12).to(DEV).requires_grad_(True)
    emb, _ = rt.get_timestamp_embeddings(a)
    assert emb.grad_fn is None and rt.get_scene_embeddings(a).grad_fn is None


def test_frozen_model_computes_data_gradients_only(monkeypatch):
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    rt = hear.load_model({"state_dict": sd}).train()
    rt.model.requires_grad_(False)
    a = oi.hear_inputs(2, 40000, seed=13).to(DEV).requires_grad_(True)
    calls = {"gemm_wgrad": 0, "colsum": 0}
    for name in calls:
        real = getattr(ops, name)

        def counted(*args, _real=real, _name=name, **kw):
            calls[_name] += 1
            return _real(*args, **kw)
        monkeypatch.setattr(ops, name, counted)
    emb = rt.get_scene_embeddings(a)
    assert emb.grad_fn is not None
    emb.square().sum().backward()
    assert calls == {"gemm_wgrad": 0, "colsum": 0}, calls
    assert all(p.grad is None for p in rt.model.parameters())
    assert a.grad is not None and torch.isfinite(a.grad).all() and a.grad.abs().max() > 0


def test_one_backward_per_graph():
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    rt = hear.load_model({"state_dict": sd}).train()
    a = oi.hear_inputs(2, 40000, seed=14).to(DEV).requires_grad_(True)
    emb, _ = rt.get_timestamp_embeddings(a)
    emb.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        emb.sum().backward()


def test_deterministic_mode_gives_bit_identical_gradients(deterministic):
    sd = jo.make_state_dict(jo.Cfg(in_channels=2, per_channel=True), seed=3)
    rt = hear.load_model_nat({"state_dict": sd}).train()
    audio = oi.hear_inputs(2, 40000, seed=15).to(DEV)
    proj = torch.randn(2, 768, generator=torch.Generator().manual_seed(1)).to(DEV)
    runs = []
    for _ in range(2):
        rt.model.zero_grad(set_to_none=True)
        a = audio.clone().requires_grad_(True)
        (rt.get_scene_embeddings(a) * proj).sum().backward()
        runs.append((a.grad.clone(), {n: p.grad.clone() for n, p in rt.model.named_parameters() if p.grad is not None}))
    assert torch.equal(runs[0][0], runs[1][0])
    assert runs[0][1].keys() == runs[1][1].keys() and len(runs[0][1]) > 100
    for n in runs[0][1]:
        assert torch.equal(runs[0][1][n], runs[1][1][n]), n


def test_hf_model_fine_tunes_with_adamw(tmp_path):
    sd = jo.make_state_dict(jo.Cfg(), seed=3)
    path = os.path.join(tmp_path, "ckpt.pt")
    torch.save({"state_dict": sd}, path)
    model = hf.WavJEPAModel.from_pretrained(path).to(DEV)
    assert not model.training and not model.runtime.training
    fe = hf.WavJEPAFeatureExtractor.from_pretrained("labhamlet/wavjepa-base")
    g = torch.Generator().manual_seed(21)
    clips_ = [torch.rand(n, generator=g) * 2 - 1 for n in (48000, 40000, 56000, 33000)]
    x = fe(clips_, return_tensors="pt")["input_values"].to(DEV)
    labels = torch.tensor([0, 1, 2, 3], device=DEV)
    head = torch.nn.Linear(768, 4).to(DEV)
    model.train()
    params = [p for n, p in model.named_parameters() if n.startswith(tuple("runtime.model." + s for s in PATH))]
    opt = torch.optim.AdamW([{"params": params, "lr": 1e-4}, {"params": list(head.parameters()), "lr": 1e-3}])
    losses = []
    for _ in range(20):
        opt.zero_grad(set_to_none=True)
        emb, _ = model(x)
        loss = F.cross_entropy(head(emb.mean(dim=1)), labels)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(np.isfinite(losses)), losses
    assert losses[-1] < 0.9 * losses[0], losses
    # the fine-tuned weights round-trip through state_dict
    model.eval()
    with torch.no_grad():
        e_tuned, _ = model(x)
    fresh = hf.WavJEPAModel.from_pretrained(path).to(DEV)
    with torch.no_grad():
        e_fresh, _ = fresh(x)
    assert not torch.equal(e_fresh, e_tuned)
    fresh.load_state_dict(model.state_dict())
    with torch.no_grad():
        e_loaded, _ = fresh(x)
    assert torch.equal(e_loaded, e_tuned)
    print(f"HF AdamW: loss {losses[0]:.4f} -> {losses[-1]:.4f}")
