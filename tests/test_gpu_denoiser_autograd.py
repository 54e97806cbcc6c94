"""The denoiser stage through autograd on the B200: `Denoiser.forward` in grad mode, `loss.backward()`, the
`wj_mse_pair_bwd` kernel and the Lightning `training_step` contract.

References: the executed reference's fixtures (tests/golden/denoiser.*, made with `o = m(gen, clean);
o["loss"].backward()`), the fused `forward_backward` / `train_step` (bit for bit in deterministic mode) and torch autograd
through the fp32 CPU oracle.  Tolerances are the project's: losses rel <= 2e-3 against the fixtures, every gradient
tensor rel-L2 <= 2e-2 (bf16 operands, fp32 accumulation)."""
import contextlib
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import wavjepa_b200 as w  # noqa: E402
from wavjepa_b200 import _lib, ops  # noqa: E402
from wavjepa_b200.denoiser import Denoiser, _MsePair  # noqa: E402
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
DEV = "cuda"
GRAD_TOL = 2e-2
STUDENT = ("extract_audio.", "feature_norms.", "post_extraction_mapper.", "encoder.")


def rel(a, b):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    if a.device != b.device:
        a, b = a.cpu(), b.cpu()
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(autouse=True, scope="module")
def _device():
    _lib.require_device()
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())


@contextlib.contextmanager
def det_mode(nbytes=256 << 20, fill=0xFF):
    """Deterministic mode with a workspace whose every byte is `fill` on entry; always switched off on exit."""
    ops.set_deterministic(True, nbytes)
    try:
        ops._det_ws.fill_(fill)
        yield
    finally:
        ops.set_deterministic(False)


def _denoiser(alpha, nr=2):
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


@pytest.fixture(scope="module")
def golden_inputs():
    """The inputs of test_gpu_model.py::test_denoiser_stage_matches_reference_goldens: the reference's batch preparation
    restated on the host with the pinned crop starts and shuffle, bf16 (what the reference's model read), on the CPU."""
    g = np.load(os.path.join(GOLD, "denoiser.npz"))
    starts, perm = torch.from_numpy(g["starts"]), torch.from_numpy(g["perm"])
    gen, clean = jo.denoiser_batch(oi.denoiser_batch(), starts, perm)
    return gen.bfloat16(), clean.bfloat16()


def _student_grads(m):
    return {n: p.grad for n, p in m.named_parameters() if n.startswith(STUDENT)}


def _fused_grads(m, gen, clean, alpha):
    a0 = m.alpha
    m.alpha = alpha
    try:
        out, grads = m.forward_backward(gen, clean)
    finally:
        m.alpha = a0
    return out, {n: g.clone() for n, g in grads.items()}


# ------------------------------------------------------------------------------------------------ reference goldens
def test_loss_backward_reproduces_reference_goldens(golden_inputs):
    """The reference's own call, `o = m(gen, clean); o["loss"].backward()`, against its fixtures."""
    g = np.load(os.path.join(GOLD, "denoiser.npz"))
    meta = json.load(open(os.path.join(GOLD, "denoiser.json")))
    m = _denoiser(meta["alpha"])
    gen, clean = (t.to(DEV) for t in golden_inputs)
    out = m(gen, clean)
    assert all(out[k].grad_fn is not None for k in ("loss", "loss_clean", "loss_denoise_dereverb"))
    with torch.no_grad():
        out_ng = m(gen, clean)
    for k in ("loss", "loss_clean", "loss_denoise_dereverb"):
        assert out_ng[k].grad_fn is None and torch.equal(out[k].detach(), out_ng[k]), k
    for k, gk in (("loss", "loss"), ("loss_clean", "loss_clean"), ("loss_denoise_dereverb", "loss_dd")):
        assert abs(out[k].item() - float(g[gk])) / float(g[gk]) < 2e-3, (k, out[k].item(), float(g[gk]))
    out["loss"].backward()
    params = dict(m.named_parameters())
    for n_, ref_norm in meta["grad_norms"].items():
        assert params[n_].grad is not None, n_
        e = abs(float(params[n_].grad.norm()) - ref_norm) / (ref_norm + 1e-12)
        assert e < GRAD_TOL, (n_, e)
    for k in g.files:
        if k.startswith("grad:"):
            e = rel(oi.subsample(params[k[5:]].grad.cpu()), g[k])
            assert e < GRAD_TOL, (k, e)
    assert all(p.grad is None for p in m.teacher.parameters())
    assert m.pos_encoding_encoder.grad is None


# ------------------------------------------------------------------------------------------------ vs the fused path
def test_autograd_gradients_are_the_fused_paths_bits(golden_inputs):
    """Deterministic mode: `loss.backward()` gives forward_backward's gradients bit for bit; loss_clean alone is the
    alpha = 1 step and loss_denoise_dereverb alone the alpha = 0 step.  Default mode: summation-order tolerance."""
    m = _denoiser(0.25)
    gen, clean = (t.to(DEV) for t in golden_inputs)

    def autograd(which):
        m.zero_grad(set_to_none=True)
        out = m(gen, clean)
        out[which].backward()
        return out, {n: gr.clone() for n, gr in _student_grads(m).items()}

    with det_mode():
        for which, alpha in (("loss", 0.25), ("loss_clean", 1.0), ("loss_denoise_dereverb", 0.0)):
            out_f, fused = _fused_grads(m, gen, clean, alpha)
            out_a, auto = autograd(which)
            assert set(auto) == set(fused), which
            for n_ in fused:
                assert torch.equal(auto[n_], fused[n_]), (which, n_)
            for k in ("loss_clean", "loss_denoise_dereverb"):
                assert torch.equal(out_a[k].detach(), out_f[k]), (which, k)
    _, fused = _fused_grads(m, gen, clean, 0.25)
    _, auto = autograd("loss")
    for n_ in fused:
        g1, g2 = fused[n_].double(), auto[n_].double()
        tol = 2e-4 if n_.endswith("in_proj_bias") else 1e-5
        assert (g1 - g2).norm().item() <= tol * g1.norm().item() + 1e-12, n_


@pytest.fixture(scope="module")
def oracle_mixed(golden_inputs):
    """torch autograd through the fp32 CPU oracle of (0.3 loss_clean + 1.7 loss_denoise_dereverb + 2 loss), alpha 0.25:
    every student gradient and the generated scene's."""
    cfg = jo.Cfg()
    sd_s = {k: v.clone().requires_grad_(v.is_floating_point() and not k.startswith(("pos_", "teacher")))
            for k, v in jo.make_state_dict(cfg, seed=11).items()}
    sd_t = jo.make_state_dict(cfg, seed=12)
    gen = golden_inputs[0].float().requires_grad_(True)
    out = jo.denoiser_forward(gen, golden_inputs[1].float(), sd_s, sd_t, cfg, 0.25)
    (0.3 * out["loss_clean"] + 1.7 * out["loss_denoise_dereverb"] + 2 * out["loss"]).backward()
    return {k: v.grad for k, v in sd_s.items() if v.grad is not None}, gen.grad


def _mixed(out):
    return 0.3 * out["loss_clean"] + 1.7 * out["loss_denoise_dereverb"] + 2 * out["loss"]


def test_mixed_upstream_matches_the_oracle(golden_inputs, oracle_mixed):
    ref, _ = oracle_mixed
    m = _denoiser(0.25)
    gen, clean = (t.to(DEV) for t in golden_inputs)
    _mixed(m(gen, clean)).backward()
    grads = _student_grads(m)
    assert set(grads) == set(ref)
    worst = max((rel(grads[n_], ref[n_]), n_) for n_ in ref)
    print(f"worst per-tensor gradient rel-L2: {worst}")
    assert worst[0] < GRAD_TOL, worst


def test_scene_gradient_matches_the_oracle(golden_inputs, oracle_mixed):
    """A generated scene that requires grad (fp32) receives the gradient of the loss through the bridge's waveform
    gradient; the clean scene, which does not, receives none.  The losses are the bits of the bf16 call."""
    _, ref_dgen = oracle_mixed
    m = _denoiser(0.25)
    gen = golden_inputs[0].float().to(DEV).requires_grad_(True)
    clean = golden_inputs[1].to(DEV)
    out = m(gen, clean)
    with torch.no_grad():
        out_ng = m(golden_inputs[0].to(DEV), clean)
    assert torch.equal(out["loss"].detach(), out_ng["loss"])
    _mixed(out).backward()
    assert gen.grad is not None and gen.grad.dtype == torch.float32 and gen.grad.shape == gen.shape
    assert clean.grad is None
    e = rel(gen.grad, ref_dgen)
    print(f"generated-scene gradient rel-L2 against the oracle: {e:.3e}")
    assert e < GRAD_TOL, e


# ------------------------------------------------------------------------------------------------ the kernel
BENCH_M = 512 * 200 * 768     # scripts/bench_denoiser.py: 512 instances per side


@pytest.mark.parametrize("M", [4, 1028, 4 * 200 * 768, BENCH_M])
@pytest.mark.parametrize("wv", [(0.25, 0.75), (0.0, -1.5), (-2.0, 0.0), (3.0, 1e-3)])
def test_mse_pair_bwd_matches_fp64(M, wv):
    g = torch.Generator(device=DEV).manual_seed(M % 9973)
    pred = torch.randn(2, M, device=DEV, generator=g)
    tgt = torch.randn(M, device=DEV, generator=g)
    wt = torch.tensor(wv, device=DEV, dtype=torch.float32)
    dp = torch.full((2, M), float("nan"), device=DEV)
    ops.mse_pair_bwd(pred, tgt, wt, dp)
    for h in range(2):
        ref = (2.0 * wt[h].double() / M) * (pred[h].double() - tgt.double())
        if wv[h] == 0.0:
            assert (dp[h] == 0).all(), h
        else:
            assert rel(dp[h], ref) < 1e-6, h
    dp2 = torch.full((2, M), float("nan"), device=DEV)
    ops.mse_pair_bwd(pred, tgt, wt, dp2)
    assert torch.equal(dp, dp2)


@pytest.mark.parametrize("alpha", [0.0, 0.25, 0.5, 1.0])
def test_mse_pair_bwd_is_mse_pairs_gradient(alpha):
    """w = (alpha, 1 - alpha), as autograd hands it to the loss Function, gives wj_mse_pair's dpred bit for bit."""
    M = 4 * 200 * 768
    pred = torch.randn(2, M, device=DEV)
    tgt = torch.randn(M, device=DEV)
    dp_f = torch.full((2, M), float("nan"), device=DEV)
    ops.mse_pair(pred, tgt, alpha, torch.zeros(2, device=DEV, dtype=torch.float64), dp_f)
    dp_b = torch.full((2, M), float("nan"), device=DEV)
    ops.mse_pair_bwd(pred, tgt, torch.tensor([alpha, 1 - alpha], device=DEV, dtype=torch.float32), dp_b)
    assert torch.equal(dp_b, dp_f)


def test_mse_pair_bwd_refuses_and_does_not_synchronise():
    M = 1001
    pred, tgt = torch.randn(2, M, device=DEV), torch.randn(M, device=DEV)
    dp = torch.full((2, M), float("nan"), device=DEV)
    with pytest.raises(_lib.WavJepaLibError, match="M % 4"):
        ops.mse_pair_bwd(pred, tgt, torch.ones(2, device=DEV), dp)
    assert torch.isnan(dp).all()
    # the kernel and the loss Function's backward read the upstream weights on the device: no host synchronisation
    M = 8 * 768
    feats = torch.randn(2, 4, M // 4, device=DEV, requires_grad=True)
    tgt = torch.randn(4 * M // 4 // 768, 768, device=DEV)
    lc, ld = _MsePair.apply(feats, tgt)
    loss = 0.25 * lc + 0.75 * ld
    dp = torch.empty(2, M, device=DEV)
    wt = torch.tensor([0.25, 0.75], device=DEV)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        ops.mse_pair_bwd(feats.detach().reshape(2, M), tgt, wt, dp)
        (dfeats,) = torch.autograd.grad(loss, feats)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert torch.equal(dfeats.reshape(2, M), dp)


# ------------------------------------------------------------------------------------------------ freezing
def test_freezing_skips_work_and_keeps_trainable_gradients(golden_inputs, monkeypatch):
    """A frozen extractor runs no conv backward and its tensors keep grad None; what is left trainable gets the full
    run's gradients bit for bit (deterministic mode).  A fully frozen student with scenes that do not require grad
    takes the no-grad path: no grad_fn, nothing saved."""
    m = _denoiser(0.25)
    gen, clean = (t.to(DEV) for t in golden_inputs)
    calls = {"conv0_bwd": 0, "conv_dgrad": 0}
    for name in calls:
        real = getattr(ops, name)

        def counted(*a, _real=real, _name=name, **k):
            calls[_name] += 1
            return _real(*a, **k)
        monkeypatch.setattr(ops, name, counted)
    with det_mode():
        m(gen, clean)["loss"].backward()
        full = {n: gr.clone() for n, gr in _student_grads(m).items()}
        assert calls == {"conv0_bwd": 1, "conv_dgrad": len(jo.Cfg().spec) - 1}
        calls.update(conv0_bwd=0, conv_dgrad=0)
        m.zero_grad(set_to_none=True)
        m.extract_audio.requires_grad_(False)
        m(gen, clean)["loss"].backward()
    assert calls == {"conv0_bwd": 0, "conv_dgrad": 0}
    for n_, gr in _student_grads(m).items():
        if n_.startswith("extract_audio."):
            assert gr is None, n_
        else:
            assert torch.equal(gr, full[n_]), n_

    m.zero_grad(set_to_none=True)
    for n_, p in m.named_parameters():
        if n_.startswith(STUDENT):
            p.requires_grad_(False)
    plans = []
    real_ff = m._core._features_forward

    def spy(x16, index, plan=None, collect=None):
        plans.append(plan)
        out, c = real_ff(x16, index, plan, collect)
        plans.append(c)
        return out, c
    monkeypatch.setattr(m._core, "_features_forward", spy)
    out = m(gen, clean)
    assert all(out[k].grad_fn is None for k in ("loss", "loss_clean", "loss_denoise_dereverb"))
    assert plans == [None, None], plans       # no plan, no saved context
    assert all(p.grad is None for p in m.parameters())


# ------------------------------------------------------------------------------------------------ Lightning loop
def test_lightning_style_loop_matches_train_step():
    """Three steps of training_step -> backward -> clip_grad_norm_(1.0) -> AdamW.step -> scheduler.step -> zero_grad with
    the optimizer and schedule of configure_optimizers, resumed at step 5000, each against the fused train_step of a
    twin that starts that step from the same weights, Adam moments and global_step.  Deterministic mode: both see the
    same gradients, so what is left is the two AdamW implementations and clip norms (the tolerance of
    test_gpu_model.py::test_denoiser_default_clip_is_the_reference_trainers)."""
    a, b = _denoiser(0.25), _denoiser(0.25)
    a.global_step = 5000
    g = torch.Generator().manual_seed(3)
    clean = torch.randn(4, 1, 32159, generator=g).bfloat16().to(DEV)
    gen = (clean.float() + 0.5 * torch.randn(4, 1, 32159, generator=g).to(DEV)).bfloat16()
    teacher_before = {n: p.detach().clone() for n, p in a.teacher.named_parameters()}
    conf = a.configure_optimizers()
    opt, sched = conf["optimizer"], conf["lr_scheduler"]["scheduler"]
    named = {n: p for n, p in a.named_parameters() if p.requires_grad}
    params = list(named.values())
    for p in params:     # a run resumed at step 5000: the scheduler's position and AdamW's step count
        opt.state[p] = dict(step=torch.tensor(5000.0), exp_avg=torch.zeros_like(p), exp_avg_sq=torch.zeros_like(p))
    sched.last_epoch = 5000
    for grp in opt.param_groups:
        grp["lr"] = a.lr_at(5000)
    core_b = b._core
    core_b._ensure_ready()
    with det_mode():
        for i in range(3):
            b.load_state_dict(a.state_dict())
            state = {n: {"exp_avg": torch.zeros_like(core_b._view(core_b._flat_p, n)),
                         "exp_avg_sq": torch.zeros_like(core_b._view(core_b._flat_p, n))} for n in core_b._train_names}
            state.update({n: {"exp_avg": opt.state[p]["exp_avg"], "exp_avg_sq": opt.state[p]["exp_avg_sq"]}
                          for n, p in named.items()})
            b.load_optimizer_state_dict({"global_step": a.global_step, "state": state})
            lr = a.lr_at(a.global_step)
            assert opt.param_groups[0]["lr"] == pytest.approx(lr, rel=1e-12)
            out = a.training_step((gen, clean), i)
            out["loss"].backward()
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
            sched.step()
            opt.zero_grad(set_to_none=True)
            b.train_step(gen, clean)
            assert a.global_step == b.global_step == 5001 + i
            pb = dict(b.named_parameters())
            for n_, p in named.items():
                d = (p.detach() - pb[n_].detach()).abs().max().item()
                assert d <= 1e-2 * lr + 2e-6 * pb[n_].detach().abs().max().item(), (i, n_, d)
    for n_, p in a.teacher.named_parameters():
        assert torch.equal(p, teacher_before[n_]), n_
    out = a.training_step((gen, clean), 3)
    out["loss"].backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        out["loss"].backward()


# ------------------------------------------------------------------------------------------------ launch count
def test_autograd_step_launches_one_kernel_more_than_forward_backward(golden_inputs):
    m = _denoiser(0.25)
    gen, clean = (t.to(DEV) for t in golden_inputs)
    m.forward_backward(gen, clean)
    m(gen, clean)["loss"].backward()
    torch.cuda.synchronize()
    n0 = _lib.kernel_launches()
    m.forward_backward(gen, clean)
    n1 = _lib.kernel_launches()
    m(gen, clean)["loss"].backward()
    n2 = _lib.kernel_launches()
    assert n2 - n1 == (n1 - n0) + 1, (n1 - n0, n2 - n1)
