"""Fine-tuning through `JEPA.get_audio_representation` on the B200: the differentiable feature path against torch autograd
through the fp32 CPU oracle, its contract (bit-identical features, grad None off the path, frozen parts skipped, one
backward per graph, tf32 stays forward-only, stock optimizers), and the odd-length conv backward of the wav2vec2
extractor.

Tolerances are the project's (tests/test_gpu_model.py): features rel-L2 <= 1e-2, every parameter gradient tensor
rel-L2 <= 2e-2 against the fp32 oracle (bf16 operands, fp32 accumulation)."""
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

DEV = "cuda"
FEAT_TOL = 1e-2
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


# name -> (cfg kwargs, seconds, size, shared extractor, batch, mask kind)
CASES = {
    "mono_dense": (dict(), 2.01, "base", False, 2, None),
    "padding_mask_ragged": (dict(), 2.01, "base", False, 3, "ragged"),
    "host_mask_hear_10s": (dict(), 2.01, "base", False, 5, "hear"),
    "nat_per_channel": (dict(in_channels=2, per_channel=True), 2.01, "base", False, 2, None),
    "nat_shared": (dict(in_channels=2, per_channel=True), 2.01, "base", True, 2, None),
    "w2v2_4s": (dict(spec=hear.W2V2_SPEC, seconds=4.02), 4.02, "base", False, 2, None),
    "large": (dict(d_model=1024, nhead=16, layers=24), 2.01, "large", False, 2, None),
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


def _oracle_grads(cfg, sd, audio, hidden, proj):
    leaves = {}
    ref_sd = {}
    for k, v in sd.items():
        if id(v) not in leaves:
            leaves[id(v)] = v.clone().requires_grad_(k.startswith(PATH))
        ref_sd[k] = leaves[id(v)]
    x = jo.local_features(audio, ref_sd, cfg)
    feats = jo.run_stack(x, ref_sd, "encoder", cfg.layers, cfg.nhead, hidden)
    (feats * proj).sum().backward()
    return feats.detach(), ref_sd


def _features(model, audio, hidden, mask):
    a = audio.to(DEV)
    if mask == "hear":
        return model.get_audio_representation(a, None, host_mask=hidden.numpy())
    return model.get_audio_representation(a, None if hidden is None else hidden.to(DEV))


@pytest.mark.parametrize("name", list(CASES))
def test_feature_path_gradients_match_the_oracle(name):
    cfg, sd, seconds, size, share, audio, hidden, mask, proj = _case(name)
    ref_feats, ref_sd = _oracle_grads(cfg, sd, audio, hidden, proj)
    model = build(cfg, sd, seconds, size, share)
    with torch.no_grad():
        f0 = _features(model, audio, hidden, mask)
    feats = _features(model, audio, hidden, mask)
    assert feats.requires_grad and feats.grad_fn is not None
    assert torch.equal(feats.detach(), f0)          # the saving forward only adds outputs
    vis = torch.ones(feats.shape[:2], dtype=torch.bool) if hidden is None else ~hidden
    assert rel(feats.detach().cpu()[vis], ref_feats[vis]) < FEAT_TOL
    if hidden is not None:
        assert not feats.detach().cpu()[hidden].any()   # padded rows stay zeros
    (feats * proj.to(DEV)).sum().backward()
    worst, n_checked = ("", 0.0), 0
    for n_, p_ in model.named_parameters():
        if not n_.startswith(PATH):
            assert p_.grad is None, n_
            continue
        assert p_.grad is not None, n_
        e = rel(p_.grad, ref_sd[n_].grad)
        worst = max(worst, (n_, e), key=lambda t: t[1])
        n_checked += 1
        assert e < GRAD_TOL, (n_, e)
    assert n_checked >= 12 * cfg.layers + 2 + 4 + len(cfg.spec) + 2, n_checked
    print(f"{name}: worst per-tensor gradient rel-L2 {worst}")


def test_product_surfaces_stay_inference_only(tmp_path):
    """HEAR, HF and ARCH call get_audio_representation under no_grad: in grad mode, with a trainable model, their
    outputs still carry no graph."""
    from wavjepa_b200 import hf
    from wavjepa_b200.arch import WavJEPAModelWrapper
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    rt = hear.load_model({"state_dict": sd})
    assert any(p.requires_grad for p in rt.model.parameters())
    audio = oi.hear_inputs(2, 48000, seed=11).to(DEV)
    emb, _ = hear.get_timestamp_embeddings(audio, rt)
    assert not emb.requires_grad
    assert not hear.get_scene_embeddings(audio, rt).requires_grad
    path = os.path.join(tmp_path, "ckpt.pt")
    torch.save({"state_dict": sd}, path)
    model = hf.WavJEPAModel.from_pretrained(path).to(DEV)
    feats = hf.WavJEPAFeatureExtractor.from_pretrained("labhamlet/wavjepa-base")(audio, return_tensors="pt")["input_values"]
    e2, _ = model(feats)
    assert not e2.requires_grad
    wrap = WavJEPAModelWrapper(build(cfg, sd), DEV, None)
    assert not wrap.get_embeddings(oi.hear_inputs(1, 40000, seed=21)[0]).requires_grad


def _grads(model):
    return {n: (None if p.grad is None else p.grad.detach().clone()) for n, p in model.named_parameters()
            if n.startswith(PATH)}


def _step(model, audio, proj):
    feats = model.get_audio_representation(audio)
    (feats * proj).sum().backward()
    return _grads(model)


@pytest.fixture
def deterministic():
    ops.set_deterministic(True)
    yield
    ops.set_deterministic(False)


def test_freezing_skips_work_and_keeps_trainable_gradients(deterministic, monkeypatch):
    """A frozen extractor runs no conv backward; the gradients of what is left trainable are those of the full run bit
    for bit; the saved activations (peak memory) shrink."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=4)
    g = torch.Generator().manual_seed(4)
    B = 16
    audio = torch.randn(B, 1, cfg.target_length, generator=g).to(DEV).bfloat16()
    proj = torch.randn(B, cfg.total_patches, cfg.d_model, generator=g).to(DEV)
    model = build(cfg, sd)
    _step(model, audio, proj)                       # warm-up (module loads, workspaces)
    model.zero_grad(set_to_none=True)

    def peak_of(fn):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = fn()
        torch.cuda.synchronize()
        return out, torch.cuda.max_memory_allocated() - base

    full, peak_full = peak_of(lambda: _step(model, audio, proj))
    calls = {"conv0_bwd": 0, "conv_dgrad": 0}
    for name in calls:
        real = getattr(ops, name)

        def counted(*a, _real=real, _name=name, **k):
            calls[_name] += 1
            return _real(*a, **k)
        monkeypatch.setattr(ops, name, counted)
    _step(model, audio, proj)
    assert calls["conv0_bwd"] == 1 and calls["conv_dgrad"] == len(cfg.spec) - 1   # the counters see the full run
    calls.update(conv0_bwd=0, conv_dgrad=0)

    model.zero_grad(set_to_none=True)
    model.extract_audio.requires_grad_(False)
    frozen, peak_frozen = peak_of(lambda: _step(model, audio, proj))
    assert calls == {"conv0_bwd": 0, "conv_dgrad": 0}
    for n_, gr in frozen.items():
        if n_.startswith("extract_audio."):
            assert gr is None, n_
        else:
            assert torch.equal(gr, full[n_]), n_

    model.zero_grad(set_to_none=True)
    model.feature_norms.requires_grad_(False)
    model.post_extraction_mapper.requires_grad_(False)
    for i in range(6):
        model.encoder.layers[i].requires_grad_(False)
    lower, peak_lower = peak_of(lambda: _step(model, audio, proj))
    for n_, gr in lower.items():
        if n_.startswith(("encoder.layers.", "encoder.norm.")) and not any(
                n_.startswith(f"encoder.layers.{i}.") for i in range(6)):
            assert torch.equal(gr, full[n_]), n_
        else:
            assert gr is None, n_
    print(f"peak allocated above the model: full {peak_full / 2**20:.0f} MiB, extractor frozen "
          f"{peak_frozen / 2**20:.0f} MiB, + 6 layers {peak_lower / 2**20:.0f} MiB")
    assert peak_frozen < peak_full and peak_lower < peak_frozen


def test_frozen_weights_inside_a_trained_layer_get_no_gradient():
    cfg = jo.Cfg()
    model = build(cfg, jo.make_state_dict(cfg, seed=6))
    lyr = model.encoder.layers[5]
    lyr.linear1.weight.requires_grad_(False)
    lyr.norm2.bias.requires_grad_(False)
    audio = torch.randn(2, 1, cfg.target_length, device=DEV).bfloat16()
    model.get_audio_representation(audio).square().mean().backward()
    assert lyr.linear1.weight.grad is None and lyr.norm2.bias.grad is None
    assert lyr.linear1.bias.grad is not None and lyr.linear2.weight.grad is not None
    assert model.extract_audio.cnn[0][0].weight.grad is not None


def test_deterministic_twins_and_gradient_accumulation(deterministic):
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=8)
    g = torch.Generator().manual_seed(8)
    a1 = torch.randn(3, 1, cfg.target_length, generator=g).to(DEV).bfloat16()
    a2 = torch.randn(3, 1, cfg.target_length, generator=g).to(DEV).bfloat16()
    proj = torch.randn(3, cfg.total_patches, cfg.d_model, generator=g).to(DEV)
    m1, m2 = build(cfg, sd), build(cfg, sd)
    g1, g1b = _step(m1, a1, proj), _step(m2, a1, proj)
    for n_ in g1:
        assert torch.equal(g1[n_], g1b[n_]), n_
    m1.zero_grad(set_to_none=True)
    g2 = _step(m1, a2, proj)
    m1.zero_grad(set_to_none=True)
    _step(m1, a1, proj)
    acc = _step(m1, a2, proj)                       # autograd adds the second backward into .grad
    for n_ in g1:
        assert torch.equal(acc[n_], g1[n_] + g2[n_]), n_


def test_limits_tf32_forward_only_and_one_backward_per_graph():
    cfg = jo.Cfg()
    model = build(cfg, jo.make_state_dict(cfg, seed=9))
    audio = torch.randn(2, 1, cfg.target_length, device=DEV).bfloat16()
    feats = model.get_audio_representation(audio)
    loss = feats.square().mean()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already backpropagated"):
        loss.backward()
    model.inference_precision = "tf32"
    t = model.get_audio_representation(audio)
    assert t.grad_fn is None and not t.requires_grad
    with torch.no_grad():
        assert torch.equal(t, model.get_audio_representation(audio))


def test_stock_adamw_loop_learns_and_the_weights_round_trip():
    """features -> mean-pool -> Linear head -> cross-entropy -> torch.optim.AdamW over the model and the head."""
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=10)
    model = build(cfg, sd)
    g = torch.Generator().manual_seed(10)
    B, n_cls = 8, 4
    audio = torch.randn(B, 1, cfg.target_length, generator=g).to(DEV).bfloat16()
    labels = torch.arange(B, device=DEV) % n_cls
    head = torch.nn.Linear(cfg.d_model, n_cls).to(DEV)
    params = [p for n, p in model.named_parameters() if n.startswith(PATH) and p.requires_grad]
    opt = torch.optim.AdamW([{"params": params}, {"params": head.parameters(), "lr": 1e-3}], lr=1e-5)
    w0 = model.encoder.layers[0].linear1.weight.detach().clone()
    c0 = model.extract_audio.cnn[3][0].weight.detach().clone()
    losses = []
    for _ in range(20):
        opt.zero_grad(set_to_none=True)
        loss = F.cross_entropy(head(model.get_audio_representation(audio).mean(dim=1)), labels)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < 0.7 * losses[0], losses
    assert not torch.equal(model.encoder.layers[0].linear1.weight, w0)
    assert not torch.equal(model.extract_audio.cnn[3][0].weight, c0)
    fresh = build(cfg, {k: v.detach().cpu() for k, v in model.state_dict().items()})
    with torch.no_grad():
        assert torch.equal(model.get_audio_representation(audio), fresh.get_audio_representation(audio))


def test_attention_backward_long_entry_takes_the_dense_nat_length():
    """The dense WavJEPA-Nat student has 2 x 200 = 400 tokens per sequence: wj_attn_varlen_bwd_bias_long keeps them
    resident (lse / delta in the Q rows' padding); the plain entry point keeps refusing them."""
    D, H, lens = 768, 12, [400, 400, 37, 385]
    cu_l = [0]
    for n in lens:
        cu_l.append(cu_l[-1] + n)
    cu = torch.tensor(cu_l, device=DEV, dtype=torch.int32)
    qkv = torch.randn(cu_l[-1], 3 * D, device=DEV).bfloat16()
    out = torch.empty(cu_l[-1], D, device=DEV, dtype=torch.bfloat16)
    lse = torch.empty(cu_l[-1], H, device=DEV)
    ops.attn_fwd(qkv, cu, len(lens), max(lens), D, H, out, lse)
    qr = qkv.float().requires_grad_(True)
    refs = []
    for s in range(len(lens)):
        x = qr[cu_l[s]:cu_l[s + 1]]
        q, k, v = (x[:, i * D:(i + 1) * D].reshape(-1, H, D // H).transpose(0, 1) for i in range(3))
        refs.append(F.scaled_dot_product_attention(q, k, v).transpose(0, 1).reshape(-1, D))
    do = torch.randn(cu_l[-1], D, device=DEV).bfloat16()
    torch.cat(refs).backward(do.float())
    dqkv = torch.full_like(qkv, float("nan"))
    dbias = torch.zeros(3 * D, device=DEV)
    ops.attn_bwd(qkv, out, do, lse, cu, len(lens), max(lens), D, H, dqkv, dbias=dbias, long_seq=True)
    assert rel(dqkv, qr.grad) < 1.5e-2
    assert rel(dbias, dqkv.float().sum(0)) < 1e-5
    with pytest.raises(_lib.WavJepaLibError):
        ops.attn_bwd(qkv, out, do, lse, cu, len(lens), max(lens), D, H, torch.empty_like(qkv))


# ------------------------------------------------------------------------------------------------ odd-length conv backward
@pytest.mark.parametrize("L_in,k", [(401, 2), (403, 3), (6429, 3)])
def test_odd_length_conv_wgrad_dgrad(L_in, k):
    Bn, Cc = 3, 512
    x = torch.randn(Bn, L_in, Cc, device=DEV).bfloat16()
    w_ = (torch.randn(Cc, Cc, k, device=DEV) * 0.03).bfloat16()
    L_out = (L_in - k) // 2 + 1
    dy = torch.randn(Bn, L_out, Cc, device=DEV).bfloat16()
    aux = (torch.rand(Bn, L_in, Cc, device=DEV) + 0.5).bfloat16()
    xf = x.float().transpose(1, 2).requires_grad_(True)
    wf = w_.float().requires_grad_(True)
    F.conv1d(xf, wf, stride=2).backward(dy.float().transpose(1, 2))
    out = torch.full((Cc, k * Cc), float("nan"), device=DEV)
    ops.gemm_wgrad(ops.make_operand(dy, Cc, L_out, Bn), ops.conv_operand_odd(x, k), L_out, Bn, out)
    assert rel(out, wf.grad.permute(0, 2, 1).reshape(Cc, k * Cc)) < 5e-5
    wk = w_.permute(0, 2, 1).reshape(Cc, k * Cc).contiguous()
    ref_dx = xf.grad.transpose(1, 2)
    dx = torch.full((Bn, L_in, Cc), float("nan"), device=DEV, dtype=torch.bfloat16)
    ops.conv_dgrad(dy, wk, dx, k)
    assert rel(dx, ref_dx) < BF16_TOL
    dx.fill_(float("nan"))
    ops.conv_dgrad(dy, wk, dx, k, act=ops.ACT_DGELU, aux=aux)     # the GELU'-factor form of the conv stack
    assert rel(dx, ref_dx * aux.float()) < BF16_TOL
    if k == 2:   # the trailing row feeds no output
        assert torch.equal(dx[:, -1].float(), torch.zeros(Bn, Cc, device=DEV))


def test_w2v2_pretraining_step_matches_the_oracle():
    """One pre-training train_step of the wav2vec2-extractor configuration (4.02 s: its last conv block reads 401 rows)
    against the live oracle: every parameter gradient tensor."""
    cfg = jo.Cfg(spec=hear.W2V2_SPEC, seconds=4.02)
    assert cfg.total_patches == 200
    sd = jo.make_state_dict(cfg, seed=12)
    inp = oi.training_inputs(cfg, 1, 2, seed=12, masker="audioset")
    ref_sd = {k: v.clone().requires_grad_(not k.startswith(("teacher_encoder.", "pos_encoding"))) for k, v in sd.items()}
    ref = jo.forward(inp["audio"], inp["ctx_masks"], inp["target_indices"], inp["ctx_and_target_masks"], ref_sd, cfg)
    ref["loss"].backward()
    model = build(cfg, sd, seconds=4.02)
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    loss = model.train_step(inp["audio"].to(DEV).bfloat16(), c_m, t_m, v_m)
    assert abs(loss.item() - ref["loss"].item()) / ref["loss"].item() < 1e-3
    n_checked = 0
    for n_, p_ in model.named_parameters():
        if not p_.requires_grad:
            continue
        e = rel(model._view(model._flat_g, n_), ref_sd[n_].grad)
        assert e < GRAD_TOL, (n_, e)
        n_checked += 1
    assert n_checked >= 300, n_checked
