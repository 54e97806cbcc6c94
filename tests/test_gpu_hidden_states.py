"""Per-layer encoder hidden states, `JEPA.get_hidden_states`, on the B200: every hidden state against the fp32 CPU oracle
(bf16 and tf32), its contract (the same bits whichever layers are requested, in grad mode or not, hidden state N under
the final LayerNorm is get_audio_representation, early exit, nothing saved without a graph, argument checks), gradients
of a loss over several hidden states against torch autograd through the oracle, frozen parts, the gather-add kernel that
injects their gradients, a SUPERB-style weighted-sum training loop, and `layer=` on the HEAR and HF loaders.

Tolerances are the project's (tests/test_gpu_finetune.py, tests/test_gpu_tf32.py): hidden states rel-L2 <= 1e-2 in bf16,
<= 2e-3 in tf32; every gradient tensor rel-L2 <= 2e-2."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import wavjepa_b200 as w
from wavjepa_b200 import _lib, hear, jepa, ops
from oracle import inputs as oi
from oracle import jepa_oracle as jo

gpu = pytest.mark.gpu
DEV = "cuda"
FEAT_TOL = 1e-2
TF32_TOL = 2e-3
GRAD_TOL = 2e-2
PATH = ("extract_audio.", "feature_norms.", "post_extraction_mapper.", "encoder.")


def rel(a, b):
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(autouse=True)
def _device(request):
    if request.node.get_closest_marker("gpu") is not None:
        _lib.require_device()
        torch.manual_seed(0)
        torch.set_num_threads(os.cpu_count())


@pytest.fixture
def deterministic():
    ops.set_deterministic(True)
    yield
    ops.set_deterministic(False)


def build(cfg: jo.Cfg, sd, seconds=2.01, size="base", share=False, device=DEV):
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
    return m.to(device)


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


# name -> (cfg kwargs, seconds, size, shared extractor, batch, mask kind): the geometries of test_gpu_finetune.py
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
    return cfg, sd, seconds, size, share, audio, hidden, mask, g


def _subset(n_layers):
    """Hidden state 0, a middle layer and the top requested one below N, in a non-sorted order."""
    return [3 * n_layers // 4, 0, n_layers // 2]


def _projections(g, subset, B, T, D, hidden):
    proj = {}
    for k in subset:
        p = torch.randn(B, T, D, generator=g)
        proj[k] = p if hidden is None else p * (~hidden)[..., None]   # the loss reads the visible rows only
    return proj


def _oracle(cfg, sd, audio, hidden, proj):
    """fp32 CPU autograd: (all N + 1 hidden states, audio.grad, {name: param grad}) for sum_k <proj_k, h_k>."""
    leaves, ref_sd = {}, {}
    for k, v in sd.items():
        if id(v) not in leaves:
            leaves[id(v)] = v.clone().requires_grad_(k.startswith(PATH))
        ref_sd[k] = leaves[id(v)]
    a = audio.clone().requires_grad_(True)
    hs = [jo.local_features(a, ref_sd, cfg)]
    jo.run_stack(hs[0], ref_sd, "encoder", cfg.layers, cfg.nhead, hidden, final_norm=False,
                 collect=lambda i, y: hs.append(y))
    sum((hs[k] * p).sum() for k, p in proj.items()).backward()
    return [h.detach() for h in hs], a.grad, {k: v.grad for k, v in ref_sd.items() if k.startswith(PATH)}


def _hidden(model, audio, hidden, mask, layers=None):
    if mask == "hear":
        return model.get_hidden_states(audio, None, host_mask=hidden.numpy(), layers=layers)
    return model.get_hidden_states(audio, None if hidden is None else hidden.to(DEV), layers=layers)


@gpu
@pytest.mark.parametrize("name", list(CASES))
def test_hidden_states_and_their_gradients_match_the_oracle(name):
    cfg, sd, seconds, size, share, audio, hidden, mask, g = _case(name)
    B, T, D, N = audio.shape[0], cfg.total_patches, cfg.d_model, cfg.layers
    subset = _subset(N)
    top = max(subset)
    proj = _projections(g, subset, B, T, D, hidden)
    ref_h, ref_dx, ref_g = _oracle(cfg, sd, audio, hidden, proj)
    model = build(cfg, sd, seconds, size, share)
    vis = torch.ones(B, T, dtype=torch.bool) if hidden is None else ~hidden
    # ---- forward parity, every hidden state, both numerics
    errs = {}
    for precision, tol in (("bf16", FEAT_TOL), ("tf32", TF32_TOL)):
        model.inference_precision = precision
        with torch.no_grad():
            hs = _hidden(model, audio.to(DEV), hidden, mask)
        assert len(hs) == N + 1
        for k, h in enumerate(hs):
            assert h.shape == (B, T, D) and h.dtype == torch.float32 and h.device.type == "cuda"
            e = rel(h.cpu()[vis], ref_h[k][vis])
            assert e <= tol, (precision, k, e)
            if hidden is not None:
                assert not h.cpu()[hidden].any(), (precision, k)   # hidden tokens' rows are constant zeros
            errs[(precision, k)] = e
    h_t = _hidden(model, audio.to(DEV).requires_grad_(True), hidden, mask, layers=subset)
    assert all(h.grad_fn is None and not h.requires_grad for h in h_t)   # tf32 stays forward-only
    model.inference_precision = "bf16"
    # ---- gradients of a loss over three hidden states, with the waveform
    with torch.no_grad():
        h0 = _hidden(model, audio.to(DEV), hidden, mask, layers=subset)
    a = audio.to(DEV).requires_grad_(True)
    hs = _hidden(model, a, hidden, mask, layers=subset)
    for h, h_ref in zip(hs, h0):
        assert h.grad_fn is not None and torch.equal(h.detach(), h_ref)   # grad mode: the same bits
    sum((h * proj[k].to(DEV)).sum() for k, h in zip(subset, hs)).backward()
    e_dx = rel(a.grad, ref_dx)
    assert e_dx <= GRAD_TOL, e_dx
    worst, n_checked = ("", 0.0), 0
    for n_, p_ in model.named_parameters():
        in_graph = n_.startswith(PATH) and not n_.startswith("encoder.norm.") and not (
            n_.startswith("encoder.layers.") and int(n_.split(".")[2]) >= top)
        if not in_graph:
            assert p_.grad is None, n_
            continue
        assert p_.grad is not None, n_
        e = rel(p_.grad, ref_g[n_])
        worst = max(worst, (n_, e), key=lambda t: t[1])
        n_checked += 1
        assert e < GRAD_TOL, (n_, e)
    assert n_checked >= 12 * top + 4 + len(cfg.spec), n_checked
    print(f"{name}: worst hidden state bf16 {max(v for (p, _), v in errs.items() if p == 'bf16'):.2e}, "
          f"tf32 {max(v for (p, _), v in errs.items() if p == 'tf32'):.2e}; audio.grad {e_dx:.2e}; "
          f"worst parameter {worst}")


# ------------------------------------------------------------------------------------------------ contract
def test_layers_are_checked_on_the_host():
    cfg = jo.Cfg()
    model = build(cfg, jo.make_state_dict(cfg, seed=1), device="cpu")
    assert model._hidden_layers(None) == list(range(13))
    assert model._hidden_layers((12, np.int64(0), 5)) == [12, 0, 5]
    audio = torch.zeros(1, 1, cfg.target_length)
    for bad in ([], [13], [-1], [3, 3], [1.0], [True], "3", 3):
        with pytest.raises(ValueError):
            model.get_hidden_states(audio, layers=bad)
    with pytest.raises(ValueError):
        hear.load_model({"state_dict": jo.make_state_dict(cfg, seed=1)}, layer=13)
    with pytest.raises(ValueError):
        hear.load_model_nat({"state_dict": jo.make_state_dict(jo.Cfg(in_channels=2, per_channel=True), seed=1)},
                            layer=-1)


@gpu
def test_contract_bits_early_exit_and_inference_saves_nothing(monkeypatch):
    cfg = jo.Cfg()
    model = build(cfg, jo.make_state_dict(cfg, seed=9))
    N = cfg.layers
    g = torch.Generator().manual_seed(9)
    B, T, D = 3, cfg.total_patches, cfg.d_model
    audio = (torch.randn(B, 1, cfg.target_length, generator=g) * 0.5).to(DEV)
    pm = ragged_mask(B, T, [T, 137, 61]).to(DEV)
    with torch.no_grad():
        every = model.get_hidden_states(audio, pm)
        for k in (0, 1, 6, N):
            assert torch.equal(model.get_hidden_states(audio, pm, layers=[k])[0], every[k]), k
        sub = model.get_hidden_states(audio, pm, layers=[N, 0, 6])
        assert all(torch.equal(s, every[k]) for s, k in zip(sub, (N, 0, 6)))
        # hidden state N through the final LayerNorm kernel is get_audio_representation, at the visible rows
        feats = model.get_audio_representation(audio, pm)
        rows = (~pm).reshape(-1)
        xN = every[N].reshape(B * T, D)[rows].contiguous()
        normed = torch.empty_like(xN)
        ops.layernorm_fwd(xN, model.encoder.norm.weight.detach(), model.encoder.norm.bias.detach(),
                          model.encoder.norm.eps, normed, None, None, None)
        assert torch.equal(normed, feats.reshape(B * T, D)[rows])
        dense = model.get_hidden_states(audio)
        dense6 = model.get_hidden_states(audio, layers=[6, 2])
        assert torch.equal(dense6[0], dense[6]) and torch.equal(dense6[1], dense[2])
    # early exit: layers=[k] runs k encoder layers and no final norm
    n_attn = []
    real_attn = ops.attn_fwd
    monkeypatch.setattr(ops, "attn_fwd", lambda *a_, **k_: n_attn.append(1) or real_attn(*a_, **k_))
    with torch.no_grad():
        for k in (0, 1, 6, N):
            n_attn.clear()
            model.get_hidden_states(audio, pm, layers=[k])
            assert len(n_attn) == k, (k, len(n_attn))
        n_attn.clear()
        model.get_audio_representation(audio, pm)
        assert len(n_attn) == N
    n_tf = []
    real_tf = ops.attn_fwd_f32
    monkeypatch.setattr(ops, "attn_fwd_f32", lambda *a_, **k_: n_tf.append(1) or real_tf(*a_, **k_))
    model.inference_precision = "tf32"
    with torch.no_grad():
        model.get_hidden_states(audio, pm, layers=[4])
        assert len(n_tf) == 4
        n_tf.clear()
        model.get_hidden_states(audio, pm, layers=[0])
        assert not n_tf
    model.inference_precision = "bf16"
    # no graph: nothing saved, no Function, no final norm
    model.requires_grad_(False)
    calls, saves = [], []
    real_bridge = jepa._FeatureBridge.apply
    monkeypatch.setattr(jepa._FeatureBridge, "apply", lambda *a_, **k_: calls.append(1) or real_bridge(*a_, **k_))
    real_stack, real_conv, real_ln = model._enc_stack.forward, jepa.conv_stack_forward, ops.layernorm_fwd
    monkeypatch.setattr(model._enc_stack, "forward", lambda *a_, **k_: saves.append(a_[6]) or real_stack(*a_, **k_))
    monkeypatch.setattr(jepa, "conv_stack_forward", lambda *a_, **k_: saves.append(a_[6]) or real_conv(*a_, **k_))
    monkeypatch.setattr(ops, "layernorm_fwd", lambda *a_, **k_: saves.append(a_[6] is not None) or real_ln(*a_, **k_))
    hs = model.get_hidden_states(audio, pm, layers=[6])
    assert hs[0].grad_fn is None and not calls
    assert len(saves) == 3 and not any(saves), saves   # conv stack, feature norm, encoder; no final norm
    assert torch.equal(hs[0], every[6])
    # a graph supports one backward; the waveform gradient comes back in audio's dtype and device
    a = audio.cpu().bfloat16().requires_grad_(True)
    h = model.get_hidden_states(a, pm, layers=[0, 3])
    assert calls and all(t.grad_fn is not None for t in h)
    loss = h[1].square().sum() + h[0].sum()
    loss.backward(retain_graph=True)
    assert a.grad.dtype == torch.bfloat16 and a.grad.device.type == "cpu" and a.grad.shape == a.shape
    with pytest.raises(RuntimeError, match="already backpropagated"):
        loss.backward()
    # one of several returned hidden states feeding the loss: the others arrive as None
    model.encoder.layers[2].requires_grad_(True)
    h = model.get_hidden_states(audio, pm, layers=[1, 3, 5])
    h[1].square().sum().backward()
    assert model.encoder.layers[2].linear1.weight.grad is not None


@gpu
def test_frozen_plans_give_the_same_gradients_and_skip_weight_work(deterministic, monkeypatch):
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=4)
    g = torch.Generator().manual_seed(4)
    B, T, D = 4, cfg.total_patches, cfg.d_model
    audio = (torch.randn(B, 1, cfg.target_length, generator=g) * 0.5).to(DEV)
    layers = [0, 4, 9]
    proj = [torch.randn(B, T, D, generator=g).to(DEV) for _ in layers]
    model = build(cfg, sd)

    def step(audio_grad=False):
        a = audio.clone().requires_grad_(audio_grad)
        hs = model.get_hidden_states(a, layers=layers)
        sum((h * p).sum() for h, p in zip(hs, proj)).backward()
        grads = {n: None if p.grad is None else p.grad.clone() for n, p in model.named_parameters() if n.startswith(PATH)}
        model.zero_grad(set_to_none=True)
        return (a.grad.clone() if audio_grad else None), grads

    dx_full, full = step(True)
    assert all((full[n] is None) == (n.startswith("encoder.norm.") or (n.startswith("encoder.layers.") and
                                                                        int(n.split(".")[2]) >= 9)) for n in full)
    model.extract_audio.requires_grad_(False)
    _, frozen = step()
    for n_, gr in frozen.items():
        if n_.startswith("extract_audio."):
            assert gr is None, n_
        elif full[n_] is not None:
            assert torch.equal(gr, full[n_]), n_
    model.feature_norms.requires_grad_(False)
    model.post_extraction_mapper.requires_grad_(False)
    for i in range(4):
        model.encoder.layers[i].requires_grad_(False)
    _, lower = step()
    for n_, gr in lower.items():
        if n_.startswith("encoder.layers.") and 4 <= int(n_.split(".")[2]) < 9:
            assert torch.equal(gr, full[n_]), n_
        else:
            assert gr is None, n_
    # frozen model, waveform gradient only: no weight-gradient GEMM and no bias column sum
    model.requires_grad_(False)
    calls = {"gemm_wgrad": 0, "colsum": 0, "add_rows": 0}
    for name in calls:
        real = getattr(ops, name)

        def counted(*a_, _real=real, _name=name, **k_):
            calls[_name] += 1
            return _real(*a_, **k_)
        monkeypatch.setattr(ops, name, counted)
    dx_frozen, g_frozen = step(True)
    assert calls["gemm_wgrad"] == 0 and calls["colsum"] == 0, calls
    assert calls["add_rows"] == 2, calls   # hidden states 4 and 0 join the backward; 9 starts it
    assert all(v is None for v in g_frozen.values())
    assert torch.equal(dx_frozen, dx_full)


# ------------------------------------------------------------------------------------------------ kernel
@gpu
@pytest.mark.parametrize("N,D", [(1, 4), (37, 768), (1000, 1024)])
def test_add_rows_matches_torch(N, D):
    g = torch.Generator(device=DEV).manual_seed(N)
    a = torch.randn(N, D, device=DEV, generator=g)
    b = torch.randn(3 * N, D, device=DEV, generator=g)
    idx = torch.randperm(3 * N, device=DEV, generator=g)[:N].to(torch.int32)
    out = a.clone()
    ops.add_rows(out, b, idx, N)
    assert torch.equal(out, a + b[idx.long()])
    out = a.clone()
    ops.add_rows(out, b, None, N)
    assert torch.equal(out, a + b[:N])
    with pytest.raises(_lib.WavJepaLibError):
        ops.add_rows(a[:, :D - 2].contiguous(), b[:, :D - 2].contiguous(), None, N)


# ------------------------------------------------------------------------------------------------ training loop
@gpu
def test_superb_weighted_sum_head_trains():
    """softmax-weighted sum of all 13 hidden states -> mean-pool -> Linear -> cross-entropy; the top four encoder
    layers, the layer weights and the head train with torch.optim.AdamW (the loss fell 1.45 -> 1.29 over the 20 steps
    on a B200; the bound asks for a clear decrease, not a rate)."""
    cfg = jo.Cfg()
    model = build(cfg, jo.make_state_dict(cfg, seed=10))
    model.requires_grad_(False)
    for i in range(8, 12):
        model.encoder.layers[i].requires_grad_(True)
    g = torch.Generator().manual_seed(10)
    B, n_cls = 8, 4
    audio = torch.randn(B, 1, cfg.target_length, generator=g).to(DEV).bfloat16()
    labels = torch.arange(B, device=DEV) % n_cls
    head = torch.nn.Linear(cfg.d_model, n_cls).to(DEV)
    mix = torch.nn.Parameter(torch.zeros(cfg.layers + 1, device=DEV))
    trainable = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.AdamW([{"params": trainable}, {"params": [*head.parameters(), mix], "lr": 1e-3}], lr=1e-5)
    w0 = model.encoder.layers[10].linear1.weight.detach().clone()
    losses = []
    for _ in range(20):
        opt.zero_grad(set_to_none=True)
        hs = model.get_hidden_states(audio)
        x = sum(wk * h for wk, h in zip(torch.softmax(mix, 0), hs))
        loss = F.cross_entropy(head(x.mean(dim=1)), labels)
        loss.backward()
        assert model.encoder.layers[7].linear1.weight.grad is None and model.encoder.norm.weight.grad is None
        opt.step()
        losses.append(loss.item())
    assert all(np.isfinite(losses)), losses
    assert losses[-1] < 0.95 * losses[0], losses
    assert not torch.equal(model.encoder.layers[10].linear1.weight, w0)
    assert not torch.equal(mix.detach(), torch.zeros_like(mix))


# ------------------------------------------------------------------------------------------------ HEAR / HF
@gpu
@pytest.mark.parametrize("nat", [False, True])
def test_hear_layer_option_matches_the_oracle(nat, tmp_path, monkeypatch):
    from wavjepa_b200 import hf
    cfg = jo.Cfg(in_channels=2, per_channel=True) if nat else jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    k = 5
    audio = oi.hear_inputs(2, 48000, seed=11)
    load = hear.load_model_nat if nat else hear.load_model
    rt = load({"state_dict": sd}, layer=k)
    emb, ts = hear.get_timestamp_embeddings(audio.to(DEV), rt)
    # the oracle's HEAR computation reading hidden state k instead of the final features
    real_stack = jo.run_stack
    monkeypatch.setattr(jo, "run_stack", lambda x, sd_, prefix, n, nhead, m, **kw:
                        real_stack(x, sd_, prefix, k, nhead, m, final_norm=False))
    with torch.no_grad():
        ref, ref_ts = (jo.hear_nat_timestamp_embeddings if nat else jo.hear_timestamp_embeddings)(audio, sd, cfg)
    monkeypatch.undo()
    assert emb.shape == ref.shape and torch.allclose(ts, ref_ts)
    e = rel(emb, ref)
    assert e <= FEAT_TOL, e
    # layer=None is today's output bit for bit; another layer is another output
    base, _ = hear.get_timestamp_embeddings(audio.to(DEV), load({"state_dict": sd}))
    none, _ = hear.get_timestamp_embeddings(audio.to(DEV), load({"state_dict": sd}, layer=None))
    assert torch.equal(base, none) and not torch.equal(base, emb)
    # hf.WavJEPAModel.from_pretrained forwards layer= to the HEAR loader
    path = os.path.join(tmp_path, "ckpt.pt")
    torch.save({"state_dict": sd}, path)
    model = hf.WavJEPAModel.from_pretrained(path, layer=k)
    fe = hf.WavJEPAFeatureExtractor.from_pretrained("labhamlet/wavjepa-nat-base" if nat else "labhamlet/wavjepa-base")
    e2, _ = model(fe(audio, return_tensors="pt")["input_values"].to(DEV))
    assert torch.equal(e2, emb)
    with pytest.raises(ValueError):
        load({"state_dict": sd}, layer=cfg.layers + 1)
    print(f"HEAR layer {k} ({'nat' if nat else 'mono'}): rel-L2 {e:.2e} against the oracle")
