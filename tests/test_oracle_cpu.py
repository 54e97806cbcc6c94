"""CPU suite (no GPU): pins the oracle restatements against the golden fixtures produced by the executed reference
(tests/golden/make_golden.py), and checks host-side logic and the C-ABI surface."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import inputs as oi
from oracle import jepa_oracle as jo
from oracle import masks_oracle as mo

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
ROOT = os.path.dirname(HERE)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


# ------------------------------------------------------------------------------------------------- masks
def _unpack(a, shape):
    return np.unpackbits(a)[:int(np.prod(shape))].reshape(shape).astype(bool)


@pytest.mark.parametrize("span", [mo.span_mask_np, mo.span_mask_py])
def test_mask_oracle_matches_reference_goldens(span):
    g = np.load(os.path.join(GOLD, "masks.npz"))
    c, t, v, a = mo.time_inverse_masks(1234, 100, 64, 200, span=span)
    assert np.array_equal(c, _unpack(g["ti_ctx"], c.shape)) and np.array_equal(t, _unpack(g["ti_tgt"], t.shape))
    assert np.array_equal(v, _unpack(g["ti_vis"], v.shape)) and np.array_equal(a, g["ti_att"])
    c, t, v, a = mo.speech_masks(99, 0, 64, 200, tgt_prob=0.1, tgt_len=10, cutoff=0.5, min_context_len=5, span=span)
    assert np.array_equal(c, _unpack(g["sp_ctx"], c.shape)) and np.array_equal(t, _unpack(g["sp_tgt"], t.shape))
    assert np.array_equal(v, _unpack(g["sp_vis"], v.shape)) and np.array_equal(a, g["sp_att"])
    c, t, v, a = mo.time_inverse_masks(5, 7, 32, 400, in_channels=2, channel_based=True, span=span)
    assert c.shape == (32, 400)
    assert np.array_equal(c, _unpack(g["nat_ctx"], c.shape)) and np.array_equal(t, _unpack(g["nat_tgt"], t.shape))
    assert np.array_equal(v, _unpack(g["nat_vis"], v.shape)) and np.array_equal(a, g["nat_att"])
    c, t, v, a = mo.time_inverse_masks(77, 0, 64, 200, cutoff=0.2, span=span)
    assert np.array_equal(c, _unpack(g["hard_ctx"], c.shape)) and np.array_equal(a, g["hard_att"])
    assert a.max() > 1  # the rejection loop is exercised


def test_mask_invariants():
    c, t, v, _ = mo.time_inverse_masks(3, 0, 128, 200)
    ctx_visible = ~c
    assert not (ctx_visible[:, None, :] & t).any()                       # context and targets are disjoint
    assert np.array_equal(v, ~(ctx_visible[:, None, :] | t))             # predictor sees context U target group
    assert (ctx_visible.sum(1) / 200 >= 0.1).all()


def test_pcg64_chain_matches_numpy():
    for words in ([0], [1234, 5, 6], [2**32 - 1, 0, 99]):
        mine = mo.Pcg64(words)
        theirs = np.random.default_rng(list(words))
        assert [mine.random() for _ in range(4)] == [theirs.random() for _ in range(4)]
        mine = mo.Pcg64(words)
        theirs = np.random.default_rng(list(words))
        assert sorted(mine.choice_no_replace(190, 13)) == sorted(theirs.choice(190, 13, replace=False).tolist())


# ------------------------------------------------------------------------------------------------- model oracle
def _run_oracle(cfg, n_clips, crops, seed, masker, backward=True):
    sd = jo.make_state_dict(cfg, seed=3)
    names = [k for k in sd if not k.startswith(("teacher_encoder.", "pos_encoding"))]
    for k in names:
        sd[k].requires_grad_(backward)
    inp = oi.training_inputs(cfg, n_clips, crops, seed=seed, masker=masker)
    out = jo.forward(inp["audio"], inp["ctx_masks"], inp["target_indices"], inp["ctx_and_target_masks"], sd, cfg)
    if backward:
        out["loss"].backward()
    return sd, inp, out


@pytest.mark.parametrize("name,cfg,crops,seed,masker", [
    ("train_c1", jo.Cfg(), 4, 1234, "audioset"),
    ("train_speech", jo.Cfg(), 2, 4321, "librispeech"),
    ("train_nat", jo.Cfg(in_channels=2, per_channel=True), 2, 55, "audioset"),
])
def test_oracle_forward_backward_matches_reference(name, cfg, crops, seed, masker):
    torch.set_num_threads(os.cpu_count())
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    meta = json.load(open(os.path.join(GOLD, f"{name}.json")))
    sd, inp, out = _run_oracle(cfg, 1, crops, seed, masker)
    assert abs(out["loss"].item() - float(g["loss"])) / float(g["loss"]) < 2e-5
    B, G, T = inp["target_indices"].shape
    preds_t = out["preds"].view(B, G, T, -1)[inp["target_indices"]]
    for k, t in (("local_features", out["local_features"]), ("contextual_features", out["contextual_features"]),
                 ("targets", out["targets"]), ("preds_at_targets", preds_t)):
        assert list(t.shape) == meta[k]["shape"], k
        assert rel(oi.subsample(t), g[k]) < 2e-4, k
        assert abs(float(t.detach().norm()) - meta[k]["l2"]) / meta[k]["l2"] < 2e-4, k
    for n_, ref_norm in meta["grad_norms"].items():
        gr = sd[n_].grad
        assert gr is not None, n_
        assert abs(float(gr.norm()) - ref_norm) / (ref_norm + 1e-12) < 2e-3, n_
    for k in g.files:
        if k.startswith("grad::"):
            assert rel(oi.subsample(sd[k[6:]].grad), g[k]) < 2e-3, k
    with torch.no_grad():
        jo.ema_update(sd, step=0)
    assert np.array_equal(oi.subsample(sd["teacher_encoder.layers.3.linear1.weight"]),
                          g["teacher_after_ema::layers.3.linear1.weight"])


def test_oracle_hear_matches_reference():
    torch.set_num_threads(os.cpu_count())
    g = np.load(os.path.join(GOLD, "hear.npz"))
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    with torch.no_grad():
        for tag, n in (("3s", 48000), ("exact", 64318)):
            emb, ts = jo.hear_timestamp_embeddings(oi.hear_inputs(2, n, seed=11), sd, cfg)
            assert list(emb.shape) == g[f"{tag}_shape"].tolist()
            assert rel(oi.subsample(emb), g[f"{tag}_emb"]) < 2e-4
            assert np.allclose(ts[0].numpy(), g[f"{tag}_ts"], rtol=1e-6, atol=1e-4)
            if tag == "3s":
                assert rel(emb.mean(1).numpy(), g["3s_scene"]) < 2e-4
    # frame geometry of hear_api/runtime.py:98-145 (SURVEY.md H3): 10 s -> 996 frames, 64318 -> 400, 1 s -> 100
    assert jo.hear_geometry(160000, 32159, 16000, 200)[:3] == (795, 5, 996)
    assert g["10s_shape"].tolist() == [2, 996, 768]
    assert jo.hear_geometry(64318, 32159, 16000, 200)[2] == 400
    assert jo.hear_geometry(16000, 32159, 16000, 200)[2] == 100


# ------------------------------------------------------------------------------------------------- host-side logic
def _model():
    import wavjepa_b200 as w

    ex = w.ConvFeatureExtractor(conv_layers_spec=jo.BASE_SPEC, in_channels=1)
    return w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
                  transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                  transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
                  transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
                  process_audio_seconds=2.01, nr_samples_per_audio=8, average_top_k_layers=8, lr=4e-4,
                  adam_weight_decay=0.04)


def test_state_dict_is_the_references():
    keys = json.load(open(os.path.join(GOLD, "ref_state_dict_keys.json")))
    m = _model()
    sd = m.state_dict()
    assert [[k, list(v.shape)] for k, v in sd.items()] == keys
    assert m.total_patches == 200 and m.target_length == 32159 and m.encoder_embedding_dim == 768
    assert sum(p.numel() for p in m.parameters() if p.requires_grad) == 111012864
    # a reference-format checkpoint loads strictly, including the torch.compile `_orig_mod` free names
    m.load_state_dict(jo.make_state_dict(jo.Cfg(), seed=3), strict=True)
    assert torch.equal(m.pos_encoding_encoder, jo.sincos_table(200, 768))


def test_schedules_and_geometry():
    from transformers import get_cosine_schedule_with_warmup
    from wavjepa_b200.extractors import out_length

    m = _model()
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.AdamW([p], lr=4e-4)
    sch = get_cosine_schedule_with_warmup(opt, num_warmup_steps=100000, num_training_steps=375000)
    for step in (0, 1, 50000, 100000, 200000, 374999):
        assert abs(m.lr_at(step) - 4e-4 * sch.lr_lambdas[0](step)) < 1e-12
    for step in (0, 1, 99999, 100000, 200000):
        assert m._get_ema_decay(step) == jo.ema_decay(step)
    assert m._get_ema_decay(0) == pytest.approx(0.999)
    assert out_length(jo.BASE_SPEC, 32159) == 200 and out_length(jo.BASE_SPEC, 64319) == 401
    assert m.extract_audio.receptive_fields[0] == 240
    m.global_step = 93750   # wavjepa/jepa.py:272-273: 1 - global_step / max_steps (375000 by default)
    assert m.get_aug_prob() == pytest.approx(0.75)
    m.global_step = 0


def test_hear_padding_pattern_is_a_function_of_the_geometry_only():
    """hear.embed_chunks hands the key-padding mask to the model as a HOST pattern that repeats per clip (no device
    read-back).  It must be the reference's mask (hear_api/runtime.py:19-35,125-131: frames [cut_off, total_steps) hidden,
    chunked into n_chunks x steps) for every clip length, including exact multiples of the unit and sub-unit clips."""
    from wavjepa_b200.hear import hear_geometry

    unit, steps, sr = 32159, 200, 16000
    for n_samples in (160000, 32159, 64318, 5000, 47999, 96477, 100000):
        pad, n_chunks, cut_off, total_steps = hear_geometry(n_samples, unit, sr, steps)
        # the reference's construction, per clip
        ref = torch.zeros(1, total_steps, dtype=torch.bool)
        ref[:, cut_off:] = True
        ref = torch.nn.functional.pad(ref, (0, max(0, n_chunks * steps - total_steps)))[:, :n_chunks * steps]
        ref = ref.reshape(n_chunks, steps)
        # ours (wavjepa_b200/hear.py: embed_chunks)
        mask = torch.zeros(max(total_steps, n_chunks * steps), dtype=torch.bool)
        mask[cut_off:total_steps] = True
        mask = mask[:n_chunks * steps].reshape(n_chunks, steps)
        assert torch.equal(mask, ref), n_samples
        assert 0 < cut_off <= total_steps and n_chunks * unit == n_samples + pad


def test_no_cpu_fallback():
    from wavjepa_b200 import _lib

    m = _model()
    with pytest.raises(_lib.WavJepaLibError):
        m.get_audio_representation(torch.zeros(1, 1, 32159), None)


def test_c_abi_exports_every_declared_symbol():
    from wavjepa_b200 import _lib

    hdr = open(os.path.join(ROOT, "include", "wavjepa_b200.h")).read()
    names = sorted(set(re.findall(r"\b(wj_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 25
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/wavjepa_b200.h but not exported"
    assert lib.wj_version() >= 1


def test_oracle_interop_rows_match_reference():
    """SURVEY.md 8(f)-3 rows, pinned by the executed reference (tests/golden/interop.npz): ARCH wrapper embedding,
    wav2vec2-extractor HEAR model (4.02 s windows), size="large" forward."""
    torch.set_num_threads(os.cpu_count())
    g = np.load(os.path.join(GOLD, "interop.npz"))
    cfg = jo.Cfg()
    sd = jo.make_state_dict(cfg, seed=3)
    with torch.no_grad():
        for tag, n in (("a", 40000), ("b", 64318)):
            v = jo.arch_get_embeddings(oi.hear_inputs(1, n, seed=21)[0], sd, cfg)
            assert v.shape == (768,) and rel(v.numpy(), g[f"arch_{tag}"]) < 2e-4, tag
        w2v2 = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)] * 2
        cfg2 = jo.Cfg(spec=w2v2, seconds=4.02)
        assert cfg2.target_length == 64319 and cfg2.total_patches == 200
        emb, ts = jo.hear_timestamp_embeddings(oi.hear_inputs(2, 100000, seed=12), jo.make_state_dict(cfg2, seed=3), cfg2)
        assert list(emb.shape) == g["w2v2_shape"].tolist() == [2, 311, 768]
        assert rel(oi.subsample(emb), g["w2v2_emb"]) < 2e-4
        assert np.allclose(ts[0].numpy(), g["w2v2_ts"], rtol=1e-6, atol=1e-4)
        cfgL = jo.Cfg(d_model=1024, nhead=16, layers=24)
        inp = oi.training_inputs(cfgL, 1, 2, seed=77, masker="audioset")
        o = jo.forward(inp["audio"], inp["ctx_masks"], inp["target_indices"], inp["ctx_and_target_masks"],
                       jo.make_state_dict(cfgL, seed=3), cfgL)
        assert abs(o["loss"].item() - float(g["large_loss"])) / float(g["large_loss"]) < 2e-5
        assert rel(oi.subsample(o["local_features"]), g["large_local"]) < 2e-4
        assert rel(oi.subsample(o["targets"]), g["large_targets"]) < 2e-4


def test_sinc_table_is_torchaudios():
    """The host-side restatement of torchaudio's polyphase Kaiser-sinc table (the reference's resampler,
    WebAudioDataModule.py:49-57) is bit-identical to the library's for the reference's arguments."""
    taf = pytest.importorskip("torchaudio.functional.functional")
    import math
    from wavjepa_b200.preprocess import BETA, LOWPASS_FILTER_WIDTH, ROLLOFF, sinc_resample_table

    for asr in (48000, 44100, 32000, 22050, 8000, 24000, 11025):
        g = math.gcd(asr, 16000)
        k_ref, w_ref = taf._get_sinc_resample_kernel(asr, 16000, g, LOWPASS_FILTER_WIDTH, ROLLOFF, "sinc_interp_kaiser", BETA,
                                                     dtype=torch.float32)
        k, w, o, n = sinc_resample_table(asr, 16000)
        assert w == w_ref and (o, n) == (asr // g, 16000 // g)
        assert torch.equal(k, k_ref[:, 0, :])


# ------------------------------------------------------------------------------------------------- denoiser stage
def test_oracle_denoiser_matches_reference():
    """SURVEY.md 8(f)-4: the restated scene generation / batch preparation / Denoiser.forward + backward against the
    fixtures produced by the executed reference (tests/golden/make_golden.py::golden_denoiser)."""
    torch.set_num_threads(os.cpu_count())
    g = np.load(os.path.join(GOLD, "denoiser.npz"))
    meta = json.load(open(os.path.join(GOLD, "denoiser.json")))
    batch = oi.denoiser_batch()
    starts, perm = torch.from_numpy(g["starts"]), torch.from_numpy(g["perm"])
    gen, clean = jo.denoiser_batch(batch, starts, perm)
    gen16, clean16 = gen.bfloat16().float(), clean.bfloat16().float()
    assert rel(oi.subsample(gen16), g["gen"]) < 2e-3 and rel(oi.subsample(clean16), g["clean"]) < 2e-3
    assert abs(float(gen16.norm()) - float(g["gen_l2"])) / float(g["gen_l2"]) < 1e-4
    cfg = jo.Cfg()
    sd_s = {k: v.clone().requires_grad_(v.is_floating_point() and not k.startswith(("pos_", "teacher")))
            for k, v in jo.make_state_dict(cfg, seed=11).items()}
    sd_t = jo.make_state_dict(cfg, seed=12)
    out = jo.denoiser_forward(gen16, clean16, sd_s, sd_t, cfg, meta["alpha"])
    for k, gk in (("loss", "loss"), ("loss_clean", "loss_clean"), ("loss_denoise_dereverb", "loss_dd")):
        assert abs(out[k].item() - float(g[gk])) / float(g[gk]) < 2e-4, (k, out[k].item(), float(g[gk]))
    out["loss"].backward()
    for n, ref_norm in meta["grad_norms"].items():
        gr = sd_s[n].grad
        assert gr is not None, n
        assert abs(float(gr.norm()) - ref_norm) / (ref_norm + 1e-12) < 5e-3, n
    for k in g.files:
        if k.startswith("grad:"):
            assert rel(oi.subsample(sd_s[k[5:]].grad), g[k]) < 5e-3, k


def test_denoiser_state_dict_is_the_references():
    import wavjepa_b200 as w
    from wavjepa_b200.denoiser import Denoiser
    keys = json.load(open(os.path.join(GOLD, "ref_denoiser_state_dict_keys.json")))
    ext = w.ConvFeatureExtractor(conv_layers_spec=[(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)], in_channels=1)
    m = Denoiser(feature_extractor=ext, transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                 transformer_encoder_cfg=w.TransformerEncoderCFG.create(), nr_samples_per_audio=2, alpha=0.25)
    own = [k for k in keys if not k.startswith("teacher.")]
    assert list(m.state_dict().keys()) == own
    m._set_teacher({"state_dict": jo.make_state_dict(jo.Cfg(), seed=12)})
    assert list(m.state_dict().keys()) == keys
    assert all(not p.requires_grad for p in m.teacher.parameters())
    assert abs(m.lr_at(2500) - 0.5e-4) < 1e-12 and m.lr_at(0) == 0.0      # 5000 warm-up steps (denoiser.py:208-209)


# ------------------------------------------------------------------------------------------------- round-2 additions
def test_oracle_hear_nat_matches_reference():
    """oracle restatement of hear_api/runtime_natjepa.py against fixtures made by executing the reference's (unmodified)
    RuntimeNatJEPA.get_timestamp_embeddings (tests/golden/make_golden.py::golden_hear_nat)."""
    torch.set_num_threads(os.cpu_count())
    g = np.load(os.path.join(GOLD, "hear_nat.npz"))
    cfg = jo.Cfg(in_channels=2, per_channel=True)
    sd = jo.make_state_dict(cfg, seed=3)
    stereo = torch.rand(2, 2, 48000, generator=torch.Generator().manual_seed(17)) * 2 - 1
    with torch.no_grad():
        emb, ts = jo.hear_nat_timestamp_embeddings(stereo, sd, cfg)
    assert list(emb.shape) == list(g["stereo_shape"]) and np.allclose(ts[0].numpy(), g["stereo_ts"], rtol=1e-6)
    assert rel(oi.subsample(emb), g["stereo_emb"]) < 2e-4
    assert rel(emb.mean(dim=1).numpy(), g["stereo_scene"]) < 2e-4


def test_lightning_base_is_used_when_available():
    """VERDICT r1 missing 4: JEPA / Denoiser derive from pytorch_lightning.LightningModule when Lightning is importable
    (checked in a fresh interpreter with a stand-in `pytorch_lightning` package, since the image has none), and from the
    shim otherwise; either way the members the reference's loop touches exist."""
    import subprocess
    import sys
    import textwrap
    code = textwrap.dedent("""
        import sys, types, torch
        from torch import nn
        pl = types.ModuleType("pytorch_lightning")
        class LightningModule(nn.Module):
            def __init__(self):
                super().__init__(); self._hp = {}; self._trainer = None
            def save_hyperparameters(self, *a, **k):
                for x in a: self._hp.update(x)
            @property
            def hparams(self):
                return types.SimpleNamespace(**self._hp)
            @property
            def trainer(self):
                if self._trainer is None: raise RuntimeError("not attached")
                return self._trainer
            @trainer.setter
            def trainer(self, t): self._trainer = t
            @property
            def global_step(self): return self.trainer.global_step
            def log_dict(self, *a, **k): pass
        pl.LightningModule = LightningModule
        sys.modules["pytorch_lightning"] = pl
        import wavjepa_b200 as w
        from wavjepa_b200 import _lightning
        assert _lightning.HAVE_LIGHTNING and issubclass(w.JEPA, LightningModule) and issubclass(w.Denoiser, LightningModule)
        spec = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)]
        m = w.JEPA(feature_extractor=w.ConvFeatureExtractor(conv_layers_spec=spec, in_channels=1),
                   transformer_encoder_cfg=w.TransformerEncoderCFG.create(num_layers=1),
                   transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
                   transformer_decoder_cfg=w.TransformerEncoderCFG.create(num_layers=1),
                   transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384))
        assert m.hparams.lr == 0.0002 and m.global_step == 0          # detached: our own counter
        m.trainer = types.SimpleNamespace(global_step=123, max_steps=10)
        assert m.global_step == 123 and abs(m._get_ema_decay() - (0.99999 - 0.00099 * (1 - 123 / 100000))) < 1e-12
        print("OK")
    """)
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]
    from wavjepa_b200 import _lightning
    import wavjepa_b200 as w
    assert issubclass(w.JEPA, _lightning.Base) and hasattr(w.JEPA, "log_dict") and hasattr(w.JEPA, "save_hyperparameters")


def test_hf_feature_extractor_and_reference_staging(tmp_path):
    from wavjepa_b200 import hf
    ext = hf.WavJEPAFeatureExtractor.from_pretrained("labhamlet/wavjepa-base", trust_remote_code=True)
    out = ext([torch.ones(5), torch.ones(8)], return_tensors="pt")
    assert tuple(out["input_values"].shape) == (2, 8) and out.input_values[0, 5:].abs().sum() == 0
    assert tuple(ext(torch.zeros(160000))["input_values"].shape) == (1, 160000)
    with pytest.raises(ValueError):
        ext(torch.zeros(10), sampling_rate=44100)
    # the staged reference copy (bench.py's reference arms) is a byte-identical copy of a checkout's hot-path packages,
    # with a sha256 manifest; checked on a small stand-in checkout in the reference's flat layout
    import hashlib
    from oracle import stage_reference
    src, dest = tmp_path / "reference", tmp_path / "staged"
    staged = {"wavjepa/jepa.py": b"class JEPA: pass\n", "wavjepa/extractors/__init__.py": b"",
              "hear_api/runtime.py": b"def load_model(): pass\n", "hear_configs/WavJEPA.py": b"# config\n",
              "data_modules/__init__.py": b"", "utils.py": b"def util(): pass\n", "LICENSE": b"MIT\n"}
    left_out = {"train.py": b"main()\n", "wavjepa/__pycache__/jepa.cpython-312.pyc": b"\0", "wavjepa/clip.wav": b"RIFF",
                "hear_api/model.ckpt": b"\0"}
    for rel_path, data in {**staged, **left_out}.items():
        (src / rel_path).parent.mkdir(parents=True, exist_ok=True)
        (src / rel_path).write_bytes(data)
    assert stage_reference.stage(str(src), str(dest)) == str(dest)
    man = json.load(open(dest / "MANIFEST.json"))["files"]
    assert sorted(man) == sorted(staged)
    for rel_path, data in staged.items():
        assert (dest / rel_path).read_bytes() == data and man[rel_path] == hashlib.sha256(data).hexdigest(), rel_path
    assert stage_reference.stage(str(tmp_path / "absent"), str(tmp_path / "none")) is None
    assert not (tmp_path / "none").exists()
