"""WavJEPA-Nat denoiser stage (SURVEY.md 8(f)-4) on the sm_100a kernels.

Mirrors, with the same names / arguments / state_dict keys:
  wavjepa/denoiser.py:43-376         Denoiser (student = extractor + LayerNorm + mapper + 12-layer encoder on FULL
                                     200-token sequences; frozen WavJEPA-Clean teacher; two dense latent MSE losses)
  wavjepa/denoiser.py:29-41          resample (Kaiser-sinc, 32 kHz -> 16 kHz)
  data_modules/scene_module/generate_scenes_batch.py:12-188   generate_scene (RIR convolution, noise aggregation,
                                     segmental-SNR mixing)

B200-first differences (results identical up to the documented tolerances):
  * the reference runs the student twice (clean, generated) and the teacher once; here the two student passes are ONE
    packed batch of 2N sequences through the same kernels (no cross-sequence interaction anywhere in the stack), the
    teacher is `JEPA.get_audio_representation` on the same kernels;
  * forward, hand-written backward, AdamW (+ cosine schedule with 5000 warm-up steps, denoiser.py:208-209) and the bf16
    weight refresh are one fused `train_step`; there is no autograd graph;
  * scene generation: the RIR convolutions are FFT convolutions of full length (`torch.fft`, i.e. cuFFT as a plain
    library, exactly torchaudio.functional.fftconvolve's rfft -> product -> irfft with n = L1 + L2 - 1); the segmental
    SNR mix, the resampler, the crop + normalise pass are kernels of libwavjepa_b200.so.
The flat-buffer / weight-view / conv machinery is `JEPA`'s: the student lives in a private JEPA core whose parameter
objects are registered here under the reference's Denoiser names (its predictor is a one-layer stub that is never run).
"""
from __future__ import annotations

import math
from typing import Any, Optional, Tuple

import torch
from torch import nn

from . import ops
from ._lib import WavJepaLibError
from .extractors import ConvFeatureExtractor
from .hear import fix_state_dict_keys
from ._lightning import Base as _ModuleBase
from .jepa import JEPA
from .preprocess import sinc_resample_table
from .types import ForwardReturn, TransformerEncoderCFG, TransformerLayerCFG

ORIGINAL_SR = 32000
BASE_SPEC = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)]


# ------------------------------------------------------------------------------------------------- scene generation
def convolve_with_rir(waveform: torch.Tensor, rir: torch.Tensor) -> torch.Tensor:
    """generate_scenes_batch.py:12-45: waveform [B, T], rir [B, C, R] -> [B, C, T] = fftconvolve(w_b, rir_b,c)[:T]."""
    B, T = waveform.shape
    R = rir.shape[-1]
    n = T + R - 1
    fw = torch.fft.rfft(waveform.float(), n=n)                       # [B, n/2+1]
    fr = torch.fft.rfft(rir.float(), n=n)                            # [B, C, n/2+1]
    return torch.fft.irfft(fw.unsqueeze(1) * fr, n=n)[..., :T].contiguous()


def aggregate_noise(noise_rirs: torch.Tensor, noise_source: torch.Tensor) -> torch.Tensor:
    """generate_scenes_batch.py:48-73: noise_rirs [B, S, C, R], noise_source [B, T] -> sum over the S sources."""
    B, T = noise_source.shape
    S, R = noise_rirs.shape[1], noise_rirs.shape[-1]
    n = T + R - 1
    fw = torch.fft.rfft(noise_source.float(), n=n)                   # [B, n/2+1]
    agg = None
    for i in range(S):   # summed in the time domain in the reference's order (fp32 rounding)
        y = torch.fft.irfft(fw.unsqueeze(1) * torch.fft.rfft(noise_rirs[:, i].float(), n=n), n=n)[..., :T]
        agg = y if agg is None else agg + y
    return agg.contiguous()


def add_noise(source: torch.Tensor, noise: torch.Tensor, snr, start_idx, real_noise_length) -> torch.Tensor:
    """generate_scenes_batch.py:107-146 on the snr_mix kernel.  source, noise [B, 1, T]."""
    B, C, T = source.shape
    if C != 1:
        raise WavJepaLibError("add_noise is built for mono scenes (the reference asserts one channel, denoiser.py:270)")
    dev = source.device
    as_i32 = lambda v: (v.to(dev) if isinstance(v, torch.Tensor) else torch.full((B,), int(v), device=dev)).reshape(B).to(torch.int32)
    snr_t = (snr.to(dev) if isinstance(snr, torch.Tensor) else torch.full((B,), float(snr), device=dev)).reshape(B).float()
    out = torch.empty(B, T, device=dev, dtype=torch.float32)
    ops.snr_mix(source.reshape(B, T).float().contiguous(), noise.reshape(B, T).float().contiguous(), as_i32(start_idx),
                as_i32(real_noise_length), snr_t.contiguous(), out)
    return out.view(B, 1, T)


def generate_scene(source_rir, noise_rirs, source, noise, real_noise_length, noise_start_idx, snr) -> torch.Tensor:
    """generate_scenes_batch.py:148-188 (the four cases; output [B, 1, T])."""
    has_rir = source_rir is not None and source_rir[0] is not None
    has_noise = noise is not None and noise[0] is not None
    if has_rir and has_noise:
        conv = convolve_with_rir(source, source_rir[:, [0], :])
        agg = aggregate_noise(noise_rirs[:, :, [0], :], noise)[:, :, :source.shape[-1]]
        return add_noise(conv, agg, snr, noise_start_idx, real_noise_length)
    if has_rir:
        return convolve_with_rir(source, source_rir[:, [0], :])
    if has_noise:
        src = source if source.dim() == 3 else source.unsqueeze(1)
        nz = noise if noise.dim() == 3 else noise.unsqueeze(1)
        return add_noise(src, nz, snr, noise_start_idx, real_noise_length)
    return source


_RESAMPLE_TABLES = {}


def resample(audio: torch.Tensor, resample_sr: int, original_sr: int = ORIGINAL_SR) -> torch.Tensor:
    """wavjepa/denoiser.py:29-41 (torchaudio Kaiser-sinc resampling) on the resample kernel.  audio [..., L] fp32."""
    if resample_sr == original_sr:
        return audio
    dev = audio.device
    key = (original_sr, resample_sr, dev)
    if key not in _RESAMPLE_TABLES:
        k, width, orig, new = sinc_resample_table(original_sr, resample_sr)
        _RESAMPLE_TABLES[key] = (k.t().contiguous().to(dev), width, orig, new)
    table_t, width, orig, new = _RESAMPLE_TABLES[key]
    lead, L = audio.shape[:-1], audio.shape[-1]
    target = -((-new * L) // orig)
    x = audio.reshape(-1, L).float().contiguous()
    out = torch.empty(x.shape[0], target, device=dev, dtype=torch.float32)
    scratch = torch.zeros(1, device=dev, dtype=torch.float64)
    for i in range(x.shape[0]):
        ops.resample_sinc(x[i], table_t, orig, new, width, target, out[i], scratch)
    return out.view(*lead, target)


# ------------------------------------------------------------------------------------------------- the module
class Denoiser(_ModuleBase):
    """reference wavjepa/denoiser.py:43-376."""
    TARGET_SECONDS: int = 10
    ORIGINAL_SR = ORIGINAL_SR

    def __init__(self, feature_extractor, transformer_encoder_layers_cfg: TransformerLayerCFG,
                 transformer_encoder_cfg: TransformerEncoderCFG, lr: float = 0.0001, adam_betas: tuple = (0.9, 0.98),
                 adam_eps: float = 1e-06, adam_weight_decay: float = 0.0, resample_sr: int = 16000,
                 process_audio_seconds: float = 2.01, nr_samples_per_audio: int = 16, size: str = "base",
                 alpha: float = 0.0, max_steps: int = 375000, grad_clip: float = 1.0, **kwargs: Any):
        super().__init__()
        # grad_clip: the reference trains this stage with gradient_clip_val=1.0, gradient_clip_algorithm='norm'
        # (denoise.py:125-126); 0 disables clipping
        self.alpha = alpha
        self.sr = resample_sr
        self.target_audio_length = self.TARGET_SECONDS * self.sr
        self.process_audio_seconds = process_audio_seconds
        self.nr_samples_per_audio = nr_samples_per_audio
        self.target_length = int(resample_sr * process_audio_seconds)
        self.total_patches = feature_extractor.total_patches(self.target_length)
        self.save_hyperparameters(dict(lr=lr, adam_betas=tuple(adam_betas), adam_eps=adam_eps,
                                       adam_weight_decay=adam_weight_decay, resample_sr=resample_sr,
                                       process_audio_seconds=process_audio_seconds,
                                       nr_samples_per_audio=nr_samples_per_audio, size=size, alpha=alpha))
        self.max_steps = max_steps
        core = JEPA(feature_extractor=feature_extractor, transformer_encoder_cfg=transformer_encoder_cfg,
                    transformer_encoder_layers_cfg=transformer_encoder_layers_cfg,
                    transformer_decoder_cfg=TransformerEncoderCFG.create(num_layers=1),
                    transformer_decoder_layers_cfg=TransformerLayerCFG.create(d_model=384), lr=lr,
                    adam_betas=adam_betas, adam_eps=adam_eps, adam_weight_decay=adam_weight_decay,
                    resample_sr=resample_sr, process_audio_seconds=process_audio_seconds,
                    nr_samples_per_audio=nr_samples_per_audio, size=size, max_steps=max_steps, grad_clip=grad_clip)
        self.__dict__["_core"] = core          # engine only: NOT a registered sub-module (keys stay the reference's)
        self.n_encoder_heads = core.n_encoder_heads
        self.encoder_embedding_dim = core.encoder_embedding_dim
        # registration order = the reference's (wavjepa/denoiser.py:120-139)
        self.extract_audio = core.extract_audio
        self.feature_norms = core.feature_norms
        self.encoder = core.encoder
        self.post_extraction_mapper = core.post_extraction_mapper
        self.pos_encoding_encoder = core.pos_encoding_encoder
        self.teacher: Optional[JEPA] = None
        self.collate_fn = lambda batch: batch.flatten(start_dim=0, end_dim=1)

    # the engine core follows .to() / .cuda() of the module it serves
    def _apply(self, fn, *a, **k):
        super()._apply(fn, *a, **k)
        self._core._apply(fn, *a, **k)
        return self

    @property
    def device(self) -> torch.device:
        return self.pos_encoding_encoder.device

    @property
    def global_step(self) -> int:
        return self._core.global_step

    @global_step.setter
    def global_step(self, v: int) -> None:
        self._core.global_step = v

    # ------------------------------------------------------------------------------------------- teacher
    def _set_teacher(self, weights_ckpt) -> None:
        """wavjepa/denoiser.py:143-181: a frozen WavJEPA-base (`JEPA`) loaded from a Lightning checkpoint (path or an
        already loaded dict with 'state_dict'; torch.compile's `_orig_mod` infixes are stripped)."""
        weights = weights_ckpt if isinstance(weights_ckpt, dict) else torch.load(weights_ckpt, weights_only=False,
                                                                                 map_location="cpu")
        model = JEPA(feature_extractor=ConvFeatureExtractor(conv_layers_spec=BASE_SPEC, in_channels=1),
                     transformer_encoder_cfg=TransformerEncoderCFG.create(),
                     transformer_encoder_layers_cfg=TransformerLayerCFG.create(),
                     transformer_decoder_cfg=TransformerEncoderCFG.create(),
                     transformer_decoder_layers_cfg=TransformerLayerCFG.create(d_model=384), resample_sr=self.sr,
                     size="base", process_audio_seconds=self.process_audio_seconds)
        model.load_state_dict(fix_state_dict_keys(weights["state_dict"]), strict=False)
        for p in model.parameters():
            p.requires_grad = False
        model.eval()
        self.teacher = model.to(self.device)

    # ------------------------------------------------------------------------------------------- optimisation
    def lr_at(self, step: int) -> float:
        """transformers.get_cosine_schedule_with_warmup(opt, 5000, max_steps) (wavjepa/denoiser.py:208-209)."""
        warm = 5000
        if step < warm:
            return self.hparams.lr * step / max(1, warm)
        prog = (step - warm) / max(1, self.max_steps - warm)
        return self.hparams.lr * max(0.0, 0.5 * (1.0 + math.cos(math.pi * 2.0 * 0.5 * prog)))

    def configure_optimizers(self):
        trainables = [p for p in self.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(trainables, lr=self.hparams.lr, betas=self.hparams.adam_betas,
                                eps=self.hparams.adam_eps, weight_decay=self.hparams.adam_weight_decay)
        sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: self.lr_at(s) / self.hparams.lr)
        return {"optimizer": opt, "lr_scheduler": {"scheduler": sched, "interval": "step"}}

    # ------------------------------------------------------------------------------------------- batch preparation
    @torch.no_grad()
    def on_after_batch_transfer(self, batch, dataloader_idx: int = 0, starts: Optional[torch.Tensor] = None,
                                perm: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """wavjepa/denoiser.py:215-290: scene generation at 32 kHz, resampling of the generated and the clean scene,
        the SAME random crops of both (nr_samples_per_audio per clip), per-crop normalisation, bf16, one shuffle.
        `starts` [B, nr] and `perm` [B * nr] replace the random draws (tests)."""
        audio, source_rir, noise, noise_length, noise_start_idx, noise_rirs, snr = batch
        dev = self.device
        to = lambda t: t.to(dev) if isinstance(t, torch.Tensor) else t
        audio = to(audio)
        scene = generate_scene(source_rir=to(source_rir), source=audio, noise=to(noise),
                               real_noise_length=to(noise_length), noise_start_idx=to(noise_start_idx),
                               noise_rirs=to(noise_rirs), snr=to(snr))
        if audio.ndim != 3:
            audio = audio.unsqueeze(1)
        if scene.ndim != 3:
            scene = scene.unsqueeze(1)
        clean = audio
        if self.sr != self.ORIGINAL_SR:
            scene = resample(scene, self.sr, self.ORIGINAL_SR)
            clean = resample(clean, self.sr, self.ORIGINAL_SR)
        if scene.shape[1] != 1:
            raise WavJepaLibError(f"Generated scene has more channels than in channels, {tuple(scene.shape)}, 1")
        B, C, L_full = scene.shape
        nr, tl = self.nr_samples_per_audio, self.target_length
        if starts is None:
            starts = torch.randint(0, L_full - tl + 1, (B, nr), device=dev)
        st = starts.to(dev).reshape(-1).to(torch.int32).contiguous()
        outs = []
        for x in (scene, clean):
            o16 = torch.empty(B * nr, C, tl, device=dev, dtype=torch.bfloat16)
            ops.crop_norm(x.float().contiguous(), st, nr, tl, o16, None)
            outs.append(o16)
        if perm is None:
            perm = torch.randperm(B * nr)
        idx = perm.to(dev)
        return outs[0][idx], outs[1][idx]

    # ------------------------------------------------------------------------------------------- forward / backward
    def _run(self, generated_scene: torch.Tensor, clean_scene: torch.Tensor, backward: bool):
        if self.teacher is None:
            raise WavJepaLibError("Denoiser needs its frozen teacher: call _set_teacher(checkpoint) first "
                                  "(the reference has no attribute `teacher` before that either)")
        core = self._core
        core._ensure_ready()
        core._sync_weights()
        dev = self.device
        bf = torch.bfloat16
        gen16 = generated_scene.to(dev, bf)
        clean16 = clean_scene.to(dev, bf)
        N = gen16.shape[0]
        T, D = self.total_patches, self.encoder_embedding_dim
        x16 = torch.cat([clean16, gen16], dim=0).contiguous()          # halves: [clean | generated]
        # the student (wavjepa/denoiser.py:338-346) on 2N full sequences; the backward computes every gradient of the
        # feature path, whatever requires_grad says
        plan = core._feature_plan(core._train_names) if backward else None
        feats, saved = core._features_forward(x16, None, plan)
        with torch.no_grad():
            targets = self.teacher.get_audio_representation(clean16, padding_mask=None).reshape(N * T, D)
        M = N * T * D
        sums = torch.zeros(2, device=dev, dtype=torch.float64)
        dfe = torch.empty(2 * N * T, D, device=dev) if backward else None
        ops.mse_pair(feats, targets.contiguous(), float(self.alpha), sums, dfe)
        lc = (sums[0] / M).float()
        ld = (sums[1] / M).float()
        out = ForwardReturn(loss=self.alpha * lc + (1 - self.alpha) * ld, loss_clean=lc, loss_denoise_dereverb=ld)
        if not backward:
            return out, None
        # ---- backward: final norm -> 12 layers -> mapper / feature norm / conv stack
        gflat = core._flat_g
        gflat.zero_()
        ddp = core._ddp
        if ddp is not None:
            ddp.begin(gflat)
        on_ready = ddp.ready if ddp is not None else None
        core._features_backward(saved, dfe, gflat, on_ready)
        if on_ready is not None:
            on_ready(0)
        world = 1
        if ddp is not None:
            ddp.finish()
            world = ddp.world_size
        return out, world

    @torch.no_grad()
    def forward(self, generated_scene: torch.Tensor, clean_scene: torch.Tensor) -> ForwardReturn:
        """reference Denoiser.forward (wavjepa/denoiser.py:308-364): dict with loss, loss_clean,
        loss_denoise_dereverb (device scalars)."""
        return self._run(generated_scene, clean_scene, backward=False)[0]

    @torch.no_grad()
    def forward_backward(self, generated_scene: torch.Tensor, clean_scene: torch.Tensor):
        """Losses + every parameter gradient (name -> fp32 view into the flat gradient buffer, world-summed)."""
        out, _ = self._run(generated_scene, clean_scene, backward=True)
        core = self._core
        grads = {n: core._view(core._flat_g, n) for n, p in self.named_parameters()
                 if p.requires_grad and not n.startswith("teacher.")}
        return out, grads

    def attach_data_parallel(self, reducer, sync: bool = True) -> None:
        self._core.attach_data_parallel(reducer, sync=sync)

    def optimizer_state_dict(self) -> dict:
        """Adam moments + global_step of the fused optimizer path (see JEPA.optimizer_state_dict)."""
        return self._core.optimizer_state_dict()

    def load_optimizer_state_dict(self, sd: dict) -> None:
        self._core.load_optimizer_state_dict(sd)

    def reserve_workspace(self, n_bytes: int) -> int:
        return self._core.reserve_workspace(n_bytes)

    @torch.no_grad()
    def train_step(self, generated_scene: torch.Tensor, clean_scene: torch.Tensor) -> ForwardReturn:
        """One optimisation step (training_step + backward + AdamW with the 5000-step warm-up cosine schedule)."""
        out, world = self._run(generated_scene, clean_scene, backward=True)
        core = self._core
        core._optimizer_tail(core._flat_g, world, self.lr_at(core.global_step))
        return out

    def training_step(self, batch, batch_idx: int = 0) -> ForwardReturn:
        generated_scene, clean_scene = batch
        return self.train_step(generated_scene, clean_scene)
