"""HEAR-2021 / HF-style inference entry points on the sm_100a kernels.

Mirrors, with the same names / arguments / return shapes:
  hear_configs/WavJEPA.py:11-43       load_model, get_scene_embeddings, get_timestamp_embeddings
  hear_configs/WavJEPA_w2v2.py:11-43  (7-layer extractor, process_seconds=4.02) -> load_model_w2v2
  hear_api/runtime.py:39-155          RuntimeJEPA (checkpoint key fix-up, geometry, padding mask, timestamps)
  hear_api/feature_helper.py:5-88     loudness normalisation to -14 dBFS + channel fix-up
  hear_configs/WavJEPA_huggingface.py:19-39 / README.md:72-108   model(input_values) -> (embeddings, timestamps)

B200-first differences (results identical at every returned frame):
  * the reference loops over clips in Python (RMS gain, host syncs) and over 2.01 s chunks sequentially; here the
    per-clip gain is one kernel, the chunking + per-chunk normalisation (mean / unbiased std INCLUDING the zero
    padding, runtime.py:12-16,133-137) is one kernel, and all B * n_chunks chunks go through the encoder as one
    packed batch whose padded tokens are dropped (they are key-masked in the reference and cut off afterwards);
  * two numerics, chosen with `precision=` on the loaders (hear-eval-kit passes model options through
    load_model(path, **opts)) or `JEPA.inference_precision`:
      "bf16" (default)  bf16 operands / fp32 accumulate and a packed-fp16 GELU (the reference runs this path in fp32):
                        features agree with the fp32 reference to <= 1e-2 relative L2 (tests/test_gpu_model.py);
      "tf32"            the reference's fp32 feature extraction with every GEMM operand rounded to nearest tf32, fp32
                        accumulation, residual stream and chunk audio, exact erf GELU: <= 2e-3 relative L2
                        (tests/test_gpu_tf32.py), at a lower throughput (DESIGN.md 2.1);
  * `layer=k` on the loaders embeds encoder hidden state k (JEPA.get_hidden_states) instead of the final features, so a
    layer sweep is one more runner option; only the first k encoder layers run (DESIGN.md 2.4);
  * whole clips are differentiable in training mode (DESIGN.md 2.5): the loaders return the runtime in eval mode, and
    after `.train()` a call in grad mode with precision "bf16" builds a graph when a feature-path parameter or the audio
    requires grad -- loudness gain, down-mix / channel fix-up, chunking and per-chunk normalisation, encoder, cut-off,
    channel and scene means all backpropagate, to the parameters and to the audio.  The embeddings are bit-identical to
    the eval-mode call; every other case runs under no_grad.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import nn

from . import ops
from ._lib import WavJepaLibError
from .extractors import ConvFeatureExtractor
from .jepa import _FEATURE_PATH, JEPA
from .types import TransformerEncoderCFG, TransformerLayerCFG

SR = 16000
BASE_SPEC = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)]
W2V2_SPEC = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)] * 2


def fix_state_dict_keys(sd):
    """torch.compile leaves `_orig_mod` in the checkpoint keys of the compiled sub-modules (hear_api/runtime.py:63-75,
    ARCH/evaluate_wavjepa_model.py:79-91)."""
    return {k.replace("._orig_mod", ""): v for k, v in sd.items()}


def hear_geometry(n_samples: int, unit: int, sr: int, steps: int) -> Tuple[int, int, int, int]:
    """(pad_frames, n_chunks, cut_off, total_steps) of hear_api/runtime.py:107-124 + calculate_padding_mask (:19-35).
    Quirks preserved: a full extra chunk when n_samples is an exact multiple of the unit; process_seconds is the
    INTEGER 32159 // 16000 = 2."""
    pad = unit - (n_samples % unit)
    total = n_samples + pad
    proc = unit // sr
    n_units = int((total / sr) / proc)
    total_steps = steps * n_units
    out_sr = int(steps / proc)
    pad_steps = int((pad / sr) * out_sr)
    return pad, total // unit, total_steps - pad_steps, total_steps


def get_timestamps(sample_rate: int, B: int, input_audio_len: int, n_frames: int) -> torch.Tensor:
    """hear_api/runtime.py:148-155 (python-float arithmetic, then fp32)."""
    step = (input_audio_len / sample_rate) / n_frames * 1000
    return torch.tensor([step * i for i in range(n_frames)]).unsqueeze(0).repeat(B, 1)


class _ClipGain(torch.autograd.Function):
    """The -14 dBFS loudness gain of `to_feature` (ops.clip_gain over the whole [B, C, L] clip) under autograd.  The
    gain comes out once per chunk, [B, n_chunks] (a broadcast view of [B]), so that `_ChunkNorm` hands back each chunk's
    share of the gain gradient and the backward (ops.clip_gain_bwd) sums them in a fixed order."""

    @staticmethod
    def forward(ctx, a, n_chunks):
        gain = ops.clip_gain(a, -14.0)
        ctx.save_for_backward(a, gain)
        return gain[:, None].expand(-1, n_chunks)

    @staticmethod
    def backward(ctx, dgain):
        a, gain = ctx.saved_tensors
        return ops.clip_gain_bwd(a, gain, dgain.contiguous()), None


class _ChunkNorm(torch.autograd.Function):
    """The chunking + per-chunk normalisation of `embed_chunks` (ops.crop_norm at starts i * unit) under autograd: a
    [B, C, L] fp32, gain [B, n_chunks] from `_ClipGain` -> the fp32 chunks [B * n_chunks, C, unit].  The backward
    (ops.crop_norm_bwd) returns (da, dgain), dgain per chunk."""

    @staticmethod
    def forward(ctx, a, gain, unit):
        B, C, _ = a.shape
        n_chunks = gain.shape[1]
        g = gain[:, 0]   # the clip's gain: [B], contiguous (gain is a broadcast view)
        starts = (torch.arange(n_chunks, device=a.device, dtype=torch.int32) * unit).repeat(B)
        out = torch.empty(B * n_chunks, C, unit, device=a.device, dtype=torch.float32)
        ops.crop_norm(a, starts, n_chunks, unit, None, out, gain=g)
        ctx.save_for_backward(a, g)
        ctx.unit = unit
        return out

    @staticmethod
    def backward(ctx, dy):
        a, g = ctx.saved_tensors
        da, dgain = ops.crop_norm_bwd(a, g, dy.contiguous(), ctx.unit)
        return da, dgain, None


def embed_chunks(model: JEPA, a: torch.Tensor, gain: Optional[torch.Tensor], unit: int, steps: int, sr: int,
                 channel_tokens: int = 1, layer: Optional[int] = None, graph: bool = False):
    """The chunk loop of hear_api/runtime.py:107-142 (and ARCH/configs/wavjepa_wrapper.py:67-110) as ONE batched pass:
    a [B, C, L] fp32 on the device, gain [B] or None.  Chunk i of clip b = gain * a[b, :, i*unit:(i+1)*unit] (zeros past
    L), normalised per chunk (mean / unbiased std including the zero padding, runtime.py:12-16); the frames that fall
    into the padding are key-masked and cut off.  layer: embed hidden state `layer` of `JEPA.get_hidden_states`
    instead of the final features (None).  Returns (emb [B, cut_off, D] fp32, cut_off).
    graph: build the autograd graph (DESIGN.md 2.5; "bf16" only): gain is then `_ClipGain`'s [B, n_chunks], the chunks
    are `_ChunkNorm`'s fp32 output, which the model rounds to the bf16 the kernel would write; otherwise the pass runs
    under no_grad."""
    B, C, L = a.shape
    pad, n_chunks, cut_off, total_steps = hear_geometry(L, unit, sr, steps)
    # The padding mask depends on the geometry only (the same for every clip), so it is built on the HOST and handed over as
    # a pattern that repeats every n_chunks sequences: the packed-token index then needs no device read-back, and calls
    # can be issued back to back without a host synchronisation.
    mask = torch.zeros(max(total_steps, n_chunks * steps), dtype=torch.bool)
    mask[cut_off:total_steps] = True
    mask = mask[:n_chunks * steps].reshape(n_chunks, steps)
    with torch.set_grad_enabled(graph):
        dev = a.device
        if graph:
            x = _ChunkNorm.apply(a, gain, unit)
        else:
            starts = (torch.arange(n_chunks, device=dev, dtype=torch.int32) * unit).repeat(B)
            if model.inference_precision == "tf32":   # conv block 0 reads the fp32 chunks
                x = torch.empty(B * n_chunks, C, unit, device=dev, dtype=torch.float32)
                ops.crop_norm(a, starts, n_chunks, unit, None, x, gain=gain)
            else:
                x = torch.empty(B * n_chunks, C, unit, device=dev, dtype=torch.bfloat16)
                ops.crop_norm(a, starts, n_chunks, unit, x, None, gain=gain)

        def features(host_mask):
            if layer is None:
                return model.get_audio_representation(x, None, host_mask=host_mask)
            return model.get_hidden_states(x, None, host_mask=host_mask, layers=[layer])[0]
        if channel_tokens > 1:
            # WavJEPA-Nat (hear_api/runtime_natjepa.py:142-147): the model emits channel-major tokens [c0 t0.., c1 t0..];
            # the time mask is repeated "B E -> B (C E)" and the per-channel embeddings are averaged
            emb = features(mask.repeat(1, channel_tokens).numpy())   # [B*n_chunks, C*steps, D]
            emb = emb.view(B * n_chunks, channel_tokens, steps, -1).mean(dim=1)
        else:
            emb = features(mask.numpy())   # [B*n_chunks, steps, D] fp32
        return emb.reshape(B, n_chunks * steps, -1)[:, :cut_off], cut_off


class RuntimeJEPA(nn.Module):
    """reference hear_api/runtime.py:39-155.

    Built in eval mode: `get_timestamp_embeddings` / `get_scene_embeddings` / `forward` run under no_grad and their
    outputs carry no graph, whatever requires grad.  After `.train()` (the flag of this module: the inner `model` is
    always run in eval mode), a call in grad mode with precision "bf16" is differentiable when a feature-path parameter
    of `model` (extract_audio, feature_norms, post_extraction_mapper, encoder) or the audio requires grad: `backward()`
    fills `.grad` of the trainable path parameters and, when the audio requires grad, `audio.grad` (fp32, on the
    audio's device) through the loudness gain, the channel fix-up, the chunking and the per-chunk normalisation.  The
    embeddings are bit-identical to the eval-mode call.  Frozen parts, layer=, one backward per graph: as in
    `JEPA.get_audio_representation` / `JEPA.get_hidden_states`; precision "tf32" stays forward-only (DESIGN.md 2.5)."""

    def __init__(self, in_channels: int, weights, is_spectrogram: bool, process_seconds: float, extractor,
                 model_size: str, sr: int, device: Optional[str] = None, precision: str = "bf16",
                 layer: Optional[int] = None, **kwargs) -> None:
        super().__init__()
        if is_spectrogram:
            raise WavJepaLibError("spectrogram front-ends are not part of WavJEPA")
        if in_channels != 1 and not isinstance(self, RuntimeNatJEPA):
            raise WavJepaLibError("RuntimeJEPA is the mono runtime (in_channels=1); use RuntimeNatJEPA for WavJEPA-Nat")
        self.sample_rate = sr
        self.in_channels = in_channels
        self.model = JEPA(feature_extractor=extractor, transformer_encoder_cfg=TransformerEncoderCFG.create(),
                          transformer_encoder_layers_cfg=TransformerLayerCFG.create(),
                          transformer_decoder_cfg=TransformerEncoderCFG.create(),
                          transformer_decoder_layers_cfg=TransformerLayerCFG.create(d_model=384), resample_sr=sr,
                          size=model_size, process_audio_seconds=process_seconds)
        self.model.inference_precision = precision   # "bf16" or "tf32" (ValueError otherwise), see the module docstring
        if layer is not None:
            self.model._hidden_layers([layer])        # ValueError unless an int in [0, N]
        self.layer = layer
        if weights is None:
            raise TypeError("load_model needs a checkpoint: weights['state_dict'] (the reference fails here too, "
                            "hear_api/runtime.py:64)")
        self.model.load_state_dict(fix_state_dict_keys(weights["state_dict"]), strict=False)
        self.embedding_size = self.model.encoder_embedding_dim
        self.scene_embedding_size = self.embedding_size
        self.timestamp_embedding_size = self.embedding_size
        self.unit_frames = int(process_seconds * self.sample_rate)
        self.output_steps = self.model.extract_audio.total_patches(self.unit_frames)
        self.model.to(device or "cuda")   # no CPU path: a machine without a B200 fails on the first call
        self.eval()

    def _graph(self, audio) -> bool:
        """Whether a call builds an autograd graph: grad mode, training mode, precision "bf16", and the audio or a
        feature-path parameter requires grad."""
        if not (torch.is_grad_enabled() and self.training and self.model.inference_precision == "bf16"):
            return False
        return (torch.is_tensor(audio) and audio.requires_grad) or \
            any(p.requires_grad for n, p in self.model.named_parameters() if n.startswith(_FEATURE_PATH))

    def _gain(self, a: torch.Tensor, graph: bool) -> torch.Tensor:
        """The loudness gain of the [B, C, L] clips before the channel fix-up: [B], or `_ClipGain`'s [B, n_chunks]."""
        if not graph:
            return ops.clip_gain(a, -14.0)
        return _ClipGain.apply(a, hear_geometry(a.shape[2], self.unit_frames, self.sample_rate, self.output_steps)[1])

    # ---- hear_api/feature_helper.py:35-88 for tensors that are already batched [B, L] / [B, C, L]
    def to_feature(self, audio: torch.Tensor, graph: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
        """-> (audio [B, 1, L] fp32 on the device, gain [B]); the gain is applied inside the chunk kernel.  graph: the
        differentiable form of a graph-building call (gain [B, n_chunks], see `embed_chunks`)."""
        dev = self.model.device
        a = torch.as_tensor(audio).to(dev, torch.float32)
        if a.dim() == 2:
            a = a.unsqueeze(1)
        if a.dim() != 3:
            raise ValueError("audio input tensor must be (n_sounds, num_samples) or (n_sounds, n_channels, num_samples)")
        if a.shape[1] > 100 and a.shape[2] <= 100:      # [B, T, C] -> [B, C, T]   (feature_helper.py:49-50)
            a = a.transpose(1, 2)
        a = a.contiguous()
        gain = self._gain(a, graph)                      # RMS over the whole (C, L) clip BEFORE the channel fix-up (:53)
        return self._fix_channels(a), gain

    def _fix_channels(self, a: torch.Tensor) -> torch.Tensor:
        """The channel fix-up of FeatureExtractor(in_channels=1): [B, C, L] -> the mono [B, 1, L]."""
        if a.shape[1] == 2:
            return a.mean(dim=1, keepdim=True).contiguous()   # :66-67
        if a.shape[1] == 4:
            return a[:, :1].contiguous()                      # :73-74
        if a.shape[1] != 1:
            raise WavJepaLibError("Unknown channel count")
        return a

    def get_timestamp_embeddings(self, audio: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        graph = self._graph(audio)
        with torch.set_grad_enabled(graph):
            a, gain = self.to_feature(audio, graph)
        B, C, L = a.shape
        emb, _ = embed_chunks(self.model, a, gain, self.unit_frames, self.output_steps, self.sample_rate,
                              channel_tokens=C, layer=self.layer, graph=graph)
        ts = get_timestamps(self.sample_rate, B, L, emb.shape[1])
        return emb, ts

    def get_scene_embeddings(self, audio: torch.Tensor) -> torch.Tensor:
        emb, _ = self.get_timestamp_embeddings(audio)
        return emb.mean(dim=1)

    def forward(self, input_values: torch.Tensor):
        """HF remote-code call shape (README.md:72-108): model(input_values) -> (embeddings, timestamps)."""
        return self.get_timestamp_embeddings(input_values)


class RuntimeNatJEPA(RuntimeJEPA):
    """reference hear_api/runtime_natjepa.py:39-155: the binaural WavJEPA-Nat runtime.  Same geometry as the mono runtime
    with (1) the channel fix-up of FeatureExtractor(in_channels=2) (feature_helper.py:55-81: mono is duplicated, stereo
    passes, the first of 4 channels is duplicated), (2) output_steps = tokens per CHANNEL (:83-86), (3) per-chunk
    normalisation over both channels jointly (:12-16), (4) the time mask repeated over the channel-major token layout and
    the two channels' embeddings averaged (:142-147)."""

    def __init__(self, in_channels: int, weights, is_spectrogram: bool, process_seconds: float, extractor,
                 model_size: str, sr: int, device: Optional[str] = None, precision: str = "bf16", **kwargs) -> None:
        if in_channels != 2:
            raise WavJepaLibError("RuntimeNatJEPA is built for the binaural model (in_channels=2)")
        super().__init__(in_channels, weights, is_spectrogram, process_seconds, extractor, model_size, sr, device,
                         precision, **kwargs)
        self.output_steps = self.model.extract_audio.total_patches(self.unit_frames) // in_channels

    def _fix_channels(self, a: torch.Tensor) -> torch.Tensor:
        """The channel fix-up of FeatureExtractor(in_channels=2): [B, C, L] -> [B, 2, L]."""
        if a.shape[1] == 1:
            return a.expand(-1, 2, -1).contiguous()           # feature_helper.py:57-58
        if a.shape[1] == 4:
            return a[:, :1].expand(-1, 2, -1).contiguous()    # :75-77
        if a.shape[1] != 2:
            raise WavJepaLibError("Unknown channel count")
        return a


def _load_weights(args):
    if len(args) == 0:
        return None
    w = args[0]
    if isinstance(w, dict):
        return w
    import sys
    import wavjepa_b200
    sys.modules.setdefault("sjepa", wavjepa_b200)    # old pickles name the module `sjepa` (hear_configs/WavJEPA.py:5-8)
    return torch.load(w, weights_only=False, map_location="cpu")


def load_model(*args, precision: str = "bf16", layer: Optional[int] = None, **kwargs) -> RuntimeJEPA:
    """hear_configs/WavJEPA.py:11-35.  args[0]: checkpoint path (or an already loaded dict with 'state_dict').
    precision: "bf16" (default) or "tf32" (reference-precision features, see the module docstring).
    layer: None (default) embeds the final features; an int k in [0, N] embeds encoder hidden state k
    (`JEPA.get_hidden_states`: 0 the encoder input, k the output of layer k - 1), for layer-wise probing."""
    extractor = ConvFeatureExtractor(conv_layers_spec=BASE_SPEC, in_channels=1)
    return RuntimeJEPA(in_channels=1, process_seconds=2.01, weights=_load_weights(args), sr=SR, model_size="base",
                       is_spectrogram=False, extractor=extractor, precision=precision, layer=layer, **kwargs)


def load_model_w2v2(*args, precision: str = "bf16", layer: Optional[int] = None, **kwargs) -> RuntimeJEPA:
    """hear_configs/WavJEPA_w2v2.py:11-35: 7-layer wav2vec2 extractor (stride 320), 4.02 s windows -> 200 tokens.
    precision, layer: as in load_model."""
    extractor = ConvFeatureExtractor(conv_layers_spec=W2V2_SPEC, in_channels=1)
    return RuntimeJEPA(in_channels=1, process_seconds=4.02, weights=_load_weights(args), sr=SR, model_size="base",
                       is_spectrogram=False, extractor=extractor, precision=precision, layer=layer, **kwargs)


def load_model_nat(*args, share_weights_over_channels: bool = False, precision: str = "bf16",
                   layer: Optional[int] = None, **kwargs) -> RuntimeNatJEPA:
    """WavJEPA-Nat counterpart of load_model (README.md:93-108 `labhamlet/wavjepa-nat-base`): per-channel extractors
    (wavjepa/extractors/audio_channel_feature_extractor.py), 2 x 200 tokens per 2.01 s window.  precision, layer: as
    in load_model (the hidden state is averaged over the two channels like the final features)."""
    from .extractors import ConvChannelFeatureExtractor
    extractor = ConvChannelFeatureExtractor(conv_layers_spec=BASE_SPEC, in_channels=2,
                                            share_weights_over_channels=share_weights_over_channels)
    return RuntimeNatJEPA(in_channels=2, process_seconds=2.01, weights=_load_weights(args), sr=SR, model_size="base",
                          is_spectrogram=False, extractor=extractor, precision=precision, layer=layer, **kwargs)


def get_scene_embeddings(audio, model):
    return model.get_scene_embeddings(audio)


def get_timestamp_embeddings(audio, model):
    return model.get_timestamp_embeddings(audio)
