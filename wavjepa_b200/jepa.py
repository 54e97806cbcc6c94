"""WavJEPA model with the reference's module API (wavjepa/jepa.py:22-467), executed on the sm_100a kernels.

What is kept from the reference: the constructor signature, attribute names, `state_dict` keys/shapes (457 tensors for
WavJEPA-base), `forward(audio, ctx_masks, target_indices, ctx_and_target_masks) -> dict`, `training_step`,
`on_after_batch_transfer`, `configure_optimizers`, `get_audio_representation`, the EMA schedule, and every numerical
quirk listed in SURVEY.md Appendix C (joint (D,T) target norm, teacher skips its final norm, eps 1e-6 / 1e-5, ...).

What is different by design (B200-first):
  * no nn.TransformerEncoder / cuDNN / SDPA: parameters live in plain containers, compute is csrc/*.cu through the C ABI;
  * the student runs on the VISIBLE context tokens only, the predictor on context+target tokens only, packed with
    cu_seqlens -- identical results at every position the loss reads (key-padding masks only hide keys);
  * all parameters are views into flat fp32 / bf16 buffers so that EMA, AdamW, the bf16 weight refresh and the
    gradient all-reduce buckets are single launches over contiguous memory;
  * `train_step` is the fused fast path (crop+normalise -> forward -> backward with overlapped bucketed all-reduce ->
    clip + AdamW -> EMA); `forward()` + `loss.backward()` still work for a stock optimizer / Lightning loop.
There is no PyTorch/CPU fallback: without libwavjepa_b200.so and an sm_100 device every compute call raises.
"""
from __future__ import annotations

import copy
import math
from typing import Any, Callable, List, Optional

import numpy as np
import torch
from torch import nn

from . import ops
from ._lib import WavJepaLibError, require_device
from ._lightning import Base as _ModuleBase
from ._lightning import attached_trainer
from .engine import LayerViews, TransformerStack
from .extractors import (ConvChannelFeatureExtractor, ConvFeatureExtractor, conv_stack_backward, conv_stack_forward,
                         conv_stack_forward_tf32, kmajor_weight)
from .pos_embed import get_1d_sincos_pos_embed_from_grid
from .types import ForwardReturn, TransformerEncoderCFG, TransformerLayerCFG

_PAD = 64  # every parameter starts on a 64-element boundary of the flat buffers (TMA needs 16-byte alignment)


# =================================================================================================== containers
class _LinearParams(nn.Module):
    def __init__(self, n_in: int, n_out: int, bias: bool = True):
        super().__init__()
        self.in_features, self.out_features = n_in, n_out
        self.weight = nn.Parameter(torch.empty(n_out, n_in))
        self.bias = nn.Parameter(torch.zeros(n_out)) if bias else None
        nn.init.trunc_normal_(self.weight, std=0.02, a=-2.0, b=2.0)  # JEPA._init_weights, wavjepa/jepa.py:150-154


class _LayerNormParams(nn.Module):
    def __init__(self, dim: int, eps: float = 1e-5):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(dim))
        self.bias = nn.Parameter(torch.zeros(dim))


class _SelfAttnParams(nn.Module):
    """Parameter layout of nn.MultiheadAttention: packed in_proj ([Wq; Wk; Wv]) keeps torch's xavier-uniform init
    (the reference's _init_weights only touches nn.Linear / nn.LayerNorm, SURVEY.md 3.3)."""

    def __init__(self, d: int):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * d, d))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * d))
        self.out_proj = _LinearParams(d, d)
        nn.init.xavier_uniform_(self.in_proj_weight)


class _EncoderLayerParams(nn.Module):
    def __init__(self, d: int, ff: int, eps: float):
        super().__init__()
        self.self_attn = _SelfAttnParams(d)
        self.linear1 = _LinearParams(d, ff)
        self.linear2 = _LinearParams(ff, d)
        self.norm1 = _LayerNormParams(d, eps)
        self.norm2 = _LayerNormParams(d, eps)


class _EncoderParams(nn.Module):
    """Parameter container with nn.TransformerEncoder's names: layers.{i}.*, norm.* (wavjepa/jepa.py:126-130)."""

    def __init__(self, d: int, ff: int, n_layers: int, eps: float):
        super().__init__()
        self.layers = nn.ModuleList([_EncoderLayerParams(d, ff, eps) for _ in range(n_layers)])
        self.norm = _LayerNormParams(d, 1e-5)


class _AttrDict(dict):
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


def _check_layer_cfg(cfg) -> None:
    if cfg.get("norm_first", False) or not cfg.get("bias", True) or cfg.get("dropout", 0.0) != 0.0:
        raise WavJepaLibError("only post-norm, bias=True, dropout=0 transformer layers are built")
    act = cfg.get("activation", "gelu")
    if not (act == "gelu" or type(act).__name__ == "GELU"):
        raise WavJepaLibError("only GELU(erf) activation is built")


def collate_fn(t: torch.Tensor) -> torch.Tensor:
    return t.flatten(0, 1)


class _Ctx:
    """Everything the backward needs from one forward."""
    pass


class _LossBridge(torch.autograd.Function):
    """Makes `out['loss'].backward()` work with a stock optimizer: runs the hand-written backward and returns the
    parameter gradients to autograd."""

    @staticmethod
    def forward(ctx, model, fctx, *params):
        ctx.model = model
        ctx.fctx = fctx
        return fctx.loss.detach().clone().reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        model, fctx = ctx.model, ctx.fctx
        gflat = torch.zeros_like(model._flat_p)
        model._backward_impl(fctx, gflat, loss_scale=grad_out)
        grads = [model._view(gflat, name) for name in model._train_names]
        return (None, None, *grads)


# parameters that `get_audio_representation` reads: the leading span of the flat layout (see JEPA._layout_names)
_FEATURE_PATH = ("extract_audio.", "feature_norms.", "post_extraction_mapper.", "encoder.")


class _FeaturePlan:
    """Which parts of the feature path a backward through `_features_forward` trains: a differentiable
    `get_audio_representation` call, or the denoiser's student.  conv / norm / mapper / final_norm / layer_w[i]: some
    tensor of that part trains (its weight gradients are computed); dx: the waveform gradient is wanted (the data
    gradient runs down to it through every part, trainable or not)."""
    __slots__ = ("names", "conv", "norm", "mapper", "final_norm", "layer_w", "local", "first_layer", "dx")


class _FeatureBridge(torch.autograd.Function):
    """Makes the features of `get_audio_representation` (collect None) or the hidden states `collect` of
    `get_hidden_states` (a tuple) differentiable: the forward runs the saving kernels, the backward runs the hand-written
    chain (final LayerNorm or the hidden states' gradients -> encoder layers -> mapper / feature norm / conv stack, down
    to conv block 0's data gradient when the waveform requires grad) into a gradient buffer owned by this call and hands
    autograd the gradients of the inputs it asks for.  `audio` is the waveform on the model's device in the caller's
    dtype; its gradient is returned in that dtype."""

    @staticmethod
    def forward(ctx, model, audio, index, plan, collect, *params):
        ctx.model = model
        ctx.audio_dtype = audio.dtype
        out, ctx.fctx = model._features_forward(audio.to(torch.bfloat16).contiguous(), index, plan, collect)
        if collect is None:
            return out
        ctx.set_materialize_grads(False)   # hidden states the loss does not read arrive as None and cost nothing
        return tuple(out)

    @staticmethod
    def backward(ctx, *grad_out):
        c = ctx.fctx
        if c is None:
            raise RuntimeError("get_audio_representation / get_hidden_states: this graph was already backpropagated "
                               "and its saved activations are freed; run the forward again (retain_graph is not "
                               "supported)")
        ctx.fctx = None
        model = ctx.model
        gflat, dx = model._features_backward(c, grad_out[0] if c.collect is None else list(grad_out))
        needs = ctx.needs_input_grad[5:]
        grads = [model._view(gflat, n) if needs[i] else None for i, n in enumerate(c.plan.names)]
        daudio = dx.to(ctx.audio_dtype) if dx is not None and ctx.needs_input_grad[1] else None
        return (None, daudio, None, None, None, *grads)


# =================================================================================================== model
class JEPA(_ModuleBase):
    """A `pytorch_lightning.LightningModule` when Lightning is installed (drop-in for `pl.Trainer.fit`, train.py:244),
    a plain nn.Module with the same members otherwise (wavjepa_b200/_lightning.py)."""
    teacher_encoder: nn.Module

    def __init__(self, feature_extractor, transformer_encoder_layers_cfg: TransformerLayerCFG,
                 transformer_encoder_cfg: TransformerEncoderCFG, transformer_decoder_layers_cfg: TransformerLayerCFG,
                 transformer_decoder_cfg: TransformerEncoderCFG, decoder_embedding_dim: int = 512, loss_fn: Any = None,
                 lr: float = 0.0002, adam_betas: tuple = (0.9, 0.98), adam_eps: float = 1e-06,
                 adam_weight_decay: float = 0.01, ema_decay: float = 0.999, ema_end_decay: float = 0.99999,
                 ema_anneal_end_step: int = 100000, average_top_k_layers: int = 12, resample_sr: int = 16000,
                 process_audio_seconds: float = 2.00, nr_samples_per_audio: int = 16,
                 use_gradient_checkpointing: bool = False, compile_modules: bool = False, size: str = "base",
                 max_steps: int = 375000, grad_clip: float = 5.0, **kwargs):
        super().__init__()
        self.sr = resample_sr
        self.nr_samples_per_audio = nr_samples_per_audio
        self.ema_end_step = ema_anneal_end_step
        self.target_length = int(resample_sr * process_audio_seconds)
        self.total_patches = feature_extractor.total_patches(self.target_length)
        self.use_compiled_forward = False          # torch.compile is not part of this build
        self.use_gradient_checkpointing = False    # activations fit: 180 GB HBM, packed tokens
        self.save_hyperparameters(dict(lr=lr, adam_betas=tuple(adam_betas), adam_eps=adam_eps,
                                       adam_weight_decay=adam_weight_decay, ema_decay=ema_decay,
                                       ema_end_decay=ema_end_decay, ema_anneal_end_step=ema_anneal_end_step,
                                       average_top_k_layers=average_top_k_layers, resample_sr=resample_sr,
                                       process_audio_seconds=process_audio_seconds,
                                       nr_samples_per_audio=nr_samples_per_audio, size=size,
                                       decoder_embedding_dim=decoder_embedding_dim))
        self._step = 0
        self.max_steps = max_steps
        self.grad_clip = grad_clip
        self.shuffle_crops = False   # True: shuffle the audio rows after cropping like the reference (jepa.py:314-316)
        if not isinstance(feature_extractor, (ConvFeatureExtractor, ConvChannelFeatureExtractor)):
            raise WavJepaLibError("feature_extractor must be a wavjepa_b200 ConvFeatureExtractor / ConvChannelFeatureExtractor")

        enc_cfg = dict(transformer_encoder_layers_cfg)
        enc_n = dict(transformer_encoder_cfg)
        dec_cfg = dict(transformer_decoder_layers_cfg)
        dec_n = dict(transformer_decoder_cfg)
        if size == "large":  # wavjepa/jepa.py:113-118
            enc_cfg["nhead"], enc_cfg["d_model"], enc_cfg["dim_feedforward"] = 16, 1024, 4096
            enc_n["num_layers"] = 24
        _check_layer_cfg(enc_cfg)
        _check_layer_cfg(dec_cfg)
        self.n_encoder_heads = enc_cfg["nhead"]
        self.encoder_embedding_dim = enc_cfg["d_model"]
        self.n_decoder_heads = dec_cfg["nhead"]
        self.decoder_embedding_dim = dec_cfg["d_model"]
        D, Dp = self.encoder_embedding_dim, self.decoder_embedding_dim
        if feature_extractor.embedding_dim == D:
            raise WavJepaLibError("extractor dim == encoder dim (no post_extraction_mapper) is not built")

        # registration order = the reference's, so state_dict() enumerates identically (wavjepa/jepa.py:108-143)
        self.mask_token = nn.Parameter(torch.zeros(1, 1, Dp))
        torch.nn.init.normal_(self.mask_token, std=0.02)
        self.pos_encoding_encoder = self._get_pos_embed_params(D)
        self.pos_encoding_decoder = self._get_pos_embed_params(Dp)
        self.extract_audio = feature_extractor
        self.feature_norms = _LayerNormParams(feature_extractor.embedding_dim, 1e-5)
        self.encoder = _EncoderParams(D, enc_cfg["dim_feedforward"], enc_n["num_layers"], enc_cfg["layer_norm_eps"])
        self.post_extraction_mapper = _LinearParams(feature_extractor.embedding_dim, D)
        self.decoder = _EncoderParams(Dp, dec_cfg["dim_feedforward"], dec_n["num_layers"], dec_cfg["layer_norm_eps"])
        self.decoder_to_encoder_mapper = _LinearParams(Dp, D)
        self.encoder_to_decoder_mapper = _LinearParams(D, Dp)
        self._init_teacher()

        self._enc_stack = TransformerStack(D, enc_cfg["nhead"], enc_cfg["dim_feedforward"], enc_n["num_layers"],
                                           enc_cfg["layer_norm_eps"])
        self._dec_stack = TransformerStack(Dp, dec_cfg["nhead"], dec_cfg["dim_feedforward"], dec_n["num_layers"],
                                           dec_cfg["layer_norm_eps"])
        self._flat_p = None
        self._ddp = None
        self.collate_fn = collate_fn
        self.return_dense_preds = True
        self.inference_precision = "bf16"

    @property
    def inference_precision(self) -> str:
        """Numerics of `get_audio_representation`: "bf16" (the default) runs the encoder with bf16 operands and the
        packed-fp16 tanh-form GELU, ~1e-2 relative L2 from the reference's fp32 features; "tf32" runs the reference's fp32
        feature extraction with every GEMM operand rounded to nearest tf32, fp32 accumulation and the exact erf GELU
        (DESIGN.md 2.1).  `forward`, `train_step`, the teacher and the denoiser ignore it.  "tf32" is inference-only:
        its features never carry a grad_fn, whether parameters or the waveform require grad; fine-tuning and the waveform
        gradient through `get_audio_representation` run in "bf16" (DESIGN.md 2.2, 2.3)."""
        return self.__dict__.get("_inference_precision", "bf16")

    @inference_precision.setter
    def inference_precision(self, value: str) -> None:
        if value not in ("bf16", "tf32"):
            raise ValueError(f"inference_precision must be 'bf16' or 'tf32', got {value!r}")
        self.__dict__["_inference_precision"] = value

    # ------------------------------------------------------------------------------------------- reference helpers
    def _get_pos_embed_params(self, embedding_dim: int) -> nn.Parameter:
        table = get_1d_sincos_pos_embed_from_grid(embedding_dim, np.arange(self.total_patches, dtype=np.float64))
        return nn.Parameter(torch.from_numpy(table).float().unsqueeze(0), requires_grad=False)

    def _init_teacher(self) -> None:
        self.teacher_encoder = copy.deepcopy(self.encoder)
        self.teacher_encoder.requires_grad_(False)

    def _get_ema_decay(self, step: Optional[int] = None) -> float:
        step = self.global_step if step is None else step
        if step >= self.ema_end_step:
            return self.hparams.ema_end_decay
        r = self.hparams.ema_end_decay - self.hparams.ema_decay
        pct_remaining = 1 - step / self.ema_end_step
        return self.hparams.ema_end_decay - r * pct_remaining

    def get_aug_prob(self) -> float:
        """wavjepa/jepa.py:272-273 (unused by the reference's own step; kept for API parity).  Reads the attached
        trainer's max_steps like the reference, else the module's own."""
        from ._lightning import attached_trainer
        tr = attached_trainer(self)
        max_steps = getattr(tr, "max_steps", None) if tr is not None else None
        return 1 - (self.global_step / (max_steps if max_steps else self.max_steps))

    def lr_at(self, step: int) -> float:
        """transformers.get_cosine_schedule_with_warmup(opt, 100000, max_steps) (wavjepa/jepa.py:224-225)."""
        warm = 100000
        if step < warm:
            return self.hparams.lr * step / max(1, warm)
        prog = (step - warm) / max(1, self.max_steps - warm)
        return self.hparams.lr * max(0.0, 0.5 * (1.0 + math.cos(math.pi * 2.0 * 0.5 * prog)))

    @property
    def device(self) -> torch.device:
        return self.mask_token.device

    @property
    def global_step(self) -> int:
        """The trainer's step counter when a pl.Trainer drives the module (wavjepa/jepa.py:186-191 reads
        LightningModule.global_step), otherwise the counter the fused / stock optimizer paths advance."""
        t = attached_trainer(self)
        return int(t.global_step) if t is not None and hasattr(t, "global_step") else self._step

    @global_step.setter
    def global_step(self, value: int) -> None:
        self._step = int(value)

    def configure_optimizers(self):
        """Stock-PyTorch optimizer over the same parameters (for a Lightning-style loop); `train_step` uses the
        fused AdamW kernel instead."""
        trainables = [p for p in self.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(trainables, lr=self.hparams.lr, betas=self.hparams.adam_betas,
                                eps=self.hparams.adam_eps, weight_decay=self.hparams.adam_weight_decay)
        sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: self.lr_at(s) / self.hparams.lr)

        # In the reference `global_step` is the Lightning trainer's counter; it drives the EMA anneal
        # (wavjepa/jepa.py:186-191).  Without a trainer nobody would advance it on this path: count optimizer steps.
        def _count(optimizer, args, kwargs):
            if attached_trainer(self) is None:
                self._step += 1

        opt.register_step_post_hook(_count)
        return {"optimizer": opt, "lr_scheduler": {"scheduler": sched, "interval": "step"}}

    # ------------------------------------------------------------------------------------------- flat buffers
    def _layout_names(self) -> List[str]:
        names = dict(self.named_parameters())
        order = [n for n in names if n.startswith("extract_audio.")]
        order += [n for n in names if n.startswith("feature_norms.")]
        order += [n for n in names if n.startswith("post_extraction_mapper.")]
        order += [n for n in names if n.startswith("encoder.")]
        order += [n for n in names if n.startswith("encoder_to_decoder_mapper.")]
        order += ["mask_token"]
        order += [n for n in names if n.startswith("decoder.")]
        order += [n for n in names if n.startswith("decoder_to_encoder_mapper.")]
        return order

    def _ensure_ready(self) -> None:
        """(Re)builds the flat fp32 / bf16 buffers when the parameters moved (first use, .to(), .cuda())."""
        dev = self.mask_token.device
        if dev.type != "cuda":
            raise WavJepaLibError("wavjepa_b200.JEPA needs its parameters on a CUDA device (no CPU fallback)")
        if self._flat_p is not None and self._flat_p.device == dev and \
                self.mask_token.data_ptr() == self._view(self._flat_p, "mask_token").data_ptr():
            return
        require_device()
        params = dict(self.named_parameters())
        order = self._layout_names()
        self._train_names = order
        self._offsets = {}
        off = 0
        for n in order:
            self._offsets[n] = (off, params[n].numel(), tuple(params[n].shape))
            off += (params[n].numel() + _PAD - 1) // _PAD * _PAD
        total = off
        flat = torch.zeros(total, device=dev, dtype=torch.float32)
        for n in order:
            o, cnt, shp = self._offsets[n]
            flat[o:o + cnt].copy_(params[n].detach().reshape(-1))
            params[n].data = flat[o:o + cnt].view(shp)
        # Adam moments follow the parameters: a rebuild (first use, .to(), .cuda()) keeps them when the layout is unchanged
        old_m, old_v = getattr(self, "_adam_m", None), getattr(self, "_adam_v", None)
        keep = old_m is not None and old_m.numel() == total and getattr(self, "_layout_sig", None) == tuple(order)
        self._layout_sig = tuple(order)
        self._flat_p = flat
        self._flat_g = torch.zeros(total, device=dev, dtype=torch.float32)
        self._flat_w16 = torch.empty(total, device=dev, dtype=torch.bfloat16)
        self._adam_m = old_m.to(dev) if keep else None
        self._adam_v = old_v.to(dev) if keep else None
        # encoder slice (EMA source) and the teacher's mirror of it
        enc_names = [n for n in order if n.startswith("encoder.")]
        e0 = self._offsets[enc_names[0]][0]
        last = self._offsets[enc_names[-1]]
        e1 = (last[0] + last[1] + _PAD - 1) // _PAD * _PAD
        self._enc_range = (e0, e1)
        tflat = torch.zeros(e1 - e0, device=dev, dtype=torch.float32)
        tparams = dict(self.teacher_encoder.named_parameters())
        self._t_offsets = {}
        for n in enc_names:
            o, cnt, shp = self._offsets[n]
            tn = n[len("encoder."):]
            self._t_offsets[tn] = (o - e0, cnt, shp)
            tflat[o - e0:o - e0 + cnt].copy_(tparams[tn].detach().reshape(-1))
            tparams[tn].data = tflat[o - e0:o - e0 + cnt].view(shp)
        self._flat_t = tflat
        self._flat_t16 = torch.empty(e1 - e0, device=dev, dtype=torch.bfloat16)
        # conv working weights (tap-major bf16) live outside the flat copy
        self._conv_names = [n for n in order if n.startswith("extract_audio.") and n.endswith(".0.weight")]
        self._w_sig = None
        self._gviews_cache = None
        self._pos_enc = self.pos_encoding_encoder.detach().reshape(self.total_patches, -1).contiguous()
        self._pos_dec = self.pos_encoding_decoder.detach().reshape(self.total_patches, -1).contiguous()
        self._sync_weights(force=True)

    def _view(self, flat: torch.Tensor, name: str) -> torch.Tensor:
        o, cnt, shp = self._offsets[name]
        return flat[o:o + cnt].view(shp)

    def _tview(self, flat: torch.Tensor, name: str) -> torch.Tensor:
        o, cnt, shp = self._t_offsets[name]
        return flat[o:o + cnt].view(shp)

    def _signature(self):
        return tuple(p._version for p in self.parameters())

    def _sync_weights(self, force: bool = False) -> None:
        """Refreshes the bf16 working copies when any fp32 master parameter changed (load_state_dict, optimizer)."""
        sig = self._signature()
        if not force and sig == self._w_sig:
            return
        ops.cast_bf16(self._flat_p, self._flat_w16)
        ops.cast_bf16(self._flat_t, self._flat_t16)
        self._refresh_conv_weights()
        self._build_weight_views()
        self._w_sig = sig

    def _conv_streams(self, wk: Optional[dict] = None) -> list:
        """(prefix, weights) of the CNN that serves each conv stream, in channel order: the mono extractor runs one
        stream over every input channel, the per-channel (Nat) extractor one mono stream per input channel, all through
        `extract_audio.cnns.0` when it shares weights over channels.  weights: the tap-major working copies of blocks
        1.. taken from `wk` (`_conv_wk`, or the tf32 copy), or their parameter names when wk is None."""
        ex = self.extract_audio
        if isinstance(ex, ConvChannelFeatureExtractor):
            prefixes = [f"extract_audio.cnns.{0 if ex.share_weights_over_channels else c}" for c in range(ex.in_channels)]
        else:
            prefixes = ["extract_audio.cnn"]
        names = lambda p: [f"{p}.{i}.0.weight" for i in range(1, len(ex.conv_layers_spec))]
        return [(p, names(p) if wk is None else [wk[n] for n in names(p)]) for p in prefixes]

    def _tap_major(self, flat: torch.Tensor, dtype: torch.dtype, old: Optional[dict] = None) -> dict:
        """Tap-major working copies (kmajor_weight) of the conv weights of blocks 1.. in `flat`, by name, written into
        the buffers of `old` where it has them."""
        out = {}
        for _, names in self._conv_streams():
            for name in names:
                if name not in out:   # a CNN shared over channels serves several streams
                    out[name] = kmajor_weight(self._view(flat, name), (old or {}).get(name), dtype=dtype)
        return out

    def _refresh_conv_weights(self) -> None:
        self._conv_wk = self._tap_major(self._flat_p, torch.bfloat16, getattr(self, "_conv_wk", None))

    @staticmethod
    def _stack_views(prefix: str, n_layers: int, mat: Callable, vec: Callable) -> List[LayerViews]:
        """Per-layer views of a stack: `mat(name)` views a weight matrix, `vec(name)` a bias or LayerNorm vector (for
        gradients both are the gradient view)."""
        out = []
        for i in range(n_layers):
            b = f"{prefix}layers.{i}."
            w = LayerViews()
            w.w_in, w.b_in = mat(b + "self_attn.in_proj_weight"), vec(b + "self_attn.in_proj_bias")
            w.w_o, w.b_o = mat(b + "self_attn.out_proj.weight"), vec(b + "self_attn.out_proj.bias")
            w.w1, w.b1 = mat(b + "linear1.weight"), vec(b + "linear1.bias")
            w.w2, w.b2 = mat(b + "linear2.weight"), vec(b + "linear2.bias")
            w.g1, w.be1 = vec(b + "norm1.weight"), vec(b + "norm1.bias")
            w.g2, w.be2 = vec(b + "norm2.weight"), vec(b + "norm2.bias")
            out.append(w)
        return out

    def _build_weight_views(self) -> None:
        p16 = lambda n: self._view(self._flat_w16, n)
        p32 = lambda n: self._view(self._flat_p, n)
        self._W_enc = self._stack_views("encoder.", self._enc_stack.n_layers, p16, p32)
        self._W_dec = self._stack_views("decoder.", self._dec_stack.n_layers, p16, p32)
        self._W_tea = self._stack_views("", self._enc_stack.n_layers, lambda n: self._tview(self._flat_t16, n),
                                        lambda n: self._tview(self._flat_t, n))

    def _grad_views(self, gflat: torch.Tensor):
        if gflat is self._flat_g and self._gviews_cache is not None:
            return self._gviews_cache
        g = lambda n: self._view(gflat, n)
        views = (self._stack_views("encoder.", self._enc_stack.n_layers, g, g),
                 self._stack_views("decoder.", self._dec_stack.n_layers, g, g), g)
        if gflat is self._flat_g:
            self._gviews_cache = views
        return views

    # ------------------------------------------------------------------------------------------- local features
    def _local_features(self, x16: torch.Tensor, save: bool, save_conv: Optional[bool] = None):
        """Waveform encoder -> LayerNorm(512) -> Linear 512->D (+bias, bf16) -> + positional table (fp32).
        reference wavjepa/jepa.py:391-396.  Returns (local32 [B*T, D], ctx pieces for the backward).
        save_conv=False (with save): a frozen extractor keeps no activations; only the feature norm saves its stats."""
        save_conv = save if save_conv is None else (save and save_conv)
        ex = self.extract_audio
        B = x16.shape[0]
        T, D = self.total_patches, self.encoder_embedding_dim
        C = ex.embedding_dim
        p32 = lambda n: self._view(self._flat_p, n)
        streams = self._conv_streams(self._conv_wk)
        conv_saved = []
        if isinstance(ex, ConvChannelFeatureExtractor):
            Tc = T // ex.in_channels
            feats = torch.empty(B, T, C, device=x16.device, dtype=torch.bfloat16)
            xs = x16.transpose(0, 1).contiguous()  # [Cin, B, L]: one mono stream per CNN
            for c, (prefix, wks) in enumerate(streams):
                f, sv = conv_stack_forward(ex.conv_layers_spec, xs[c].unsqueeze(1), p32(f"{prefix}.0.0.weight"),
                                           p32(f"{prefix}.0.2.weight"), p32(f"{prefix}.0.2.bias"), wks, save_conv)
                feats[:, c * Tc:(c + 1) * Tc].copy_(f)  # channel-major token order (audio_channel_feature_extractor.py:177-178)
                conv_saved.append(sv)
        else:
            (prefix, wks), = streams
            feats, sv = conv_stack_forward(ex.conv_layers_spec, x16, p32(f"{prefix}.0.0.weight"),
                                           p32(f"{prefix}.0.2.weight"), p32(f"{prefix}.0.2.bias"), wks, save_conv)
            conv_saved.append(sv)
        f2 = feats.view(B * T, C)
        ln16 = torch.empty(B * T, C, device=x16.device, dtype=torch.bfloat16)
        st = torch.empty(B * T, 2, device=x16.device) if save else None
        ops.layernorm_fwd(f2, p32("feature_norms.weight"), p32("feature_norms.bias"), self.feature_norms.eps, None,
                          ln16, st, None)
        local32 = torch.empty(B * T, D, device=x16.device)
        ops.gemm(ops.plain_operand(ln16), self._view(self._flat_w16, "post_extraction_mapper.weight"), B * T, 1,
                 local32, bias=p32("post_extraction_mapper.bias"), act=ops.ACT_BF16, resid=self._pos_enc,
                 resid_mod=T)
        return local32, (conv_saved, f2, ln16, st)

    # ------------------------------------------------------------------------------------------- teacher
    @torch.no_grad()
    def _forward_teacher_packed(self, local32: torch.Tensor, local16: torch.Tensor, B: int) -> torch.Tensor:
        """JEPA._forward_teacher + _make_targets (wavjepa/jepa.py:230-270): dense T tokens per instance, no mask,
        NO final norm; targets = mean over the top-K layers of the per-(layer, instance) instance norm over (T, D)."""
        T, D = self.total_patches, self.encoder_embedding_dim
        nl = self._enc_stack.n_layers
        K = self.hparams.average_top_k_layers
        first_layer = max(0, nl - K)
        dev = local32.device
        cu = torch.arange(0, (B + 1) * T, T, device=dev, dtype=torch.int32)
        targets = torch.empty(B * T, D, device=dev)
        if K > 1:
            n_used = nl - first_layer
            inst = torch.empty(n_used, B, 2, device=dev)
            outs, sums = [], []

            def hook(i, x32, rowsum):
                if i >= first_layer:   # keep the layer output (it is the next layer's residual anyway) and its row sums
                    outs.append(x32)
                    sums.append(rowsum)

            self._enc_stack.forward(self._W_tea, local32, local16, cu, B, T, False, hook, rowsum_from=first_layer)
            # one pass over the K layer outputs instead of K read-modify-write passes over the targets
            ops.target_combine(outs, sums, B, T, D, 1.0 / n_used, inst, targets)
        else:
            x32, _, _ = self._enc_stack.forward(self._W_tea, local32, local16, cu, B, T, False)
            targets = x32
        return targets

    # ------------------------------------------------------------------------------------------- forward
    def _forward_impl(self, x16: torch.Tensor, mi: "ops.MaskIndex", save: bool) -> _Ctx:
        B = x16.shape[0]
        T, D, Dp = self.total_patches, self.encoder_embedding_dim, self.decoder_embedding_dim
        dev = x16.device
        bf = torch.bfloat16
        p32 = lambda n: self._view(self._flat_p, n)
        p16 = lambda n: self._view(self._flat_w16, n)
        c = _Ctx()
        c.mi, c.B = mi, B
        local32, c.local_saved = self._local_features(x16, save)
        c.local32 = local32
        Nc, Nv, Nt = mi.Nc, mi.Nv, mi.Nt
        # ---- student on the visible context tokens (wavjepa/jepa.py:397-399)
        xc32 = torch.empty(Nc, D, device=dev)
        xc16 = torch.empty(Nc, D, device=dev, dtype=bf)
        ops.gather_rows(local32, mi.ctx_rows, Nc, xc32, xc16)
        xs32, _, c.enc_saved = self._enc_stack.forward(self._W_enc, xc32, xc16, mi.cu_c, B, mi.max_nc, save)
        cf16 = torch.empty(Nc, D, device=dev, dtype=bf)
        c.enc_norm_st = torch.empty(Nc, 2, device=dev) if save else None
        ops.layernorm_fwd(xs32, p32("encoder.norm.weight"), p32("encoder.norm.bias"), self.encoder.norm.eps, None,
                          cf16, c.enc_norm_st, None)
        c.xs32, c.cf16 = (xs32, cf16) if save else (None, None)
        # ---- encoder_to_decoder_mapper (wavjepa/jepa.py:400)
        ctx16 = torch.empty(Nc, Dp, device=dev, dtype=bf)
        ops.gemm(ops.plain_operand(cf16), p16("encoder_to_decoder_mapper.weight"), Nc, 1, ctx16,
                 bias=p32("encoder_to_decoder_mapper.bias"))
        c.contextual_features = ctx16
        # ---- predictor on context + target tokens of every target group (wavjepa/jepa.py:422-440)
        x0_32 = torch.empty(Nv, Dp, device=dev)
        x0_16 = torch.empty(Nv, Dp, device=dev, dtype=bf)
        ops.predictor_assemble(ctx16, p32("mask_token").view(-1), self._pos_dec, mi.vis_src, mi.vis_pos, Nv, Dp,
                               x0_32, x0_16)
        xp32, _, c.dec_saved = self._dec_stack.forward(self._W_dec, x0_32, x0_16, mi.cu_v, B * mi.G, mi.max_nv, save)
        pf16 = torch.empty(Nv, Dp, device=dev, dtype=bf)
        c.dec_norm_st = torch.empty(Nv, 2, device=dev) if save else None
        ops.layernorm_fwd(xp32, p32("decoder.norm.weight"), p32("decoder.norm.bias"), self.decoder.norm.eps, None,
                          pf16, c.dec_norm_st, None)
        c.xp32 = xp32 if save else None
        pt16 = torch.empty(Nt, Dp, device=dev, dtype=bf)
        ops.gather_rows(pf16, mi.tgt_vrow, Nt, None, pt16)
        c.pt16 = pt16 if save else None
        pred16 = torch.empty(Nt, D, device=dev, dtype=bf)
        ops.gemm(ops.plain_operand(pt16), p16("decoder_to_encoder_mapper.weight"), Nt, 1, pred16,
                 bias=p32("decoder_to_encoder_mapper.bias"))
        c.pred16 = pred16
        # ---- teacher targets on the detached local features (wavjepa/jepa.py:408-409)
        local16 = torch.empty(B * T, D, device=dev, dtype=bf)
        ops.gather_rows(local32, None, B * T, None, local16)
        c.targets = self._forward_teacher_packed(local32, local16, B)
        # ---- masked latent MSE over the target rows (wavjepa/jepa.py:335-362)
        c.loss = torch.zeros(1, device=dev)
        c.dpred = torch.empty(Nt, D, device=dev, dtype=bf) if save else None
        ops.masked_mse(pred16, c.targets, mi.tgt_trow, Nt, D, c.loss, c.dpred)
        return c

    # ------------------------------------------------------------------------------------------- backward
    def _backward_impl(self, c: _Ctx, gflat: torch.Tensor, loss_scale=None, on_ready: Optional[Callable] = None):
        """Hand-written backward of `_forward_impl`.  `gflat` (zeroed, same layout as the flat parameters) receives
        every parameter gradient; on_ready(offset) announces that gflat[offset:] is final (bucketed all-reduce)."""
        mi, B = c.mi, c.B
        T, D, Dp = self.total_patches, self.encoder_embedding_dim, self.decoder_embedding_dim
        dev = gflat.device
        bf = torch.bfloat16
        Nc, Nv, Nt = mi.Nc, mi.Nv, mi.Nt
        p32 = lambda n: self._view(self._flat_p, n)
        p16 = lambda n: self._view(self._flat_w16, n)
        G_enc, G_dec, g = self._grad_views(gflat)
        ready = (lambda name: on_ready(self._offsets[name][0])) if on_ready is not None else (lambda name: None)

        dpred = c.dpred
        if loss_scale is not None:
            s = torch.as_tensor(loss_scale, device=dev, dtype=torch.float32).reshape(1)
            ops.scale_bf16(dpred, s)
        # ---- decoder_to_encoder_mapper
        ops.colsum(dpred, g("decoder_to_encoder_mapper.bias"))
        ops.gemm_wgrad(ops.plain_operand(dpred), ops.plain_operand(c.pt16), Nt, 1, g("decoder_to_encoder_mapper.weight"),
                       accumulate=True)
        ready("decoder_to_encoder_mapper.weight")
        dpf = torch.zeros(Nv, Dp, device=dev)  # rows that are not targets get no gradient
        ops.gemm_dgrad(ops.plain_operand(dpred), p16("decoder_to_encoder_mapper.weight"), Nt, 1, dpf, K=D, N=Dp,
                       out_rows=mi.tgt_vrow)
        # ---- predictor final norm + stack
        dxp = torch.empty(Nv, Dp, device=dev)
        ops.layernorm_bwd(dpf, c.xp32, c.dec_norm_st, p32("decoder.norm.weight"), dxp, None,
                          g("decoder.norm.weight"), g("decoder.norm.bias"), None)
        ready("decoder.norm.weight")
        dx0 = self._dec_stack.backward(self._W_dec, G_dec, c.dec_saved, dxp, mi.cu_v, B * mi.G, mi.max_nv,
                                       lambda i: ready(f"decoder.layers.{i}.self_attn.in_proj_weight"))
        # ---- predictor input assembly: context rows and the mask token
        # (the mask-token gradient by block sums + atomics; the context rows by a fixed-order gather over the target
        # groups, so the bf16 gradient entering the student's backward is bit-identical from run to run)
        ops.predictor_assemble_bwd(dx0, mi.vis_src, Nv, Dp, None, g("mask_token").view(-1))
        ready("mask_token")
        dctx16 = torch.empty(Nc, Dp, device=dev, dtype=bf)
        ops.predictor_ctx_grad(dx0, mi.vis_src, mi.cu_v, mi.B * mi.G, mi.G, Nc, Dp, None, dctx16)
        # ---- encoder_to_decoder_mapper
        ops.colsum(dctx16, g("encoder_to_decoder_mapper.bias"))
        ops.gemm_wgrad(ops.plain_operand(dctx16), ops.plain_operand(c.cf16), Nc, 1,
                       g("encoder_to_decoder_mapper.weight"), accumulate=True)
        ready("encoder_to_decoder_mapper.weight")
        dcf = torch.empty(Nc, D, device=dev)
        ops.gemm_dgrad(ops.plain_operand(dctx16), p16("encoder_to_decoder_mapper.weight"), Nc, 1, dcf, K=Dp, N=D)
        # ---- student final norm + stack
        dxs = torch.empty(Nc, D, device=dev)
        ops.layernorm_bwd(dcf, c.xs32, c.enc_norm_st, p32("encoder.norm.weight"), dxs, None,
                          g("encoder.norm.weight"), g("encoder.norm.bias"), None)
        ready("encoder.norm.weight")
        dxc = self._enc_stack.backward(self._W_enc, G_enc, c.enc_saved, dxs, mi.cu_c, B, mi.max_nc,
                                       lambda i: ready(f"encoder.layers.{i}.self_attn.in_proj_weight"))
        # ---- scatter to the dense token grid: the mapper output is bf16 (autocast), so is its gradient
        dlocal16 = torch.zeros(B * T, D, device=dev, dtype=bf)
        ops.scatter_dgelu(dxc, mi.ctx_rows, None, Nc, dlocal16)
        self._local_backward(c.local_saved, dlocal16, B, g, ready)
        if on_ready is not None:
            on_ready(0)

    def _local_backward(self, local_saved, dlocal16: torch.Tensor, B: int, g, ready, norm: bool = True,
                        conv: bool = True, dx: Optional[torch.Tensor] = None, wg_mapper: bool = True,
                        wg_norm: bool = True, wg_conv: bool = True) -> None:
        """Backward of `_local_features` from the (bf16) gradient of the mapper output on the dense token grid:
        post_extraction_mapper -> feature_norms -> conv stack(s).  norm=False stops after the mapper, conv=False after
        the feature norm (frozen parts below them: no data gradient flows there).  dx (fp32 [B, Cin, L], overwritten):
        continue through conv block 0 to the waveform.  wg_* False: that part is frozen, its weight gradients (and bias
        column sums) are not computed; the data gradient still passes through it."""
        T, D = self.total_patches, self.encoder_embedding_dim
        dev = dlocal16.device
        p32 = lambda n: self._view(self._flat_p, n)
        p16 = lambda n: self._view(self._flat_w16, n)
        conv_saved, f2, ln16, st = local_saved
        C = f2.shape[1]
        if wg_mapper:
            ops.colsum(dlocal16, g("post_extraction_mapper.bias"))
            ops.gemm_wgrad(ops.plain_operand(dlocal16), ops.plain_operand(ln16), B * T, 1,
                           g("post_extraction_mapper.weight"), accumulate=True)
        ready("post_extraction_mapper.weight")
        if not (norm or conv):
            return
        dln = torch.empty(B * T, C, device=dev)
        ops.gemm_dgrad(ops.plain_operand(dlocal16), p16("post_extraction_mapper.weight"), B * T, 1, dln, K=D, N=C)
        dfeat = torch.empty(B * T, C, device=dev)
        ops.layernorm_bwd(dln, f2, st, p32("feature_norms.weight"), dfeat, None,
                          *((g("feature_norms.weight"), g("feature_norms.bias")) if wg_norm else (None, None)), None)
        ready("feature_norms.weight")
        if not conv:
            return
        # ---- conv stack(s)
        ex = self.extract_audio
        streams = self._conv_streams(self._conv_wk)
        if isinstance(ex, ConvChannelFeatureExtractor):
            Tc = T // ex.in_channels
            dfeat3 = dfeat.view(B, T, C)
            for ch in range(ex.in_channels - 1, -1, -1):
                prefix, wks = streams[ch]
                sv = conv_saved[ch]
                dfc = dfeat3[:, ch * Tc:(ch + 1) * Tc].contiguous().view(B * Tc, C)
                # with shared weights every channel pass adds into the SAME gradient region: it is final (and may be
                # all-reduced) only after the last pass
                last = (not ex.share_weights_over_channels) or ch == 0
                # each mono stream's waveform gradient lands in its channel
                dxc = None if dx is None else torch.empty(B, 1, dx.shape[2], device=dev)
                self._conv_backward(prefix, wks, ex.conv_layers_spec, sv, dfc, B, Tc, C, g,
                                    ready if last else (lambda name: None), dxc, wg_conv)
                if dx is not None:
                    dx[:, ch:ch + 1].copy_(dxc)
        else:
            (prefix, wks), = streams
            self._conv_backward(prefix, wks, ex.conv_layers_spec, conv_saved[0], dfeat, B, T, C, g, ready, dx, wg_conv)

    def _conv_backward(self, prefix, wks, spec, sv, dfeat, B, T, C, g, ready, dx=None, weights: bool = True):
        n = len(spec)
        dev = dfeat.device
        p32 = lambda nm: self._view(self._flat_p, nm)
        dh = torch.empty(B, T, C, device=dev, dtype=torch.bfloat16)
        ops.scatter_dgelu(dfeat, None, sv.pre[n - 1].view(B * T, C), B * T, dh.view(B * T, C))
        gw = g if weights else (lambda nm: None)
        conv_stack_backward(spec, sv, dh, p32(f"{prefix}.0.0.weight"), p32(f"{prefix}.0.2.weight"),
                            p32(f"{prefix}.0.2.bias"), wks, gw(f"{prefix}.0.0.weight"), gw(f"{prefix}.0.2.weight"),
                            gw(f"{prefix}.0.2.bias"), [gw(f"{prefix}.{i}.0.weight") for i in range(1, n)],
                            on_layer_done=lambda i: ready(f"{prefix}.{i}.0.weight"), dx=dx, weights=weights)

    # ------------------------------------------------------------------------------------------- public API
    def forward(self, audio: torch.Tensor, ctx_masks: torch.Tensor, target_indices: torch.Tensor,
                ctx_and_target_masks: torch.Tensor) -> ForwardReturn:
        """reference JEPA.forward (wavjepa/jepa.py:365-419).  audio [B, C, L] (bf16 or fp32), ctx_masks [B, T] bool
        (True = hidden), target_indices [B, G, T] bool (True = predict), ctx_and_target_masks [B, G, T] bool
        (True = hidden from the predictor).  Returns the reference's dict; `preds` holds the predictions at the
        positions selected by target_indices (all other positions are zero -- the reference computes them but
        nothing reads them)."""
        self._ensure_ready()
        self._sync_weights()
        dev = self.device
        if audio.dim() != 3:
            raise ValueError("audio must be [B, C, L]")
        x16 = audio.to(device=dev, dtype=torch.bfloat16).contiguous()
        mi = ops.mask_indices(ctx_masks.to(dev), target_indices.to(dev), ctx_and_target_masks.to(dev))
        B, G, T, D = x16.shape[0], mi.G, self.total_patches, self.encoder_embedding_dim
        if mi.T != T:
            raise ValueError(f"masks cover {mi.T} tokens but the model produces {T}")
        want_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        c = self._forward_impl(x16, mi, save=want_grad)
        if want_grad:
            params = [dict(self.named_parameters())[n] for n in self._train_names]
            loss = _LossBridge.apply(self, c, *params)
        else:
            loss = c.loss.reshape(())
        out = ForwardReturn(local_features=c.local32.view(B, T, D), contextual_features=c.contextual_features,
                            loss=loss, targets=c.targets.view(B, T, D))
        if self.return_dense_preds:
            preds = torch.zeros(B * G * T, D, device=dev, dtype=torch.bfloat16)
            preds[target_indices.to(dev).reshape(-1)] = c.pred16
            out["preds"] = preds.view(B * G, T, D)
        else:
            out["preds"] = c.pred16
        return out

    def on_after_batch_transfer(self, batch, dataloader_idx: int = 0, starts: Optional[torch.Tensor] = None):
        """reference wavjepa/jepa.py:275-316: nr_samples_per_audio random crops of target_length per clip,
        per-crop normalisation, bf16, flattened; masks flattened.  One fused kernel (crop + Welford + scale).
        The reference additionally shuffles the audio rows only (masks are i.i.d., so this changes nothing
        statistically); here the crops stay in clip order unless `self.shuffle_crops` is set."""
        audio, ctx_masks, target_indices, ctx_and_target_masks = batch
        if audio.dim() != 3:
            audio = audio.unsqueeze(1)
        audio = audio.to(self.device, torch.float32).contiguous()
        n_clips, C, L_full = audio.shape
        S = self.nr_samples_per_audio
        if starts is None:
            starts = torch.randint(0, L_full - self.target_length + 1, (n_clips, S), device=self.device)
        starts = starts.to(self.device, torch.int32).reshape(-1).contiguous()
        x16 = torch.empty(n_clips * S, C, self.target_length, device=self.device, dtype=torch.bfloat16)
        ops.crop_norm(audio, starts, S, self.target_length, x16, None)
        if self.shuffle_crops:   # the reference permutes the AUDIO rows only (masks stay in place), jepa.py:314-316;
            x16 = x16[torch.randperm(x16.shape[0], device=self.device)]   # on the device: no host round trip
        return x16, collate_fn(ctx_masks), collate_fn(target_indices), collate_fn(ctx_and_target_masks)

    def training_step(self, batch, batch_idx: int = 0) -> ForwardReturn:
        """reference wavjepa/jepa.py:318-333: forward, then the EMA teacher update with the PRE-step student."""
        audio_input, ctx_masks, target_indices, ctx_and_target_masks = batch
        out = self(audio_input, ctx_masks, target_indices, ctx_and_target_masks)
        self._step_teacher()
        return out

    @torch.no_grad()
    def _step_teacher(self) -> None:
        """teacher = r * teacher + (1 - r) * student over the whole encoder in ONE launch (wavjepa/jepa.py:193-198)."""
        self._ensure_ready()
        r = self._get_ema_decay()
        e0, e1 = self._enc_range
        ops.ema_update(self._flat_t, self._flat_p[e0:e1], r)
        ops.cast_bf16(self._flat_t, self._flat_t16)

    # ------------------------------------------------------------------------------------------- fused train step
    def reserve_workspace(self, n_bytes: int) -> int:
        """Pre-sizes PyTorch's caching allocator pool on this device: the activation buffers of a step are allocated
        through it, their sizes follow the masks (token counts differ from step to step), and a pool that is still
        growing makes some rank call into the driver (cudaMalloc / cuMemMap, synchronising) in the middle of a step --
        at N GPUs every such stall is paid by all ranks at the next all-reduce.  Returns the bytes reserved."""
        dev = self.device
        free, _ = torch.cuda.mem_get_info(dev)
        n = int(min(n_bytes, 0.8 * free))
        if n > 0:
            block = torch.empty(n, dtype=torch.uint8, device=dev)
            del block
        return n

    def attach_data_parallel(self, reducer, sync: bool = True) -> None:
        """reducer: wavjepa_b200.dist.BucketedAllReduce (or None).  With sync (default) rank 0's student / teacher
        parameters, Adam moments and global_step are broadcast first, as Lightning's DDP strategy does at setup
        (train.py:174-179): the gradient all-reduce alone would never repair replicas that started different."""
        self._ddp = reducer
        if reducer is not None and sync and self.mask_token.device.type == "cuda":
            self._ensure_ready()
            reducer.broadcast_([self._flat_p, self._flat_t])
            has_m = reducer.any_rank(self._adam_m is not None)
            if has_m:
                if self._adam_m is None:
                    self._adam_m = torch.zeros_like(self._flat_p)
                    self._adam_v = torch.zeros_like(self._flat_p)
                reducer.broadcast_([self._adam_m, self._adam_v])
            self.global_step = reducer.broadcast_int(self.global_step)
            self._sync_weights(force=True)

    @torch.no_grad()
    def train_step(self, x16: torch.Tensor, ctx_masks: torch.Tensor, target_indices: torch.Tensor,
                   ctx_and_target_masks: torch.Tensor) -> torch.Tensor:
        """One full optimisation step on pre-cropped bf16 instances: forward, hand-written backward with the
        bucketed gradient all-reduce overlapped (if a reducer is attached), EMA with the pre-step student
        (wavjepa/jepa.py:330-331), global-norm clip (train.py:177-178) + AdamW (wavjepa/jepa.py:215-222) fused into
        one pass that also refreshes the bf16 working weights.  Returns the (device) loss tensor, no host sync
        besides the mask totals."""
        self._ensure_ready()
        self._sync_weights()
        mi = ops.mask_indices(ctx_masks, target_indices, ctx_and_target_masks)
        self._last_mi = mi
        c = self._forward_impl(x16, mi, save=True)
        gflat = self._flat_g
        gflat.zero_()
        ddp = self._ddp
        if ddp is not None:
            ddp.begin(gflat)
        self._backward_impl(c, gflat, None, ddp.ready if ddp is not None else None)
        world = 1
        if ddp is not None:
            ddp.finish()
            world = ddp.world_size
        # the EMA uses the student weights BEFORE the optimizer step (wavjepa/jepa.py:330-331): folded into the
        # AdamW pass, which reads every parameter once anyway (SURVEY.md 8(f)-1)
        self._optimizer_tail(gflat, world, self.lr_at(self.global_step), ema_decay=self._get_ema_decay())
        return c.loss

    def _optimizer_tail(self, gflat: torch.Tensor, world: int, lr: float, ema_decay: Optional[float] = None) -> None:
        """Global-norm clip + AdamW over the flat buffers (+ bf16 working-weight refresh) and, when `ema_decay` is
        given, the EMA teacher update with the pre-step student in the same pass; the lr of optimizer step k is the
        scheduler's value at k = global_step (LambdaLR)."""
        if self._adam_m is None:
            self._adam_m = torch.zeros_like(self._flat_p)
            self._adam_v = torch.zeros_like(self._flat_p)
        ss = torch.zeros(1, device=gflat.device, dtype=torch.float64)
        ops.sumsq(gflat, 1.0 / world, ss)
        b1, b2 = self.hparams.adam_betas
        if ema_decay is None:
            ops.adamw_step(self._flat_p, gflat, self._adam_m, self._adam_v, lr, b1, b2,
                           self.hparams.adam_eps, self.hparams.adam_weight_decay, self.global_step + 1, 1.0 / world,
                           self.grad_clip, ss, self._flat_w16)
        else:
            e0, e1 = self._enc_range
            ops.adamw_ema_step(self._flat_p, gflat, self._adam_m, self._adam_v, lr, b1, b2,
                               self.hparams.adam_eps, self.hparams.adam_weight_decay, self.global_step + 1,
                               1.0 / world, self.grad_clip, ss, self._flat_w16, self._flat_t, self._flat_t16, e0, e1,
                               ema_decay)
        self._refresh_conv_weights()
        self._tf32_cache = None   # the tf32 working weights are rebuilt from the updated parameters on their next use
        self._step = self.global_step + 1

    # ------------------------------------------------------------------------------------------- optimizer state
    def optimizer_state_dict(self) -> dict:
        """State of the fused optimizer path, in the shape of a Lightning checkpoint's `optimizer_states[0]` plus the
        step counter that drives the LR and EMA schedules (the reference's checkpoints carry both, train.py
        ModelCheckpoint): {'global_step', 'state': {name: {'exp_avg', 'exp_avg_sq'}}, 'param_names'}.  Tensors are
        detached copies on the parameters' device."""
        self._ensure_ready()
        st = {}
        if self._adam_m is not None:
            for n in self._train_names:
                st[n] = {"exp_avg": self._view(self._adam_m, n).clone(), "exp_avg_sq": self._view(self._adam_v, n).clone()}
        return {"global_step": int(self.global_step), "state": st, "param_names": list(self._train_names)}

    def load_optimizer_state_dict(self, sd: dict) -> None:
        """Inverse of optimizer_state_dict(): restores Adam moments and global_step so that a resumed run continues the
        warm-up / cosine LR schedule and the EMA anneal where it stopped instead of restarting them at step 0."""
        self._ensure_ready()
        self.global_step = int(sd["global_step"])
        state = sd.get("state", {})
        if not state:
            self._adam_m = self._adam_v = None
            return
        missing = [n for n in self._train_names if n not in state]
        if missing:
            raise KeyError(f"optimizer state lacks {len(missing)} parameters, e.g. {missing[:3]}")
        self._adam_m = torch.zeros_like(self._flat_p)
        self._adam_v = torch.zeros_like(self._flat_p)
        for n in self._train_names:
            self._view(self._adam_m, n).copy_(state[n]["exp_avg"])
            self._view(self._adam_v, n).copy_(state[n]["exp_avg_sq"])

    def checkpoint(self) -> dict:
        """Lightning-shaped checkpoint dict ({'state_dict', 'global_step', 'optimizer_states'}) of a fused-path run."""
        return {"state_dict": {k: v.detach().clone() for k, v in self.state_dict().items()},
                "global_step": int(self.global_step), "optimizer_states": [self.optimizer_state_dict()]}

    def load_checkpoint(self, ckpt: dict, strict: bool = True) -> None:
        self.load_state_dict({k.replace("._orig_mod", ""): v for k, v in ckpt["state_dict"].items()}, strict=strict)
        if ckpt.get("optimizer_states"):
            self.load_optimizer_state_dict(ckpt["optimizer_states"][0])
        elif "global_step" in ckpt:
            self.global_step = int(ckpt["global_step"])

    # ------------------------------------------------------------------------------------------- inference
    @torch.no_grad()
    def _periodic_index(self, host_mask, B: int, T: int):
        """Packed-row index of a padding mask that is known on the HOST and repeats every P sequences (the HEAR chunk
        geometry: the same for every clip): (ctx_rows, cu, Nc, max_n) without reading anything back from the device,
        cached per (pattern, batch)."""
        import numpy as np
        hm = np.ascontiguousarray(np.asarray(host_mask, dtype=bool))
        if hm.ndim != 2 or hm.shape[1] != T or B % hm.shape[0] != 0:
            raise ValueError(f"host_mask must be [P, {T}] with P dividing the batch ({B}); got {hm.shape}")
        key = (hm.tobytes(), hm.shape[0], B, str(self.device))
        cache = self.__dict__.setdefault("_periodic_index_cache", {})
        if key not in cache:
            P, reps = hm.shape[0], B // hm.shape[0]
            vis = ~hm
            n_per = vis.sum(1)
            rows_1 = np.flatnonzero(vis.reshape(-1)).astype(np.int64)
            cu_1 = np.concatenate([[0], np.cumsum(n_per)]).astype(np.int64)
            dev = self.device
            rep = torch.arange(reps, device=dev, dtype=torch.int64)[:, None]
            rows = (torch.from_numpy(rows_1).to(dev)[None, :] + rep * (P * T)).reshape(-1).to(torch.int32)
            cu = (torch.from_numpy(cu_1[:-1]).to(dev)[None, :] + rep * int(rows_1.size)).reshape(-1)
            cu = torch.cat([cu, torch.tensor([reps * int(rows_1.size)], device=dev)]).to(torch.int32)
            if len(cache) >= 16:
                cache.clear()
            cache[key] = (rows.contiguous(), cu.contiguous(), reps * int(rows_1.size), int(n_per.max()) if n_per.size else 0)
        return cache[key]

    def _visible_index(self, B: int, padding_mask, host_mask):
        """None when every token is visible, else the packed index (ctx_rows, cu, Nc, max_len) of the visible rows of a
        batch of B sequences: from host_mask when given (`_periodic_index`), else from padding_mask."""
        T = self.total_patches
        if host_mask is not None:
            return self._periodic_index(host_mask, B, T)
        if padding_mask is None:
            return None
        pm = padding_mask.to(self.device).reshape(B, 1, T).contiguous()
        mi = ops.mask_indices(pm.view(B, T), torch.zeros_like(pm), pm)
        return mi.ctx_rows, mi.cu_c, mi.Nc, mi.max_nc

    def _tf32_weights(self) -> dict:
        """fp32 working copy of the extractor, mapper and encoder weight matrices rounded to nearest tf32 (conv weights
        tap-major), built on first use and rebuilt when a parameter changed (load_state_dict, optimizer steps) or the flat
        buffers moved.  Bias and LayerNorm vectors are read from the fp32 masters."""
        sig = (self._signature(), self._flat_p.data_ptr())
        cache = self.__dict__.get("_tf32_cache")
        if cache is not None and cache[0] == sig:
            return cache[1]
        self._tf32_cache = None
        flat = ops.tf32_round(self._flat_p[:self._enc_range[1]])   # extractor .. encoder: the leading part of the layout
        v32 = lambda n: self._view(flat, n)
        p32 = lambda n: self._view(self._flat_p, n)
        w = dict(layers=self._stack_views("encoder.", self._enc_stack.n_layers, v32, p32),
                 conv=self._tap_major(flat, torch.float32), mapper=v32("post_extraction_mapper.weight"))
        self._tf32_cache = (sig, w)
        return w

    def _local_features_tf32(self, x32: torch.Tensor, w: dict) -> torch.Tensor:
        """_local_features at reference precision (inference only): fp32 waveform -> conv stack (tf32) -> LayerNorm(512)
        -> tf32 Linear 512->D (+bias) + positional table, all fp32.  Returns local32 [B*T, D]."""
        ex = self.extract_audio
        B = x32.shape[0]
        T, D = self.total_patches, self.encoder_embedding_dim
        C = ex.embedding_dim
        p32 = lambda n: self._view(self._flat_p, n)

        def stack(prefix, wks, x):
            return conv_stack_forward_tf32(ex.conv_layers_spec, x, p32(f"{prefix}.0.0.weight"), p32(f"{prefix}.0.2.weight"),
                                           p32(f"{prefix}.0.2.bias"), wks)

        streams = self._conv_streams(w["conv"])
        if isinstance(ex, ConvChannelFeatureExtractor):
            Tc = T // ex.in_channels
            feats = torch.empty(B, T, C, device=x32.device)
            xs = x32.transpose(0, 1).contiguous()  # [Cin, B, L]: one mono stream per CNN
            for c, (prefix, wks) in enumerate(streams):
                feats[:, c * Tc:(c + 1) * Tc].copy_(stack(prefix, wks, xs[c].unsqueeze(1)))
        else:
            feats = stack(*streams[0], x32)
        ln = torch.empty(B * T, C, device=x32.device)
        ops.add_layernorm_fwd_f32(feats.view(B * T, C), None, p32("feature_norms.weight"), p32("feature_norms.bias"),
                                  self.feature_norms.eps, None, ln)
        local32 = torch.empty(B * T, D, device=x32.device)
        ops.gemm_tf32(ops.plain_operand(ln), w["mapper"], B * T, 1, local32, bias=p32("post_extraction_mapper.bias"),
                      resid=self._pos_enc, resid_mod=T)
        return local32

    def _visible_rows(self, local32: torch.Tensor, index, bf16: bool):
        """The encoder's input rows: all of local32 [B*T, D] (index None) or an fp32 copy of its visible rows, and with
        bf16 their bf16 copy.  Returns (x32, x16 | None, cu, max_len)."""
        T, D = self.total_patches, self.encoder_embedding_dim
        dev = local32.device
        if index is None:
            rows, x32, M = None, local32, local32.shape[0]
            cu, max_len = torch.arange(0, M + T, T, device=dev, dtype=torch.int32), T
        else:
            rows, cu, M, max_len = index
            x32 = torch.empty(M, D, device=dev)
        x16 = torch.empty(M, D, device=dev, dtype=torch.bfloat16) if bf16 else None
        if index is not None or bf16:
            ops.gather_rows(local32, rows, M, None if index is None else x32, x16)
        return x32, x16, cu, max_len

    def _final_norm(self, xs32: torch.Tensor, index, B: int, st: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The encoder's final LayerNorm of its output rows into the features [B, T, D] fp32, scattered to the visible
        rows when packed (padded rows are zeros); st: LayerNorm statistics for the backward."""
        T, D = self.total_patches, self.encoder_embedding_dim
        dev = xs32.device
        M = xs32.shape[0]
        out = torch.empty(B, T, D, device=dev) if index is None else torch.zeros(B, T, D, device=dev)
        packed = out.view(B * T, D) if index is None else torch.empty(M, D, device=dev)
        ops.layernorm_fwd(xs32, self._view(self._flat_p, "encoder.norm.weight"),
                          self._view(self._flat_p, "encoder.norm.bias"), self.encoder.norm.eps, packed, None, st, None)
        if index is not None:
            ops.scatter_rows(packed, index[0], M, out.view(B * T, D))
        return out

    def _audio_representation_tf32(self, audio: torch.Tensor, index) -> torch.Tensor:
        """get_audio_representation with inference_precision == "tf32" (same masking semantics)."""
        w = self._tf32_weights()
        x32 = audio.to(device=self.device, dtype=torch.float32).contiguous()
        B = x32.shape[0]
        xv32, _, cu, max_len = self._visible_rows(self._local_features_tf32(x32, w), index, bf16=False)
        xs32 = self._enc_stack.forward_tf32(w["layers"], xv32, ops.tf32_round(xv32), cu, B, max_len)
        return self._final_norm(xs32, index, B)

    # ------------------------------------------------------------------------------------------- fine-tuning
    def _feature_plan(self, trainable, audio_grad: bool = False, top: Optional[int] = None) -> Optional[_FeaturePlan]:
        """What a backward through the features computes: the weight gradients of the feature-path parameters named in
        `trainable` (other names are ignored) and, with audio_grad, the waveform gradient.  None when it computes
        neither.  top (hidden states up to `top`): the path ends at the output of encoder layer top - 1, so the layers
        from `top` on and the final norm are not part of it."""
        trainable = set(trainable)
        names = [n for n in self._train_names if n.startswith(_FEATURE_PATH)]
        if top is not None:
            names = [n for n in names if not n.startswith("encoder.") or
                     (n.startswith("encoder.layers.") and int(n.split(".")[2]) < top)]
        trainable = [n for n in names if n in trainable]
        if not (trainable or audio_grad):
            return None
        plan = _FeaturePlan()
        plan.names = names
        plan.dx = audio_grad
        plan.conv = any(n.startswith("extract_audio.") for n in trainable)
        plan.norm = any(n.startswith("feature_norms.") for n in trainable)
        plan.mapper = any(n.startswith("post_extraction_mapper.") for n in trainable)
        plan.final_norm = any(n.startswith("encoder.norm.") for n in trainable)
        plan.local = plan.conv or plan.norm or plan.mapper or plan.dx
        n_layers = self._enc_stack.n_layers
        layers = [int(n.split(".")[2]) for n in trainable if n.startswith("encoder.layers.")]
        plan.layer_w = [i in layers for i in range(n_layers)]
        plan.first_layer = 0 if plan.local else min(layers, default=n_layers)
        return plan

    def _dense_rows(self, x32: torch.Tensor, index, B: int, copy: bool = False) -> torch.Tensor:
        """Encoder rows [M, D] fp32 on the token grid [B, T, D]: scattered into zeros when packed (a fresh buffer);
        dense: x32 itself, or with `copy` a copy of it (a buffer the backward reads must not be handed out)."""
        T, D = self.total_patches, self.encoder_embedding_dim
        if index is None:
            if copy:
                out = torch.empty_like(x32)
                ops.gather_rows(x32, None, x32.shape[0], out, None)
                x32 = out
            return x32.view(B, T, D)
        out = torch.zeros(B, T, D, device=x32.device)
        ops.scatter_rows(x32, index[0], x32.shape[0], out.view(B * T, D))
        return out

    def _features_forward(self, x16: torch.Tensor, index, plan: Optional[_FeaturePlan] = None,
                          collect: Optional[List[int]] = None):
        """The bf16 feature forward (bf16 [B, Cin, L] waveform -> features [B, T, D] fp32) of get_audio_representation,
        of `_FeatureBridge` and of the denoiser's student.  index: None (dense) or (ctx_rows, cu, Nc, max_len) of the
        visible rows.  collect (get_hidden_states): instead of the features, the list of hidden states `collect` [B, T, D]
        fp32 (0: the encoder input, k: the output of layer k - 1); only the layers below max(collect) run and the final
        norm does not.  Without a plan nothing is saved and the context is None; with one, the activations the backward
        needs are kept from the lowest trainable point upward.  Returns (features or hidden states, context)."""
        B = x16.shape[0]
        save = plan is not None
        top = self._enc_stack.n_layers if collect is None else max(collect)
        # (the waveform gradient runs the whole conv stack backward: its GELU' copies are kept even when it is frozen)
        local32, local_saved = self._local_features(x16, save=save and plan.local,
                                                    save_conv=save and (plan.conv or plan.dx))
        x32, xv16, cu, max_len = self._visible_rows(local32, index, bf16=top > 0)
        del local32
        M = x32.shape[0]
        hook, hidden = None, {}
        if collect is not None:
            # every hidden state below the top is an input the backward reads (the top one nothing else holds)
            if 0 in collect:
                hidden[0] = self._dense_rows(x32, index, B, copy=save and top > 0)

            def hook(i, y, _):
                if i + 1 in collect:
                    hidden[i + 1] = self._dense_rows(y, index, B, copy=save and i + 1 < top)
        xs32, _, enc_saved = self._enc_stack.forward(self._W_enc[:top], x32, xv16, cu, B, max_len, save, hook,
                                                     save_from=plan.first_layer if save else 0)
        norm_st = None
        if collect is None:
            norm_st = torch.empty(M, 2, device=x16.device) if save else None
            out = self._final_norm(xs32, index, B, norm_st)
        else:
            out = [hidden[k] for k in collect]
        if not save:
            return out, None
        c = _Ctx()
        c.B, c.index, c.plan, c.x_shape, c.cu, c.max_len, c.M = B, index, plan, x16.shape, cu, max_len, M
        c.collect = collect
        c.local_saved = local_saved if plan.local else None
        c.enc_saved, c.xs32, c.norm_st = enc_saved, (xs32 if collect is None else None), norm_st
        return out, c

    def _features_backward(self, c: _Ctx, grad_out, gflat: Optional[torch.Tensor] = None,
                           on_ready: Optional[Callable] = None):
        """Backward of `_features_forward` from the fp32 gradient of the features [B, T, D], or (a context with
        `collect`) from the list of the gradients of the hidden states, None for those the loss does not read: the
        highest one that is read starts the encoder backward, every other one is added to the gradient at its layer
        boundary (ops.add_rows).  gflat: the gradient buffer (zeroed, flat layout), by default one owned by this call over
        the extractor..encoder span (several graphs may be alive); on_ready(offset) announces that gflat[offset:] is
        final (bucketed all-reduce).  Returns (gflat, the fp32 gradient of the bf16 waveform [B, Cin, L] when plan.dx,
        else None).  Only the parts with a trainable tensor compute weight gradients."""
        dev = self._flat_p.device
        B, M, plan = c.B, c.M, c.plan
        T, D = self.total_patches, self.encoder_embedding_dim
        n_layers = self._enc_stack.n_layers
        p32 = lambda n: self._view(self._flat_p, n)
        if gflat is None:
            gflat = torch.zeros(self._enc_range[1], device=dev)
        g = lambda n: self._view(gflat, n)
        ready = (lambda name: on_ready(self._offsets[name][0])) if on_ready is not None else (lambda name: None)
        rows = None if c.index is None else c.index[0]

        def dense(gr):
            return gr.to(device=dev, dtype=torch.float32).contiguous().view(B * T, D)

        def packed(dy):   # padded rows are constants: only the visible rows' gradient enters
            if rows is None:
                return dy
            dyp = torch.empty(M, D, device=dev)
            ops.gather_rows(dy, rows, M, dyp, None)
            return dyp

        daudio = torch.empty(c.x_shape, device=dev) if plan.dx else None
        inject, dh0 = None, None
        if c.collect is None:
            top = n_layers
            dx = torch.empty(M, D, device=dev)
            ops.layernorm_bwd(packed(dense(grad_out)), c.xs32, c.norm_st, p32("encoder.norm.weight"), dx, None,
                              *((g("encoder.norm.weight"), g("encoder.norm.bias")) if plan.final_norm else (None, None)),
                              None)
            ready("encoder.norm.weight")
            c.xs32 = None
        else:
            # a hidden state at or below the lowest layer the backward visits reaches nothing trainable, unless the
            # local features or the waveform want their gradient
            low = 0 if plan.local else plan.first_layer + 1
            dh = {k: dense(gr) for k, gr in zip(c.collect, grad_out) if gr is not None and k >= low}
            if not dh:
                c.enc_saved = c.local_saved = None
                return gflat, (daudio.zero_() if plan.dx else None)
            top = max(dh)
            dx = packed(dh.pop(top))
            dh0 = dh.pop(0, None) if top > 0 else None

            def inject(i, x):
                if i + 1 in dh:
                    ops.add_rows(x, dh[i + 1], rows, M)
        if plan.first_layer < top:
            # (the cached views of _grad_views slice the whole layout: a call-owned buffer gets its own encoder views)
            G_enc = self._grad_views(gflat)[0] if gflat is self._flat_g else \
                self._stack_views("encoder.", n_layers, g, g)
            dx = self._enc_stack.backward(self._W_enc[:top], G_enc, c.enc_saved, dx, c.cu, B, c.max_len,
                                          lambda i: ready(f"encoder.layers.{i}.self_attn.in_proj_weight"),
                                          stop_at=plan.first_layer, need_dx=plan.local, need_wgrad=plan.layer_w,
                                          inject=inject)
        if plan.local:
            if dh0 is not None:
                ops.add_rows(dx, dh0, rows, M)
            # the mapper output is bf16 (autocast), so is its gradient on the dense token grid
            if c.index is None:
                dlocal16 = torch.empty(B * T, D, device=dev, dtype=torch.bfloat16)
                ops.gather_rows(dx, None, M, None, dlocal16)
            else:
                dlocal16 = torch.zeros(B * T, D, device=dev, dtype=torch.bfloat16)
                ops.scatter_dgelu(dx, rows, None, M, dlocal16)
            del dx
            self._local_backward(c.local_saved, dlocal16, B, g, ready,
                                 norm=plan.norm or plan.conv or plan.dx, conv=plan.conv or plan.dx, dx=daudio,
                                 wg_mapper=plan.mapper, wg_norm=plan.norm, wg_conv=plan.conv)
        c.enc_saved = c.local_saved = None
        return gflat, daudio

    def get_audio_representation(self, audio: torch.Tensor, padding_mask: Optional[torch.Tensor] = None,
                                 host_mask=None) -> torch.Tensor:
        """reference wavjepa/jepa.py:456-467: student encoder (incl. final norm) features [B, T, D] fp32.  Tokens
        hidden by padding_mask (True) are excluded as keys exactly like the reference's key-padding mask; their own
        output rows (which the callers cut off, hear_api/runtime.py:141-142) are returned as zeros.
        host_mask (optional, CPU bool [P, T], P | B): the same padding mask given as a pattern known on the host that
        repeats every P sequences -- the packed index then needs no device read-back (padding_mask is ignored).

        Fine-tuning: in grad mode, when a parameter of the feature path (extract_audio, feature_norms,
        post_extraction_mapper, encoder) requires grad, the features carry a grad_fn and `backward()` fills `.grad` of
        the trainable path parameters (everything else keeps grad None).  The values are bit-identical to the no-grad
        call.  Rows hidden by a padding mask stay constant zeros: gradient flows from the visible rows only (the
        reference computes values at padded query positions, but no caller reads them).  Frozen parts save nothing and
        are not backpropagated: a frozen extractor, or encoder layers below the lowest trainable one; frozen layers
        above it pass the gradient on without computing weight gradients.

        Waveform gradient: in grad mode, when `audio` requires grad (a frozen encoder used as a perceptual or
        feature-matching loss, input saliency, a network in front of a trainable encoder), the features carry a
        grad_fn and `backward()` also fills `audio.grad` -- on audio's device, in its dtype (fp32 or bf16): the
        gradient with respect to the bf16 waveform the model reads, through every block down to conv block 0.  Only
        the parts with a trainable tensor compute weight gradients, so a fully frozen encoder runs data gradients only.
        Padded samples still receive the gradient the GroupNorm of block 0 couples them to.  No gradient reaches
        padding_mask / host_mask.

        One graph supports one backward.  inference_precision "tf32" stays forward-only (no grad_fn, whatever
        requires grad): fine-tuning and the waveform gradient run in the "bf16" training numerics (DESIGN.md 2.2,
        2.3)."""
        self.eval()
        self._ensure_ready()
        self._sync_weights()
        index = self._visible_index(audio.shape[0], padding_mask, host_mask)
        if self.inference_precision == "tf32":
            return self._audio_representation_tf32(audio, index)
        dev = self.device
        plan = None
        if torch.is_grad_enabled():   # the rule of `forward`
            plan = self._feature_plan([n for n, p in self.named_parameters() if p.requires_grad], audio.requires_grad)
        if plan is None:
            return self._features_forward(audio.to(device=dev, dtype=torch.bfloat16).contiguous(), index)[0]
        params = dict(self.named_parameters())
        # audio moves to the device outside the Function: autograd's copy backward takes the gradient back to audio.device
        return _FeatureBridge.apply(self, audio.to(device=dev), index, plan, None, *[params[n] for n in plan.names])

    def _hidden_layers(self, layers) -> List[int]:
        """The hidden-state indices of `get_hidden_states(layers=...)`: None -> all N + 1, else a non-empty sequence of
        distinct ints in [0, N] (ValueError otherwise).  Host-side only."""
        n = self._enc_stack.n_layers
        if layers is None:
            return list(range(n + 1))
        if isinstance(layers, (str, bytes)) or not hasattr(layers, "__iter__"):
            raise ValueError(f"layers must be a sequence of ints in [0, {n}], got {layers!r}")
        out = []
        for k in layers:
            if isinstance(k, bool) or not isinstance(k, (int, np.integer)):
                raise ValueError(f"layers must hold ints in [0, {n}], got {k!r}")
            if not 0 <= int(k) <= n:
                raise ValueError(f"hidden state {int(k)} is out of range: this encoder has {n} layers, [0, {n}]")
            if int(k) in out:
                raise ValueError(f"hidden state {int(k)} is requested twice")
            out.append(int(k))
        if not out:
            raise ValueError("layers is empty: request at least one hidden state (None requests all)")
        return out

    def _hidden_states_tf32(self, audio: torch.Tensor, index, collect: List[int]) -> List[torch.Tensor]:
        """get_hidden_states with inference_precision == "tf32" (the path of _audio_representation_tf32, stopped after
        layer max(collect) - 1)."""
        w = self._tf32_weights()
        x32 = audio.to(device=self.device, dtype=torch.float32).contiguous()
        B = x32.shape[0]
        top = max(collect)
        xv32, _, cu, max_len = self._visible_rows(self._local_features_tf32(x32, w), index, bf16=False)
        hidden = {}
        if 0 in collect:
            hidden[0] = self._dense_rows(xv32, index, B)

        def hook(i, y):
            if i + 1 in collect:
                hidden[i + 1] = self._dense_rows(y, index, B)
        if top > 0:
            self._enc_stack.forward_tf32(w["layers"][:top], xv32, ops.tf32_round(xv32), cu, B, max_len, hook)
        return [hidden[k] for k in collect]

    def get_hidden_states(self, audio: torch.Tensor, padding_mask: Optional[torch.Tensor] = None, host_mask=None,
                          layers=None) -> List[torch.Tensor]:
        """The student encoder's per-layer hidden states (the `hidden_states` convention of HF transformers), fp32
        [B, T, D] each on the model's device, in the order of `layers`:
          hidden state 0        the encoder input: post_extraction_mapper output + pos_encoding_encoder;
          hidden state k        the output of encoder.layers[k-1] (after its norm2), 1 <= k <= N (12 base, 24 large);
        so `get_audio_representation == encoder.norm(hidden state N)`.  layers: distinct ints in [0, N] (None: all
        N + 1); anything else raises ValueError before any device work.  Only the layers below max(layers) run, and
        the final norm never does: layers=[6] runs 6 encoder layers, layers=[0] none.

        Token layout, padding_mask / host_mask and the zero rows of hidden tokens are those of
        `get_audio_representation`; so is inference_precision ("tf32": the reference-precision forward, no grad_fn).

        Gradients ("bf16"): under the rule of `get_audio_representation` (some feature-path parameter requires grad,
        or audio does) the hidden states carry a grad_fn, and any subset of them may feed the loss.  The graph holds the
        path up to layer max(layers) - 1: the parameters of the layers above and of encoder.norm keep grad None.  A
        hidden state the loss does not read costs nothing in the backward; the others' gradients are added at their
        layer boundaries of the one encoder backward.  Frozen parts save nothing, the waveform gradient arrives in
        audio's dtype on audio's device, one graph supports one backward (DESIGN.md 2.4)."""
        collect = self._hidden_layers(layers)
        self.eval()
        self._ensure_ready()
        self._sync_weights()
        index = self._visible_index(audio.shape[0], padding_mask, host_mask)
        if self.inference_precision == "tf32":
            return self._hidden_states_tf32(audio, index, collect)
        dev = self.device
        plan = None
        if torch.is_grad_enabled():
            plan = self._feature_plan([n for n, p in self.named_parameters() if p.requires_grad], audio.requires_grad,
                                      top=max(collect))
        if plan is None:
            return self._features_forward(audio.to(device=dev, dtype=torch.bfloat16).contiguous(), index, None,
                                          collect)[0]
        params = dict(self.named_parameters())
        return list(_FeatureBridge.apply(self, audio.to(device=dev), index, plan, collect,
                                         *[params[n] for n in plan.names]))
