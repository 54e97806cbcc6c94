"""Waveform encoders with the reference's class API, running on the sm_100a kernels.

Mirrors wavjepa/extractors/: `Extractor` (audio_extractor.py:6-20), `ConvFeatureExtractor`
(audio_feature_extractor.py:13-154) and `ConvChannelFeatureExtractor` (audio_channel_feature_extractor.py:13-179).
Parameter names and shapes are the reference's (`cnn.{i}.0.weight [out, in, k]`, `cnn.0.2.{weight,bias}`;
`cnns.{c}.{i}.0.weight` for the per-channel variant) so checkpoints interchange.

Execution (no PyTorch compute anywhere):
  block 0      Conv1d(Cin, C, 10, 5) + GroupNorm(C, C) + GELU   -> one fused HBM-bound kernel  (csrc/conv0.cu)
  blocks 1..n  Conv1d(C, C, k in {2,3}, 2) + GELU                -> implicit-GEMM tcgen05 tiles over channels-last
                                                                    activations, GELU in the epilogue (csrc/gemm_tcgen05.cu)
Activations are channels-last bf16 [B, L, C] end to end, so the reference's final `B C T -> B T C` rearrange
(audio_feature_extractor.py:137) is free.
"""
from __future__ import annotations

import math
from abc import ABC, abstractmethod
from typing import List, Optional, Sequence

import torch
from torch import nn

from . import ops
from ._lib import WavJepaLibError


class Extractor(ABC):
    """reference wavjepa/extractors/audio_extractor.py:6-20"""

    embedding_dim: int

    @abstractmethod
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        ...

    @abstractmethod
    def total_patches(self, time: int) -> int:
        ...


class _ConvParams(nn.Module):
    """Holds `weight` [out, in, k] of one Conv1d (kaiming_normal_ init, audio_feature_extractor.py:70-72)."""

    def __init__(self, n_in: int, n_out: int, k: int, stride: int):
        super().__init__()
        self.in_channels, self.out_channels, self.kernel_size, self.stride = n_in, n_out, k, stride
        self.weight = nn.Parameter(torch.empty(n_out, n_in, k))
        nn.init.kaiming_normal_(self.weight)


class _GroupNormParams(nn.Module):
    """Affine parameters of GroupNorm(C, C) (audio_feature_extractor.py:94); eps 1e-5."""

    def __init__(self, channels: int, eps: float = 1e-5):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(channels))
        self.bias = nn.Parameter(torch.zeros(channels))


class _Slot(nn.Module):
    """Parameter-free placeholder keeping the reference's Sequential indices (Dropout(0) / GELU positions)."""


def _check_spec(spec: Sequence[Sequence[int]]) -> None:
    if len(spec) < 2:
        raise WavJepaLibError("conv_layers_spec needs at least two layers")
    dim0, k0, s0 = spec[0]
    if (k0, s0) != (10, 5):
        raise WavJepaLibError(f"block 0 must be (dim, 10, 5) -- the fused conv0 kernel is built for k=10, stride=5; got {spec[0]}")
    for (dim, k, s) in spec[1:]:
        if dim != dim0 or s != 2 or k not in (2, 3):
            raise WavJepaLibError(f"blocks 1.. must be ({dim0}, k in (2,3), 2); got {(dim, k, s)}")
    if dim0 % 128 != 0:
        raise WavJepaLibError("channel count must be a multiple of 128")


def out_length(spec: Sequence[Sequence[int]], time: int) -> int:
    """Closed form of ConvFeatureExtractor.total_patches (audio_feature_extractor.py:140-145): valid convs, no padding."""
    L = time
    for (_, k, s) in spec:
        L = (L - k) // s + 1
    return L


# =============================================================================================== kernel orchestration
def kmajor_weight(w: torch.Tensor, out: Optional[torch.Tensor] = None, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """[O, C, k] fp32 master weight -> [O, k*C] (tap-major) working copy used by the implicit GEMM (bf16, or fp32 for the
    tf32 GEMM)."""
    O, C, k = w.shape
    if out is None:
        out = torch.empty(O, k * C, device=w.device, dtype=dtype)
    out.view(O, k, C).copy_(w.detach().permute(0, 2, 1))
    return out


class ConvSaved:
    __slots__ = ("x16", "moments", "stats", "acts", "pre")


def conv_stack_forward(spec, x16: torch.Tensor, w0: torch.Tensor, gn_w: torch.Tensor, gn_b: torch.Tensor,
                       wks: List[torch.Tensor], save: bool, gn_eps: float = 1e-5):
    """x16 [B, Cin, L] bf16 -> (features [B, T, C] bf16, ConvSaved | None)."""
    assert x16.dtype == torch.bfloat16 and x16.is_contiguous()
    B, Cin, L = x16.shape
    C = spec[0][0]
    dev = x16.device
    L0 = (L - 10) // 5 + 1
    if L0 <= 0:
        raise WavJepaLibError("input shorter than the first conv kernel")
    a = torch.empty(B, L0, C, device=dev, dtype=torch.bfloat16)
    moments, stats = ops.conv0_workspaces(B, Cin, C, dev)
    # (block 0 saves nothing the size of its output: its backward recomputes GELU'(z) from the input window)
    ops.conv0_fwd(x16, w0, gn_w, gn_b, a, moments, stats, eps=gn_eps)
    acts, pre = [a], [None]
    for i, (_, k, _) in enumerate(spec[1:], start=1):
        x = acts[-1]
        L_in = x.shape[1]
        L_out = (L_in - k) // 2 + 1
        g = torch.empty(B, L_out, C, device=dev, dtype=torch.bfloat16)
        h = torch.empty(B, L_out, C, device=dev, dtype=torch.bfloat16) if save else None
        if L_in % 2 == 0:
            a_op = ops.conv_operand(x, k)
        else:
            a_op = ops.conv_operand_odd(x, k)
        ops.gemm(a_op, wks[i - 1], L_out, B, g.view(-1, C), act=ops.ACT_GELU,
                 out2=h.view(-1, C) if save else None)
        if not save:
            acts[-1] = None  # free as we go
        acts.append(g)
        pre.append(h)
    sv = None
    if save:
        sv = ConvSaved()
        sv.x16, sv.moments, sv.stats, sv.acts, sv.pre = x16, moments, stats, acts, pre
    return acts[-1], sv


def conv_stack_forward_tf32(spec, x32: torch.Tensor, w0: torch.Tensor, gn_w: torch.Tensor, gn_b: torch.Tensor,
                            wks: List[torch.Tensor], gn_eps: float = 1e-5) -> torch.Tensor:
    """Inference at reference precision: x32 [B, Cin, L] fp32 -> features [B, T, C] fp32.  Block 0 in fp32 on the CUDA
    cores, blocks 1..n as tf32 implicit GEMMs (wks: fp32 tap-major weights rounded to nearest tf32) with the exact GELU.
    Every block output that feeds another conv is rounded to nearest tf32; the last one (LayerNorm input) is not."""
    assert x32.dtype == torch.float32 and x32.is_contiguous()
    B, Cin, L = x32.shape
    C = spec[0][0]
    dev = x32.device
    L0 = (L - 10) // 5 + 1
    if L0 <= 0:
        raise WavJepaLibError("input shorter than the first conv kernel")
    x = torch.empty(B, L0, C, device=dev, dtype=torch.float32)
    moments, stats = ops.conv0_workspaces(B, Cin, C, dev)
    ops.conv0_fwd_f32(x32, w0, gn_w, gn_b, x, moments, stats, eps=gn_eps)
    n = len(spec)
    for i, (_, k, _) in enumerate(spec[1:], start=1):
        L_in = x.shape[1]
        L_out = (L_in - k) // 2 + 1
        g = torch.empty(B, L_out, C, device=dev, dtype=torch.float32)
        if L_in % 2 == 0:
            a_op = ops.conv_operand(x, k)
        else:
            a_op = ops.conv_operand_odd(x, k)
        ops.gemm_tf32(a_op, wks[i - 1], L_out, B, g.view(-1, C), act=ops.ACT_GELU_ERF, round_out=i < n - 1)
        x = g
    return x


def conv_stack_backward(spec, sv: ConvSaved, dh_last: torch.Tensor, w0, gn_w, gn_b, wks, g_w0, g_gn_w, g_gn_b,
                        g_ws: List[torch.Tensor], gn_eps: float = 1e-5, on_layer_done=None) -> None:
    """dh_last: bf16 [B, T, C] gradient w.r.t. the PRE-activation of the last conv block.  Accumulates into the fp32
    gradient tensors g_* (shapes of the parameters).

    Odd input lengths (the wav2vec2 extractor's 401-row input of its last block): the weight gradient reads the
    activations through the forward's strided view (k*C columns per output row, batch pitch L_in*C), and conv_dgrad
    writes dx with that batch pitch; the trailing input row of a k = 2 block feeds no output and gets a zero gradient."""
    n = len(spec)
    B = dh_last.shape[0]
    C = spec[0][0]
    dev = dh_last.device
    dh = dh_last
    for i in range(n - 1, 0, -1):
        k = spec[i][1]
        x = sv.acts[i - 1]
        L_in = x.shape[1]
        L_out = dh.shape[1]
        dwk = torch.empty(C, k * C, device=dev, dtype=torch.float32)
        x_op = ops.conv_operand(x, k) if L_in % 2 == 0 else ops.conv_operand_odd(x, k)
        ops.gemm_wgrad(ops.make_operand(dh, C, L_out, B), x_op, L_out, B, dwk)
        g_ws[i - 1].add_(dwk.view(C, k, C).permute(0, 2, 1))
        dx = torch.empty(B, L_in, C, device=dev, dtype=torch.bfloat16)
        if i - 1 >= 1:
            ops.conv_dgrad(dh, wks[i - 1], dx, k, act=ops.ACT_DGELU, aux=sv.pre[i - 1])
        else:
            ops.conv_dgrad(dh, wks[i - 1], dx, k)
        sv.acts[i] = None
        sv.pre[i] = None
        dh = dx
        if on_layer_done is not None:
            on_layer_done(i)
    red = torch.empty(B, 2 + sv.x16.shape[1] * 10, C, device=dev, dtype=torch.float64)
    ops.conv0_bwd(sv.x16, w0, gn_w, gn_b, sv.moments, sv.stats, dh, red, g_w0, g_gn_w, g_gn_b, eps=gn_eps)
    if on_layer_done is not None:
        on_layer_done(0)


# =============================================================================================== modules
class ConvFeatureExtractor(Extractor, nn.Module):
    """reference wavjepa/extractors/audio_feature_extractor.py:13-154 (mode="default", no bias, not depthwise)."""

    def __init__(self, *args, conv_layers_spec: list, in_channels: int = 2, dropout: float = 0.0,
                 mode: str = "default", conv_bias: bool = False, depthwise: bool = False, **kwargs):
        nn.Module.__init__(self)
        if mode != "default" or conv_bias or depthwise or dropout != 0.0:
            raise WavJepaLibError("only mode='default', conv_bias=False, depthwise=False, dropout=0 is built "
                                  "(the configuration of configs/extractor/*.yaml)")
        spec = [tuple(int(v) for v in cl) for cl in conv_layers_spec]
        _check_spec(spec)
        if in_channels not in (1, 2):
            raise WavJepaLibError("in_channels must be 1 or 2")
        self.in_channels = in_channels
        self.depthwise = depthwise
        self.conv_layers_spec = spec
        blocks = []
        in_d = in_channels
        for i, (dim, k, stride) in enumerate(spec):
            if i == 0:
                blocks.append(nn.Sequential(_ConvParams(in_d, dim, k, stride), _Slot(), _GroupNormParams(dim), _Slot()))
            else:
                blocks.append(nn.Sequential(_ConvParams(in_d, dim, k, stride), _Slot(), _Slot()))
            in_d = dim
        self.cnn = nn.Sequential(*blocks)
        self.embedding_dim = spec[-1][0]
        self._wk_cache = None

    # ---- weight access used by the JEPA engine
    def conv_params(self):
        return [blk[0].weight for blk in self.cnn]

    def gn_params(self):
        return self.cnn[0][2].weight, self.cnn[0][2].bias

    def _working_weights(self):
        ws = self.conv_params()
        sig = tuple((w.data_ptr(), w._version) for w in ws)
        if self._wk_cache is None or self._wk_cache[0] != sig:
            self._wk_cache = (sig, [kmajor_weight(w) for w in ws[1:]])
        return self._wk_cache[1]

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [B, Cin, L] -> local features [B, T, C] (bf16).  Inference only; training goes through JEPA, whose
        backward owns the saved activations."""
        if x.dim() != 3 or x.shape[1] != self.in_channels:
            raise ValueError(f"expected [B, {self.in_channels}, L], got {tuple(x.shape)}")
        x16 = x.to(torch.bfloat16).contiguous()
        gw, gb = self.gn_params()
        feats, _ = conv_stack_forward(self.conv_layers_spec, x16, self.conv_params()[0].detach(), gw.detach(),
                                      gb.detach(), self._working_weights(), save=False)
        return feats

    def total_patches(self, time: int, device: str = "cuda") -> int:
        return out_length(self.conv_layers_spec, time)

    @property
    def receptive_fields(self) -> List[int]:
        rf = 1
        fields = [rf]
        for _, width, stride in reversed(self.conv_layers_spec):
            rf = (rf - 1) * stride + width
            fields.append(rf)
        return list(reversed(fields))

    def description(self, sfreq: Optional[int] = None, dummy_time: Optional[int] = None) -> str:
        dims, _, strides = zip(*self.conv_layers_spec)
        rf = self.receptive_fields[0]
        ds = math.prod(strides)
        desc = f"Receptive field: {rf} samples"
        if sfreq is not None:
            desc += f", {rf / sfreq:.2f} seconds"
        desc += f" | Downsampled by {ds}"
        if sfreq is not None:
            desc += f", new sfreq: {sfreq / ds:.2f} Hz"
        desc += f" | Overlap of {rf - ds} samples"
        if dummy_time is not None:
            desc += f" | {self.total_patches(dummy_time)} encoded samples/trial"
        return desc


class ConvChannelFeatureExtractor(Extractor, nn.Module):
    """reference wavjepa/extractors/audio_channel_feature_extractor.py:13-179 (WavJEPA-Nat): one mono CNN per input
    channel (or one shared CNN), tokens concatenated channel-major: [c0 t0..t(T-1), c1 t0..t(T-1), ...] (:177-178)."""

    def __init__(self, *args, conv_layers_spec: list, in_channels: int = 2, dropout: float = 0.0,
                 mode: str = "default", conv_bias: bool = False, depthwise: bool = False,
                 share_weights_over_channels: bool = False, **kwargs):
        nn.Module.__init__(self)
        self.in_channels = in_channels
        self.share_weights_over_channels = share_weights_over_channels
        spec = [tuple(int(v) for v in cl) for cl in conv_layers_spec]
        n_cnn = 1 if share_weights_over_channels else in_channels
        subs = [ConvFeatureExtractor(conv_layers_spec=spec, in_channels=1, dropout=dropout, mode=mode,
                                     conv_bias=conv_bias, depthwise=depthwise) for _ in range(n_cnn)]
        self._spec = spec
        self.conv_layers_spec = spec
        self.cnns = nn.ModuleList([s.cnn for s in subs])
        self._subs = subs  # plain list: the parameters are registered through self.cnns only
        self.embedding_dim = spec[-1][0]

    def sub(self, c: int) -> ConvFeatureExtractor:
        return self._subs[0 if self.share_weights_over_channels else c]

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 3 or x.shape[1] != self.in_channels:
            raise ValueError(f"expected [B, {self.in_channels}, L], got {tuple(x.shape)}")
        outs = [self.sub(c)(x[:, c:c + 1].contiguous()) for c in range(self.in_channels)]
        return torch.cat(outs, dim=1)

    def total_patches(self, time: int, device: str = "cuda") -> int:
        return out_length(self._spec, time) * self.in_channels
