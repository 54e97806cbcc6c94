"""Forward / backward orchestration of the transformer stacks on the sm_100a kernels (host side only: buffer
allocation through PyTorch's caching allocator and kernel sequencing on the current stream).

One `TransformerStack` serves the student encoder, the EMA teacher and the predictor of wavjepa/jepa.py:126-130:
post-norm nn.TransformerEncoderLayer semantics (wavjepa/types/wavjepa_configs.py:29-47)

    o1 = bf16(out_proj(MHA(x)))                  x1 = LN1(x  + o1)      (eps 1e-6)
    o2 = bf16(W2 GELU(bf16(W1 x1 + b1)) + b2)    x2 = LN2(x1 + o2)

over PACKED variable-length token sets (cu_seqlens), which reproduces the reference's key-padding-masked dense
computation at every visible position (SURVEY.md 3.1).  Precision policy = the reference's bf16 autocast: GEMM /
attention operands bf16 with fp32 accumulation, residual stream / LayerNorm / softmax statistics fp32.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import torch

from . import ops


class LayerViews:
    """Views of one layer's tensors into the model's flat buffers: the bf16 working weights + fp32 vectors, or the fp32
    gradients."""
    __slots__ = ("w_in", "b_in", "w_o", "b_o", "w1", "b1", "w2", "b2", "g1", "be1", "g2", "be2")


class LayerSaved:
    __slots__ = ("x32", "x16", "qkv", "att", "lse", "o1", "st1", "x1_32", "x1_16", "h", "g", "o2", "st2")


def _empty(shape, dtype, dev):
    return torch.empty(shape, device=dev, dtype=dtype)


class TransformerStack:
    def __init__(self, d_model: int, nhead: int, dim_ff: int, n_layers: int, ln_eps: float):
        if d_model % nhead != 0 or (d_model // nhead) not in (32, 64):
            raise ValueError(f"head dim {d_model}/{nhead} unsupported (attention kernel is built for 32 and 64)")
        if d_model % 128 != 0 or dim_ff % 128 != 0:
            raise ValueError("d_model and dim_feedforward must be multiples of 128")
        self.d, self.H, self.ff, self.n_layers, self.eps = d_model, nhead, dim_ff, n_layers, ln_eps

    # ------------------------------------------------------------------------------------------------ forward
    def forward(self, layers: List[LayerViews], x32: torch.Tensor, x16: torch.Tensor, cu: torch.Tensor, n_seqs: int,
                max_len: int, save: bool, layer_hook: Optional[Callable] = None, rowsum_from: int = 1 << 30,
                save_from: int = 0):
        """x32/x16: [M, d] fp32 residual stream and its bf16 copy.  Returns (x32, x16, saved list).
        layer_hook(i, x32, rowsum) is called after layer i (teacher target accumulation); rowsum is produced for
        layers i >= rowsum_from.  With `save`, layers i >= save_from keep what the backward needs and the saved list
        holds None for the layers below (a frozen prefix that `backward(stop_at=save_from)` never reaches).

        Every Linear writes its output as bf16 (what autocast makes it) through the TMA-store epilogue; the fp32
        residual sum y = x + bf16(Linear) is formed inside the LayerNorm kernel and never stored: the backward
        re-forms it from the saved (x, o) pair."""
        d, H, ff = self.d, self.H, self.ff
        M = x32.shape[0]
        dev = x32.device
        bf, f32 = torch.bfloat16, torch.float32
        saved = []
        keep_all = save
        for i, w in enumerate(layers):
            save = keep_all and i >= save_from
            if keep_all and not save:
                saved.append(None)
            qkv = _empty((M, 3 * d), bf, dev)
            ops.gemm(ops.plain_operand(x16), w.w_in, M, 1, qkv, bias=w.b_in)
            att = _empty((M, d), bf, dev)
            lse = _empty((M, H), f32, dev) if save else None
            ops.attn_fwd(qkv, cu, n_seqs, max_len, d, H, att, lse)
            o1 = _empty((M, d), bf, dev)
            ops.gemm(ops.plain_operand(att), w.w_o, M, 1, o1, bias=w.b_o)
            x1_32 = _empty((M, d), f32, dev)
            x1_16 = _empty((M, d), bf, dev)
            st1 = _empty((M, 2), f32, dev) if save else None
            ops.add_layernorm_fwd(x32, o1, w.g1, w.be1, self.eps, x1_32, x1_16, st1, None)
            g = _empty((M, ff), bf, dev)
            h = _empty((M, ff), bf, dev) if save else None
            ops.gemm(ops.plain_operand(x1_16), w.w1, M, 1, g, bias=w.b1, act=ops.ACT_GELU, out2=h)
            o2 = _empty((M, d), bf, dev)
            ops.gemm(ops.plain_operand(g), w.w2, M, 1, o2, bias=w.b2)
            x2_32 = _empty((M, d), f32, dev)
            x2_16 = _empty((M, d), bf, dev)
            st2 = _empty((M, 2), f32, dev) if save else None
            rowsum = _empty((M, 2), f32, dev) if i >= rowsum_from else None
            ops.add_layernorm_fwd(x1_32, o2, w.g2, w.be2, self.eps, x2_32, x2_16, st2, rowsum)
            if save:
                s = LayerSaved()
                s.x32, s.x16, s.qkv, s.att, s.lse, s.o1, s.st1, s.x1_32, s.x1_16, s.h, s.g, s.o2, s.st2 = \
                    x32, x16, qkv, att, lse, o1, st1, x1_32, x1_16, h, g, o2, st2
                saved.append(s)
            if layer_hook is not None:
                layer_hook(i, x2_32, rowsum)
            x32, x16 = x2_32, x2_16
        return x32, x16, saved

    def forward_tf32(self, layers: List[LayerViews], x32: torch.Tensor, xop: torch.Tensor, cu: torch.Tensor, n_seqs: int,
                     max_len: int, layer_hook: Optional[Callable] = None) -> torch.Tensor:
        """Inference forward at reference precision (the reference's fp32 feature extraction): the same packed layout,
        `layers` hold fp32 weight matrices rounded to nearest tf32.  x32: [M, d] fp32 residual stream, xop: its copy
        rounded to nearest tf32.  Returns the fp32 output of the last layer; layer_hook(i, x32) is called with the
        output of layer i (a buffer the stack does not write again).

        Every GEMM runs on the tf32 tensor cores with operands rounded to nearest as they are written (the tensor core
        would truncate raw fp32); attention keeps bf16 Q/K/V and P but writes O in fp32; the Linear outputs stay fp32
        into the residual add; GELU is the exact erf form."""
        d, H, ff = self.d, self.H, self.ff
        M = x32.shape[0]
        dev = x32.device
        bf, f32 = torch.bfloat16, torch.float32
        for i, w in enumerate(layers):
            qkv = _empty((M, 3 * d), bf, dev)
            ops.gemm_tf32(ops.plain_operand(xop), w.w_in, M, 1, qkv, bias=w.b_in)
            att = _empty((M, d), f32, dev)
            ops.attn_fwd_f32(qkv, cu, n_seqs, max_len, d, H, att)
            del qkv
            o1 = _empty((M, d), f32, dev)
            ops.gemm_tf32(ops.plain_operand(att), w.w_o, M, 1, o1, bias=w.b_o)
            del att
            x1_32 = _empty((M, d), f32, dev)
            x1_op = _empty((M, d), f32, dev)
            ops.add_layernorm_fwd_f32(x32, o1, w.g1, w.be1, self.eps, x1_32, x1_op)
            del o1
            g = _empty((M, ff), f32, dev)
            ops.gemm_tf32(ops.plain_operand(x1_op), w.w1, M, 1, g, bias=w.b1, act=ops.ACT_GELU_ERF, round_out=True)
            o2 = _empty((M, d), f32, dev)
            ops.gemm_tf32(ops.plain_operand(g), w.w2, M, 1, o2, bias=w.b2)
            del g
            x32 = _empty((M, d), f32, dev)
            xop = _empty((M, d), f32, dev)
            ops.add_layernorm_fwd_f32(x1_32, o2, w.g2, w.be2, self.eps, x32, xop)
            if layer_hook is not None:
                layer_hook(i, x32)
        return x32

    # ------------------------------------------------------------------------------------------------ backward
    def backward(self, layers: List[LayerViews], grads: List[LayerViews], saved: List[LayerSaved], dx: torch.Tensor,
                 cu: torch.Tensor, n_seqs: int, max_len: int, on_layer_done: Optional[Callable] = None,
                 stop_at: int = 0, need_dx: bool = True, need_wgrad: Optional[Sequence[bool]] = None,
                 inject: Optional[Callable] = None):
        """dx: fp32 [M, d] gradient w.r.t. the stack output (before any final norm), only read.  Accumulates parameter
        gradients into `grads` (pre-zeroed) and returns the gradient w.r.t. the stack input (fp32).

        inject(i, dx): called at the top of the iteration of every layer i below the last one, before its LayerNorm
        backward, with the fp32 half of the gradient w.r.t. layer i's output (a buffer of the stack); it may add a
        gradient of that output which reaches it from outside the stack (a returned hidden state).

        Between layers the gradient travels as a pair (fp32 residual branch, bf16 Linear data gradient -- bf16 is
        what autocast's Linear backward returns); the pair is summed inside the next LayerNorm backward.

        Layers below `stop_at` are not visited.  need_dx=False: nothing below the lowest visited layer wants its input
        gradient, so its last data-gradient GEMM is skipped and None is returned.  need_wgrad[i] False (a frozen layer):
        layer i runs its data-gradient chain only -- no weight-gradient GEMM, no LayerNorm, bias or attention-bias
        gradient; `grads[i]` is not touched and may be None.  The data gradients are the same bits either way."""
        d, H, ff = self.d, self.H, self.ff
        M = dx.shape[0]
        dev = dx.device
        bf, f32 = torch.bfloat16, torch.float32
        dx_b = None   # bf16 half of the gradient w.r.t. the current layer's output
        for i in range(len(layers) - 1, stop_at - 1, -1):
            w, gw, s = layers[i], grads[i], saved[i]
            wg = need_wgrad is None or need_wgrad[i]
            if inject is not None and dx_b is not None:
                inject(i, dx)
            # ---- LN2 and the MLP
            dy2 = _empty((M, d), f32, dev)
            dy2_16 = _empty((M, d), bf, dev)
            ops.add_layernorm_bwd(dx, dx_b, s.x1_32, s.o2, s.st2, w.g2, dy2, dy2_16,
                                  *((gw.g2, gw.be2, gw.b2) if wg else ()))
            if wg:
                ops.gemm_wgrad(ops.plain_operand(dy2_16), ops.plain_operand(s.g), M, 1, gw.w2, accumulate=True)
            dh = _empty((M, ff), bf, dev)
            ops.gemm_dgrad(ops.plain_operand(dy2_16), w.w2, M, 1, dh, K=d, N=ff, act=ops.ACT_DGELU, aux=s.h,
                           colsum=gw.b1 if wg else None)
            if wg:
                ops.gemm_wgrad(ops.plain_operand(dh), ops.plain_operand(s.x1_16), M, 1, gw.w1, accumulate=True)
            dx1_b = _empty((M, d), bf, dev)
            ops.gemm_dgrad(ops.plain_operand(dh), w.w1, M, 1, dx1_b, K=ff, N=d)
            del dh, dy2_16
            # ---- LN1 and the attention block
            dy1 = _empty((M, d), f32, dev)
            dy1_16 = _empty((M, d), bf, dev)
            ops.add_layernorm_bwd(dy2, dx1_b, s.x32, s.o1, s.st1, w.g1, dy1, dy1_16,
                                  *((gw.g1, gw.be1, gw.b_o) if wg else ()))
            del dy2, dx1_b
            if wg:
                ops.gemm_wgrad(ops.plain_operand(dy1_16), ops.plain_operand(s.att), M, 1, gw.w_o, accumulate=True)
            datt = _empty((M, d), bf, dev)
            ops.gemm_dgrad(ops.plain_operand(dy1_16), w.w_o, M, 1, datt, K=d, N=d)
            dqkv = _empty((M, 3 * d), bf, dev)
            ops.attn_bwd(s.qkv, s.att, datt, s.lse, cu, n_seqs, max_len, d, H, dqkv, dbias=gw.b_in if wg else None,
                         long_seq=True)
            if wg:
                ops.gemm_wgrad(ops.plain_operand(dqkv), ops.plain_operand(s.x16), M, 1, gw.w_in, accumulate=True)
            dx = dy1
            saved[i] = None
            if i == stop_at and not need_dx:
                if on_layer_done is not None:
                    on_layer_done(i)
                return None
            dx_b = _empty((M, d), bf, dev)
            ops.gemm_dgrad(ops.plain_operand(dqkv), w.w_in, M, 1, dx_b, K=3 * d, N=d)
            if on_layer_done is not None:
                on_layer_done(i)
        if not need_dx:
            return None
        if dx_b is not None:
            ops.add_bf16(dx, dx_b)
        return dx
