"""Python-side launchers for the C-ABI kernels (raw pointers + the current PyTorch CUDA stream).

PyTorch is used only for device memory and streams.  Every function here fails loudly if the CUDA library is
missing or a tensor is not on a CUDA device -- there is no eager fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import Epilogue, Operand, check

ACT_NONE, ACT_GELU, ACT_DGELU, ACT_BF16 = 0, 1, 2, 3
ACT_GELU_ERF = 4   # tf32 GEMM only: exact erf GELU in fp32


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.WavJepaLibError("wavjepa_b200 ops need CUDA tensors (no CPU fallback)")
    return t.data_ptr()


def make_operand(t: torch.Tensor, cols: int, rows: int, batch: int = 1, *, row_stride: Optional[int] = None,
                 batch_stride: Optional[int] = None, nq: int = 1, q_stride: Optional[int] = None,
                 seg_width: int = 0, seg_q: Sequence[int] = (), seg_p: Sequence[int] = (),
                 offset: int = 0) -> Operand:
    """4-D strided view (see wj_operand_t) of a bf16 tensor (wj_gemm_bf16) or an fp32 one (wj_gemm_tf32).  Strides are
    in ELEMENTS here."""
    assert t.dtype in (torch.bfloat16, torch.float32)
    esz = t.element_size()
    op = Operand()
    op.ptr = _ptr(t) + offset * esz
    row_stride = cols if row_stride is None else row_stride
    q_stride = row_stride if q_stride is None else q_stride
    batch_stride = rows * row_stride if batch_stride is None else batch_stride
    op.dim[0], op.dim[1], op.dim[2], op.dim[3] = cols, nq, rows, batch
    op.stride_bytes[0], op.stride_bytes[1], op.stride_bytes[2] = q_stride * esz, row_stride * esz, max(batch_stride, 8) * esz
    op.seg_width = seg_width
    for i, v in enumerate(seg_q):
        op.seg_q[i] = v
    for i, v in enumerate(seg_p):
        op.seg_p[i] = v
    return op


def plain_operand(t: torch.Tensor) -> Operand:
    """Row-major [M, K] matrix (last dim contiguous)."""
    assert t.dim() == 2 and t.stride(1) == 1
    return make_operand(t, t.shape[1], t.shape[0], 1, row_stride=t.stride(0))


def gemm(a: Operand, w: torch.Tensor, L: int, batch: int, out: torch.Tensor, *, K: Optional[int] = None,
         N: Optional[int] = None, ld_out: Optional[int] = None, out_offset: int = 0,
         bias: Optional[torch.Tensor] = None, act: int = ACT_NONE, out2: Optional[torch.Tensor] = None,
         ld_out2: Optional[int] = None, out2_offset: int = 0,
         resid: Optional[torch.Tensor] = None, ld_resid: Optional[int] = None, resid_mod: int = 0,
         resid_offset: int = 0, aux: Optional[torch.Tensor] = None, ld_aux: Optional[int] = None, aux_offset: int = 0,
         accumulate: bool = False, out_rows: Optional[torch.Tensor] = None, block_n: int = 0,
         colsum: Optional[torch.Tensor] = None) -> None:
    """out[b*L+t, :] = epilogue(A(t,b) @ w.T); w is bf16 [N, K] (row-major)."""
    assert w.dtype == torch.bfloat16 and w.stride(-1) == 1
    N = w.shape[0] if N is None else N
    K = w.shape[1] if K is None else K
    e = Epilogue()
    esz = out.element_size()
    e.out = _ptr(out) + out_offset * esz
    e.ld_out = out.stride(-2) if ld_out is None else ld_out
    e.out_f32 = 1 if out.dtype == torch.float32 else 0
    assert out.dtype in (torch.float32, torch.bfloat16)
    e.accumulate = 1 if accumulate else 0
    if out2 is not None:
        assert out2.dtype == torch.bfloat16
        e.out2 = _ptr(out2) + out2_offset * 2
        e.ld_out2 = out2.stride(-2) if ld_out2 is None else ld_out2
    if bias is not None:
        assert bias.dtype == torch.float32
        e.bias = _ptr(bias)
    if resid is not None:
        e.resid = _ptr(resid) + resid_offset * resid.element_size()
        e.resid_f32 = 1 if resid.dtype == torch.float32 else 0
        e.ld_resid = resid.stride(-2) if ld_resid is None else ld_resid
        e.resid_mod = resid_mod
    if aux is not None:
        assert aux.dtype == torch.bfloat16
        e.aux = _ptr(aux) + aux_offset * 2
        e.ld_aux = aux.stride(-2) if ld_aux is None else ld_aux
    e.act = act
    if out_rows is not None:
        assert out_rows.dtype == torch.int32
        e.out_rows = _ptr(out_rows)
    if colsum is not None:
        assert colsum.dtype == torch.float32
        e.colsum = _ptr(colsum)
    lib = _lib.load()
    if _lib._profile is not None:
        _lib._profile.meta = (2.0 * L * batch * N * K, L * batch, N, K, e.act, int(e.out_f32))
        _lib._profile.nbytes = (L * batch * K * 2 + N * K * 2 + L * batch * N * (esz + 2 * (out2 is not None)) +
                                (L * batch * N * resid.element_size() if resid is not None and resid_mod == 0 else 0) +
                                (L * batch * N * 2 if aux is not None else 0))
    check(lib.wj_gemm_bf16(C.byref(a), C.c_void_p(_ptr(w)), C.c_int64(w.stride(0)), L, batch, N, K, C.byref(e),
                           block_n, _stream()))


def gemm_tf32(a: Operand, w: torch.Tensor, L: int, batch: int, out: torch.Tensor, *, bias: Optional[torch.Tensor] = None,
              act: int = ACT_NONE, resid: Optional[torch.Tensor] = None, resid_mod: int = 0,
              round_out: bool = False) -> None:
    """out[b*L+t, :] = epilogue(A(t,b) @ w.T) on the tf32 tensor cores: A over an fp32 tensor, w fp32 [N, K], both
    already rounded to nearest tf32.  act: ACT_NONE or ACT_GELU_ERF; out bf16 or fp32 (round_out: rounded to nearest
    tf32, for an output that is the next GEMM's operand)."""
    assert w.dtype == torch.float32 and w.dim() == 2 and w.stride(-1) == 1
    assert out.dtype in (torch.float32, torch.bfloat16) and out.stride(-1) == 1
    N, K = w.shape
    e = Epilogue()
    e.out = _ptr(out)
    e.ld_out = out.stride(-2)
    e.out_f32 = 1 if out.dtype == torch.float32 else 0
    if bias is not None:
        assert bias.dtype == torch.float32
        e.bias = _ptr(bias)
    if resid is not None:
        assert resid.dtype == torch.float32 and resid.stride(-1) == 1
        e.resid = _ptr(resid)
        e.resid_f32 = 1
        e.ld_resid = resid.stride(-2)
        e.resid_mod = resid_mod
    e.act = act
    lib = _lib.load()
    if _lib._profile is not None:
        _lib._profile.meta = (2.0 * L * batch * N * K, L * batch, N, K, e.act, int(e.out_f32))
        _lib._profile.nbytes = L * batch * K * 4 + N * K * 4 + L * batch * N * out.element_size()
    check(lib.wj_gemm_tf32(C.byref(a), C.c_void_p(_ptr(w)), C.c_int64(w.stride(0)), L, batch, N, K, C.byref(e),
                           1 if round_out else 0, _stream()))


def gemm_wgrad(dy: Operand, x: Operand, L: int, batch: int, out: torch.Tensor, *, M: Optional[int] = None,
               N: Optional[int] = None, ld_out: Optional[int] = None, out_offset: int = 0, accumulate: bool = False,
               splits: int = 0) -> None:
    """out[m, n] (+)= sum_{b,t} dY[b,t,m] * X(n; t, b); out fp32 [M, N]."""
    assert out.dtype == torch.float32
    M = out.shape[0] if M is None else M
    N = out.shape[1] if N is None else N
    ld = out.stride(0) if ld_out is None else ld_out
    lib = _lib.load()
    if _lib._profile is not None:
        _lib._profile.meta = (2.0 * L * batch * M * N, L * batch, M, N, 0, 1)
        _lib._profile.nbytes = L * batch * (M + N) * 2 + M * N * 4
    check(lib.wj_gemm_wgrad_bf16(C.byref(dy), C.byref(x), L, batch, M, N, C.c_void_p(_ptr(out) + out_offset * 4),
                                 C.c_int64(ld), 1 if accumulate else 0, splits, _stream()))


_det_ws: Optional[torch.Tensor] = None


def set_deterministic(on: bool, workspace_bytes: int = 256 << 20, device=None) -> None:
    """Bit-reproducible reductions (wj_set_deterministic): per-block / per-split partial results in a workspace plus a
    fixed-order second pass instead of floating-point atomics.  Costs a few percent of step time; all calls must then be
    issued on one stream.  The reference has no equivalent switch (torch's own deterministic-algorithms flag is the
    closest); off by default."""
    global _det_ws
    lib = _lib.load()
    if not on:
        check(lib.wj_set_deterministic(None, C.c_size_t(0)))
        _det_ws = None
        return
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    _det_ws = torch.empty(workspace_bytes, dtype=torch.uint8, device=dev)
    check(lib.wj_set_deterministic(C.c_void_p(_det_ws.data_ptr()), C.c_size_t(workspace_bytes)))


def gemm_option(name: str, value: int) -> None:
    """Routing switch of the GEMM entry points (A/B measurements, tests): 'pair_wgrad' / 'pair_dgrad' = 1 (default) lets
    the weight- / data-gradient GEMMs use the CTA-pair kernel where the shape allows, 0 keeps them on single CTAs."""
    check(_lib.load().wj_gemm_option({"pair_wgrad": 1, "pair_dgrad": 2}[name], int(value)))


def gemm_dgrad(a: Operand, w: torch.Tensor, L: int, batch: int, out: torch.Tensor, *, K: int, N: int,
               w_col_offset: int = 0, w_cols: Optional[int] = None, seg_col_off: Sequence[int] = (),
               ld_out: Optional[int] = None, out_offset: int = 0, act: int = ACT_NONE,
               aux: Optional[torch.Tensor] = None, ld_aux: Optional[int] = None, aux_offset: int = 0,
               resid: Optional[torch.Tensor] = None, ld_resid: Optional[int] = None, resid_offset: int = 0,
               accumulate: bool = False, out_rows: Optional[torch.Tensor] = None, block_n: int = 0,
               colsum: Optional[torch.Tensor] = None) -> None:
    """out[b*L+t, n] = epilogue(sum_r A(r; t, b) * w[r, w_col_offset + seg_col_off[s] + n]); w bf16 [R, cols] row-major."""
    assert w.dtype == torch.bfloat16 and w.dim() == 2 and w.stride(1) == 1
    e = Epilogue()
    esz = out.element_size()
    e.out = _ptr(out) + out_offset * esz
    e.ld_out = out.stride(-2) if ld_out is None else ld_out
    e.out_f32 = 1 if out.dtype == torch.float32 else 0
    e.accumulate = 1 if accumulate else 0
    if resid is not None:
        e.resid = _ptr(resid) + resid_offset * resid.element_size()
        e.resid_f32 = 1 if resid.dtype == torch.float32 else 0
        e.ld_resid = resid.stride(-2) if ld_resid is None else ld_resid
    if aux is not None:
        assert aux.dtype == torch.bfloat16
        e.aux = _ptr(aux) + aux_offset * 2
        e.ld_aux = aux.stride(-2) if ld_aux is None else ld_aux
    e.act = act
    if out_rows is not None:
        e.out_rows = _ptr(out_rows)
    if colsum is not None:
        assert colsum.dtype == torch.float32
        e.colsum = _ptr(colsum)
    seg = (C.c_int32 * 4)(*([int(v) for v in seg_col_off] + [0] * (4 - len(seg_col_off))))
    w_cols = (w.shape[1] - w_col_offset) if w_cols is None else w_cols
    lib = _lib.load()
    if _lib._profile is not None:
        _lib._profile.meta = (2.0 * L * batch * N * K, L * batch, N, K, e.act, int(e.out_f32))
        _lib._profile.nbytes = (L * batch * K * 2 + N * K * 2 + L * batch * N * esz +
                                (L * batch * N * resid.element_size() if resid is not None else 0) +
                                (L * batch * N * 2 if aux is not None else 0))
    check(lib.wj_gemm_dgrad_bf16(C.byref(a), C.c_void_p(_ptr(w) + w_col_offset * 2), C.c_int64(w.stride(0)),
                                 w.shape[0], w_cols, seg, L, batch, N, K, C.byref(e), block_n, _stream()))


def conv_operand(x: torch.Tensor, k: int) -> Operand:
    """Implicit-GEMM view of channels-last activations x [B, L_in, C] (L_in even) for a stride-2 Conv1d of width k
    (reference nn.Conv1d(512,512,k,2), wavjepa/extractors/audio_feature_extractor.py:70): virtual column j*C + c of
    output row t is x[b, 2t + j, c] = pair-view (c, parity j&1, row t + j//2)."""
    B, L_in, C = x.shape
    if L_in % 2 != 0 or k not in (2, 3):
        raise _lib.WavJepaLibError(f"conv_operand: stride-2 implicit GEMM needs an even input length and k in (2,3); got L={L_in} k={k}")
    return make_operand(x, C, L_in // 2, B, nq=2, q_stride=C, row_stride=2 * C, batch_stride=L_in * C,
                        seg_width=C, seg_q=(0, 1, 0)[:k], seg_p=(0, 0, 1)[:k])


def conv_operand_odd(x: torch.Tensor, k: int) -> Operand:
    """Implicit-GEMM view of channels-last activations x [B, L_in, C] with L_in odd, for a stride-2 Conv1d of width k:
    output row t reads the k*C contiguous values x[b, 2t : 2t + k, :] (row pitch 2C, batch pitch L_in*C).  Every
    element it addresses lies inside x: for k = 2 the trailing row x[b, L_in - 1] is never read."""
    B, L_in, C = x.shape
    if L_in % 2 == 0 or k not in (2, 3):
        raise _lib.WavJepaLibError(f"conv_operand_odd: needs an odd input length and k in (2,3); got L={L_in} k={k}")
    L_out = (L_in - k) // 2 + 1
    return make_operand(x, k * C, L_out, B, row_stride=2 * C, batch_stride=L_in * C)


_conv_rows_cache: dict = {}


def _conv_rows(B: int, L_in: int, n: int, parity: int, device) -> torch.Tensor:
    """int32 [B * n]: physical row b*L_in + 2m + parity of logical output row b*n + m (odd-length conv_dgrad)."""
    key = (B, L_in, n, parity, str(device))
    t = _conv_rows_cache.get(key)
    if t is None:
        m = torch.arange(n, device=device, dtype=torch.int32)
        b = torch.arange(B, device=device, dtype=torch.int32)[:, None]
        t = (b * L_in + 2 * m[None, :] + parity).reshape(-1).contiguous()
        if len(_conv_rows_cache) >= 16:
            _conv_rows_cache.clear()
        _conv_rows_cache[key] = t
    return t


def conv_dgrad(dy: torch.Tensor, wk: torch.Tensor, dx: torch.Tensor, k: int, *, act: int = ACT_NONE,
               aux: Optional[torch.Tensor] = None) -> None:
    """Data gradient of the stride-2 Conv1d: dy [B, L_out, O] bf16, wk [O, k*C] bf16 (k-major), dx [B, L_in, C].
    Even input positions 2m receive taps j=0 (t=m) and j=2 (t=m-1); odd positions 2m+1 receive tap j=1 (t=m):
    two GEMMs over (shifted) views of dy, written with row pitch 2C.  act/aux: optional x aux epilogue
    (aux = GELU' of the layer below saved by its forward epilogue, same layout as dx).

    Odd L_in: the batch pitch L_in*C is not a multiple of the 2C row pitch, so both GEMMs write (and read aux) through
    an explicit output-row index (the generic epilogue).  For k = 2 the trailing row L_in - 1 feeds no output: it is
    written with zeros."""
    B, L_out, O = dy.shape
    _, L_in, C = dx.shape
    assert dy.is_contiguous() and dx.is_contiguous() and wk.shape == (O, k * C)
    taps_even = (0, 2) if k == 3 else (0,)
    a_even = make_operand(dy, O, L_out, B, seg_width=O, seg_q=(0,) * len(taps_even), seg_p=(0, -1)[:len(taps_even)])
    a_odd = make_operand(dy, O, L_out, B, seg_width=O, seg_q=(0,), seg_p=(0,))
    if L_in % 2 != 0:
        assert aux is None or (aux.is_contiguous() and aux.shape == dx.shape)
        n_even = L_out + 1 if k == 3 else L_out     # k = 3: row L_in - 1 = 2 L_out receives tap 2 of t = L_out - 1
        n_odd = L_out
        kw = dict(ld_out=C, act=act, aux=aux, ld_aux=C)
        gemm_dgrad(a_even, wk, n_even, B, dx, K=len(taps_even) * O, N=C, seg_col_off=[j * C for j in taps_even],
                   out_rows=_conv_rows(B, L_in, n_even, 0, dx.device), **kw)
        gemm_dgrad(a_odd, wk, n_odd, B, dx, K=O, N=C, seg_col_off=[C], out_rows=_conv_rows(B, L_in, n_odd, 1, dx.device),
                   **kw)
        if k == 2:
            dx[:, L_in - 1].zero_()
        return
    half = L_in // 2
    kw = dict(ld_out=2 * C, act=act, aux=aux, ld_aux=2 * C)
    gemm_dgrad(a_even, wk, half, B, dx, K=len(taps_even) * O, N=C, seg_col_off=[j * C for j in taps_even],
               out_offset=0, aux_offset=0, **kw)
    gemm_dgrad(a_odd, wk, half, B, dx, K=O, N=C, seg_col_off=[C], out_offset=C, aux_offset=C, **kw)


# ----------------------------------------------------------------------------------------------------- masks
def masks_generate(kind: int, batch: int, n_times: int, in_channels: int, channel_based: bool, n_targets: int,
                   ctx_prob: float, ctx_len: int, tgt_prob: float, tgt_len: int, cutoff: float, min_context_len: int,
                   base_seed: int, row0: int, device):
    T = n_times // in_channels
    t_out = n_times if channel_based else T
    ctx = torch.empty(batch, t_out, dtype=torch.bool, device=device)
    tgt = torch.empty(batch, n_targets, t_out, dtype=torch.bool, device=device)
    vis = torch.empty(batch, n_targets, t_out, dtype=torch.bool, device=device)
    attempts = torch.zeros(batch, dtype=torch.int32, device=device)
    err = torch.zeros(1, dtype=torch.int32, device=device)
    lib = _lib.load()
    check(lib.wj_masks_generate(kind, batch, n_times, in_channels, 1 if channel_based else 0, n_targets,
                                C.c_double(ctx_prob), ctx_len, C.c_double(tgt_prob), tgt_len, C.c_float(cutoff),
                                min_context_len, C.c_uint32(base_seed & 0xFFFFFFFF), C.c_uint32(row0 & 0xFFFFFFFF),
                                C.c_void_p(_ptr(ctx)), C.c_void_p(_ptr(tgt)), C.c_void_p(_ptr(vis)),
                                C.c_void_p(_ptr(attempts)), C.c_void_p(_ptr(err)), _stream()))
    return ctx, tgt, vis, attempts, err


class MaskIndex:
    """Packed index lists built by wj_mask_indices (all int32, on device) + host-side totals."""
    __slots__ = ("B", "G", "T", "n_c", "n_v", "n_t", "cu_c", "cu_v", "cu_t", "totals", "ctx_rows", "vis_src",
                 "vis_pos", "tgt_vrow", "tgt_trow", "Nc", "Nv", "Nt", "max_nc", "max_nv")


def mask_indices(ctx_hidden: torch.Tensor, tgt: torch.Tensor, vis_hidden: torch.Tensor) -> MaskIndex:
    """ctx_hidden [B,T] bool, tgt [B,G,T] bool, vis_hidden [B,G,T] bool.  One small D2H copy (the totals)."""
    assert ctx_hidden.dtype == torch.bool and tgt.dtype == torch.bool and vis_hidden.dtype == torch.bool
    ctx_hidden, tgt, vis_hidden = ctx_hidden.contiguous(), tgt.contiguous(), vis_hidden.contiguous()
    B, T = ctx_hidden.shape
    G = tgt.shape[1]
    dev = ctx_hidden.device
    mi = MaskIndex()
    mi.B, mi.G, mi.T = B, G, T
    i32 = dict(dtype=torch.int32, device=dev)
    mi.n_c = torch.empty(B, **i32); mi.n_v = torch.empty(B * G, **i32); mi.n_t = torch.empty(B * G, **i32)
    mi.cu_c = torch.empty(B + 1, **i32); mi.cu_v = torch.empty(B * G + 1, **i32); mi.cu_t = torch.empty(B * G + 1, **i32)
    mi.totals = torch.empty(8, **i32)
    mi.ctx_rows = torch.empty(B * T, **i32)
    mi.vis_src = torch.empty(B * G * T, **i32); mi.vis_pos = torch.empty(B * G * T, **i32)
    mi.tgt_vrow = torch.empty(B * G * T, **i32); mi.tgt_trow = torch.empty(B * G * T, **i32)
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_mask_indices(p(ctx_hidden), p(tgt), p(vis_hidden), B, G, T, p(mi.n_c), p(mi.n_v), p(mi.n_t),
                              p(mi.cu_c), p(mi.cu_v), p(mi.cu_t), p(mi.totals), p(mi.ctx_rows), p(mi.vis_src),
                              p(mi.vis_pos), p(mi.tgt_vrow), p(mi.tgt_trow), _stream()))
    tot = mi.totals.tolist()  # the one host sync of the step: grid sizes of the varlen kernels
    mi.Nc, mi.Nv, mi.Nt, viol, mi.max_nc, mi.max_nv = tot[0], tot[1], tot[2], tot[3], tot[4], tot[5]
    if viol:
        raise _lib.WavJepaLibError(f"{viol} target positions are hidden from the predictor (ctx_and_target_masks); "
                                   "unsupported by the packed path")
    return mi


# ----------------------------------------------------------------------------------------------------- conv0
def conv0_workspaces(B: int, Cin: int, C: int, device, backward: bool = False):
    """(moments fp64 [B, n], stats fp32 [B, C, 2][, red_scratch fp64 [B, 2 + Cin*10, C]]) for conv0_fwd / conv0_bwd."""
    n = int(_lib.load().wj_conv0_moment_count(Cin))
    mom = torch.empty(B, n, device=device, dtype=torch.float64)
    stats = torch.empty(B, C, 2, device=device, dtype=torch.float32)
    if backward:
        return mom, stats, torch.empty(B, 2 + Cin * 10, C, device=device, dtype=torch.float64)
    return mom, stats


def conv0_fwd(x: torch.Tensor, w: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, out: torch.Tensor,
              moments: torch.Tensor, stats: torch.Tensor, k: int = 10, stride: int = 5, eps: float = 1e-5) -> None:
    """Conv1d(Cin->C, 10, 5) + GroupNorm(C, C) + GELU -> out [B, L_out, C] bf16; moments / stats feed the backward."""
    B, Cin, L = x.shape
    assert x.dtype == torch.bfloat16 and x.is_contiguous() and w.dtype == torch.float32
    assert moments.dtype == torch.float64 and stats.dtype == torch.float32
    lib = _lib.load()
    if _lib._profile is not None:
        L_out = (L - k) // stride + 1
        _lib._profile.nbytes = B * (Cin * L * 2 + L_out * w.shape[0] * 2)
    check(lib.wj_conv0_gn_gelu_fwd(C.c_void_p(_ptr(x)), C.c_void_p(_ptr(w)), C.c_void_p(_ptr(gamma)),
                                   C.c_void_p(_ptr(beta)), B, Cin, L, w.shape[0], k, stride, C.c_float(eps),
                                   C.c_void_p(_ptr(moments)), C.c_void_p(_ptr(stats)), C.c_void_p(_ptr(out)),
                                   None, _stream()))


def conv0_fwd_f32(x: torch.Tensor, w: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, out: torch.Tensor,
                  moments: torch.Tensor, stats: torch.Tensor, k: int = 10, stride: int = 5, eps: float = 1e-5) -> None:
    """conv0_fwd of the TF32 inference path: x fp32 [B, Cin, L], unrounded fp32 weights, exact GELU -> out fp32
    [B, L_out, C] rounded to nearest tf32."""
    B, Cin, L = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous() and w.dtype == torch.float32
    assert out.dtype == torch.float32 and out.is_contiguous()
    assert moments.dtype == torch.float64 and stats.dtype == torch.float32
    lib = _lib.load()
    if _lib._profile is not None:
        L_out = (L - k) // stride + 1
        _lib._profile.nbytes = B * (Cin * L * 4 + L_out * w.shape[0] * 4)
    check(lib.wj_conv0_gn_gelu_fwd_f32(C.c_void_p(_ptr(x)), C.c_void_p(_ptr(w)), C.c_void_p(_ptr(gamma)),
                                       C.c_void_p(_ptr(beta)), B, Cin, L, w.shape[0], k, stride, C.c_float(eps),
                                       C.c_void_p(_ptr(moments)), C.c_void_p(_ptr(stats)), C.c_void_p(_ptr(out)),
                                       _stream()))


def conv0_bwd(x, w, gamma, beta, moments, stats, dy, red_scratch, dw, dgamma, dbeta, k: int = 10, stride: int = 5,
              eps: float = 1e-5) -> None:
    """Backward of conv0_fwd from dy (bf16 [B, L_out, C]); GELU' is recomputed from x, nothing else is read."""
    B, Cin, L = x.shape
    assert red_scratch.dtype == torch.float64 and red_scratch.numel() >= B * (2 + Cin * 10) * w.shape[0]
    assert dy.dtype == torch.bfloat16 and dy.is_contiguous()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.nbytes = B * Cin * L * 2 + dy.numel() * 2
    check(lib.wj_conv0_gn_gelu_bwd(p(x), p(w), p(gamma), p(beta), B, Cin, L, w.shape[0], k, stride, C.c_float(eps),
                                   p(moments), p(stats), p(dy), None, p(red_scratch), p(dw), p(dgamma), p(dbeta),
                                   _stream()))


# ----------------------------------------------------------------------------------------------------- norms
def layernorm_fwd(x: torch.Tensor, gamma, beta, eps: float, out_f32=None, out_bf16=None, stats=None, rowsum=None):
    M, D = x.shape
    assert x.is_contiguous()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, M, D, str(x.dtype)[6:], out_f32 is not None, out_bf16 is not None)
        _lib._profile.nbytes = M * D * (x.element_size() + 4 * (out_f32 is not None) + 2 * (out_bf16 is not None))
    check(lib.wj_layernorm_fwd(p(x), 1 if x.dtype == torch.bfloat16 else 0, p(gamma), p(beta), C.c_float(eps), M, D,
                               p(out_f32), p(out_bf16), p(stats), p(rowsum), _stream()))


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, stats, gamma, dx_f32=None, dx_bf16=None, dgamma=None, dbeta=None,
                  colsum=None):
    M, D = x.shape
    assert dy.dtype == torch.float32 and dy.is_contiguous() and x.is_contiguous()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, M, D, colsum is not None)
        _lib._profile.nbytes = M * D * (4 + x.element_size() + 4 * (dx_f32 is not None) + 2 * (dx_bf16 is not None))
    check(lib.wj_layernorm_bwd(p(dy), p(x), 1 if x.dtype == torch.bfloat16 else 0, p(stats), p(gamma), M, D, p(dx_f32),
                               p(dx_bf16), p(dgamma), p(dbeta), p(colsum), _stream()))


def add_layernorm_fwd(x: torch.Tensor, add: Optional[torch.Tensor], gamma, beta, eps: float, out_f32=None, out_bf16=None,
                      stats=None, rowsum=None):
    """LayerNorm(x + add): x fp32 residual stream, add bf16 (the Linear output as autocast rounds it) or None."""
    M, D = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous()
    assert add is None or (add.dtype == torch.bfloat16 and add.is_contiguous() and add.shape == x.shape)
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, M, D, add is not None, out_f32 is not None, out_bf16 is not None)
        _lib._profile.nbytes = M * D * (4 + 2 * (add is not None) + 4 * (out_f32 is not None) + 2 * (out_bf16 is not None))
    check(lib.wj_add_layernorm_fwd(p(x), p(add), p(gamma), p(beta), C.c_float(eps), M, D, p(out_f32), p(out_bf16),
                                   p(stats), p(rowsum), _stream()))


def add_layernorm_fwd_f32(x: torch.Tensor, add: Optional[torch.Tensor], gamma, beta, eps: float, out_f32=None,
                          out_tf32=None):
    """LayerNorm(x + add) of the TF32 inference path: x and add fp32 (add may be None); out_f32 unrounded, out_tf32 the
    same values rounded to nearest tf32 (the next GEMM's operand)."""
    M, D = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous()
    assert add is None or (add.dtype == torch.float32 and add.is_contiguous() and add.shape == x.shape)
    for o in (out_f32, out_tf32):
        assert o is None or (o.dtype == torch.float32 and o.is_contiguous() and o.shape == x.shape)
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.nbytes = M * D * (4 + 4 * (add is not None) + 4 * (out_f32 is not None) + 4 * (out_tf32 is not None))
    check(lib.wj_add_layernorm_fwd_f32(p(x), p(add), p(gamma), p(beta), C.c_float(eps), M, D, p(out_f32), p(out_tf32),
                                       _stream()))


def tf32_round(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x (fp32) rounded to nearest tf32 (into `out`, which may be x)."""
    assert x.dtype == torch.float32 and x.is_contiguous()
    out = torch.empty_like(x) if out is None else out
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == x.numel()
    check(_lib.load().wj_tf32_round(C.c_void_p(_ptr(x)), C.c_void_p(_ptr(out)), C.c_int64(x.numel()), _stream()))
    return out


def add_layernorm_bwd(dy_f32: Optional[torch.Tensor], dy_bf16: Optional[torch.Tensor], x: torch.Tensor,
                      add: Optional[torch.Tensor], stats, gamma, dx_f32=None, dx_bf16=None, dgamma=None, dbeta=None,
                      colsum=None):
    """Backward of add_layernorm_fwd; the output gradient is dy_f32 + dy_bf16 (either may be None)."""
    M, D = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous()
    assert dy_f32 is None or (dy_f32.dtype == torch.float32 and dy_f32.is_contiguous())
    assert dy_bf16 is None or (dy_bf16.dtype == torch.bfloat16 and dy_bf16.is_contiguous())
    assert add is None or (add.dtype == torch.bfloat16 and add.is_contiguous())
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, M, D, dy_f32 is not None, dy_bf16 is not None, colsum is not None)
        _lib._profile.nbytes = M * D * (4 * (dy_f32 is not None) + 2 * (dy_bf16 is not None) + 4 + 2 * (add is not None) +
                                        4 * (dx_f32 is not None) + 2 * (dx_bf16 is not None))
    check(lib.wj_add_layernorm_bwd(p(dy_f32), p(dy_bf16), p(x), p(add), p(stats), p(gamma), M, D, p(dx_f32), p(dx_bf16),
                                   p(dgamma), p(dbeta), p(colsum), _stream()))


def add_bf16(a: torch.Tensor, b: torch.Tensor):
    """a (fp32) += b (bf16), in place."""
    assert a.dtype == torch.float32 and b.dtype == torch.bfloat16 and a.numel() == b.numel()
    assert a.is_contiguous() and b.is_contiguous()
    lib = _lib.load()
    check(lib.wj_add_bf16(C.c_void_p(_ptr(a)), C.c_void_p(_ptr(b)), C.c_int64(a.numel()), _stream()))


def crop_norm(audio: torch.Tensor, starts: Optional[torch.Tensor], crops_per_clip: int, crop_len: int,
              out_bf16=None, out_f32=None, gain: Optional[torch.Tensor] = None):
    n_clips, ch, clip_len = audio.shape
    assert audio.dtype == torch.float32 and audio.is_contiguous()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:   # crop read 3x by design? no: algorithmic = read the crops once, write them once
        n_out = n_clips * crops_per_clip * ch * crop_len
        _lib._profile.nbytes = n_out * (4 + 2 * (out_bf16 is not None) + 4 * (out_f32 is not None))
    check(lib.wj_crop_norm(p(audio), p(starts), p(gain), n_clips, ch, C.c_int64(clip_len), crops_per_clip, crop_len,
                           p(out_bf16), p(out_f32), _stream()))


def clip_gain(audio: torch.Tensor, target_dbfs: float = -14.0) -> torch.Tensor:
    n_clips, ch, clip_len = audio.shape
    assert audio.dtype == torch.float32 and audio.is_contiguous()
    gain = torch.empty(n_clips, device=audio.device, dtype=torch.float32)
    lib = _lib.load()
    check(lib.wj_clip_gain(C.c_void_p(_ptr(audio)), n_clips, ch, C.c_int64(clip_len), C.c_float(target_dbfs),
                           C.c_void_p(_ptr(gain)), _stream()))
    return gain


def scatter_rows(src: torch.Tensor, idx: torch.Tensor, N: int, out: torch.Tensor):
    assert src.dtype == torch.float32 and out.dtype == torch.float32 and idx.dtype == torch.int32
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_scatter_rows(p(src), p(idx), N, src.shape[-1], p(out), _stream()))


def target_accum(x: torch.Tensor, rowsum, B: int, T: int, D: int, scale: float, first: bool, inst_stats, targets,
                 eps: float = 1e-5):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:   # read x, read-modify-write targets (write only for the first layer)
        _lib._profile.nbytes = B * T * D * (4 + (4 if first else 8))
    check(lib.wj_target_accum(p(x), p(rowsum), B, T, D, C.c_float(eps), C.c_float(scale), 1 if first else 0,
                              p(inst_stats), p(targets), _stream()))


def target_combine(xs, rowsums, B: int, T: int, D: int, scale: float, inst_stats, targets, eps: float = 1e-5):
    """targets = scale * sum_l instance_norm(xs[l]) over all layers in one pass (JEPA._make_targets, wavjepa/jepa.py:230-253)."""
    n = len(xs)
    assert n == len(rowsums) and inst_stats.numel() >= n * B * 2
    lib = _lib.load()
    px = (C.c_void_p * n)(*[_ptr(t) for t in xs])
    pr = (C.c_void_p * n)(*[_ptr(t) for t in rowsums])
    if _lib._profile is not None:
        _lib._profile.nbytes = B * T * D * 4 * (n + 1)
    check(lib.wj_target_combine(px, pr, n, B, T, D, C.c_float(eps), C.c_float(scale), C.c_void_p(_ptr(inst_stats)),
                                C.c_void_p(_ptr(targets)), _stream()))


# ----------------------------------------------------------------------------------------------------- attention
def attn_fwd(qkv: torch.Tensor, cu: torch.Tensor, n_seqs: int, max_len: int, D: int, H: int, out: torch.Tensor,
             lse2=None):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, n_seqs, max_len, D, H, qkv.shape[0])
    check(lib.wj_attn_varlen_fwd(p(qkv), p(cu), n_seqs, max_len, C.c_int64(qkv.shape[0]), D, H, p(out), p(lse2), _stream()))


def attn_fwd_f32(qkv: torch.Tensor, cu: torch.Tensor, n_seqs: int, max_len: int, D: int, H: int, out: torch.Tensor):
    """attn_fwd with O written as fp32 rounded to nearest tf32 (head dim 64, <= 512 tokens)."""
    assert out.dtype == torch.float32 and out.is_contiguous()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, n_seqs, max_len, D, H, qkv.shape[0])
    check(lib.wj_attn_varlen_fwd_f32out(p(qkv), p(cu), n_seqs, max_len, C.c_int64(qkv.shape[0]), D, H, p(out),
                                        _stream()))


def attn_bwd(qkv, out, dout, lse2, cu, n_seqs: int, max_len: int, D: int, H: int, dqkv, dbias=None,
             long_seq: bool = False):
    """dbias (optional, fp32 [3 D]) += column sums of dqkv: the in_proj bias gradient, formed in the kernel's epilogue.
    long_seq: also take head-dim-64 sequences of 385..400 tokens (wj_attn_varlen_bwd_bias_long), which the plain entry
    point refuses."""
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, n_seqs, max_len, D, H, qkv.shape[0])
    assert dbias is None or (dbias.dtype == torch.float32 and dbias.numel() == 3 * D)
    fn = lib.wj_attn_varlen_bwd_bias_long if long_seq else lib.wj_attn_varlen_bwd_bias
    check(fn(p(qkv), p(out), p(dout), p(lse2), p(cu), n_seqs, max_len, C.c_int64(qkv.shape[0]), D, H, p(dqkv), p(dbias),
             _stream()))


# ----------------------------------------------------------------------------------------------------- misc
def gather_rows(src: torch.Tensor, idx: Optional[torch.Tensor], N: int, out_f32=None, out_bf16=None):
    D = src.shape[-1]
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_gather_rows(p(src), 1 if src.dtype == torch.bfloat16 else 0, p(idx), N, D, p(out_f32), p(out_bf16),
                             _stream()))


def scatter_dgelu(src: torch.Tensor, idx: torch.Tensor, h: Optional[torch.Tensor], N: int, out_bf16: torch.Tensor):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_scatter_dgelu(p(src), p(idx), p(h), N, src.shape[-1], p(out_bf16), _stream()))


def predictor_assemble(ctx_bf16, mask_token, pos, vis_src, vis_pos, N: int, D: int, out_f32, out_bf16):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_predictor_assemble(p(ctx_bf16), p(mask_token), p(pos), p(vis_src), p(vis_pos), N, D, p(out_f32),
                                    p(out_bf16), _stream()))


def predictor_assemble_bwd(dx0, vis_src, N: int, D: int, d_ctx, d_mask_token):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_predictor_assemble_bwd(p(dx0), p(vis_src), N, D, p(d_ctx), p(d_mask_token), _stream()))


def predictor_ctx_grad(dx0, vis_src, cu_v, n_seqs: int, G: int, Nc: int, D: int, d_ctx_f32=None, d_ctx_bf16=None):
    """d_ctx[s] = sum over the G target groups (fixed order) of the predictor-input gradient rows that copy context row s
    (the context part of predictor_assemble_bwd, without atomics).  Either output may be None."""
    assert dx0.dtype == torch.float32 and dx0.is_contiguous()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    ws = torch.empty(Nc * G, device=dx0.device, dtype=torch.int32)
    check(lib.wj_predictor_ctx_grad(p(dx0), p(vis_src), p(cu_v), n_seqs, G, Nc, D, p(ws), p(d_ctx_f32), p(d_ctx_bf16),
                                    _stream()))


def masked_mse(pred_bf16, targets, tgt_rows, Nt: int, D: int, loss, dpred_bf16=None):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.nbytes = Nt * D * (2 + 4 + 2 * (dpred_bf16 is not None))
    check(lib.wj_masked_mse(p(pred_bf16), p(targets), p(tgt_rows), Nt, D, p(loss), p(dpred_bf16), _stream()))


def ema_update(teacher_flat: torch.Tensor, student_flat: torch.Tensor, decay: float):
    assert teacher_flat.numel() == student_flat.numel()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.nbytes = teacher_flat.numel() * 12
    check(lib.wj_ema_update(p(teacher_flat), p(student_flat), C.c_int64(teacher_flat.numel()), C.c_double(decay),
                            _stream()))


def sumsq(x: torch.Tensor, scale: float, out_f64: torch.Tensor):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.nbytes = x.numel() * 4
    check(lib.wj_sumsq(p(x), C.c_int64(x.numel()), C.c_float(scale), p(out_f64), _stream()))


def adamw_step(p_, g, m, v, lr, beta1, beta2, eps, wd, step, grad_scale=1.0, max_norm=0.0, grad_sumsq=None, p_bf16=None):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.nbytes = p_.numel() * (28 + 2 * (p_bf16 is not None))
    check(lib.wj_adamw_step(p(p_), p(g), p(m), p(v), C.c_int64(p_.numel()), C.c_float(lr), C.c_float(beta1),
                            C.c_float(beta2), C.c_float(eps), C.c_float(wd), int(step), C.c_float(grad_scale),
                            C.c_float(max_norm), p(grad_sumsq), p(p_bf16), _stream()))


def adamw_ema_step(p_, g, m, v, lr, beta1, beta2, eps, wd, step, grad_scale, max_norm, grad_sumsq, p_bf16, teacher,
                   teacher_bf16, ema_lo: int, ema_hi: int, ema_decay: float):
    """adamw_step with the EMA teacher update (pre-step student values of p_[ema_lo:ema_hi]) folded into the same pass."""
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    assert teacher.numel() == ema_hi - ema_lo
    if _lib._profile is not None:   # p, m, v read+write, g read, bf16 copy; teacher read+write + bf16 copy
        _lib._profile.nbytes = p_.numel() * (28 + 2 * (p_bf16 is not None)) + teacher.numel() * (8 + 2 * (teacher_bf16 is not None))
    check(lib.wj_adamw_ema_step(p(p_), p(g), p(m), p(v), C.c_int64(p_.numel()), C.c_float(lr), C.c_float(beta1),
                                C.c_float(beta2), C.c_float(eps), C.c_float(wd), int(step), C.c_float(grad_scale),
                                C.c_float(max_norm), p(grad_sumsq), p(p_bf16), p(teacher), p(teacher_bf16),
                                C.c_int64(ema_lo), C.c_int64(ema_hi), C.c_double(ema_decay), _stream()))


def cast_bf16(x: torch.Tensor, y: torch.Tensor):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_cast_bf16(p(x), p(y), C.c_int64(x.numel()), _stream()))


def colsum(x: torch.Tensor, out: torch.Tensor, M: Optional[int] = None):
    M = x.shape[0] if M is None else M
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    if _lib._profile is not None:
        _lib._profile.meta = (0.0, M, x.shape[1], str(x.dtype)[6:])
        _lib._profile.nbytes = M * x.shape[1] * x.element_size()
    check(lib.wj_colsum(p(x), 1 if x.dtype == torch.bfloat16 else 0, C.c_int64(M), x.shape[1], C.c_int64(x.stride(0)),
                        p(out), _stream()))


def scale_bf16(x: torch.Tensor, scale_dev: torch.Tensor):
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_scale_bf16(p(x), p(scale_dev), C.c_int64(x.numel()), _stream()))


# ----------------------------------------------------------------------------------------------------- input pipeline
def resample_sinc(x: torch.Tensor, table_t: torch.Tensor, orig: int, new: int, width: int, target_length: int,
                  out_row: torch.Tensor, sumsq_slot: torch.Tensor):
    """x [L] fp32 -> out_row [cap] fp32 (resampled, zero-padded / cropped), sumsq_slot [1] fp64 += sum of squares."""
    assert x.dtype == torch.float32 and x.is_contiguous() and out_row.dtype == torch.float32 and out_row.is_contiguous()
    assert table_t.dtype == torch.float32 and table_t.is_contiguous() and table_t.shape == (2 * width + orig, new)
    assert sumsq_slot.dtype == torch.float64
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_resample_sinc(p(x), C.c_int64(x.numel()), p(table_t), orig, new, width, C.c_int64(target_length),
                               p(out_row), C.c_int64(out_row.numel()), p(sumsq_slot), _stream()))


def rms_gain_rows(clips: torch.Tensor, sumsq: torch.Tensor, counts: torch.Tensor, target_dbfs: float = -14.0):
    assert clips.dtype == torch.float32 and clips.dim() == 2 and clips.is_contiguous()
    assert sumsq.dtype == torch.float64 and counts.dtype == torch.int64
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_rms_gain_rows(p(clips), p(sumsq), p(counts), clips.shape[0], C.c_int64(clips.shape[1]),
                               C.c_float(target_dbfs), _stream()))


# ----------------------------------------------------------------------------------------------------- denoiser stage
def mse_pair(pred: torch.Tensor, target: torch.Tensor, alpha: float, sums_f64: torch.Tensor, dpred=None):
    """pred fp32 [2, M] (clean half, generated half), target fp32 [M]; sums_f64 [2] += squared-error sums."""
    assert pred.dtype == torch.float32 and target.dtype == torch.float32 and sums_f64.dtype == torch.float64
    M = target.numel()
    assert pred.numel() == 2 * M and pred.is_contiguous() and target.is_contiguous()
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_mse_pair(p(pred), p(target), C.c_int64(M), C.c_float(alpha), p(sums_f64), p(dpred), _stream()))


def snr_mix(source: torch.Tensor, noise: torch.Tensor, start: torch.Tensor, length: torch.Tensor, snr: torch.Tensor,
            out: torch.Tensor):
    """source, noise, out fp32 [B, T]; start, length int32 [B]; snr fp32 [B]."""
    B, T = source.shape
    assert source.dtype == torch.float32 and noise.shape == source.shape and source.is_contiguous() and noise.is_contiguous()
    assert start.dtype == torch.int32 and length.dtype == torch.int32 and snr.dtype == torch.float32
    energy = torch.empty(B, 2, device=source.device, dtype=torch.float64)
    lib = _lib.load()
    p = lambda t: C.c_void_p(_ptr(t))
    check(lib.wj_snr_mix(p(source), p(noise), p(start), p(length), p(snr), B, C.c_int64(T), p(energy), p(out), _stream()))
    return energy
