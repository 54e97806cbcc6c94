"""Deterministic mode (ops.set_deterministic) at the kernel level on the B200: every entry point whose reduction would end
in floating-point atomics takes the workspace + fixed-order path instead.  Each test checks that path

  (a) against a plain fp64 torch restatement of the operation,
  (b) for bit-identical results across two runs on a NaN-poisoned workspace (0xFF bytes are NaN as fp32 and as fp64, so a
      partial slot that is read without being written poisons the result) and one run on a finite-poisoned one (0x7F
      bytes: huge finite values), so the result cannot depend on stale workspace contents, and
  (c) against the default (atomic) mode: summation-order tolerance, or exact equality where no atomics touch the output.

Reduction destinations are pre-filled with a random tensor wherever the API says `+=`; overwrite destinations with NaN."""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import wavjepa_b200 as w  # noqa: E402
from wavjepa_b200 import _lib, ops  # noqa: E402
from oracle import inputs as oi  # noqa: E402
from oracle import jepa_oracle as jo  # noqa: E402

DEV = "cuda"
BF16_TOL = 4e-3   # rel-L2 of a bf16-rounded result against fp32 (bf16 eps = 3.9e-3, rel-L2 of rounding ~1.7e-3)
NAN = float("nan")


def rel(a, b):
    a = a.double()
    b = b.double()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def rel_acc(out, pre, ref):
    """Error of an accumulating output (out = pre + ref) relative to the accumulated part alone."""
    ref = ref.double()
    return ((out.double() - pre.double() - ref).norm() / (ref.norm() + 1e-30)).item()


@pytest.fixture(autouse=True, scope="module")
def _device():
    _lib.require_device()
    torch.manual_seed(0)


@contextlib.contextmanager
def det_mode(nbytes=256 << 20, fill=0xFF):
    """Deterministic mode with a workspace whose every byte is `fill` on entry; always switched off on exit."""
    ops.set_deterministic(True, nbytes)
    try:
        ops._det_ws.fill_(fill)
        yield
    finally:
        ops.set_deterministic(False)


def det_runs(fn, nbytes=256 << 20):
    """fn() -> tuple of output tensors (fresh, pre-filled buffers).  Runs it twice on a NaN-poisoned workspace and once on
    a finite-poisoned one; all three runs must agree bit for bit.  Returns the first run's outputs."""
    runs = []
    for fill in (0xFF, 0xFF, 0x7F):
        with det_mode(nbytes, fill):
            runs.append(fn())
    for other in runs[1:]:
        for a, b in zip(runs[0], other):
            assert torch.equal(a, b)
    return runs[0]


def assert_refused(call):
    with pytest.raises(_lib.WavJepaLibError, match="too small"):
        call()


@contextlib.contextmanager
def pair_wgrad(on):
    ops.gemm_option("pair_wgrad", 1 if on else 0)
    try:
        yield
    finally:
        ops.gemm_option("pair_wgrad", 1)


# ------------------------------------------------------------------------------------------------------- weight gradient
WGRAD_SHAPES = [(1000, 256, 384, 0), (64, 128, 128, 1), (50000, 768, 3072, 0), (333, 1152, 384, 0),
                # the default mode swaps operands here (N = 384 allows only 128-wide tiles, M = 1536 allows 256)
                (20000, 1536, 384, 0), (700, 512, 128, 3),
                (1000, 256, 256, 0), (19906, 2304, 768, 0), (700, 512, 768, 3), (300, 768, 768, 1)]


@pytest.mark.parametrize("pair", [1, 0])
@pytest.mark.parametrize("M,Nw,Kw,splits", WGRAD_SHAPES)
def test_wgrad(M, Nw, Kw, splits, pair):
    dy = torch.randn(M, Nw, device=DEV).bfloat16()
    x = torch.randn(M, Kw, device=DEV).bfloat16()
    ref = dy.double().t() @ x.double()
    pre = torch.randn(Nw, Kw, device=DEV)
    with pair_wgrad(pair):
        for acc in (False, True):
            def run():
                out = pre.clone() if acc else torch.full((Nw, Kw), NAN, device=DEV)
                ops.gemm_wgrad(ops.plain_operand(dy), ops.plain_operand(x), M, 1, out, splits=splits, accumulate=acc)
                return (out,)
            (out,) = det_runs(run)
            (base,) = run()
            if acc:
                assert rel_acc(out, pre, ref) < 5e-5
                assert rel_acc(out, pre, base.double() - pre.double()) < 1e-5
            else:
                assert rel(out, ref) < 5e-5
                if splits == 1:     # one split, overwrite: plain stores in both modes
                    assert torch.equal(out, base)
                else:
                    assert rel(out, base) < 1e-5


@pytest.mark.parametrize("pair", [1, 0])
@pytest.mark.parametrize("M,Nw,Kw,splits", [(700, 512, 128, 3), (20000, 1536, 384, 0), (19906, 512, 768, 0)])
def test_wgrad_into_column_window(M, Nw, Kw, splits, pair):
    """The output is a column window of a wider buffer (ld_out > N, out_offset): the columns around it stay untouched."""
    off, ld = 64, Kw + 192
    dy = torch.randn(M, Nw, device=DEV).bfloat16()
    x = torch.randn(M, Kw, device=DEV).bfloat16()
    ref = dy.double().t() @ x.double()
    buf0 = torch.randn(Nw, ld, device=DEV)
    with pair_wgrad(pair):
        for acc in (False, True):
            def run():
                buf = buf0.clone()
                if not acc:
                    buf[:, off:off + Kw] = NAN
                ops.gemm_wgrad(ops.plain_operand(dy), ops.plain_operand(x), M, 1, buf, N=Kw, ld_out=ld,
                               out_offset=off, splits=splits, accumulate=acc)
                return (buf,)
            (buf,) = det_runs(run)
            (base,) = run()
            assert torch.equal(buf[:, :off], buf0[:, :off]) and torch.equal(buf[:, off + Kw:], buf0[:, off + Kw:])
            win, pre = buf[:, off:off + Kw], buf0[:, off:off + Kw]
            if acc:
                assert rel_acc(win, pre, ref) < 5e-5
            else:
                assert rel(win, ref) < 5e-5
            assert rel(win, base[:, off:off + Kw]) < 1e-5


def _conv_operand(x, L_in, k):
    Bn, _, Cc = x.shape
    return ops.make_operand(x, Cc, L_in // 2, Bn, nq=2, q_stride=Cc, row_stride=2 * Cc, batch_stride=L_in * Cc,
                            seg_width=Cc, seg_q=(0, 1, 0)[:k], seg_p=(0, 0, 1)[:k])


@pytest.mark.parametrize("pair", [1, 0])
@pytest.mark.parametrize("L_in,k", [(402, 3), (400, 2)])
def test_conv_wgrad(L_in, k, pair):
    Bn, Cc = 3, 512
    x = torch.randn(Bn, L_in, Cc, device=DEV).bfloat16()
    L_out = (L_in - k) // 2 + 1
    dy = torch.randn(Bn, L_out, Cc, device=DEV).bfloat16()
    # dW[o, j*C + c] = sum_{b,t} dy[b, t, o] * x[b, 2t + j, c]
    xd, dyd = x.double(), dy.double()
    ref = torch.cat([torch.einsum("bto,btc->oc", dyd, xd[:, j:j + 2 * L_out - 1:2]) for j in range(k)], dim=1)
    pre = torch.randn(Cc, k * Cc, device=DEV)
    with pair_wgrad(pair):
        for acc in (False, True):
            def run():
                out = pre.clone() if acc else torch.full((Cc, k * Cc), NAN, device=DEV)
                ops.gemm_wgrad(ops.make_operand(dy, Cc, L_out, Bn), _conv_operand(x, L_in, k), L_out, Bn, out,
                               accumulate=acc)
                return (out,)
            (out,) = det_runs(run)
            (base,) = run()
            if acc:
                assert rel_acc(out, pre, ref) < 5e-5
                assert rel_acc(out, pre, base.double() - pre.double()) < 1e-5
            else:
                assert rel(out, ref) < 5e-5
                assert rel(out, base) < 1e-5


# ------------------------------------------------------------------------------------------------------- GEMM column sums
def _check_gemm_colsum(run, cs0, fused_gelu=False):
    """run(colsum buffer or None) -> stored output(s); the colsum must equal the fp64 column sum of the stored output and,
    bit for bit, the deterministic ops.colsum of that output into a copy of the same pre-filled buffer (it is the same
    code).  The stored output equals, bit for bit, the default mode's GEMM without column sums: that is the GEMM the
    deterministic mode runs."""
    def det():
        cs = cs0.clone()
        outs = run(cs)
        c = cs0.clone()
        ops.colsum(outs[0], c)
        return (cs, c) + outs
    cs, c, *outs = det_runs(det)
    assert torch.equal(cs, c)
    assert rel_acc(cs, cs0, outs[0].double().sum(0)) < 1e-5
    for a, b in zip(outs, run(None)):   # no atomics touch the GEMM output
        assert torch.equal(a, b)
    cs_def = cs0.clone()
    outs_def = run(cs_def)
    if fused_gelu:
        # the default mode's fused column sums move a GELU GEMM from the TMA-store epilogue (packed-half tanh-form GELU,
        # ptx.cuh gelu_h2) to the generic one (fp32 erfc-form GELU, gelu_fast): the two forms differ by one bf16 ulp on
        # some outputs, so compare those outputs at bf16 tolerance and the column sums over the same stored output
        for a, b in zip(outs, outs_def):
            assert rel(a, b) < BF16_TOL
        cs_def = cs0.clone()
        ops.colsum(outs[0], cs_def)
    else:
        for a, b in zip(outs, outs_def):
            assert torch.equal(a, b)
    assert rel_acc(cs, cs0, cs_def.double() - cs0.double()) < 1e-5
    return outs


def test_gemm_colsum_epilogues():
    M, N, K = 1000, 1536, 384
    a = torch.randn(M, K, device=DEV).bfloat16()
    wt = (torch.randn(N, K, device=DEV) * 0.05).bfloat16()
    bias = torch.randn(N, device=DEV)
    res = torch.randn(M, N, device=DEV)
    base = a.double() @ wt.double().t() + bias.double()
    cs0 = torch.randn(N, device=DEV)

    def bf16_out(cs):
        out = torch.full((M, N), NAN, device=DEV, dtype=torch.bfloat16)
        ops.gemm(ops.plain_operand(a), wt, M, 1, out, bias=bias, colsum=cs)
        return (out,)
    (out,) = _check_gemm_colsum(bf16_out, cs0)
    assert rel(out, base) < BF16_TOL

    def f32_resid(cs):
        out = torch.full((M, N), NAN, device=DEV)
        ops.gemm(ops.plain_operand(a), wt, M, 1, out, bias=bias, resid=res, colsum=cs)
        return (out,)
    (out,) = _check_gemm_colsum(f32_resid, cs0)
    assert rel(out, base + res.double()) < 2e-5

    def gelu_out2(cs):
        out = torch.full((M, N), NAN, device=DEV, dtype=torch.bfloat16)
        out2 = torch.full((M, N), NAN, device=DEV, dtype=torch.bfloat16)
        ops.gemm(ops.plain_operand(a), wt, M, 1, out, bias=bias, act=ops.ACT_GELU, out2=out2, colsum=cs)
        return (out, out2)
    out, out2 = _check_gemm_colsum(gelu_out2, cs0, fused_gelu=True)
    h = base.bfloat16().double().requires_grad_(True)
    F.gelu(h).sum().backward()
    assert rel(out, F.gelu(h.detach())) < BF16_TOL
    assert rel(out2, h.grad) < BF16_TOL


@pytest.mark.parametrize("block_n", [-256, 256])
def test_dgrad_dgelu_colsum(block_n):
    M, N, K = 4000, 3072, 768
    dy = torch.randn(M, K, device=DEV).bfloat16()
    wt = (torch.randn(K, N, device=DEV) * 0.05).bfloat16()
    aux = torch.randn(M, N, device=DEV).bfloat16()
    cs0 = torch.randn(N, device=DEV)

    def run(cs):
        out = torch.full((M, N), NAN, device=DEV, dtype=torch.bfloat16)
        ops.gemm_dgrad(ops.plain_operand(dy), wt, M, 1, out, K=K, N=N, act=ops.ACT_DGELU, aux=aux, colsum=cs,
                       block_n=block_n)
        return (out,)
    (out,) = _check_gemm_colsum(run, cs0)
    assert rel(out, (dy.double() @ wt.double()) * aux.double()) < BF16_TOL


def test_gemm_colsum_refuses_out_rows_and_accumulate():
    M, N, K = 256, 256, 128
    a = torch.randn(M, K, device=DEV).bfloat16()
    wt = (torch.randn(N, K, device=DEV) * 0.05).bfloat16()
    perm = torch.randperm(M, device=DEV).int()
    out = torch.zeros(M, N, device=DEV)
    cs = torch.zeros(N, device=DEV)
    with det_mode():
        with pytest.raises(_lib.WavJepaLibError):
            ops.gemm(ops.plain_operand(a), wt, M, 1, out, out_rows=perm, colsum=cs)
        with pytest.raises(_lib.WavJepaLibError):
            ops.gemm(ops.plain_operand(a), wt, M, 1, out, accumulate=True, colsum=cs)
        with pytest.raises(_lib.WavJepaLibError):
            ops.gemm_dgrad(ops.plain_operand(a), wt.t().contiguous(), M, 1, out, K=K, N=N, out_rows=perm, colsum=cs)
        with pytest.raises(_lib.WavJepaLibError):
            ops.gemm_dgrad(ops.plain_operand(a), wt.t().contiguous(), M, 1, out, K=K, N=N, accumulate=True, colsum=cs)
    assert torch.equal(cs, torch.zeros(N, device=DEV))


# ------------------------------------------------------------------------------------------------------- colsum
# (N, ld, first column, kernel): the 8-wide kernel needs N % 8 == 0, a 16-byte aligned base and ld % 8 == 0
COLSUM_LAYOUTS = [(768, 768, 0, "8-wide"), (1152, 1160, 0, "8-wide"), (1150, 1158, 0, "generic"),
                  (384, 390, 0, "generic"), (384, 392, 2, "generic")]


@pytest.mark.parametrize("M", [1, 7, 33, 1237, 200000])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("N,ld,c0,kernel", COLSUM_LAYOUTS)
def test_colsum(N, ld, c0, kernel, dtype, M):
    x = torch.randn(M, ld, device=DEV).to(dtype)[:, c0:c0 + N]
    assert x.stride(0) == ld
    pre = torch.randn(N, device=DEV)

    def run():
        out = pre.clone()
        ops.colsum(x, out)
        return (out,)
    (out,) = det_runs(run)
    ref = x.double().sum(0)
    assert rel_acc(out, pre, ref) < 2e-5
    (base,) = run()
    assert rel_acc(out, pre, base.double() - pre.double()) < 1e-5


# ------------------------------------------------------------------------------------------------------- LayerNorm backward
def _ln_case(kind, M, D):
    """(x, add, dy_f32, dy_bf16) of one LayerNorm-backward form: plain LN over fp32 / bf16 x, or add + LN with the
    output gradient as (fp32 + bf16) / fp32 / bf16."""
    x = torch.randn(M, D, device=DEV) * 2 + 0.5
    add = d32 = d16 = None
    if kind == "ln_bf16":
        x = x.bfloat16()
    if kind.startswith("add"):
        add = torch.randn(M, D, device=DEV).bfloat16()
    if kind in ("ln_f32", "ln_bf16", "add_d32_d16", "add_d32"):
        d32 = torch.randn(M, D, device=DEV)
    if kind in ("add_d32_d16", "add_d16"):
        d16 = torch.randn(M, D, device=DEV).bfloat16()
    return x, add, d32, d16


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("M", [1, 9, 1237, 19906])
@pytest.mark.parametrize("D", [128, 256, 384, 512, 768, 1024])
def test_layernorm_bwd(D, M, det):
    g = 1 + 0.1 * torch.randn(D, device=DEV)
    b = 0.1 * torch.randn(D, device=DEV)
    for kind in ("ln_f32", "ln_bf16", "add_d32_d16", "add_d32", "add_d16"):
        x, add, d32, d16 = _ln_case(kind, M, D)
        st = torch.empty(M, 2, device=DEV)
        if add is None:
            ops.layernorm_fwd(x, g, b, 1e-6, None, None, st, None)
        else:
            ops.add_layernorm_fwd(x, add, g, b, 1e-6, None, None, st, None)
        # fp64 reference
        xr = (x.double() + (add.double() if add is not None else 0.0)).requires_grad_(True)
        gr = g.double().requires_grad_(True)
        br = b.double().requires_grad_(True)
        dyt = (d32.double() if d32 is not None else 0.0) + (d16.double() if d16 is not None else 0.0)
        F.layer_norm(xr, (D,), gr, br, 1e-6).backward(dyt)
        refs = (gr.grad, br.grad, xr.grad.sum(0))
        pres = [torch.randn(D, device=DEV) for _ in range(3)]
        for subset in ((0,), (2,), (0, 1, 2)):     # only dgamma; only the colsum; all three reductions
            def run():
                dxf = torch.full((M, D), NAN, device=DEV)
                dxb = torch.full((M, D), NAN, device=DEV, dtype=torch.bfloat16)
                red = [pres[i].clone() if i in subset else None for i in range(3)]
                if add is None:
                    ops.layernorm_bwd(d32, x, st, g, dxf, dxb, *red)
                else:
                    ops.add_layernorm_bwd(d32, d16, x, add, st, g, dxf, dxb, *red)
                return (dxf, dxb) + tuple(r for r in red if r is not None)
            outs = det_runs(run) if det else run()
            dxf, dxb, red = outs[0], outs[1], outs[2:]
            assert rel(dxf, xr.grad) < 1e-4 and rel(dxb, xr.grad) < BF16_TOL, (kind, subset)
            for i, r in zip(subset, red):
                if i < 2:
                    assert rel_acc(r, pres[i], refs[i]) < 1e-4, (kind, subset, i)
                else:   # colsum of dx: the fp64 sum of the stored dx, and the fp64 reference (absolute, as it can cancel)
                    assert rel_acc(r, pres[i], dxf.double().sum(0)) < 1e-5, (kind, subset)
                    assert (r.double() - pres[i].double() - refs[i]).abs().max().item() < 1e-2, (kind, subset)
            if det:
                base = run()
                assert torch.equal(dxf, base[0]) and torch.equal(dxb, base[1])   # no atomics on dx
                for i, r, q in zip(subset, red, base[2:]):
                    assert rel_acc(r, pres[i], q.double() - pres[i].double()) < 1e-5, (kind, subset, i)


# ------------------------------------------------------------------------------------------------------- conv-0 backward
@pytest.mark.parametrize("L", [32159, 4000, 2577, 60])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("Cin", [1, 2])
def test_conv0_bwd(Cin, B, L):
    C = 512
    x = torch.randn(B, Cin, L, device=DEV).bfloat16()
    wt = torch.randn(C, Cin, 10, device=DEV) * math.sqrt(2.0 / (Cin * 10))
    gamma = 1.0 + 0.1 * torch.randn(C, device=DEV)
    beta = 0.1 * torch.randn(C, device=DEV)
    L_out = (L - 10) // 5 + 1
    out = torch.empty(B, L_out, C, device=DEV, dtype=torch.bfloat16)
    mom, stats, red = ops.conv0_workspaces(B, Cin, C, DEV, backward=True)
    ops.conv0_fwd(x, wt, gamma, beta, out, mom, stats)
    dy = torch.randn(B, L_out, C, device=DEV).bfloat16()
    # fp64 reference: bf16 weights, the conv output rounded to bf16 (autocast) with a straight-through gradient
    wr = wt.bfloat16().double().requires_grad_(True)
    gr = gamma.double().requires_grad_(True)
    br = beta.double().requires_grad_(True)
    h = F.conv1d(x.double(), wr, stride=5)
    hq = h + (h.bfloat16().double() - h).detach()
    F.gelu(F.group_norm(hq, C, gr, br, 1e-5)).backward(dy.double().transpose(1, 2))
    pre = (torch.randn_like(wt), torch.randn(C, device=DEV), torch.randn(C, device=DEV))

    def run():
        dw, dg, db = (p.clone() for p in pre)
        ops.conv0_bwd(x, wt, gamma, beta, mom, stats, dy, red, dw, dg, db)
        return dw, dg, db
    outs = det_runs(run)
    base = run()
    for o, p, r, q in zip(outs, pre, (wr.grad, gr.grad, br.grad), base):
        # GELU' recomputed in packed fp16 and dz in bf16 (like autograd's bf16 conv weight gradient): ~2^-9 per term
        assert rel_acc(o, p, r) < 4e-3
        # both modes reduce in fp64: only the last bits of the fp64 sums differ
        assert rel_acc(o, p, q.double() - p.double()) < 1e-6


# ------------------------------------------------------------------------------------------------------- attention backward
def _attn_ref(qkv, cu, D, H):
    dh = D // H
    outs = []
    for s in range(len(cu) - 1):
        x = qkv[cu[s]:cu[s + 1]]
        n = x.shape[0]
        if n == 0:
            continue
        q, k, v = (x[:, i * D:(i + 1) * D].reshape(n, H, dh).transpose(0, 1) for i in range(3))
        o = F.scaled_dot_product_attention(q, k, v)
        outs.append(o.transpose(0, 1).reshape(n, D))
    return torch.cat(outs)


# the backward-capable rows of test_gpu_kernels.py::test_attention_fwd_bwd; head dim 32 runs the tcgen05 backward up to
# 128 tokens and the mma.sync one above, head dim 64 the mma.sync one
ATTN_CASES = [(768, 12, [39, 72, 20, 1, 64, 65]), (384, 12, [85, 122, 128, 17]), (768, 12, [200, 200, 200]),
              (384, 12, [250, 3]), (384, 12, [5, 0, 128, 0, 33]), (768, 12, [128] * 40 + [7]),
              (768, 24, [129, 256, 1, 128]), (384, 12, [257, 5]), (768, 12, [256, 255, 130, 2]),
              (384, 12, [64] * 300 + [100] * 300), (384, 12, [400, 230, 512, 1]), (384, 12, [272, 7] * 40),
              (384, 12, [600, 5])]


@pytest.mark.parametrize("D,H,lens", ATTN_CASES)
def test_attention_bwd_dbias(D, H, lens):
    cu_l = [0]
    for n in lens:
        cu_l.append(cu_l[-1] + n)
    tot = cu_l[-1]
    cu = torch.tensor(cu_l, device=DEV, dtype=torch.int32)
    qkv = torch.randn(tot, 3 * D, device=DEV).bfloat16()
    out = torch.empty(tot, D, device=DEV, dtype=torch.bfloat16)
    lse = torch.empty(tot, H, device=DEV)
    ops.attn_fwd(qkv, cu, len(lens), max(lens), D, H, out, lse)
    do = torch.randn(tot, D, device=DEV).bfloat16()
    qr = qkv.double().requires_grad_(True)
    _attn_ref(qr, cu_l, D, H).backward(do.double())
    args = (qkv, out, do, lse, cu, len(lens), max(lens), D, H)

    def run():
        dqkv = torch.full((tot, 3 * D), NAN, device=DEV, dtype=torch.bfloat16)
        db = torch.ones(3 * D, device=DEV)
        ops.attn_bwd(*args, dqkv, dbias=db)
        c = torch.ones(3 * D, device=DEV)
        ops.colsum(dqkv, c)
        return dqkv, db, c
    dqkv, db, c = det_runs(run)
    # the bias gradient is the ordered column sum of the stored dqkv: compare the buffers (both pre-filled with 1)
    assert torch.equal(db, c)
    assert rel(dqkv, qr.grad) < 1.5e-2
    assert rel_acc(db, torch.ones_like(db), dqkv.double().sum(0)) < 1e-5
    cs = qr.grad.sum(0)
    assert (db.double() - 1.0 - cs).abs().max().item() <= 1e-2 * cs.abs().max().item() + 1e-3
    # default mode: dqkv is written with plain stores in both modes
    base = torch.full((tot, 3 * D), NAN, device=DEV, dtype=torch.bfloat16)
    db_def = torch.ones(3 * D, device=DEV)
    ops.attn_bwd(*args, base, dbias=db_def)
    assert torch.equal(dqkv, base)
    # the default tcgen05 route (head dim 32, <= 128 tokens) sums the query third from its fp32 accumulators, takes the
    # value third from dO and leaves the key third at exactly zero; the deterministic mode sums the bf16-rounded dqkv
    # instead, so the two differ by the bf16 rounding of the summands (random data: ~1e-3 of the column sums)
    tol = 1e-2 if D // H == 32 and max(lens) <= 128 else 1e-5
    assert rel_acc(db, torch.ones_like(db), db_def.double() - 1.0) < tol


# ------------------------------------------------------------------------------------------------------- predictor input
@pytest.mark.parametrize("N", [1, 900, 300000])
def test_predictor_assemble_bwd_mask_token(N):
    D, Nc = 384, 300
    vsrc = torch.randint(0, Nc, (N,), device=DEV, dtype=torch.int32)
    vsrc[torch.rand(N, device=DEV) < 0.5] = -1          # rows that hold the mask token
    if N == 1:
        vsrc.fill_(-1)
    dx0 = torch.randn(N, D, device=DEV)
    pre = torch.randn(D, device=DEV)

    def run():
        dmt = pre.clone()
        ops.predictor_assemble_bwd(dx0, vsrc, N, D, None, dmt)
        return (dmt,)
    (dmt,) = det_runs(run)
    ref = (dx0.double() * (vsrc < 0)[:, None]).sum(0)
    assert rel_acc(dmt, pre, ref) < 1e-5
    (base,) = run()
    assert rel_acc(dmt, pre, base.double() - pre.double()) < 1e-5
    # the context gradient is refused in this mode (wj_predictor_ctx_grad is its atomic-free form), before any launch
    dctx = torch.zeros(Nc, D, device=DEV)
    dmt = pre.clone()
    with det_mode():
        with pytest.raises(_lib.WavJepaLibError, match="d_ctx"):
            ops.predictor_assemble_bwd(dx0, vsrc, N, D, dctx, dmt)
    assert torch.equal(dmt, pre) and not dctx.any()


# ------------------------------------------------------------------------------------------------------- masked MSE
@pytest.mark.parametrize("D", [384, 768])
@pytest.mark.parametrize("Nt", [1, 7, 4321, 200000])
def test_masked_mse(Nt, D):
    R = 2000
    pred = torch.randn(Nt, D, device=DEV).bfloat16()
    tg = torch.randn(R, D, device=DEV)
    rows = torch.randint(0, R, (Nt,), device=DEV, dtype=torch.int32)
    pre = torch.rand(1, device=DEV)

    def run():
        loss = pre.clone()
        dp = torch.full((Nt, D), NAN, device=DEV, dtype=torch.bfloat16)
        ops.masked_mse(pred, tg, rows, Nt, D, loss, dp)
        return loss, dp
    loss, dp = det_runs(run)
    pr = pred.double().requires_grad_(True)
    ref = ((pr - tg.double()[rows.long()]) ** 2).mean(-1).sum() / (Nt + 1e-8)
    ref.backward()
    assert rel_acc(loss, pre, ref.detach()) < 1e-5
    assert rel(dp, pr.grad) < BF16_TOL
    loss_def, dp_def = run()
    assert torch.equal(dp, dp_def)
    # (up to 1184 fp32 block partials in another order: a few 1e-6 at most)
    assert rel_acc(loss, pre, loss_def.double() - pre.double()) < 1e-5


# ------------------------------------------------------------------------------------------------------- sum of squares
@pytest.mark.parametrize("n", [1, 3, 1_000_003, 50_000_000])
def test_sumsq(n):
    scale = 0.37
    x = torch.randn(n, device=DEV)
    pre = torch.rand(1, device=DEV, dtype=torch.float64)

    def run():
        out = pre.clone()
        ops.sumsq(x, scale, out)
        return (out,)
    (out,) = det_runs(run)
    v = x * scale                       # fp32 product, as the kernel forms it
    ref = (v.double() ** 2).sum()
    assert rel_acc(out, pre, ref) < 1e-12
    (base,) = run()
    assert rel_acc(out, pre, base - pre) < 1e-12


# ------------------------------------------------------------------------------------------------------- contract
def _contract_calls():
    """Entry points whose deterministic branch needs more than a 256-byte workspace: name -> (call, destinations that
    must stay untouched when the call is refused, every output buffer).  Each call re-fills its outputs first."""
    torch.manual_seed(7)
    calls = {}
    # weight gradient, three splits
    dy = torch.randn(700, 512, device=DEV).bfloat16()
    xw = torch.randn(700, 128, device=DEV).bfloat16()
    w_pre, w_out = torch.randn(512, 128, device=DEV), torch.empty(512, 128, device=DEV)

    def wgrad():
        w_out.copy_(w_pre)
        ops.gemm_wgrad(ops.plain_operand(dy), ops.plain_operand(xw), 700, 1, w_out, splits=3)
    calls["wgrad"] = (wgrad, [(w_out, w_pre)], [w_out])
    # GEMM with fused column sums (the GEMM writes `out` before the column sum is refused: only the colsum is checked)
    a = torch.randn(1000, 384, device=DEV).bfloat16()
    wt = (torch.randn(768, 384, device=DEV) * 0.05).bfloat16()
    g_out = torch.empty(1000, 768, device=DEV, dtype=torch.bfloat16)
    g_cs_pre, g_cs = torch.randn(768, device=DEV), torch.empty(768, device=DEV)

    def gemm_cs():
        g_out.fill_(NAN)
        g_cs.copy_(g_cs_pre)
        ops.gemm(ops.plain_operand(a), wt, 1000, 1, g_out, colsum=g_cs)
    calls["gemm_colsum"] = (gemm_cs, [(g_cs, g_cs_pre)], [g_out, g_cs])
    # column sums
    xc = torch.randn(1237, 1152, device=DEV)
    c_pre, c_out = torch.randn(1152, device=DEV), torch.empty(1152, device=DEV)

    def colsum():
        c_out.copy_(c_pre)
        ops.colsum(xc, c_out)
    calls["colsum"] = (colsum, [(c_out, c_pre)], [c_out])
    # LayerNorm backward, D = 768 at the student's row count
    M, D = 19906, 768
    xl = torch.randn(M, D, device=DEV) * 2 + 0.5
    gl, bl = 1 + 0.1 * torch.randn(D, device=DEV), 0.1 * torch.randn(D, device=DEV)
    st = torch.empty(M, 2, device=DEV)
    ops.layernorm_fwd(xl, gl, bl, 1e-6, None, None, st, None)
    dyl = torch.randn(M, D, device=DEV)
    dx_pre = torch.randn(M, D, device=DEV)
    l_pre = [torch.randn(D, device=DEV) for _ in range(3)]
    dx, l_out = torch.empty(M, D, device=DEV), [torch.empty(D, device=DEV) for _ in range(3)]

    def ln_bwd():
        dx.copy_(dx_pre)
        for o, p in zip(l_out, l_pre):
            o.copy_(p)
        ops.layernorm_bwd(dyl, xl, st, gl, dx, None, *l_out)
    calls["layernorm_bwd"] = (ln_bwd, [(dx, dx_pre)] + list(zip(l_out, l_pre)), [dx] + l_out)
    # conv-0 backward
    B, Cin, L, C = 3, 2, 4000, 512
    x0 = torch.randn(B, Cin, L, device=DEV).bfloat16()
    w0 = torch.randn(C, Cin, 10, device=DEV) * 0.2
    ga, be = 1.0 + 0.1 * torch.randn(C, device=DEV), 0.1 * torch.randn(C, device=DEV)
    L_out = (L - 10) // 5 + 1
    y0 = torch.empty(B, L_out, C, device=DEV, dtype=torch.bfloat16)
    mom, stats, red = ops.conv0_workspaces(B, Cin, C, DEV, backward=True)
    ops.conv0_fwd(x0, w0, ga, be, y0, mom, stats)
    dy0 = torch.randn(B, L_out, C, device=DEV).bfloat16()
    c0_pre = (torch.randn_like(w0), torch.randn(C, device=DEV), torch.randn(C, device=DEV))
    c0_out = tuple(torch.empty_like(p) for p in c0_pre)

    def conv0():
        for o, p in zip(c0_out, c0_pre):
            o.copy_(p)
        ops.conv0_bwd(x0, w0, ga, be, mom, stats, dy0, red, *c0_out)
    calls["conv0_bwd"] = (conv0, list(zip(c0_out, c0_pre)), list(c0_out))
    return calls


def test_workspace_size_does_not_change_the_bits():
    calls = _contract_calls()
    for name in ("wgrad", "colsum", "layernorm_bwd", "conv0_bwd"):
        fn, _, outs = calls[name]
        res = []
        for nbytes in (64 << 20, 256 << 20):
            with det_mode(nbytes):
                fn()
            res.append([o.clone() for o in outs])
        for a, b in zip(*res):
            assert torch.equal(a, b), name


def test_too_small_workspace_is_refused_before_any_launch():
    calls = _contract_calls()
    D, N = 384, 300000
    vsrc = torch.randint(-1, 300, (N,), device=DEV, dtype=torch.int32)
    dx0 = torch.randn(N, D, device=DEV)
    mt_pre, mt = torch.randn(D, device=DEV), torch.empty(D, device=DEV)

    def assemble_bwd():
        mt.copy_(mt_pre)
        ops.predictor_assemble_bwd(dx0, vsrc, N, D, None, mt)
    calls["predictor_assemble_bwd"] = (assemble_bwd, [(mt, mt_pre)], [mt])
    # masked MSE needs 4 bytes per block: 4321 rows are 541 blocks (2164 bytes)
    Nt = 4321
    pred = torch.randn(Nt, 768, device=DEV).bfloat16()
    tg = torch.randn(2000, 768, device=DEV)
    rows = torch.randint(0, 2000, (Nt,), device=DEV, dtype=torch.int32)
    loss_pre, loss = torch.rand(1, device=DEV), torch.empty(1, device=DEV)
    dp_pre, dp = torch.randn(Nt, 768, device=DEV).bfloat16(), torch.empty(Nt, 768, device=DEV, dtype=torch.bfloat16)

    def mse():
        loss.copy_(loss_pre)
        dp.copy_(dp_pre)
        ops.masked_mse(pred, tg, rows, Nt, 768, loss, dp)
    calls["masked_mse"] = (mse, [(loss, loss_pre), (dp, dp_pre)], [loss, dp])
    xs = torch.randn(1_000_003, device=DEV)
    ss_pre, ss = torch.rand(1, device=DEV, dtype=torch.float64), torch.empty(1, device=DEV, dtype=torch.float64)

    def sumsq():
        ss.copy_(ss_pre)
        ops.sumsq(xs, 0.5, ss)
    calls["sumsq"] = (sumsq, [(ss, ss_pre)], [ss])
    # attention backward with the bias gradient: the kernel writes dqkv, then the ordered column sum is refused
    Da, H, lens = 768, 12, [200, 200, 200]
    tot = sum(lens)
    cu = torch.tensor([0, 200, 400, 600], device=DEV, dtype=torch.int32)
    qkv = torch.randn(tot, 3 * Da, device=DEV).bfloat16()
    ao = torch.empty(tot, Da, device=DEV, dtype=torch.bfloat16)
    lse = torch.empty(tot, H, device=DEV)
    ops.attn_fwd(qkv, cu, 3, 200, Da, H, ao, lse)
    do = torch.randn(tot, Da, device=DEV).bfloat16()
    dq = torch.empty(tot, 3 * Da, device=DEV, dtype=torch.bfloat16)
    db_pre, db = torch.randn(3 * Da, device=DEV), torch.empty(3 * Da, device=DEV)

    def attn():
        db.copy_(db_pre)
        ops.attn_bwd(qkv, ao, do, lse, cu, 3, 200, Da, H, dq, dbias=db)
    calls["attn_bwd_dbias"] = (attn, [(db, db_pre)], [db])
    for name, (fn, untouched, _) in calls.items():
        with det_mode(256):
            assert_refused(fn)
        torch.cuda.synchronize()
        for o, p in untouched:
            assert torch.equal(o, p), name
        fn()                                 # default mode again: the same call succeeds
        torch.cuda.synchronize()
        assert not any(torch.equal(o, p) for o, p in untouched[-1:]), name


def test_off_is_off():
    with det_mode():
        assert ops._det_ws is not None
    assert ops._det_ws is None
    # the forms that deterministic mode refuses run again ...
    N, D, Nc = 900, 384, 300
    vsrc = torch.randint(-1, Nc, (N,), device=DEV, dtype=torch.int32)
    dx0 = torch.randn(N, D, device=DEV)
    dctx, dmt = torch.zeros(Nc, D, device=DEV), torch.zeros(D, device=DEV)
    ops.predictor_assemble_bwd(dx0, vsrc, N, D, dctx, dmt)
    ref = torch.zeros(Nc, D, device=DEV, dtype=torch.float64).index_add_(
        0, vsrc.clamp(min=0).long(), dx0.double() * (vsrc >= 0)[:, None])
    assert rel(dctx, ref) < 1e-5 and rel(dmt, (dx0.double() * (vsrc < 0)[:, None]).sum(0)) < 1e-5
    a = torch.randn(256, 128, device=DEV).bfloat16()
    wt = (torch.randn(256, 128, device=DEV) * 0.05).bfloat16()
    out, cs = torch.zeros(256, 256, device=DEV), torch.zeros(256, device=DEV)
    ops.gemm(ops.plain_operand(a), wt, 256, 1, out, accumulate=True, colsum=cs)
    assert rel(cs, out.double().sum(0)) < 1e-5
    # ... and a reduction takes the atomic path: the same result as a run that never switched the mode on
    x = torch.randn(1237, 768, device=DEV)
    c1 = torch.zeros(768, device=DEV)
    ops.colsum(x, c1)
    assert rel(c1, x.double().sum(0)) < 2e-5


# ------------------------------------------------------------------------------------------------------- model level
def _build_model(cfg, sd):
    if cfg.per_channel:
        ex = w.ConvChannelFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=cfg.in_channels,
                                           share_weights_over_channels=False)
    else:
        ex = w.ConvFeatureExtractor(conv_layers_spec=cfg.spec, in_channels=cfg.in_channels)
    m = w.JEPA(feature_extractor=ex, transformer_encoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_encoder_layers_cfg=w.TransformerLayerCFG.create(),
               transformer_decoder_cfg=w.TransformerEncoderCFG.create(),
               transformer_decoder_layers_cfg=w.TransformerLayerCFG.create(d_model=384),
               process_audio_seconds=2.01, nr_samples_per_audio=8, average_top_k_layers=cfg.top_k, lr=4e-4,
               adam_weight_decay=0.04)
    m.load_state_dict({k: v.detach() for k, v in sd.items()}, strict=True)
    return m.to(DEV)


def _grad_close(names, view_a, view_b):
    for n_ in names:
        g1, g2 = view_a(n_).double(), view_b(n_).double()
        # (the attention in_proj bias gradient is taken from the stored bf16 dqkv in this mode, from dO for the value
        # third in the default one: equal up to bf16 rounding of the summands)
        tol = 2e-4 if n_.endswith("in_proj_bias") else 1e-5
        assert (g1 - g2).norm().item() <= tol * g1.norm().item() + 1e-12, n_


def test_nat_train_step_deterministic():
    """WavJEPA-Nat (two channels, per-channel conv stacks): conv-0 with two input channels and the binaural shapes."""
    cfg = jo.Cfg(in_channels=2, per_channel=True)
    sd = jo.make_state_dict(cfg, seed=3)
    inp = oi.training_inputs(cfg, 1, 2, seed=55, masker="audioset")
    audio = inp["audio"].to(DEV).bfloat16()
    c_m, t_m, v_m = (inp[k].to(DEV) for k in ("ctx_masks", "target_indices", "ctx_and_target_masks"))
    ref = _build_model(cfg, sd)
    ref.global_step = 50000
    l_ref = ref.train_step(audio, c_m, t_m, v_m).item()
    a, b = _build_model(cfg, sd), _build_model(cfg, sd)
    a.global_step = b.global_step = 50000
    for step in range(2):     # the second step starts from the first's (identical) update
        with det_mode(fill=0xFF):
            la = a.train_step(audio, c_m, t_m, v_m).item()
        with det_mode(fill=0x7F):
            lb = b.train_step(audio, c_m, t_m, v_m).item()
        assert la == lb
        assert torch.equal(a._flat_g, b._flat_g)
        assert torch.equal(a._flat_p, b._flat_p) and torch.equal(a._flat_t, b._flat_t)
        if step == 0:
            assert abs(la - l_ref) < 1e-6
            _grad_close(ref._train_names, lambda n_: ref._view(ref._flat_g, n_), lambda n_: a._view(a._flat_g, n_))


def _denoiser(alpha, nr=2):
    from wavjepa_b200.denoiser import Denoiser
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


def test_denoiser_forward_backward_deterministic():
    batch = oi.denoiser_batch()
    m_ref, a, b = _denoiser(0.25), _denoiser(0.25), _denoiser(0.25)
    gen, clean = m_ref.on_after_batch_transfer(tuple(t.to(DEV) for t in batch), 0)

    def step(m):
        out, grads = m.forward_backward(gen, clean)
        return {k: v.item() for k, v in out.items() if torch.is_tensor(v) and v.numel() == 1}, \
            {n_: g.clone() for n_, g in grads.items()}
    out_ref, g_ref = step(m_ref)
    with det_mode(fill=0xFF):
        out_a, g_a = step(a)
    with det_mode(fill=0x7F):
        out_b, g_b = step(b)
    assert out_a == out_b and set(g_a) == set(g_b)
    for n_ in g_a:
        assert torch.equal(g_a[n_], g_b[n_]), n_
    for k, v in out_ref.items():
        assert abs(out_a[k] - v) <= 1e-6 * max(1.0, abs(v)), k
    _grad_close(list(g_ref), g_ref.__getitem__, g_a.__getitem__)
