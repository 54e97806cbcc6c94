// First block of the waveform encoder: Conv1d(Cin -> C, k=10, stride=5, no bias) + GroupNorm(C groups, C channels)
// + exact GELU, fused, writing channels-last bf16 so that the next layer's implicit GEMM can TMA it directly.
// Reference: wavjepa/extractors/audio_feature_extractor.py:70 (conv), :94 (GroupNorm, eps 1e-5), :95 (GELU); block 0
// of `self.cnn` (:107-121).  The conv is 10 MAC / output and the output is 100x larger than the input (6.58 MB of bf16
// per 2 s instance), so nothing the size of the output is ever read back or stored twice:
//
//   moments   (tiny)  per instance: s[a] = sum_t x_a(t), R[a][a'] = sum_t x_a(t) x_a'(t) over the conv windows
//                     (a = ci*10 + tap, x_a(t) = x[ci, 5t + tap]); fp32 partial sums folded into fp64.
//   stats     (tiny)  GroupNorm statistics of every (instance, channel) in closed form: mean = w.s / L,
//                     E[h^2] = w^T R w / L (fp64).  The reference takes them over the bf16-ROUNDED conv output; the
//                     closed form uses the unrounded one -- a relative difference of ~1e-6 (rounding noise is zero-mean
//                     with variance 2^-18 h^2 / 3), far below the bf16 resolution of the result.
//   forward   (one pass) conv (bf16-rounded, as autocast does) -> normalise -> affine -> GELU -> [B, L_out, C] bf16
//   backward  (one pass over dY) per (instance, channel): S1 = sum dz, S2 = sum dz hhat, P[a] = sum dz x_a with
//                     dz = dY gelu'(z), z RECOMPUTED from the input window (10 MAC on the tensor cores + the closed-form
//                     statistics) instead of read from a saved copy: the forward writes its 3.37 GB (B = 512) once and
//                     the backward reads dY once; then (tiny) dW[c,a] += rstd gamma (P[a] - S1/L s[a] - S2/L Q[a]),
//                     Q[a] = sum_t hhat x_a = rstd ((R w)[a] - mean s[a]); dgamma += S2, dbeta += S1.
// MMA column <-> channel mapping: inside a group of 64 channels, column j of n-tile nt is channel
// (j >> 1) * 16 + nt * 2 + (j & 1), so that the accumulator columns a lane owns over the 8 n-tiles (2 tg, 2 tg + 1) are 16
// CONSECUTIVE channels: a lane stores / loads 32 contiguous bytes per row, a warp 8 rows x 128 contiguous bytes.
#include "common.cuh"

namespace wj {

constexpr int kC0K = 10;      // kernel width
constexpr int kC0S = 5;       // stride
constexpr int kC0TT = 128;    // outputs per smem window
constexpr int kC0MaxCin = 2;
constexpr int kC0Win = (kC0TT - 1) * kC0S + kC0K;      // 645 samples
constexpr int kC0WinPad = (kC0Win + 3 + 3) & ~3;       // 648: float4 reads may run 3 past the last tap

struct Conv0Args {
  const bf16* x;      // [B, Cin, L]
  const float* w;     // [C, Cin, 10] fp32 master weights (rounded to bf16 on load: autocast semantics)
  int B, Cin, L, L_out, C;
  const float* xf;    // fp32 input instead of x (the TF32 inference path): neither input nor weights are rounded
};

__host__ __device__ inline int conv0_moment_count(int Cin) { const int na = Cin * kC0K; return na + na * na; }

// ------------------------------------------------------------------------------------------------ moments
// grid B, block 512: thread o < NA + NA*NA owns one moment; the instance streams through smem in windows.
// F32: the TF32 inference path (fp32 input a.xf, unrounded weights)
template <int CIN, bool F32 = false>
__global__ void __launch_bounds__(512) conv0_moments_kernel(Conv0Args a, double* __restrict__ mom) {
  constexpr int NA = CIN * kC0K;
  constexpr int NOUT = NA + NA * NA;
  constexpr int TCH = 512;                                  // outputs per window
  constexpr int WIN = (TCH - 1) * kC0S + kC0K;
  __shared__ float s_x[CIN * WIN];
  const int b = blockIdx.x;
  const int o = threadIdx.x;
  int a0 = 0, a1 = -1;
  if (o < NA) a0 = o;
  else if (o < NOUT) { a0 = (o - NA) / NA; a1 = (o - NA) % NA; }
  const int off0 = (a0 / kC0K) * WIN + (a0 % kC0K);
  const int off1 = a1 >= 0 ? (a1 / kC0K) * WIN + (a1 % kC0K) : 0;
  double total = 0.0;
  for (int t0 = 0; t0 < a.L_out; t0 += TCH) {
    const int nt = min(TCH, a.L_out - t0);
    const int win = (nt - 1) * kC0S + kC0K;
    __syncthreads();
    for (int ci = 0; ci < CIN; ++ci) {
      const bf16* src = a.x + (static_cast<size_t>(b) * CIN + ci) * a.L + static_cast<size_t>(t0) * kC0S;
      if constexpr (F32) {
        const float* srcf = a.xf + (static_cast<size_t>(b) * CIN + ci) * a.L + static_cast<size_t>(t0) * kC0S;
        for (int i = threadIdx.x; i < win; i += blockDim.x) s_x[ci * WIN + i] = srcf[i];
      } else {
        for (int i = threadIdx.x; i < win; i += blockDim.x) s_x[ci * WIN + i] = __bfloat162float(src[i]);
      }
    }
    __syncthreads();
    if (o < NOUT) {
      float acc = 0.f;
      if (a1 < 0) {
        for (int t = 0; t < nt; ++t) acc += s_x[off0 + t * kC0S];
      } else {
        for (int t = 0; t < nt; ++t) acc = fmaf(s_x[off0 + t * kC0S], s_x[off1 + t * kC0S], acc);
      }
      total += static_cast<double>(acc);
    }
  }
  if (o < NOUT) mom[static_cast<size_t>(b) * NOUT + o] = total;
}

// grid B, block C: closed-form GroupNorm statistics -> stats[b, c] = (mean, rstd)
template <int CIN, bool F32 = false>
__global__ void conv0_stats_kernel(Conv0Args a, const double* __restrict__ mom, float eps, float* __restrict__ stats) {
  constexpr int NA = CIN * kC0K;
  constexpr int NOUT = NA + NA * NA;
  __shared__ double s_m[NOUT];
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < NOUT; i += blockDim.x) s_m[i] = mom[static_cast<size_t>(b) * NOUT + i];
  __syncthreads();
  const int c = threadIdx.x;
  if (c >= a.C) return;
  double w[NA];
#pragma unroll
  for (int i = 0; i < NA; ++i) {
    const float wi = a.w[static_cast<size_t>(c) * NA + i];
    w[i] = static_cast<double>(F32 ? wi : bf16_round(wi));
  }
  double m = 0.0, q = 0.0;
#pragma unroll
  for (int i = 0; i < NA; ++i) m += w[i] * s_m[i];
  for (int i = 0; i < NA; ++i) {
    double r = 0.0;
#pragma unroll
    for (int j = 0; j < NA; ++j) r += w[j] * s_m[NA + i * NA + j];
    q += w[i] * r;
  }
  const double mean = m / a.L_out;
  double var = q / a.L_out - mean * mean;   // biased
  if (var < 0.0) var = 0.0;
  stats[(static_cast<size_t>(b) * a.C + c) * 2 + 0] = static_cast<float>(mean);
  stats[(static_cast<size_t>(b) * a.C + c) * 2 + 1] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
}

// ------------------------------------------------------------------------------------------------ main passes
// Both passes run the 10-tap convolution on the legacy tensor-core path (mma.sync.m16n8k16, bf16 in / fp32 out): the
// A operand is the [16 outputs x 16 taps] window matrix A[t][k] = x[ci, 5t + k] (taps 10..15 are zero), read straight
// from the bf16 input window in shared memory; B is the [16 taps x 8 channels] slice of the (bf16-rounded) weights.
// What is left on the CUDA cores is the epilogue: ~20 instructions per output in the forward (bf16 round, affine,
// GELU + GELU', pack, store), ~12 in the backward.
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t a) {
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}
__device__ __forceinline__ uint32_t pack2(bf16 lo, bf16 hi) {
  return static_cast<uint32_t>(__bfloat16_as_ushort(lo)) | (static_cast<uint32_t>(__bfloat16_as_ushort(hi)) << 16);
}

constexpr int kC0WinB = kC0Win + 3;   // bf16 window per input channel (odd pad keeps rows apart; zero-filled tail)

// Loads the bf16 input window of outputs [t0, t0 + kC0TT) (zero past the end of the signal).
template <int CIN>
__device__ __forceinline__ void load_window_bf16(const Conv0Args& a, int b, int t0, bf16* s_x) {
  for (int ci = 0; ci < CIN; ++ci) {
    const bf16* src = a.x + (static_cast<size_t>(b) * CIN + ci) * a.L;
    for (int i = threadIdx.x; i < kC0WinB; i += blockDim.x) {
      const long long p = static_cast<long long>(t0) * kC0S + i;
      s_x[ci * kC0WinB + i] = (i < kC0Win && p < a.L) ? src[p] : __float2bfloat16_rn(0.f);
    }
  }
}

// A fragment of the conv window matrix for outputs tl0 .. tl0+15 of the tile: A[t][k] = x[5 (tl0 + t) + k], k < 10
__device__ __forceinline__ void conv_a_frag(const bf16* sx, int tl0, int g, int tg, uint32_t (&a)[4]) {
  const bf16* r0 = sx + (tl0 + g) * kC0S + 2 * tg;
  const bf16* r1 = r0 + 8 * kC0S;
  a[0] = pack2(r0[0], r0[1]);
  a[1] = pack2(r1[0], r1[1]);
  a[2] = tg == 0 ? pack2(r0[8], r0[9]) : 0u;
  a[3] = tg == 0 ? pack2(r1[8], r1[9]) : 0u;
}

// A fragment of the TRANSPOSED window matrix: A[j][t] = x[5 (tl0 + t) + j]  (rows = taps, k = outputs), taps >= 10 zero
__device__ __forceinline__ void conv_at_frag(const bf16* sx, int tl0, int g, int tg, uint32_t (&a)[4]) {
  const bf16* c0 = sx + (tl0 + 2 * tg) * kC0S + g;          // t = 2tg, 2tg+1 ; j = g
  const bf16* c1 = c0 + 8 * kC0S;                            // t + 8
  a[0] = pack2(c0[0], c0[kC0S]);
  a[2] = pack2(c1[0], c1[kC0S]);
  a[1] = g < 2 ? pack2(c0[8], c0[kC0S + 8]) : 0u;           // j = g + 8 (taps 8, 9)
  a[3] = g < 2 ? pack2(c1[8], c1[kC0S + 8]) : 0u;
}

// channel of column j (0..7) of n-tile nt (0..7) in the 64-channel group cg
__device__ __forceinline__ int c0_chan(int cg, int nt, int j) { return cg * 64 + (j >> 1) * 16 + nt * 2 + (j & 1); }

// grid (ceil(chunks / chunks_per_block), B), block 256 = 8 warps: every warp takes one block of 16 outputs of the
// 128-output tile and ALL channels, 64 at a time.  Weights and the per-channel (scale, shift) sit in shared memory in
// FRAGMENT order ([ci][cg][nt][column g][16 taps], [cg][nt][tg]) so that the mapping above costs nothing in the loop.
template <int CIN>
__global__ void __launch_bounds__(256) conv0_fwd_kernel(Conv0Args a, const float* __restrict__ stats,
                                                        const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, bf16* __restrict__ out,
                                                        int chunks_per_block) {
  extern __shared__ __align__(16) uint8_t smem_c0[];
  bf16* s_w = reinterpret_cast<bf16*>(smem_c0);                       // [CIN][C (fragment order)][16] taps (10..15 zero)
  float4* s_p = reinterpret_cast<float4*>(s_w + CIN * a.C * 16);      // [C/2 (fragment order)] (scale0, shift0, scale1, shift1)
  bf16* s_x = reinterpret_cast<bf16*>(s_p + a.C / 2);                 // [CIN][kC0WinB]
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  for (int i = threadIdx.x; i < CIN * a.C * 16; i += blockDim.x) {
    const int k = i & 15, pos = (i >> 4) % a.C, ci = (i >> 4) / a.C;
    const int c = c0_chan(pos >> 6, (pos >> 3) & 7, pos & 7);
    s_w[i] = __float2bfloat16_rn(k < kC0K ? a.w[(static_cast<size_t>(c) * CIN + ci) * kC0K + k] : 0.f);
  }
  for (int i = threadIdx.x; i < a.C / 2; i += blockDim.x) {
    const int c = c0_chan(i >> 5, (i >> 2) & 7, 2 * (i & 3));     // pair (c, c + 1) of lane column pair tg = i & 3
    const float4 st = *reinterpret_cast<const float4*>(stats + (static_cast<size_t>(b) * a.C + c) * 2);  // m0 r0 m1 r1
    const float g0 = gamma[c] * st.y, g1 = gamma[c + 1] * st.w;
    s_p[i] = make_float4(g0, beta[c] - st.x * g0, g1, beta[c + 1] - st.z * g1);
  }
  const int n_groups = a.C / 64;
  for (int ch = 0; ch < chunks_per_block; ++ch) {
    const int t0 = (blockIdx.x * chunks_per_block + ch) * kC0TT;
    if (t0 >= a.L_out) break;
    __syncthreads();
    load_window_bf16<CIN>(a, b, t0, s_x);
    __syncthreads();
    const int tl0 = warp * 16;
    if (t0 + tl0 >= a.L_out) continue;
    uint32_t af[CIN][4];
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) conv_a_frag(s_x + ci * kC0WinB, tl0, g, tg, af[ci]);
    const int ta = t0 + tl0 + g, tb = ta + 8;
    const bool va = ta < a.L_out, vb = tb < a.L_out;
    bf16* oa = out + (static_cast<size_t>(b) * a.L_out + ta) * a.C + tg * 16;
    bf16* ob = oa + static_cast<size_t>(8) * a.C;
    for (int cg = 0; cg < n_groups; ++cg) {
      uint32_t ya[8], yb[8];   // 16 consecutive channels (cg*64 + tg*16 ..) of rows ta / tb, bf16x2 per n-tile
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
          const uint32_t* wp = reinterpret_cast<const uint32_t*>(s_w + (static_cast<size_t>(ci) * a.C + (cg * 8 + nt) * 8 + g) * 16) + tg;
          mma16816(c, af[ci], wp[0], wp[4]);
        }
        const float4 pr = s_p[(cg * 8 + nt) * 4 + tg];
        bf16_round2(c[0], c[1]);   // autocast: the conv output is bf16 before GroupNorm (fp32) sees it
        bf16_round2(c[2], c[3]);
        ya[nt] = gelu_h2(fmaf(c[0], pr.x, pr.y), fmaf(c[1], pr.z, pr.w));
        yb[nt] = gelu_h2(fmaf(c[2], pr.x, pr.y), fmaf(c[3], pr.z, pr.w));
      }
      if (va) {
        *reinterpret_cast<uint4*>(oa + cg * 64) = make_uint4(ya[0], ya[1], ya[2], ya[3]);
        *reinterpret_cast<uint4*>(oa + cg * 64 + 8) = make_uint4(ya[4], ya[5], ya[6], ya[7]);
      }
      if (vb) {
        *reinterpret_cast<uint4*>(ob + cg * 64) = make_uint4(yb[0], yb[1], yb[2], yb[3]);
        *reinterpret_cast<uint4*>(ob + cg * 64 + 8) = make_uint4(yb[4], yb[5], yb[6], yb[7]);
      }
    }
  }
}

// Backward, the one pass over dY: red[b, 0, c] += S1, red[b, 1, c] += S2, red[b, 2 + a, c] += P[a].
// Warp w owns the 64-channel group w (8 n-tiles, mapping above) and walks every 16-output block of the CTA's time
// range: conv (mma) -> hhat -> z -> gelu'(z); dz = dY * gelu'(z); S1 += dz, S2 += dz hhat;
// P^T[tap][ch] += X^T[tap][t] dz[t][ch] (mma, dz rounded to bf16 like autograd's bf16 conv weight gradient, transposed
// into a B fragment with movmatrix).  dY arrives as 2 x 16-byte loads per row per lane.
template <int CIN>
__global__ void __launch_bounds__(256, 2) conv0_bwd_kernel(Conv0Args a, const float* __restrict__ stats,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, const bf16* __restrict__ dy,
                                                           double* __restrict__ red, int chunks_per_block, int nslab) {
  constexpr int NA = CIN * kC0K;
  __shared__ __align__(16) bf16 s_x[CIN * kC0WinB];
  __shared__ float4 s_mr[256];   // (mean0, rstd0, mean1, rstd1) of channel pair i (C = 512), FRAGMENT order [warp][nt][tg]
  __shared__ float4 s_gb[256];   // (gamma0, beta0, gamma1, beta1)
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  const int c_base = warp * 64;
  // weights of this warp's 8 n-tiles as B fragments (bf16-rounded), (mean, rstd, gamma, beta) of its channel pairs
  uint32_t wb[CIN][8][2];
  for (int i = threadIdx.x; i < a.C / 2; i += blockDim.x) {
    const int c = c0_chan(i >> 5, (i >> 2) & 7, 2 * (i & 3));
    s_mr[i] = *reinterpret_cast<const float4*>(stats + (static_cast<size_t>(b) * a.C + c) * 2);
    s_gb[i] = make_float4(gamma[c], beta[c], gamma[c + 1], beta[c + 1]);
  }
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int c = c0_chan(warp, nt, g);
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) {
      const float* wr = a.w + (static_cast<size_t>(c) * CIN + ci) * kC0K;
      wb[ci][nt][0] = pack_bf16x2(wr[2 * tg], wr[2 * tg + 1]);
      wb[ci][nt][1] = tg == 0 ? pack_bf16x2(wr[8], wr[9]) : 0u;
    }
  }
  float s1[8][2], s2[8][2], pt[CIN][8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    s1[nt][0] = s1[nt][1] = s2[nt][0] = s2[nt][1] = 0.f;
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) pt[ci][nt][0] = pt[ci][nt][1] = pt[ci][nt][2] = pt[ci][nt][3] = 0.f;
  }
  for (int ch = 0; ch < chunks_per_block; ++ch) {
    const int t0 = (blockIdx.x * chunks_per_block + ch) * kC0TT;
    if (t0 >= a.L_out) break;
    __syncthreads();
    load_window_bf16<CIN>(a, b, t0, s_x);
    __syncthreads();
    const int nblk = min(kC0TT, a.L_out - t0);
    for (int tl0 = 0; tl0 < nblk; tl0 += 16) {
      uint32_t af[CIN][4], atf[CIN][4];
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) {
        conv_a_frag(s_x + ci * kC0WinB, tl0, g, tg, af[ci]);
        conv_at_frag(s_x + ci * kC0WinB, tl0, g, tg, atf[ci]);
      }
      const int ta = t0 + tl0 + g, tb = ta + 8;
      const bool va = ta < a.L_out, vb = tb < a.L_out;
      const bf16* pa = dy + (static_cast<size_t>(b) * a.L_out + ta) * a.C + c_base + tg * 16;
      const bf16* pb = pa + static_cast<size_t>(8) * a.C;
      uint32_t da[8], db[8];   // dY of this lane's 16 consecutive channels, rows ta / tb (bf16x2 per n-tile; 0 past the end)
      {
        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
        const uint4 a0 = va ? *reinterpret_cast<const uint4*>(pa) : z, a1 = va ? *reinterpret_cast<const uint4*>(pa + 8) : z;
        const uint4 b0 = vb ? *reinterpret_cast<const uint4*>(pb) : z, b1 = vb ? *reinterpret_cast<const uint4*>(pb + 8) : z;
        da[0] = a0.x; da[1] = a0.y; da[2] = a0.z; da[3] = a0.w; da[4] = a1.x; da[5] = a1.y; da[6] = a1.z; da[7] = a1.w;
        db[0] = b0.x; db[1] = b0.y; db[2] = b0.z; db[3] = b0.w; db[4] = b1.x; db[5] = b1.y; db[6] = b1.z; db[7] = b1.w;
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) mma16816(c, af[ci], wb[ci][nt][0], wb[ci][nt][1]);
        const float2 ya = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&da[nt]));
        const float2 yb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&db[nt]));
        const float4 mr = s_mr[(warp * 8 + nt) * 4 + tg];
        const float4 gb = s_gb[(warp * 8 + nt) * 4 + tg];
        bf16_round2(c[0], c[1]);
        bf16_round2(c[2], c[3]);
        const float h0 = (c[0] - mr.x) * mr.y, h1 = (c[1] - mr.z) * mr.w;
        const float h2 = (c[2] - mr.x) * mr.y, h3 = (c[3] - mr.z) * mr.w;
        const float2 ga = dgelu_h2(fmaf(h0, gb.x, gb.y), fmaf(h1, gb.z, gb.w));
        const float2 gbv = dgelu_h2(fmaf(h2, gb.x, gb.y), fmaf(h3, gb.z, gb.w));
        const float z0 = ya.x * ga.x, z1 = ya.y * ga.y, z2 = yb.x * gbv.x, z3 = yb.y * gbv.y;   // dz (0 past the end)
        s1[nt][0] += z0 + z2; s1[nt][1] += z1 + z3;
        s2[nt][0] = fmaf(z0, h0, fmaf(z2, h2, s2[nt][0]));
        s2[nt][1] = fmaf(z1, h1, fmaf(z3, h3, s2[nt][1]));
        const uint32_t b0 = movmatrix_trans(pack_bf16x2(z0, z1)), b1 = movmatrix_trans(pack_bf16x2(z2, z3));
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) mma16816(pt[ci][nt], atf[ci], b0, b1);
      }
    }
  }
  // S1 / S2: sum over the 8 lanes (g) that share a channel pair; P^T: fragments already hold sums over outputs.
  // Accumulator columns (2 tg, 2 tg + 1) of n-tile nt are channels c_base + tg * 16 + nt * 2 + {0, 1}.
  // (fp64 atomics: the weight gradient is a difference of large sums -- see the finalize kernel -- so fp32 summation-order
  // noise here showed up as ~4e-3 run-to-run differences of dW; in fp64 it is below fp32 resolution)
  // nslab > 1 (deterministic mode): every block of an instance owns a slab, so each element has ONE contributor and the
  // finalize kernel adds the slabs in order
  double* r = red + (static_cast<size_t>(b) * nslab + (nslab > 1 ? blockIdx.x : 0)) * (2 + NA) * a.C + c_base + tg * 16;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float v1 = s1[nt][e], v2 = s2[nt][e];
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        v1 += __shfl_xor_sync(0xffffffffu, v1, o);
        v2 += __shfl_xor_sync(0xffffffffu, v2, o);
      }
      if (g == 0) {
        atomicAdd(r + nt * 2 + e, static_cast<double>(v1));
        atomicAdd(r + a.C + nt * 2 + e, static_cast<double>(v2));
      }
    }
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) {
      double* rp = r + static_cast<size_t>(2 + ci * kC0K) * a.C + nt * 2;
      atomicAdd(rp + static_cast<size_t>(g) * a.C, static_cast<double>(pt[ci][nt][0]));
      atomicAdd(rp + static_cast<size_t>(g) * a.C + 1, static_cast<double>(pt[ci][nt][1]));
      if (g < 2) {
        atomicAdd(rp + static_cast<size_t>(g + 8) * a.C, static_cast<double>(pt[ci][nt][2]));
        atomicAdd(rp + static_cast<size_t>(g + 8) * a.C + 1, static_cast<double>(pt[ci][nt][3]));
      }
    }
  }
}

// Backward finalize: grid C/32, block (32, 8).  Thread (cx, by) folds instances by, by+8, ... of channel c.
template <int CIN>
__global__ void __launch_bounds__(256) conv0_bwd_finalize_kernel(Conv0Args a, const double* __restrict__ mom,
                                                                 const float* __restrict__ stats,
                                                                 const float* __restrict__ gamma,
                                                                 const double* __restrict__ red, float* __restrict__ dw,
                                                                 float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                                 int nslab) {
  constexpr int NA = CIN * kC0K;
  constexpr int NOUT = NA + NA * NA;
  __shared__ float s_m[8][NOUT];
  __shared__ float s_acc[8][32][NA + 2];
  const int cx = threadIdx.x, by = threadIdx.y;
  const int c = blockIdx.x * 32 + cx;
  const bool c_ok = c < a.C;
  float w[NA];
#pragma unroll
  for (int i = 0; i < NA; ++i) w[i] = c_ok ? bf16_round(a.w[static_cast<size_t>(c) * NA + i]) : 0.f;
  const float ga = c_ok ? gamma[c] : 0.f;
  const float invL = 1.0f / a.L_out;
  float acc[NA + 2];
#pragma unroll
  for (int i = 0; i < NA + 2; ++i) acc[i] = 0.f;
  for (int b0 = 0; b0 < a.B; b0 += 8) {
    const int b = b0 + by;
    __syncthreads();
    if (b < a.B)
      for (int i = cx; i < NOUT; i += 32) s_m[by][i] = static_cast<float>(mom[static_cast<size_t>(b) * NOUT + i]);
    __syncthreads();
    if (b < a.B && c_ok) {
      const float mean = stats[(static_cast<size_t>(b) * a.C + c) * 2], rstd = stats[(static_cast<size_t>(b) * a.C + c) * 2 + 1];
      const double* r0 = red + static_cast<size_t>(b) * nslab * (2 + NA) * a.C + c;
      // the 2 + NA sums of this (instance, channel): slabs added in slab order, the loads of one slab issued together
      double rv[2 + NA];
#pragma unroll
      for (int i = 0; i < 2 + NA; ++i) rv[i] = 0.0;
      for (int sl = 0; sl < nslab; ++sl) {
        const double* rs = r0 + static_cast<size_t>(sl) * (2 + NA) * a.C;
#pragma unroll
        for (int i = 0; i < 2 + NA; ++i) rv[i] += rs[static_cast<size_t>(i) * a.C];
      }
      const float S1 = static_cast<float>(rv[0]), S2 = static_cast<float>(rv[1]);
      const float k1 = S1 * invL, k2 = S2 * invL * rstd, sc = rstd * ga;
#pragma unroll
      for (int i = 0; i < NA; ++i) {
        float rw = 0.f;   // (R w)[i]
#pragma unroll
        for (int j = 0; j < NA; ++j) rw = fmaf(s_m[by][NA + i * NA + j], w[j], rw);
        const float q = rw - mean * s_m[by][i];            // Q[i] / rstd
        acc[i] += sc * (static_cast<float>(rv[2 + i]) - k1 * s_m[by][i] - k2 * q);
      }
      acc[NA] += S2;
      acc[NA + 1] += S1;
    }
  }
#pragma unroll
  for (int i = 0; i < NA + 2; ++i) s_acc[by][cx][i] = acc[i];
  __syncthreads();
  if (by == 0 && c_ok) {
#pragma unroll
    for (int i = 0; i < NA + 2; ++i) {
      float v = 0.f;
#pragma unroll
      for (int y = 0; y < 8; ++y) v += s_acc[y][cx][i];
      if (i < NA) dw[static_cast<size_t>(c) * NA + i] += v;
      else if (i == NA) dgamma[c] += v;
      else dbeta[c] += v;
    }
  }
}

// Data gradient, the second pass over dY (it needs S1 / S2 of every (instance, channel), which exist only after the first
// pass): per output t and channel c, with hhat, GELU' and dz recomputed exactly as in conv0_bwd_kernel,
//   dconv[t, c] = gamma rstd (dz - S1/L_out - hhat S2/L_out)          (GroupNorm backward incl. the statistics' terms)
//   part[b, t, ci*10 + j] = sum_c w_bf16[c, ci, j] dconv[t, c]          (the channel contraction, K = C, N = 10 taps)
// The accumulators of n-tiles (2p, 2p + 1) of the conv MMA are, as they stand, the A fragment of a k = 16 MMA over those 16
// channels (dconv rounded to bf16, like autocast's bf16 conv input gradient), so the contraction needs no shuffle: B is
// the bf16 weight slice [16 channels x 8 taps] (2 tap tiles, taps 10..15 zero), stored in fragment order in shared memory.
// Layout as conv0_fwd_kernel: grid (ceil(chunks / chunks_per_block), B), 8 warps each taking 16 outputs of the 128-output
// tile and all channels.  Every part row t < L_out is written by exactly one lane; the overlap-add of the two windows
// that cover a sample is left to conv0_dx_gather_kernel (no atomics: bit-identical run to run).
template <int CIN>
__global__ void __launch_bounds__(256) conv0_bwd_dx_kernel(Conv0Args a, const float* __restrict__ stats,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, const bf16* __restrict__ dy,
                                                           const double* __restrict__ red, int nslab,
                                                           float* __restrict__ part, int chunks_per_block) {
  constexpr int NA = CIN * kC0K;
  extern __shared__ __align__(16) uint8_t smem_c0[];
  uint2* s_wb = reinterpret_cast<uint2*>(smem_c0);                   // [CIN][cg 8][pair 4][tap tile 2][lane 32] (b0, b1)
  bf16* s_w = reinterpret_cast<bf16*>(s_wb + CIN * 8 * 4 * 2 * 32);   // conv weights as in conv0_fwd_kernel
  float4* s_p = reinterpret_cast<float4*>(s_w + CIN * a.C * 16);      // [C/2 (fragment order)][3]
  bf16* s_x = reinterpret_cast<bf16*>(s_p + 3 * (a.C / 2));           // [CIN][kC0WinB]
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  for (int i = threadIdx.x; i < CIN * a.C * 16; i += blockDim.x) {
    const int k = i & 15, pos = (i >> 4) % a.C, ci = (i >> 4) / a.C;
    const int c = c0_chan(pos >> 6, (pos >> 3) & 7, pos & 7);
    s_w[i] = __float2bfloat16_rn(k < kC0K ? a.w[(static_cast<size_t>(c) * CIN + ci) * kC0K + k] : 0.f);
  }
  for (int i = threadIdx.x; i < CIN * 8 * 4 * 2 * 32; i += blockDim.x) {
    const int ln = i & 31, tt = (i >> 5) & 1, p = (i >> 6) & 3, cg = (i >> 8) & 7, ci = i >> 11;
    const int tap = tt * 8 + (ln >> 2);
    const int c = c0_chan(cg, 2 * p, 2 * (ln & 3));   // k = 2tg, 2tg+1 -> c, c+1 (n-tile 2p); k + 8 -> c+2, c+3 (2p+1)
    uint2 v = make_uint2(0u, 0u);
    if (tap < kC0K) {
      const float* wc = a.w + static_cast<size_t>(c) * NA + ci * kC0K + tap;
      v.x = pack_bf16x2(wc[0], wc[NA]);
      v.y = pack_bf16x2(wc[2 * NA], wc[3 * NA]);
    }
    s_wb[i] = v;
  }
  const float invL = 1.0f / a.L_out;
  for (int i = threadIdx.x; i < a.C / 2; i += blockDim.x) {
    const int c = c0_chan(i >> 5, (i >> 2) & 7, 2 * (i & 3));
    const float4 mr = *reinterpret_cast<const float4*>(stats + (static_cast<size_t>(b) * a.C + c) * 2);
    double s[4] = {0.0, 0.0, 0.0, 0.0};   // S1(c), S1(c+1), S2(c), S2(c+1): slabs added in slab order (as the finalize)
    for (int sl = 0; sl < nslab; ++sl) {
      const double* rs = red + (static_cast<size_t>(b) * nslab + sl) * (2 + NA) * a.C + c;
      s[0] += rs[0]; s[1] += rs[1]; s[2] += rs[a.C]; s[3] += rs[a.C + 1];
    }
    s_p[3 * i + 0] = mr;                                                           // (mean0, rstd0, mean1, rstd1)
    s_p[3 * i + 1] = make_float4(gamma[c], beta[c], gamma[c + 1], beta[c + 1]);
    s_p[3 * i + 2] = make_float4(static_cast<float>(s[0]) * invL, static_cast<float>(s[2]) * invL,   // S1/L, S2/L
                                 static_cast<float>(s[1]) * invL, static_cast<float>(s[3]) * invL);
  }
  const int n_groups = a.C / 64;
  for (int ch = 0; ch < chunks_per_block; ++ch) {
    const int t0 = (blockIdx.x * chunks_per_block + ch) * kC0TT;
    if (t0 >= a.L_out) break;
    __syncthreads();
    load_window_bf16<CIN>(a, b, t0, s_x);
    __syncthreads();
    const int tl0 = warp * 16;
    if (t0 + tl0 >= a.L_out) continue;
    uint32_t af[CIN][4];
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) conv_a_frag(s_x + ci * kC0WinB, tl0, g, tg, af[ci]);
    const int ta = t0 + tl0 + g, tb = ta + 8;
    const bool va = ta < a.L_out, vb = tb < a.L_out;
    float acc[CIN][2][4];
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
      for (int tt = 0; tt < 2; ++tt) acc[ci][tt][0] = acc[ci][tt][1] = acc[ci][tt][2] = acc[ci][tt][3] = 0.f;
    for (int cg = 0; cg < n_groups; ++cg) {
      const bf16* pa = dy + (static_cast<size_t>(b) * a.L_out + ta) * a.C + cg * 64 + tg * 16;
      const bf16* pb = pa + static_cast<size_t>(8) * a.C;
      uint32_t da[8], db[8];   // dY of this lane's 16 consecutive channels, rows ta / tb (0 past the end)
      {
        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
        const uint4 a0 = va ? *reinterpret_cast<const uint4*>(pa) : z, a1 = va ? *reinterpret_cast<const uint4*>(pa + 8) : z;
        const uint4 b0 = vb ? *reinterpret_cast<const uint4*>(pb) : z, b1 = vb ? *reinterpret_cast<const uint4*>(pb + 8) : z;
        da[0] = a0.x; da[1] = a0.y; da[2] = a0.z; da[3] = a0.w; da[4] = a1.x; da[5] = a1.y; da[6] = a1.z; da[7] = a1.w;
        db[0] = b0.x; db[1] = b0.y; db[2] = b0.z; db[3] = b0.w; db[4] = b1.x; db[5] = b1.y; db[6] = b1.z; db[7] = b1.w;
      }
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        uint32_t dc[4];   // A fragment of dconv over the 16 channels of n-tiles 2p, 2p + 1
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int nt = 2 * p + h;
          float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int ci = 0; ci < CIN; ++ci) {
            const uint32_t* wp = reinterpret_cast<const uint32_t*>(s_w + (static_cast<size_t>(ci) * a.C + (cg * 8 + nt) * 8 + g) * 16) + tg;
            mma16816(c, af[ci], wp[0], wp[4]);
          }
          const float2 ya = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&da[nt]));
          const float2 yb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&db[nt]));
          const int pi = ((cg * 8 + nt) * 4 + tg) * 3;
          const float4 mr = s_p[pi], gb = s_p[pi + 1], kk = s_p[pi + 2];
          bf16_round2(c[0], c[1]);
          bf16_round2(c[2], c[3]);
          const float h0 = (c[0] - mr.x) * mr.y, h1 = (c[1] - mr.z) * mr.w;
          const float h2 = (c[2] - mr.x) * mr.y, h3 = (c[3] - mr.z) * mr.w;
          const float2 ga = dgelu_h2(fmaf(h0, gb.x, gb.y), fmaf(h1, gb.z, gb.w));
          const float2 gbv = dgelu_h2(fmaf(h2, gb.x, gb.y), fmaf(h3, gb.z, gb.w));
          const float z0 = ya.x * ga.x, z1 = ya.y * ga.y, z2 = yb.x * gbv.x, z3 = yb.y * gbv.y;   // dz
          const float sc0 = gb.x * mr.y, sc1 = gb.z * mr.w;
          // rows past the end carry no gradient (dz is 0 there, the statistics' terms are not)
          const float e0 = va ? sc0 * (z0 - kk.x - h0 * kk.y) : 0.f, e1 = va ? sc1 * (z1 - kk.z - h1 * kk.w) : 0.f;
          const float e2 = vb ? sc0 * (z2 - kk.x - h2 * kk.y) : 0.f, e3 = vb ? sc1 * (z3 - kk.z - h3 * kk.w) : 0.f;
          dc[2 * h] = pack_bf16x2(e0, e1);
          dc[2 * h + 1] = pack_bf16x2(e2, e3);
        }
        const uint32_t afr[4] = {dc[0], dc[1], dc[2], dc[3]};
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
          for (int tt = 0; tt < 2; ++tt) {
            const uint2 bw = s_wb[(((ci * 8 + cg) * 4 + p) * 2 + tt) * 32 + lane];
            mma16816(acc[ci][tt], afr, bw.x, bw.y);
          }
      }
    }
    // accumulator (row g / g + 8, taps tt*8 + 2tg, +1): taps >= 10 exist only for tt = 1, tg > 0
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
      for (int tt = 0; tt < 2; ++tt) {
        const int tap = tt * 8 + 2 * tg;
        if (tap >= kC0K) continue;
        if (va) *reinterpret_cast<float2*>(part + (static_cast<size_t>(b) * a.L_out + ta) * NA + ci * kC0K + tap) =
            make_float2(acc[ci][tt][0], acc[ci][tt][1]);
        if (vb) *reinterpret_cast<float2*>(part + (static_cast<size_t>(b) * a.L_out + tb) * NA + ci * kC0K + tap) =
            make_float2(acc[ci][tt][2], acc[ci][tt][3]);
      }
  }
}

// dx[b, ci, s] = part[b, t, ci*10 + j] + part[b, t - 1, ci*10 + j + 5] with t = s / 5, j = s % 5 (each term only where
// that output exists): the overlap-add of the two stride-5 windows covering sample s, in a fixed order.  Samples after
// the last window get 0.  One thread per sample.
template <int CIN>
__global__ void __launch_bounds__(256) conv0_dx_gather_kernel(const float* __restrict__ part, int B, int L, int L_out,
                                                              float* __restrict__ dx) {
  constexpr int NA = CIN * kC0K;
  const long long n = static_cast<long long>(B) * CIN * L;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int s = static_cast<int>(i % L);
    const long long bc = i / L;
    const int ci = static_cast<int>(bc % CIN), b = static_cast<int>(bc / CIN);
    const int t = s / kC0S, j = s - t * kC0S;
    const float* pb = part + static_cast<size_t>(b) * L_out * NA + ci * kC0K;
    float v = 0.f;
    if (t < L_out) v = pb[static_cast<size_t>(t) * NA + j];
    if (t >= 1 && t - 1 < L_out) v += pb[static_cast<size_t>(t - 1) * NA + j + kC0S];
    dx[i] = v;
  }
}

// Forward of the TF32 inference path: fp32 input and weights, fp32 FMA on the CUDA cores (Cin x 10 MAC per output),
// closed-form statistics of the unrounded conv output, exact erf GELU, fp32 channels-last [B, L_out, C] output rounded to
// nearest tf32 (it is the operand of the next conv's implicit GEMM).  (256 clips x 10 s: 16.9 GB written in 8.5 ms,
// ~2 TB/s -- short of the HBM bound; the exact erff per output is the rest, profiles/r03_bench_hear_precision.json.)
// grid (ceil(L_out / kC0F32T), B), block C / 2: thread i owns channels 2i, 2i + 1 (weights and affine in registers); a
// warp writes 256 contiguous bytes of each output row.
constexpr int kC0F32T = 64;                                 // outputs per block
constexpr int kC0F32Win = (kC0F32T - 1) * kC0S + kC0K;      // 325 samples
template <int CIN>
__global__ void __launch_bounds__(256) conv0_fwd_f32_kernel(Conv0Args a, const float* __restrict__ stats,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float* __restrict__ out) {
  constexpr int NA = CIN * kC0K;
  __shared__ float s_x[CIN][kC0F32Win];
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kC0F32T;
  const int c = 2 * threadIdx.x;
  for (int ci = 0; ci < CIN; ++ci) {
    const float* src = a.xf + (static_cast<size_t>(b) * CIN + ci) * a.L;
    for (int i = threadIdx.x; i < kC0F32Win; i += blockDim.x) {
      const long long pos = static_cast<long long>(t0) * kC0S + i;
      s_x[ci][i] = pos < a.L ? src[pos] : 0.f;
    }
  }
  float w0[NA], w1[NA];
#pragma unroll
  for (int i = 0; i < NA; ++i) {
    w0[i] = a.w[static_cast<size_t>(c) * NA + i];
    w1[i] = a.w[static_cast<size_t>(c + 1) * NA + i];
  }
  const float4 st = *reinterpret_cast<const float4*>(stats + (static_cast<size_t>(b) * a.C + c) * 2);   // m0 r0 m1 r1
  const float sc0 = gamma[c] * st.y, sc1 = gamma[c + 1] * st.w;
  const float sh0 = beta[c] - st.x * sc0, sh1 = beta[c + 1] - st.z * sc1;
  __syncthreads();
  const int nt = min(kC0F32T, a.L_out - t0);
  float* op = out + (static_cast<size_t>(b) * a.L_out + t0) * a.C + c;
#pragma unroll 4
  for (int t = 0; t < nt; ++t) {
    float y0 = 0.f, y1 = 0.f;
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) {
#pragma unroll
      for (int k = 0; k < kC0K; ++k) {
        const float xv = s_x[ci][t * kC0S + k];
        y0 = fmaf(xv, w0[ci * kC0K + k], y0);
        y1 = fmaf(xv, w1[ci * kC0K + k], y1);
      }
    }
    const float g0 = tf32_round(gelu_erf(fmaf(y0, sc0, sh0)));
    const float g1 = tf32_round(gelu_erf(fmaf(y1, sc1, sh1)));
    *reinterpret_cast<float2*>(op + static_cast<size_t>(t) * a.C) = make_float2(g0, g1);
  }
}

static int check_conv0(int Cin, int C, int k, int stride) {
  if (k != kC0K || stride != kC0S) { set_error("conv0: only k=10, stride=5 is built (got k=%d s=%d)", k, stride); return WJ_ERR_ARG; }
  if (Cin < 1 || Cin > kC0MaxCin) { set_error("conv0: Cin must be 1 or 2"); return WJ_ERR_ARG; }
  if (C != 512) { set_error("conv0: the tensor-core kernels are built for C = 512 channels (8 warps x 64); got %d", C); return WJ_ERR_ARG; }
  return WJ_OK;
}

}  // namespace wj

using namespace wj;

extern "C" int wj_conv0_moment_count(int Cin) { return conv0_moment_count(Cin); }

extern "C" int wj_conv0_gn_gelu_fwd(const void* x_bf16, const float* w, const float* gamma, const float* beta, int B,
                                    int Cin, int L, int C, int k, int stride, float eps, double* moments, float* stats,
                                    void* out_bf16, void* dgelu_bf16, void* stream) {
  if (B <= 0) return WJ_OK;
  int rc = check_conv0(Cin, C, k, stride);
  if (rc) return rc;
  cudaStream_t st = WJ_STREAM(stream);
  Conv0Args a;
  a.x = reinterpret_cast<const bf16*>(x_bf16); a.w = w; a.B = B; a.Cin = Cin; a.L = L; a.C = C; a.xf = nullptr;
  a.L_out = (L - k) / stride + 1;
  const int chunks = (a.L_out + kC0TT - 1) / kC0TT;
  const int cpb = 4;
  dim3 grid((chunks + cpb - 1) / cpb, B);
  bf16* out = reinterpret_cast<bf16*>(out_bf16);
  (void)dgelu_bf16;   // (ABI of round 1: the backward now recomputes GELU' from the input window; nothing is saved)
  const size_t smem = static_cast<size_t>(Cin) * C * 16 * 2 + static_cast<size_t>(C / 2) * 16 + static_cast<size_t>(Cin) * kC0WinB * 2 + 16;
  if (Cin == 1) {
    conv0_moments_kernel<1><<<B, 512, 0, st>>>(a, moments);
    conv0_stats_kernel<1><<<B, C, 0, st>>>(a, moments, eps, stats);
    conv0_fwd_kernel<1><<<grid, 256, smem, st>>>(a, stats, gamma, beta, out, cpb);
  } else {
    conv0_moments_kernel<2><<<B, 512, 0, st>>>(a, moments);
    conv0_stats_kernel<2><<<B, C, 0, st>>>(a, moments, eps, stats);
    conv0_fwd_kernel<2><<<grid, 256, smem, st>>>(a, stats, gamma, beta, out, cpb);
  }
  return check_launch("conv0_gn_gelu_fwd", 3);
}

extern "C" int wj_conv0_gn_gelu_bwd(const void* x_bf16, const float* w, const float* gamma, const float* beta, int B,
                                    int Cin, int L, int C, int k, int stride, float eps, const double* moments,
                                    const float* stats, const void* dy_bf16, const void* dgelu_bf16, void* red_scratch,
                                    float* dw, float* dgamma, float* dbeta, void* stream) {
  if (B <= 0) return WJ_OK;
  int rc = check_conv0(Cin, C, k, stride);
  if (rc) return rc;
  (void)eps; (void)dgelu_bf16;   // GELU' is recomputed (see the kernel); the argument is kept for ABI stability
  cudaStream_t st = WJ_STREAM(stream);
  Conv0Args a;
  a.x = reinterpret_cast<const bf16*>(x_bf16); a.w = w; a.B = B; a.Cin = Cin; a.L = L; a.C = C; a.xf = nullptr;
  a.L_out = (L - k) / stride + 1;
  const int na = Cin * kC0K;
  const int chunks = (a.L_out + kC0TT - 1) / kC0TT;
  const int cpb = 13;   // 2 + na accumulators per channel flushed with atomics at the end: few, long blocks
  dim3 grid((chunks + cpb - 1) / cpb, B);
  double* red = reinterpret_cast<double*>(red_scratch);
  int nslab = 1;
  if (det_on()) {   // one slab per block of an instance, from the deterministic-mode workspace
    nslab = static_cast<int>(grid.x);
    red = reinterpret_cast<double*>(det_ws(static_cast<size_t>(B) * nslab * (2 + na) * C * sizeof(double), &rc));
    if (rc) return rc;
  }
  cudaMemsetAsync(red, 0, static_cast<size_t>(B) * nslab * (2 + na) * C * sizeof(double), st);
  const bf16* dy = reinterpret_cast<const bf16*>(dy_bf16);
  dim3 fgrid((C + 31) / 32), fblock(32, 8);
  if (Cin == 1) {
    conv0_bwd_kernel<1><<<grid, C / 2, 0, st>>>(a, stats, gamma, beta, dy, red, cpb, nslab);
    conv0_bwd_finalize_kernel<1><<<fgrid, fblock, 0, st>>>(a, moments, stats, gamma, red, dw, dgamma, dbeta, nslab);
  } else {
    conv0_bwd_kernel<2><<<grid, C / 2, 0, st>>>(a, stats, gamma, beta, dy, red, cpb, nslab);
    conv0_bwd_finalize_kernel<2><<<fgrid, fblock, 0, st>>>(a, moments, stats, gamma, red, dw, dgamma, dbeta, nslab);
  }
  return check_launch("conv0_gn_gelu_bwd", 2);
}

// Backward of block 0 down to the waveform.  The first pass is conv0_bwd_kernel, always on per-block slabs (each sum has
// one contributor, the slabs are added in order), so S1 / S2 -- and with them dx -- are bit-identical run to run in
// either mode; then conv0_bwd_dx_kernel (second pass: the data gradient of every output's window into `part`) and the
// fixed-order overlap-add.  dw / dgamma / dbeta (all or none): the weight-gradient finalize of wj_conv0_gn_gelu_bwd.
static void conv0_dx_geometry(int B, int Cin, int L, int C, int* L_out, int* nslab, size_t* red_bytes, size_t* part_bytes) {
  *L_out = (L - kC0K) / kC0S + 1;
  const int chunks = (*L_out + kC0TT - 1) / kC0TT;
  *nslab = (chunks + 12) / 13;   // the first pass's grid.x (13 chunks per block, as wj_conv0_gn_gelu_bwd)
  *red_bytes = static_cast<size_t>(B) * *nslab * (2 + Cin * kC0K) * C * sizeof(double);
  *part_bytes = static_cast<size_t>(B) * *L_out * Cin * kC0K * sizeof(float);
}

extern "C" long long wj_conv0_bwd_dx_workspace(int B, int Cin, int L, int C) {
  if (B <= 0 || L < kC0K) return 0;
  int L_out, nslab;
  size_t rb, pb;
  conv0_dx_geometry(B, Cin, L, C, &L_out, &nslab, &rb, &pb);
  return static_cast<long long>(rb + pb);
}

extern "C" int wj_conv0_gn_gelu_bwd_dx(const void* x_bf16, const float* w, const float* gamma, const float* beta, int B,
                                       int Cin, int L, int C, int k, int stride, const double* moments, const float* stats,
                                       const void* dy_bf16, void* workspace, float* dx, float* dw, float* dgamma,
                                       float* dbeta, void* stream) {
  if (B <= 0) return WJ_OK;
  int rc = check_conv0(Cin, C, k, stride);
  if (rc) return rc;
  if (L < kC0K) { set_error("conv0_bwd_dx: input shorter than the kernel"); return WJ_ERR_ARG; }
  if (dx == nullptr || workspace == nullptr) { set_error("conv0_bwd_dx: dx and the workspace are required"); return WJ_ERR_ARG; }
  const int nw = (dw != nullptr) + (dgamma != nullptr) + (dbeta != nullptr);
  if (nw != 0 && nw != 3) { set_error("conv0_bwd_dx: dw, dgamma and dbeta are given together or not at all"); return WJ_ERR_ARG; }
  cudaStream_t st = WJ_STREAM(stream);
  Conv0Args a;
  a.x = reinterpret_cast<const bf16*>(x_bf16); a.w = w; a.B = B; a.Cin = Cin; a.L = L; a.C = C; a.xf = nullptr;
  int nslab;
  size_t red_bytes, part_bytes;
  conv0_dx_geometry(B, Cin, L, C, &a.L_out, &nslab, &red_bytes, &part_bytes);
  double* red = reinterpret_cast<double*>(workspace);
  float* part = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + red_bytes);
  cudaMemsetAsync(red, 0, red_bytes, st);
  const bf16* dy = reinterpret_cast<const bf16*>(dy_bf16);
  const int chunks = (a.L_out + kC0TT - 1) / kC0TT;
  dim3 grid1(nslab, B);
  const int cpb2 = 4;
  dim3 grid2((chunks + cpb2 - 1) / cpb2, B);
  const size_t smem2 = static_cast<size_t>(Cin) * 8 * 4 * 2 * 32 * sizeof(uint2) + static_cast<size_t>(Cin) * C * 16 * 2 +
                       static_cast<size_t>(C / 2) * 3 * 16 + static_cast<size_t>(Cin) * kC0WinB * 2 + 16;
  const long long n = static_cast<long long>(B) * Cin * L;
  const int ggrid = static_cast<int>(std::min<long long>((n + 255) / 256, 148LL * 16));
  dim3 fgrid((C + 31) / 32), fblock(32, 8);
  static bool attr_set[2] = {false, false};
  if (!attr_set[Cin - 1]) {
    const cudaError_t e = Cin == 1 ? cudaFuncSetAttribute(conv0_bwd_dx_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem2))
                                   : cudaFuncSetAttribute(conv0_bwd_dx_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem2));
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    attr_set[Cin - 1] = true;
  }
  if (Cin == 1) {
    conv0_bwd_kernel<1><<<grid1, C / 2, 0, st>>>(a, stats, gamma, beta, dy, red, 13, nslab);
    conv0_bwd_dx_kernel<1><<<grid2, 256, smem2, st>>>(a, stats, gamma, beta, dy, red, nslab, part, cpb2);
    conv0_dx_gather_kernel<1><<<ggrid, 256, 0, st>>>(part, B, L, a.L_out, dx);
    if (nw) conv0_bwd_finalize_kernel<1><<<fgrid, fblock, 0, st>>>(a, moments, stats, gamma, red, dw, dgamma, dbeta, nslab);
  } else {
    conv0_bwd_kernel<2><<<grid1, C / 2, 0, st>>>(a, stats, gamma, beta, dy, red, 13, nslab);
    conv0_bwd_dx_kernel<2><<<grid2, 256, smem2, st>>>(a, stats, gamma, beta, dy, red, nslab, part, cpb2);
    conv0_dx_gather_kernel<2><<<ggrid, 256, 0, st>>>(part, B, L, a.L_out, dx);
    if (nw) conv0_bwd_finalize_kernel<2><<<fgrid, fblock, 0, st>>>(a, moments, stats, gamma, red, dw, dgamma, dbeta, nslab);
  }
  return check_launch("conv0_gn_gelu_bwd_dx", nw ? 4 : 3);
}

// Conv block 0 of the TF32 inference path (see conv0_fwd_f32_kernel): x fp32 [B, Cin, L], out fp32 [B, L_out, C].
extern "C" int wj_conv0_gn_gelu_fwd_f32(const float* x, const float* w, const float* gamma, const float* beta, int B,
                                        int Cin, int L, int C, int k, int stride, float eps, double* moments, float* stats,
                                        float* out, void* stream) {
  if (B <= 0) return WJ_OK;
  int rc = check_conv0(Cin, C, k, stride);
  if (rc) return rc;
  if (L < k) { set_error("conv0_f32: input shorter than the kernel"); return WJ_ERR_ARG; }
  cudaStream_t st = WJ_STREAM(stream);
  Conv0Args a;
  a.x = nullptr; a.xf = x; a.w = w; a.B = B; a.Cin = Cin; a.L = L; a.C = C;
  a.L_out = (L - k) / stride + 1;
  dim3 grid((a.L_out + kC0F32T - 1) / kC0F32T, B);
  if (Cin == 1) {
    conv0_moments_kernel<1, true><<<B, 512, 0, st>>>(a, moments);
    conv0_stats_kernel<1, true><<<B, C, 0, st>>>(a, moments, eps, stats);
    conv0_fwd_f32_kernel<1><<<grid, C / 2, 0, st>>>(a, stats, gamma, beta, out);
  } else {
    conv0_moments_kernel<2, true><<<B, 512, 0, st>>>(a, moments);
    conv0_stats_kernel<2, true><<<B, C, 0, st>>>(a, moments, eps, stats);
    conv0_fwd_f32_kernel<2><<<grid, C / 2, 0, st>>>(a, stats, gamma, beta, out);
  }
  return check_launch("conv0_gn_gelu_fwd_f32", 3);
}
