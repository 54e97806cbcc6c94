// HBM-bound normalisation kernels: LayerNorm fwd/bwd (warp per row, row kept in registers), crop + per-instance
// normalisation of the waveform, and the teacher-target instance norm accumulated layer by layer.
//
//   LayerNorm        : nn.LayerNorm inside nn.TransformerEncoderLayer (post-norm, eps 1e-6,
//                      wavjepa/types/wavjepa_configs.py:29-47), feature_norms / encoder.norm / decoder.norm
//                      (eps 1e-5, wavjepa/jepa.py:109,127,130)
//   crop_norm        : JEPA.on_after_batch_transfer (wavjepa/jepa.py:291-311) and hear_api/runtime.py:12-16
//   target_accum     : JEPA._make_targets (wavjepa/jepa.py:230-253): F.instance_norm over (D,T) jointly per
//                      (layer, instance), then the mean over the top-K layers
#include "common.cuh"

namespace wj {

// ------------------------------------------------------------------------------------------------ LayerNorm
// TF32 (the reference-precision inference path): the addend is fp32 (add_f32) and the operand copy of the output is fp32
// rounded to nearest tf32 (out_tf32, the next GEMM's operand) instead of bf16.
template <int D, typename TIn, bool TF32 = false>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const TIn* __restrict__ x, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps, int M,
                                                            float* __restrict__ out_f32, bf16* __restrict__ out_bf16,
                                                            float* __restrict__ stats, float* __restrict__ rowsum,
                                                            const bf16* __restrict__ add,
                                                            const float* __restrict__ add_f32 = nullptr,
                                                            float* __restrict__ out_tf32 = nullptr) {
  // add (optional, bf16 [M, D]): the row normalised is x + add -- the residual sum y = x + bf16(Linear(...)) of the
  // post-norm layer, formed here in registers so that the GEMM writes 2 bytes per element and y never exists in HBM
  constexpr int PER = D / 32;  // elements per lane, contiguous chunks of 4
  static_assert(PER % 4 == 0, "D must be a multiple of 128");
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= M) return;
  const size_t base = static_cast<size_t>(warp) * D;
  float v[PER];
#pragma unroll
  for (int i = 0; i < PER / 4; ++i) {
    const int col = (i * 32 + lane) * 4;
    if constexpr (sizeof(TIn) == 4) {
      const float4 f = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + base + col);
      v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
    } else {
      const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(x) + base + col);
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
      const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
      v[4 * i] = a.x; v[4 * i + 1] = a.y; v[4 * i + 2] = b.x; v[4 * i + 3] = b.y;
    }
    if constexpr (TF32) {
      if (add_f32 != nullptr) {
        const float4 f = *reinterpret_cast<const float4*>(add_f32 + base + col);
        v[4 * i] += f.x; v[4 * i + 1] += f.y; v[4 * i + 2] += f.z; v[4 * i + 3] += f.w;
      }
    } else if (add != nullptr) {
      const uint2 u = *reinterpret_cast<const uint2*>(add + base + col);
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
      const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
      v[4 * i] += a.x; v[4 * i + 1] += a.y; v[4 * i + 2] += b.x; v[4 * i + 3] += b.y;
    }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) s += v[i];
  const float mean = warp_sum(s) * (1.0f / D);
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) { const float d = v[i] - mean; ss += d * d; }
  const float var = warp_sum(ss) * (1.0f / D);
  const float rstd = rsqrtf(var + eps);
  if (stats != nullptr && lane == 0) { stats[2 * warp] = mean; stats[2 * warp + 1] = rstd; }
  float osum = 0.f, osq = 0.f;
#pragma unroll
  for (int i = 0; i < PER / 4; ++i) {
    const int col = (i * 32 + lane) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + col));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + col));
    float4 o;
    o.x = (v[4 * i] - mean) * rstd * g.x + b.x;
    o.y = (v[4 * i + 1] - mean) * rstd * g.y + b.y;
    o.z = (v[4 * i + 2] - mean) * rstd * g.z + b.z;
    o.w = (v[4 * i + 3] - mean) * rstd * g.w + b.w;
    osum += o.x + o.y + o.z + o.w;
    osq += o.x * o.x + o.y * o.y + o.z * o.z + o.w * o.w;
    if (out_f32 != nullptr) *reinterpret_cast<float4*>(out_f32 + base + col) = o;
    if constexpr (TF32) {
      if (out_tf32 != nullptr)
        *reinterpret_cast<float4*>(out_tf32 + base + col) =
            make_float4(tf32_round(o.x), tf32_round(o.y), tf32_round(o.z), tf32_round(o.w));
    } else if (out_bf16 != nullptr) {
      uint2 u;
      u.x = pack_bf16x2(o.x, o.y);
      u.y = pack_bf16x2(o.z, o.w);
      *reinterpret_cast<uint2*>(out_bf16 + base + col) = u;
    }
  }
  if (rowsum != nullptr) {  // per-row sum / sum of squares of the OUTPUT (teacher-target instance norm)
    osum = warp_sum(osum);
    osq = warp_sum(osq);
    if (lane == 0) { rowsum[2 * warp] = osum; rowsum[2 * warp + 1] = osq; }
  }
}

// dx = rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat));  dgamma += sum_rows dy*xhat;  dbeta += sum_rows dy
// Optionally colsum += sum_rows dx (bias gradient of the Linear that produced x's non-residual branch).
template <int D, typename TIn>
__global__ void __launch_bounds__(256, (D == 384 || D == 256) ? 2 : 1) layernorm_bwd_kernel(const float* __restrict__ dy, const TIn* __restrict__ x,
                                                            const float* __restrict__ stats,
                                                            const float* __restrict__ gamma, int M,
                                                            float* __restrict__ dx_f32, bf16* __restrict__ dx_bf16,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                            float* __restrict__ colsum, int rows_per_warp,
                                                            const bf16* __restrict__ dy_b, const bf16* __restrict__ x_add,
                                                            float* __restrict__ part) {
  // part != NULL (deterministic mode): block sums go to part[pass][blockIdx.x][D]; an ordered reduction follows
  // dy (fp32, may be NULL) + dy_b (bf16, may be NULL) = gradient w.r.t. the LayerNorm output: the fp32 residual branch
  // plus the bf16 data gradient of the Linear that consumed the output.  x + x_add = the normalised row (see forward).
  constexpr int PER = D / 32;
  __shared__ float s_red[8][D];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * 8 + wib;
  float ag[PER], ab[PER], ac[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) { ag[i] = 0.f; ab[i] = 0.f; ac[i] = 0.f; }
  float g[PER];
#pragma unroll
  for (int i = 0; i < PER / 4; ++i) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(gamma + (i * 32 + lane) * 4));
    g[4 * i] = t.x; g[4 * i + 1] = t.y; g[4 * i + 2] = t.z; g[4 * i + 3] = t.w;
  }
  // D = 768: rows are software-pipelined -- the loads of row r + 1 are issued before row r's arithmetic, so each warp
  // keeps two rows of HBM requests in flight (only one 8-warp block fits an SM there, and one row per warp in flight
  // left the 19 906-row launches at half the bandwidth of the long ones).  Narrower rows keep two blocks per SM instead
  // (the second row buffer would cost the second block).
  constexpr bool PIPE = D == 768 || D == 384;   // (D = 1024 would spill; D = 384 keeps its two blocks per SM: launch bounds)
  auto load_row = [&](int row, float (&xs)[PER], float (&d)[PER], float& mean, float& rstd) {
    const size_t base = static_cast<size_t>(row) * D;
    mean = stats[2 * row];
    rstd = stats[2 * row + 1];
#pragma unroll
    for (int i = 0; i < PER / 4; ++i) {
      const int col = (i * 32 + lane) * 4;
      float4 xv;
      if constexpr (sizeof(TIn) == 4) {
        xv = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + base + col);
      } else {
        const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(x) + base + col);
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        xv = make_float4(a.x, a.y, b.x, b.y);
      }
      if (x_add != nullptr) {
        const uint2 u = *reinterpret_cast<const uint2*>(x_add + base + col);
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        xv.x += a.x; xv.y += a.y; xv.z += b.x; xv.w += b.y;
      }
      float4 dv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (dy != nullptr) dv = *reinterpret_cast<const float4*>(dy + base + col);
      if (dy_b != nullptr) {
        const uint2 u = *reinterpret_cast<const uint2*>(dy_b + base + col);
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        dv.x += a.x; dv.y += a.y; dv.z += b.x; dv.w += b.y;
      }
      xs[4 * i] = xv.x; xs[4 * i + 1] = xv.y; xs[4 * i + 2] = xv.z; xs[4 * i + 3] = xv.w;
      d[4 * i] = dv.x; d[4 * i + 1] = dv.y; d[4 * i + 2] = dv.z; d[4 * i + 3] = dv.w;
    }
  };
  const int row_lo = gw * rows_per_warp;
  const int row_hi = min(row_lo + rows_per_warp, M);
  float xh[PER], d[PER], mean = 0.f, rstd = 0.f;
  if constexpr (PIPE) {
    if (row_lo < row_hi) load_row(row_lo, xh, d, mean, rstd);
  }
  for (int row = row_lo; row < row_hi; ++row) {
    const size_t base = static_cast<size_t>(row) * D;
    float nx[PER], nd[PER], nmean = 0.f, nrstd = 0.f;
    if constexpr (PIPE) {
      if (row + 1 < row_hi) load_row(row + 1, nx, nd, nmean, nrstd);
    } else {
      load_row(row, xh, d, mean, rstd);
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      xh[i] = (xh[i] - mean) * rstd;
      ag[i] += d[i] * xh[i];
      ab[i] += d[i];
      const float gd = g[i] * d[i];
      s1 += gd;
      s2 += gd * xh[i];
    }
    s1 = warp_sum(s1) * (1.0f / D);
    s2 = warp_sum(s2) * (1.0f / D);
#pragma unroll
    for (int i = 0; i < PER / 4; ++i) {
      const int col = (i * 32 + lane) * 4;
      float4 o;
      o.x = rstd * (g[4 * i] * d[4 * i] - s1 - xh[4 * i] * s2);
      o.y = rstd * (g[4 * i + 1] * d[4 * i + 1] - s1 - xh[4 * i + 1] * s2);
      o.z = rstd * (g[4 * i + 2] * d[4 * i + 2] - s1 - xh[4 * i + 2] * s2);
      o.w = rstd * (g[4 * i + 3] * d[4 * i + 3] - s1 - xh[4 * i + 3] * s2);
      ac[4 * i] += o.x; ac[4 * i + 1] += o.y; ac[4 * i + 2] += o.z; ac[4 * i + 3] += o.w;
      if (dx_f32 != nullptr) *reinterpret_cast<float4*>(dx_f32 + base + col) = o;
      if (dx_bf16 != nullptr) {
        uint2 u;
        u.x = pack_bf16x2(o.x, o.y);
        u.y = pack_bf16x2(o.z, o.w);
        *reinterpret_cast<uint2*>(dx_bf16 + base + col) = u;
      }
    }
    if constexpr (PIPE) {
#pragma unroll
      for (int i = 0; i < PER; ++i) { xh[i] = nx[i]; d[i] = nd[i]; }
      mean = nmean;
      rstd = nrstd;
    }
  }
  // block reduction of the three column accumulators, then one atomic per column per block
  for (int pass = 0; pass < 3; ++pass) {
    float* dst = pass == 0 ? dgamma : (pass == 1 ? dbeta : colsum);
    if (dst == nullptr) continue;
    float* a = pass == 0 ? ag : (pass == 1 ? ab : ac);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < PER / 4; ++i) {
      const int col = (i * 32 + lane) * 4;
      s_red[wib][col] = a[4 * i]; s_red[wib][col + 1] = a[4 * i + 1];
      s_red[wib][col + 2] = a[4 * i + 2]; s_red[wib][col + 3] = a[4 * i + 3];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += 256) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += s_red[w][c];
      if (part != nullptr) part[(static_cast<size_t>(pass) * gridDim.x + blockIdx.x) * D + c] = t;
      else atomicAdd(dst + c, t);
    }
  }
}

// ------------------------------------------------------------------------------------------------ crop + normalise
// out[i, c, :] = (x[clip, c, start:start+Lc] - mean) / (std_unbiased + 1e-5) over (C, Lc) jointly; one block / instance.
__global__ void __launch_bounds__(512) crop_norm_kernel(const float* __restrict__ audio, const int* __restrict__ starts,
                                                        int C, long long Lfull, int S, int Lc, const float* __restrict__ gain,
                                                        bf16* __restrict__ out_bf16, float* __restrict__ out_f32) {
  __shared__ double s_red[32];
  __shared__ double s_val[2];
  const int inst = blockIdx.x;
  const int clip = inst / S;
  const long long start = starts ? starts[inst] : 0;
  const float* src = audio + static_cast<size_t>(clip) * C * Lfull;
  const int n = C * Lc;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const float gn = gain ? gain[clip] : 1.0f;  // loudness gain of hear_api/feature_helper.py:5-13 (inference only)
  auto at = [&](int i) -> float {
    const int c = i / Lc, t = i - c * Lc;
    const long long p = start + t;
    return p < Lfull ? __fmul_rn(src[static_cast<size_t>(c) * Lfull + p], gn) : 0.f;  // zero padding past the clip end (HEAR)
  };
  auto block_sum = [&](double v) -> double {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    if (warp == 0) {
      double t = lane < nw ? s_red[lane] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (lane == 0) s_val[0] = t;
    }
    __syncthreads();
    return s_val[0];
  };
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += at(i);
  const double mean = block_sum(s) / n;
  double ss = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { const double d = at(i) - mean; ss += d * d; }
  const double var = block_sum(ss) / (n - 1);
  const float fm = static_cast<float>(mean);
  const float inv = 1.0f / (static_cast<float>(sqrt(var)) + 1e-5f);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = (at(i) - fm) * inv;
    if (out_bf16) out_bf16[static_cast<size_t>(inst) * n + i] = __float2bfloat16_rn(v);
    if (out_f32) out_f32[static_cast<size_t>(inst) * n + i] = v;
  }
}

// ------------------------------------------------------------------------------------------------ teacher targets
// inst_stats[b] = {mean, rstd} over the T*D values of instance b, from per-row (sum, sumsq) pairs.
__global__ void __launch_bounds__(256) instance_stats_kernel(const float* __restrict__ rowsum, int B, int T, int D,
                                                             float eps, float* __restrict__ inst_stats) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  double s = 0.0, q = 0.0;
  for (int t = lane; t < T; t += 32) {
    s += rowsum[2 * (static_cast<size_t>(b) * T + t)];
    q += rowsum[2 * (static_cast<size_t>(b) * T + t) + 1];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  if (lane == 0) {
    const double n = static_cast<double>(T) * D;
    const double mean = s / n;
    double var = q / n - mean * mean;  // biased (F.instance_norm)
    if (var < 0.0) var = 0.0;
    inst_stats[2 * b] = static_cast<float>(mean);
    inst_stats[2 * b + 1] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  }
}

// targets (+)= scale * (x - mean_b) * rstd_b
__global__ void __launch_bounds__(256) target_accum_kernel(const float* __restrict__ x,
                                                           const float* __restrict__ inst_stats, long long n4,
                                                           int per_inst4, float scale, int first,
                                                           float* __restrict__ targets) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / per_inst4);
    const float mean = inst_stats[2 * b], rs = inst_stats[2 * b + 1] * scale;
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    float4 t = first ? make_float4(0.f, 0.f, 0.f, 0.f) : reinterpret_cast<float4*>(targets)[i];
    t.x += (v.x - mean) * rs; t.y += (v.y - mean) * rs; t.z += (v.z - mean) * rs; t.w += (v.w - mean) * rs;
    reinterpret_cast<float4*>(targets)[i] = t;
  }
}

// All K layers at once: targets = scale * sum_l (x_l - mean_{l,b}) * rstd_{l,b}: every layer output is read ONCE and the
// targets are written ONCE ((K + 1) * 4 bytes per element instead of K * 12 with the layer-by-layer accumulation).
constexpr int kMaxTargetLayers = 16;
struct TargetLayers {
  const float* x[kMaxTargetLayers];
  const float* rowsum[kMaxTargetLayers];
};
__global__ void __launch_bounds__(256) instance_stats_multi_kernel(TargetLayers L, int B, int T, int D, float eps,
                                                                   float* __restrict__ inst_stats) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31, l = blockIdx.y;
  if (b >= B) return;
  const float* rowsum = L.rowsum[l];
  double s = 0.0, q = 0.0;
  for (int t = lane; t < T; t += 32) {
    s += rowsum[2 * (static_cast<size_t>(b) * T + t)];
    q += rowsum[2 * (static_cast<size_t>(b) * T + t) + 1];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  if (lane == 0) {
    const double n = static_cast<double>(T) * D;
    const double mean = s / n;
    double var = q / n - mean * mean;  // biased (F.instance_norm)
    if (var < 0.0) var = 0.0;
    inst_stats[2 * (static_cast<size_t>(l) * B + b)] = static_cast<float>(mean);
    inst_stats[2 * (static_cast<size_t>(l) * B + b) + 1] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  }
}
template <int K>
__global__ void __launch_bounds__(256) target_combine_kernel(TargetLayers L, const float* __restrict__ inst_stats, int B,
                                                             long long n4, int per_inst4, float scale,
                                                             float* __restrict__ targets) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / per_inst4);
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int l = 0; l < K; ++l) {
      const float2 st = *reinterpret_cast<const float2*>(inst_stats + 2 * (static_cast<size_t>(l) * B + b));
      const float rs = st.y * scale;
      const float4 v = reinterpret_cast<const float4*>(L.x[l])[i];
      t.x += (v.x - st.x) * rs; t.y += (v.y - st.x) * rs; t.z += (v.z - st.x) * rs; t.w += (v.w - st.x) * rs;
    }
    reinterpret_cast<float4*>(targets)[i] = t;
  }
}

template <typename TIn>
static int launch_ln_fwd(const void* x, const float* g, const float* b, float eps, int M, int D, float* of, bf16* ob,
                         float* stats, float* rowsum, cudaStream_t st, const bf16* add = nullptr) {
  const int blocks = (M + 7) / 8;
  const TIn* xi = reinterpret_cast<const TIn*>(x);
  switch (D) {
    case 128: layernorm_fwd_kernel<128, TIn><<<blocks, 256, 0, st>>>(xi, g, b, eps, M, of, ob, stats, rowsum, add); break;
    case 256: layernorm_fwd_kernel<256, TIn><<<blocks, 256, 0, st>>>(xi, g, b, eps, M, of, ob, stats, rowsum, add); break;
    case 384: layernorm_fwd_kernel<384, TIn><<<blocks, 256, 0, st>>>(xi, g, b, eps, M, of, ob, stats, rowsum, add); break;
    case 512: layernorm_fwd_kernel<512, TIn><<<blocks, 256, 0, st>>>(xi, g, b, eps, M, of, ob, stats, rowsum, add); break;
    case 768: layernorm_fwd_kernel<768, TIn><<<blocks, 256, 0, st>>>(xi, g, b, eps, M, of, ob, stats, rowsum, add); break;
    case 1024: layernorm_fwd_kernel<1024, TIn><<<blocks, 256, 0, st>>>(xi, g, b, eps, M, of, ob, stats, rowsum, add); break;
    default: set_error("layernorm: unsupported D=%d (128,256,384,512,768,1024)", D); return WJ_ERR_ARG;
  }
  return check_launch("layernorm_fwd");
}

}  // namespace wj

using namespace wj;

extern "C" int wj_layernorm_fwd(const void* x, int x_is_bf16, const float* gamma, const float* beta, float eps, int M,
                                int D, float* out_f32, void* out_bf16, float* stats, float* rowsum, void* stream) {
  if (M <= 0) return WJ_OK;
  if (x_is_bf16) return launch_ln_fwd<bf16>(x, gamma, beta, eps, M, D, out_f32, reinterpret_cast<bf16*>(out_bf16), stats, rowsum, WJ_STREAM(stream));
  return launch_ln_fwd<float>(x, gamma, beta, eps, M, D, out_f32, reinterpret_cast<bf16*>(out_bf16), stats, rowsum, WJ_STREAM(stream));
}

template <typename TIn>
static int launch_ln_bwd(const float* dy, const void* xv, const float* stats, const float* gamma, int M, int D,
                         float* dx_f32, bf16* db, float* dgamma, float* dbeta, float* colsum, cudaStream_t st,
                         const bf16* dy_b = nullptr, const bf16* x_add = nullptr) {
  // Each warp walks a contiguous run of rows (amortises the column reductions).  Blocks are equal-sized, so the grid should
  // fill whole waves of the resident slots (1 block per SM for D >= 512, 2 below: registers): take the wave count in 4..1
  // with the fullest last wave (19 906 rows at D = 768: 147 blocks of 17 rows per warp instead of 498 = 3.4 waves,
  // 59.5 -> 48.3 us).
  const int slots = sm_count() * (D >= 512 ? 1 : 2);
  int rows_per_warp = 1;
  double best = -1.0;
  for (int w = 4; w >= 1; --w) {   // (finer blocks win ties: 172 953 rows at D = 384 measured 187 us in 2 waves, 196 in 1)
    int rpw = static_cast<int>((static_cast<long long>(M) + static_cast<long long>(slots) * 8 * w - 1) / (static_cast<long long>(slots) * 8 * w));
    if (rpw < 1) rpw = 1;
    const int nb = (M + rpw * 8 - 1) / (rpw * 8);
    const double eff = static_cast<double>(nb) / (static_cast<double>((nb + slots - 1) / slots) * slots);
    if (eff > best + 0.01) { best = eff; rows_per_warp = rpw; }
  }
  const int blocks = (M + rows_per_warp * 8 - 1) / (rows_per_warp * 8);
  const TIn* x = reinterpret_cast<const TIn*>(xv);
  int rc = WJ_OK;
  float* part = reinterpret_cast<float*>(det_ws(static_cast<size_t>(3) * blocks * D * sizeof(float), &rc));
  if (rc) return rc;
  switch (D) {
    case 128: layernorm_bwd_kernel<128, TIn><<<blocks, 256, 0, st>>>(dy, x, stats, gamma, M, dx_f32, db, dgamma, dbeta, colsum, rows_per_warp, dy_b, x_add, part); break;
    case 256: layernorm_bwd_kernel<256, TIn><<<blocks, 256, 0, st>>>(dy, x, stats, gamma, M, dx_f32, db, dgamma, dbeta, colsum, rows_per_warp, dy_b, x_add, part); break;
    case 384: layernorm_bwd_kernel<384, TIn><<<blocks, 256, 0, st>>>(dy, x, stats, gamma, M, dx_f32, db, dgamma, dbeta, colsum, rows_per_warp, dy_b, x_add, part); break;
    case 512: layernorm_bwd_kernel<512, TIn><<<blocks, 256, 0, st>>>(dy, x, stats, gamma, M, dx_f32, db, dgamma, dbeta, colsum, rows_per_warp, dy_b, x_add, part); break;
    case 768: layernorm_bwd_kernel<768, TIn><<<blocks, 256, 0, st>>>(dy, x, stats, gamma, M, dx_f32, db, dgamma, dbeta, colsum, rows_per_warp, dy_b, x_add, part); break;
    case 1024: layernorm_bwd_kernel<1024, TIn><<<blocks, 256, 0, st>>>(dy, x, stats, gamma, M, dx_f32, db, dgamma, dbeta, colsum, rows_per_warp, dy_b, x_add, part); break;
    default: set_error("layernorm_bwd: unsupported D=%d", D); return WJ_ERR_ARG;
  }
  rc = check_launch("layernorm_bwd");
  if (part != nullptr) {   // deterministic mode: add the block sums in block order
    float* dst[3] = {dgamma, dbeta, colsum};
    for (int pass = 0; pass < 3 && rc == WJ_OK; ++pass)
      if (dst[pass] != nullptr) rc = det_reduce_f32(part + static_cast<size_t>(pass) * blocks * D, blocks, 1, D, dst[pass], D, st);
  }
  return rc;
}

extern "C" int wj_layernorm_bwd(const float* dy, const void* x, int x_is_bf16, const float* stats, const float* gamma,
                                int M, int D, float* dx_f32, void* dx_bf16, float* dgamma, float* dbeta, float* colsum,
                                void* stream) {
  if (M <= 0) return WJ_OK;
  bf16* db = reinterpret_cast<bf16*>(dx_bf16);
  if (x_is_bf16) return launch_ln_bwd<bf16>(dy, x, stats, gamma, M, D, dx_f32, db, dgamma, dbeta, colsum, WJ_STREAM(stream));
  return launch_ln_bwd<float>(dy, x, stats, gamma, M, D, dx_f32, db, dgamma, dbeta, colsum, WJ_STREAM(stream));
}

extern "C" int wj_add_layernorm_fwd(const float* x, const void* add_bf16, const float* gamma, const float* beta, float eps,
                                    int M, int D, float* out_f32, void* out_bf16, float* stats, float* rowsum,
                                    void* stream) {
  if (M <= 0) return WJ_OK;
  return launch_ln_fwd<float>(x, gamma, beta, eps, M, D, out_f32, reinterpret_cast<bf16*>(out_bf16), stats, rowsum,
                              WJ_STREAM(stream), reinterpret_cast<const bf16*>(add_bf16));
}

// LayerNorm(x + add) of the TF32 inference path: x fp32, add fp32 or NULL; out_f32 = the unrounded result (residual
// stream), out_tf32 = the result rounded to nearest tf32 (the next GEMM's operand); either may be NULL.
extern "C" int wj_add_layernorm_fwd_f32(const float* x, const float* add_f32, const float* gamma, const float* beta,
                                        float eps, int M, int D, float* out_f32, float* out_tf32, void* stream) {
  if (M <= 0) return WJ_OK;
  const int blocks = (M + 7) / 8;
  cudaStream_t st = WJ_STREAM(stream);
  switch (D) {
#define WJ_LNF(DD) case DD: layernorm_fwd_kernel<DD, float, true><<<blocks, 256, 0, st>>>(x, gamma, beta, eps, M, out_f32, nullptr, nullptr, nullptr, nullptr, add_f32, out_tf32); break;
    WJ_LNF(128) WJ_LNF(256) WJ_LNF(384) WJ_LNF(512) WJ_LNF(768) WJ_LNF(1024)
#undef WJ_LNF
    default: set_error("add_layernorm_fwd_f32: unsupported D=%d (128,256,384,512,768,1024)", D); return WJ_ERR_ARG;
  }
  return check_launch("add_layernorm_fwd_f32");
}

extern "C" int wj_add_layernorm_bwd(const float* dy_f32, const void* dy_bf16, const float* x, const void* add_bf16,
                                    const float* stats, const float* gamma, int M, int D, float* dx_f32, void* dx_bf16,
                                    float* dgamma, float* dbeta, float* colsum, void* stream) {
  if (M <= 0) return WJ_OK;
  if (dy_f32 == nullptr && dy_bf16 == nullptr) { set_error("wj_add_layernorm_bwd: no output gradient given"); return WJ_ERR_ARG; }
  return launch_ln_bwd<float>(dy_f32, x, stats, gamma, M, D, dx_f32, reinterpret_cast<bf16*>(dx_bf16), dgamma, dbeta, colsum,
                              WJ_STREAM(stream), reinterpret_cast<const bf16*>(dy_bf16),
                              reinterpret_cast<const bf16*>(add_bf16));
}

extern "C" int wj_crop_norm(const float* audio, const int* starts, const float* gain, int n_clips, int channels,
                            int64_t clip_len, int crops_per_clip, int crop_len, void* out_bf16, float* out_f32,
                            void* stream) {
  const int n = n_clips * crops_per_clip;
  if (n <= 0) return WJ_OK;
  crop_norm_kernel<<<n, 512, 0, WJ_STREAM(stream)>>>(audio, starts, channels, clip_len, crops_per_clip, crop_len, gain,
                                                    reinterpret_cast<bf16*>(out_bf16), out_f32);
  return check_launch("crop_norm");
}

extern "C" int wj_target_combine(const float* const* xs, const float* const* rowsums, int n_layers, int B, int T, int D,
                                 float eps, float scale, float* inst_stats, float* targets, void* stream) {
  if (B <= 0 || n_layers <= 0) return WJ_OK;
  if (D % 4 != 0 || n_layers > kMaxTargetLayers) { set_error("wj_target_combine: D %% 4 != 0 or more than %d layers", kMaxTargetLayers); return WJ_ERR_ARG; }
  TargetLayers L;
  for (int l = 0; l < kMaxTargetLayers; ++l) { L.x[l] = l < n_layers ? xs[l] : nullptr; L.rowsum[l] = l < n_layers ? rowsums[l] : nullptr; }
  cudaStream_t st = WJ_STREAM(stream);
  instance_stats_multi_kernel<<<dim3((B + 7) / 8, n_layers), 256, 0, st>>>(L, B, T, D, eps, inst_stats);
  const long long n4 = static_cast<long long>(B) * T * D / 4;
  long long blocks = (n4 + 255) / 256;
  const long long cap = static_cast<long long>(sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  const int g = static_cast<int>(blocks);
  switch (n_layers) {
#define WJ_TC(K) case K: target_combine_kernel<K><<<g, 256, 0, st>>>(L, inst_stats, B, n4, T * D / 4, scale, targets); break;
    WJ_TC(1) WJ_TC(2) WJ_TC(3) WJ_TC(4) WJ_TC(5) WJ_TC(6) WJ_TC(7) WJ_TC(8) WJ_TC(9) WJ_TC(10) WJ_TC(11) WJ_TC(12)
    WJ_TC(13) WJ_TC(14) WJ_TC(15) WJ_TC(16)
#undef WJ_TC
  }
  return check_launch("target_combine", 2);
}

extern "C" int wj_target_accum(const float* x, const float* rowsum, int B, int T, int D, float eps, float scale,
                               int first, float* inst_stats, float* targets, void* stream) {
  if (B <= 0) return WJ_OK;
  if (D % 4 != 0) { set_error("wj_target_accum: D %% 4 != 0"); return WJ_ERR_ARG; }
  cudaStream_t st = WJ_STREAM(stream);
  instance_stats_kernel<<<(B + 7) / 8, 256, 0, st>>>(rowsum, B, T, D, eps, inst_stats);
  const long long n4 = static_cast<long long>(B) * T * D / 4;
  long long blocks = (n4 + 255) / 256;
  const long long cap = static_cast<long long>(sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  target_accum_kernel<<<static_cast<int>(blocks), 256, 0, st>>>(x, inst_stats, n4, T * D / 4, scale, first, targets);
  return check_launch("target_accum", 2);
}
