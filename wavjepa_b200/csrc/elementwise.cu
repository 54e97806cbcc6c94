// HBM-bound elementwise / gather / reduction kernels of the WavJEPA step.
//
//   gather_rows / scatter_dgelu : contextual_features[~ctx_masks] (wavjepa/jepa.py:399) and its backward
//   predictor_assemble fwd/bwd  : JEPA.decoder_forward input assembly (wavjepa/jepa.py:425-435)
//   masked_mse                  : JEPA.masked_loss (wavjepa/jepa.py:335-362), forward and d(loss)/d(pred) in one pass
//   ema_update                  : JEPA._step_teacher (wavjepa/jepa.py:193-198)
//   adamw_step / sumsq          : torch.optim.AdamW + clip_grad_norm_(5.0) (wavjepa/jepa.py:215-222, train.py:177-178)
//   cast / colsum               : bf16 working copies of the fp32 master weights; bias gradients
#include "common.cuh"

namespace wj {

__device__ __forceinline__ float4 load4(const void* p, bool is_bf16, size_t idx) {
  if (is_bf16) {
    const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(p) + idx);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
  return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + idx);
}
__device__ __forceinline__ void store4(float* of, bf16* ob, size_t idx, float4 v) {
  if (of != nullptr) *reinterpret_cast<float4*>(of + idx) = v;
  if (ob != nullptr) {
    uint2 u;
    u.x = pack_bf16x2(v.x, v.y);
    u.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(ob + idx) = u;
  }
}

__global__ void __launch_bounds__(256) gather_rows_kernel(const void* __restrict__ src, int src_bf16,
                                                          const int* __restrict__ idx, long long n4, int D4,
                                                          float* __restrict__ out_f32, bf16* __restrict__ out_bf16) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / D4;
    const int c = static_cast<int>(i - r * D4);
    const long long sr = idx ? idx[r] : r;
    const float4 v = load4(src, src_bf16, static_cast<size_t>(sr) * D4 * 4 + c * 4);
    store4(out_f32, out_bf16, static_cast<size_t>(i) * 4, v);
  }
}

// out_bf16[idx[r], :] = src_f32[r, :] * h[idx[r], :]   (h = GELU' saved by the forward epilogue; rows not listed stay as
// the caller zeroed them)
__global__ void __launch_bounds__(256) scatter_dgelu_kernel(const float* __restrict__ src, const int* __restrict__ idx,
                                                            const bf16* __restrict__ h, long long n4, int D4,
                                                            bf16* __restrict__ out) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / D4;
    const int c = static_cast<int>(i - r * D4);
    const size_t o = static_cast<size_t>(idx ? idx[r] : r) * D4 * 4 + c * 4;
    float4 v = reinterpret_cast<const float4*>(src)[i];
    if (h != nullptr) {
      const float4 hv = load4(h, true, o);
      v.x *= hv.x; v.y *= hv.y; v.z *= hv.z; v.w *= hv.w;
    }
    store4(nullptr, out, o, v);
  }
}

// out_f32[idx[r], :] = src_f32[r, :]
__global__ void __launch_bounds__(256) scatter_rows_kernel(const float* __restrict__ src, const int* __restrict__ idx,
                                                           long long n4, int D4, float* __restrict__ out) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / D4;
    const int c = static_cast<int>(i - r * D4);
    reinterpret_cast<float4*>(out)[static_cast<long long>(idx[r]) * D4 + c] = reinterpret_cast<const float4*>(src)[i];
  }
}

// a[r, :] += b[idx ? idx[r] : r, :]: one warp per row, float4 loads and stores.  Every element has one writer, so the
// sum is the same bits from run to run without a deterministic-mode variant.
__global__ void __launch_bounds__(256) add_rows_f32_kernel(float* __restrict__ a, const float* __restrict__ b,
                                                           const int* __restrict__ idx, int N, int D4) {
  const int lane = threadIdx.x & 31;
  const long long warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long r = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5; r < N; r += warps) {
    const long long sr = idx ? idx[r] : r;
    float4* ar = reinterpret_cast<float4*>(a) + r * D4;
    const float4* br = reinterpret_cast<const float4*>(b) + sr * D4;
    for (int c = lane; c < D4; c += 32) {
      float4 x = ar[c];
      const float4 y = br[c];
      x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w;
      ar[c] = x;
    }
  }
}

// gain[clip] = 10^((target_dbfs - 20 log10(rms)) / 20), rms over all channels and samples of the clip; 1 if rms == 0
__global__ void __launch_bounds__(512) clip_gain_kernel(const float* __restrict__ audio, long long per_clip,
                                                        float target_dbfs, float* __restrict__ gain) {
  __shared__ double s_red[16];
  const float* src = audio + static_cast<size_t>(blockIdx.x) * per_clip;
  double acc = 0.0;
  for (long long i = threadIdx.x; i < per_clip; i += blockDim.x) { const double v = src[i]; acc += v * v; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 16; ++w) t += s_red[w];
    const float rms = sqrtf(static_cast<float>(t / static_cast<double>(per_clip)));
    float g = 1.0f;
    if (rms != 0.f) {
      const float cur = 20.0f * log10f(rms);
      g = powf(10.0f, (target_dbfs - cur) / 20.0f);
    }
    gain[blockIdx.x] = g;
  }
}

// x0[r, :] = (src[r] >= 0 ? ctx[src[r], :] : bf16(mask_token)) + pos[pos_idx[r], :]
__global__ void __launch_bounds__(256) predictor_assemble_kernel(const bf16* __restrict__ ctx,
                                                                 const float* __restrict__ mask_token,
                                                                 const float* __restrict__ pos,
                                                                 const int* __restrict__ vis_src,
                                                                 const int* __restrict__ vis_pos, long long n4, int D4,
                                                                 float* __restrict__ out_f32,
                                                                 bf16* __restrict__ out_bf16) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / D4;
    const int c = static_cast<int>(i - r * D4) * 4;
    const int s = vis_src[r];
    float4 v;
    if (s >= 0) {
      v = load4(ctx, true, static_cast<size_t>(s) * D4 * 4 + c);
    } else {
      const float4 m = *reinterpret_cast<const float4*>(mask_token + c);
      v = make_float4(bf16_round(m.x), bf16_round(m.y), bf16_round(m.z), bf16_round(m.w));  // .type_as(bf16)
    }
    const float4 p = *reinterpret_cast<const float4*>(pos + static_cast<size_t>(vis_pos[r]) * D4 * 4 + c);
    v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
    store4(out_f32, out_bf16, static_cast<size_t>(i) * 4, v);
  }
}

// d_ctx[src[r], :] += dx0[r, :] (src >= 0);  d_mask_token += sum over rows with src < 0
__global__ void __launch_bounds__(256) predictor_assemble_bwd_kernel(const float* __restrict__ dx0,
                                                                     const int* __restrict__ vis_src, int N, int D,
                                                                     int rows_per_block, float* __restrict__ d_ctx,
                                                                     float* __restrict__ d_mask, float* __restrict__ part) {
  // thread t owns columns t, t+256, ... ; the block walks rows_per_block rows
  const int r0 = blockIdx.x * rows_per_block;
  const int r1 = min(N, r0 + rows_per_block);
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float acc = 0.f;
    for (int r = r0; r < r1; ++r) {
      const int s = vis_src[r];
      const float v = dx0[static_cast<size_t>(r) * D + c];
      if (s >= 0) {
        if (d_ctx != nullptr) atomicAdd(d_ctx + static_cast<size_t>(s) * D + c, v);
      } else {
        acc += v;
      }
    }
    if (part != nullptr) part[static_cast<size_t>(blockIdx.x) * D + c] = acc;   // deterministic mode: ordered reduce follows
    else atomicAdd(d_mask + c, acc);
  }
}

// Inverse of vis_src: ctx_vrow[src * G + g] = predictor row of context row `src` in target group g's sequence (-1 when the
// sequence does not hold it).  One block per predictor sequence.
__global__ void __launch_bounds__(128) ctx_vrows_kernel(const int* __restrict__ vis_src, const int* __restrict__ cu_v,
                                                        int G, int* __restrict__ ctx_vrow) {
  const int s = blockIdx.x, g = s % G;
  for (int r = cu_v[s] + threadIdx.x; r < cu_v[s + 1]; r += blockDim.x) {
    const int src = vis_src[r];
    if (src >= 0) ctx_vrow[static_cast<size_t>(src) * G + g] = r;
  }
}

// d_ctx[s, :] = sum over the target groups g (in order) of dx0[ctx_vrow[s * G + g], :]: the gradient of a context row is the
// sum of its copies in the G predictor sequences of its instance.  A gather with a fixed summation order -- no atomics, so
// the bf16 value handed to the student's backward is the same in every run.
__global__ void __launch_bounds__(256) predictor_ctx_grad_kernel(const float* __restrict__ dx0,
                                                                 const int* __restrict__ ctx_vrow, long long n4, int D4,
                                                                 int G, float* __restrict__ out_f32,
                                                                 bf16* __restrict__ out_bf16) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long s = i / D4;
    const int c = static_cast<int>(i - s * D4) * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int g = 0; g < G; ++g) {
      const int r = ctx_vrow[s * G + g];
      if (r >= 0) {
        const float4 v = *reinterpret_cast<const float4*>(dx0 + static_cast<size_t>(r) * D4 * 4 + c);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    }
    store4(out_f32, out_bf16, static_cast<size_t>(i) * 4, acc);
  }
}

// loss += sum_i mean_d (pred[i,d] - tgt[trow[i],d])^2 / (Nt + 1e-8);  dpred = 2 (pred - tgt) / (D (Nt + 1e-8))
__global__ void __launch_bounds__(256) masked_mse_kernel(const bf16* __restrict__ pred, const float* __restrict__ tgt,
                                                         const int* __restrict__ trow, int Nt, int D,
                                                         float* __restrict__ loss, bf16* __restrict__ dpred,
                                                         float* __restrict__ part) {
  __shared__ float s_part[8];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float denom = static_cast<float>(Nt) + 1e-8f;
  const float inv = 1.0f / (static_cast<float>(D) * denom);
  float acc = 0.f;
  for (int i = blockIdx.x * 8 + wib; i < Nt; i += gridDim.x * 8) {
    const size_t pb = static_cast<size_t>(i) * D, tb = static_cast<size_t>(trow[i]) * D;
    for (int c = lane * 4; c < D; c += 128) {
      const float4 p = load4(pred, true, pb + c);
      const float4 t = *reinterpret_cast<const float4*>(tgt + tb + c);
      const float4 d = make_float4(p.x - t.x, p.y - t.y, p.z - t.z, p.w - t.w);
      acc += d.x * d.x + d.y * d.y + d.z * d.z + d.w * d.w;
      if (dpred != nullptr) {
        const float k = 2.0f * inv;
        store4(nullptr, dpred, pb + c, make_float4(d.x * k, d.y * k, d.z * k, d.w * k));
      }
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) s_part[wib] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += s_part[w];
    if (part != nullptr) part[blockIdx.x] = t * inv;
    else atomicAdd(loss, t * inv);
  }
}

// teacher = fl(fl(teacher * r) + fl(student * q)) -- exactly teacher.mul_(r).add_((1 - r) * student) in fp32
__global__ void __launch_bounds__(256) ema_kernel(float* __restrict__ teacher, const float* __restrict__ student, float r,
                                                  float q, long long n4, long long n) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 t = reinterpret_cast<float4*>(teacher)[i];
    const float4 s = reinterpret_cast<const float4*>(student)[i];
    t.x = __fadd_rn(__fmul_rn(t.x, r), __fmul_rn(s.x, q));
    t.y = __fadd_rn(__fmul_rn(t.y, r), __fmul_rn(s.y, q));
    t.z = __fadd_rn(__fmul_rn(t.z, r), __fmul_rn(s.z, q));
    t.w = __fadd_rn(__fmul_rn(t.w, r), __fmul_rn(s.w, q));
    reinterpret_cast<float4*>(teacher)[i] = t;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (long long i = n4 * 4; i < n; ++i) teacher[i] = __fadd_rn(__fmul_rn(teacher[i], r), __fmul_rn(student[i], q));
}

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ x, long long n, float scale,
                                                    double* __restrict__ out, double* __restrict__ part) {
  __shared__ double s_part[8];
  double acc = 0.0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float v = x[i] * scale;
    acc += static_cast<double>(v) * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += s_part[w];
    if (part != nullptr) part[blockIdx.x] = t;
    else atomicAdd(out, t);
  }
}

// torch.optim.AdamW (non-amsgrad, decoupled decay) with the clip_grad_norm_ coefficient folded in:
//   g *= grad_scale * min(1, max_norm / (sqrt(sumsq) + 1e-6));  p *= 1 - lr*wd;  m,v updates;  p -= lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps)
// and, folded into the same pass over the parameters (SURVEY.md 8(f)-1): the EMA teacher update with the PRE-step
// student value, teacher[i - ema_lo] = fl(fl(teacher * r) + fl(p_old * q)) for i in [ema_lo, ema_hi)
// (JEPA._step_teacher, wavjepa/jepa.py:193-198, runs before the optimizer step in training_step :330-331), plus the bf16
// working copies of both.  One float4 per thread per array (n, ema_lo, ema_hi are multiples of 4).
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                    float* __restrict__ m, float* __restrict__ v, long long n4, float lr,
                                                    float beta1, float beta2, float eps, float wd, float bc1,
                                                    float bc2_sqrt, float grad_scale, float max_norm,
                                                    const double* __restrict__ sumsq, bf16* __restrict__ p_bf16,
                                                    float* __restrict__ teacher, bf16* __restrict__ teacher_bf16,
                                                    long long ema_lo4, long long ema_hi4, float ema_r, float ema_q,
                                                    long long n) {
  float coef = grad_scale;
  if (sumsq != nullptr && max_norm > 0.f) {
    const float total = static_cast<float>(sqrt(*sumsq));
    const float c = max_norm / (total + 1e-6f);
    coef *= fminf(c, 1.0f);
  }
  const float step = lr / bc1;
  const float decay = 1.0f - lr * wd;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 g4 = reinterpret_cast<const float4*>(g)[i];
    float4 p4 = reinterpret_cast<float4*>(p)[i];
    float4 m4 = reinterpret_cast<float4*>(m)[i];
    float4 v4 = reinterpret_cast<float4*>(v)[i];
    if (teacher != nullptr && i >= ema_lo4 && i < ema_hi4) {
      float4 t = reinterpret_cast<float4*>(teacher)[i - ema_lo4];
      t.x = __fadd_rn(__fmul_rn(t.x, ema_r), __fmul_rn(p4.x, ema_q));
      t.y = __fadd_rn(__fmul_rn(t.y, ema_r), __fmul_rn(p4.y, ema_q));
      t.z = __fadd_rn(__fmul_rn(t.z, ema_r), __fmul_rn(p4.z, ema_q));
      t.w = __fadd_rn(__fmul_rn(t.w, ema_r), __fmul_rn(p4.w, ema_q));
      reinterpret_cast<float4*>(teacher)[i - ema_lo4] = t;
      if (teacher_bf16 != nullptr) store4(nullptr, teacher_bf16, static_cast<size_t>(i - ema_lo4) * 4, t);
    }
    float* pp = reinterpret_cast<float*>(&p4);
    float* mm = reinterpret_cast<float*>(&m4);
    float* vv = reinterpret_cast<float*>(&v4);
    const float* gg = reinterpret_cast<const float*>(&g4);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gr = gg[k] * coef;
      float pv = pp[k] * decay;
      const float mv = beta1 * mm[k] + (1.0f - beta1) * gr;
      const float v2 = beta2 * vv[k] + (1.0f - beta2) * gr * gr;
      mm[k] = mv;
      vv[k] = v2;
      const float denom = sqrtf(v2) / bc2_sqrt + eps;
      pv -= step * (mv / denom);
      pp[k] = pv;
    }
    reinterpret_cast<float4*>(m)[i] = m4;
    reinterpret_cast<float4*>(v)[i] = v4;
    reinterpret_cast<float4*>(p)[i] = p4;
    if (p_bf16 != nullptr) store4(nullptr, p_bf16, static_cast<size_t>(i) * 4, p4);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {   // scalar tail (n not a multiple of 4; never inside the EMA range)
    for (long long i = n4 * 4; i < n; ++i) {
      const float gr = g[i] * coef;
      float pv = p[i] * decay;
      const float mv = beta1 * m[i] + (1.0f - beta1) * gr;
      const float v2 = beta2 * v[i] + (1.0f - beta2) * gr * gr;
      m[i] = mv;
      v[i] = v2;
      pv -= step * (mv / (sqrtf(v2) / bc2_sqrt + eps));
      p[i] = pv;
      if (p_bf16 != nullptr) p_bf16[i] = __float2bfloat16_rn(pv);
    }
  }
}

// a (fp32) += b (bf16): joins the two halves of a gradient (fp32 residual branch + bf16 Linear data gradient) where a
// consumer wants one fp32 tensor (the bottom of a transformer stack)
__global__ void __launch_bounds__(256) add_bf16_kernel(float* __restrict__ a, const bf16* __restrict__ b, long long n4) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 x = reinterpret_cast<float4*>(a)[i];
    const float4 y = load4(b, true, static_cast<size_t>(i) * 4);
    x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w;
    reinterpret_cast<float4*>(a)[i] = x;
  }
}

__global__ void __launch_bounds__(256) cast_kernel(const float* __restrict__ x, bf16* __restrict__ y, long long n) {
  const long long n4 = n / 4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    store4(nullptr, y, static_cast<size_t>(i) * 4, v);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (long long i = n4 * 4; i < n; ++i) y[i] = __float2bfloat16_rn(x[i]);
}

// out[n] += sum_m x[m, n]  (x bf16 or fp32, row-major with leading dimension ld; N % 8 == 0 fast path).
// Block (32, 8): thread (tx, ty) owns 8 consecutive columns (one 16-byte bf16 vector / two fp32 vectors) and every
// 8th row of the block's row range, 4 rows in flight; the 8 row-partials meet in smem, one atomic per column per block.
__global__ void __launch_bounds__(256) colsum8_kernel(const void* __restrict__ x, int is_bf16, long long M, int N,
                                                      long long ld, int rows_per_block, float* __restrict__ out,
                                                      float* __restrict__ part) {
  // part != NULL (deterministic mode): this row block's sums go to part[blockIdx.y][N] instead of atomics on out
  __shared__ float s_acc[8][32][9];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int c = (blockIdx.x * 32 + tx) * 8;
  const long long r0 = static_cast<long long>(blockIdx.y) * rows_per_block;
  const long long r1 = min(M, r0 + rows_per_block);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  if (c < N) {
    if (is_bf16) {
      const bf16* p = reinterpret_cast<const bf16*>(x) + c;
      long long r = r0 + ty;
      for (; r + 24 < r1; r += 32) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const uint4*>(p + (r + 8 * u) * ld);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v[u]);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 f = __bfloat1622float2(h2[t]);
            acc[2 * t] += f.x; acc[2 * t + 1] += f.y;
          }
        }
      }
      for (; r < r1; r += 8) {
        const uint4 v = *reinterpret_cast<const uint4*>(p + r * ld);
        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 f = __bfloat1622float2(h2[t]);
          acc[2 * t] += f.x; acc[2 * t + 1] += f.y;
        }
      }
    } else {
      const float* p = reinterpret_cast<const float*>(x) + c;
      for (long long r = r0 + ty; r < r1; r += 8) {
        const float4 a = *reinterpret_cast<const float4*>(p + r * ld);
        const float4 b = *reinterpret_cast<const float4*>(p + r * ld + 4);
        acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
        acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) s_acc[ty][tx][i] = acc[i];
  __syncthreads();
  // 256 threads finish 32 x 8 columns: thread (tx, ty) sums column ty of group tx over the 8 row-partials
  if (c < N) {
    float v = 0.f;
#pragma unroll
    for (int y = 0; y < 8; ++y) v += s_acc[y][tx][ty];
    if (part != nullptr) part[static_cast<size_t>(blockIdx.y) * N + c + ty] = v;
    else atomicAdd(out + c + ty, v);
  }
}

// generic fallback (N even)
__global__ void __launch_bounds__(256) colsum_kernel(const void* __restrict__ x, int is_bf16, long long M, int N,
                                                     long long ld, int rows_per_block, float* __restrict__ out,
                                                     float* __restrict__ part) {
  const long long r0 = static_cast<long long>(blockIdx.y) * rows_per_block;
  const long long r1 = min(M, r0 + rows_per_block);
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 2;
  if (c >= N) return;
  float a0 = 0.f, a1 = 0.f;
  if (is_bf16) {
    const bf16* p = reinterpret_cast<const bf16*>(x);
    for (long long r = r0; r < r1; ++r) {
      const float2 v = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p + r * ld + c));
      a0 += v.x; a1 += v.y;
    }
  } else {
    const float* p = reinterpret_cast<const float*>(x);
    for (long long r = r0; r < r1; ++r) {
      const float2 v = *reinterpret_cast<const float2*>(p + r * ld + c);
      a0 += v.x; a1 += v.y;
    }
  }
  if (part != nullptr) {
    part[static_cast<size_t>(blockIdx.y) * N + c] = a0;
    part[static_cast<size_t>(blockIdx.y) * N + c + 1] = a1;
  } else {
    atomicAdd(out + c, a0);
    atomicAdd(out + c + 1, a1);
  }
}

__global__ void __launch_bounds__(256) scale_kernel(bf16* __restrict__ x, const float* __restrict__ s, long long n) {
  const float k = *s;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    x[i] = __float2bfloat16_rn(__bfloat162float(x[i]) * k);
}

static int grid_for(long long work_items, int threads = 256, int waves = 16) {
  long long blocks = (work_items + threads - 1) / threads;
  const long long cap = static_cast<long long>(sm_count()) * waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace wj

using namespace wj;

extern "C" int wj_gather_rows(const void* src, int src_is_bf16, const int* idx, int N, int D, float* out_f32,
                              void* out_bf16, void* stream) {
  if (N <= 0) return WJ_OK;
  if (D % 4) { set_error("wj_gather_rows: D %% 4 != 0"); return WJ_ERR_ARG; }
  const long long n4 = static_cast<long long>(N) * (D / 4);
  gather_rows_kernel<<<grid_for(n4), 256, 0, WJ_STREAM(stream)>>>(src, src_is_bf16, idx, n4, D / 4, out_f32,
                                                                 reinterpret_cast<bf16*>(out_bf16));
  return check_launch("gather_rows");
}

extern "C" int wj_scatter_dgelu(const float* src, const int* idx, const void* h_bf16, int N, int D, void* out_bf16,
                                void* stream) {
  if (N <= 0) return WJ_OK;
  if (D % 4) { set_error("wj_scatter_dgelu: D %% 4 != 0"); return WJ_ERR_ARG; }
  const long long n4 = static_cast<long long>(N) * (D / 4);
  scatter_dgelu_kernel<<<grid_for(n4), 256, 0, WJ_STREAM(stream)>>>(src, idx, reinterpret_cast<const bf16*>(h_bf16), n4,
                                                                   D / 4, reinterpret_cast<bf16*>(out_bf16));
  return check_launch("scatter_dgelu");
}

extern "C" int wj_scatter_rows(const float* src, const int* idx, int N, int D, float* out, void* stream) {
  if (N <= 0) return WJ_OK;
  if (D % 4 || idx == nullptr) { set_error("wj_scatter_rows: D %% 4 != 0 or idx NULL"); return WJ_ERR_ARG; }
  const long long n4 = static_cast<long long>(N) * (D / 4);
  scatter_rows_kernel<<<grid_for(n4), 256, 0, WJ_STREAM(stream)>>>(src, idx, n4, D / 4, out);
  return check_launch("scatter_rows");
}

extern "C" int wj_add_rows_f32(float* a, const float* b, const int* idx, int N, int D, void* stream) {
  if (N <= 0) return WJ_OK;
  if (D % 4) { set_error("wj_add_rows_f32: D %% 4 != 0"); return WJ_ERR_ARG; }
  add_rows_f32_kernel<<<grid_for(static_cast<long long>(N) * 32), 256, 0, WJ_STREAM(stream)>>>(a, b, idx, N, D / 4);
  return check_launch("add_rows_f32");
}

extern "C" int wj_clip_gain(const float* audio, int n_clips, int channels, int64_t clip_len, float target_dbfs,
                            float* gain, void* stream) {
  if (n_clips <= 0) return WJ_OK;
  clip_gain_kernel<<<n_clips, 512, 0, WJ_STREAM(stream)>>>(audio, static_cast<long long>(channels) * clip_len,
                                                          target_dbfs, gain);
  return check_launch("clip_gain");
}

extern "C" int wj_predictor_assemble(const void* ctx_bf16, const float* mask_token, const float* pos,
                                     const int* vis_src, const int* vis_pos, int N, int D, float* out_f32,
                                     void* out_bf16, void* stream) {
  if (N <= 0) return WJ_OK;
  if (D % 4) { set_error("wj_predictor_assemble: D %% 4 != 0"); return WJ_ERR_ARG; }
  const long long n4 = static_cast<long long>(N) * (D / 4);
  predictor_assemble_kernel<<<grid_for(n4), 256, 0, WJ_STREAM(stream)>>>(
      reinterpret_cast<const bf16*>(ctx_bf16), mask_token, pos, vis_src, vis_pos, n4, D / 4, out_f32,
      reinterpret_cast<bf16*>(out_bf16));
  return check_launch("predictor_assemble");
}

extern "C" int wj_predictor_assemble_bwd(const float* dx0, const int* vis_src, int N, int D, float* d_ctx,
                                         float* d_mask_token, void* stream) {
  if (N <= 0) return WJ_OK;
  int rows_per_block = (N + sm_count() * 8 - 1) / (sm_count() * 8);
  if (rows_per_block < 1) rows_per_block = 1;
  const int blocks = (N + rows_per_block - 1) / rows_per_block;
  int rc = WJ_OK;
  float* part = reinterpret_cast<float*>(det_ws(static_cast<size_t>(blocks) * D * sizeof(float), &rc));
  if (rc) return rc;
  if (part != nullptr && d_ctx != nullptr) {
    set_error("wj_predictor_assemble_bwd: deterministic mode takes d_ctx = NULL (use wj_predictor_ctx_grad)");
    return WJ_ERR_ARG;
  }
  predictor_assemble_bwd_kernel<<<blocks, 256, 0, WJ_STREAM(stream)>>>(dx0, vis_src, N, D, rows_per_block, d_ctx,
                                                                      d_mask_token, part);
  rc = check_launch("predictor_assemble_bwd");
  if (rc == WJ_OK && part != nullptr) rc = det_reduce_f32(part, blocks, 1, D, d_mask_token, D, WJ_STREAM(stream));
  return rc;
}

extern "C" int wj_predictor_ctx_grad(const float* dx0, const int* vis_src, const int* cu_v, int n_seqs, int G, int Nc, int D,
                                     int* ctx_vrow, float* d_ctx_f32, void* d_ctx_bf16, void* stream) {
  if (Nc <= 0 || n_seqs <= 0) return WJ_OK;
  if (D % 4 || G <= 0) { set_error("wj_predictor_ctx_grad: D %% 4 != 0 or G <= 0"); return WJ_ERR_ARG; }
  cudaStream_t st = WJ_STREAM(stream);
  cudaMemsetAsync(ctx_vrow, 0xFF, static_cast<size_t>(Nc) * G * sizeof(int), st);
  ctx_vrows_kernel<<<n_seqs, 128, 0, st>>>(vis_src, cu_v, G, ctx_vrow);
  const long long n4 = static_cast<long long>(Nc) * (D / 4);
  predictor_ctx_grad_kernel<<<grid_for(n4), 256, 0, st>>>(dx0, ctx_vrow, n4, D / 4, G, d_ctx_f32,
                                                         reinterpret_cast<bf16*>(d_ctx_bf16));
  return check_launch("predictor_ctx_grad", 2);
}

extern "C" int wj_masked_mse(const void* pred_bf16, const float* targets, const int* tgt_rows, int Nt, int D,
                             float* loss, void* dpred_bf16, void* stream) {
  if (Nt <= 0) return WJ_OK;
  if (D % 4) { set_error("wj_masked_mse: D %% 4 != 0"); return WJ_ERR_ARG; }
  int blocks = (Nt + 7) / 8;
  const int cap = sm_count() * 8;
  if (blocks > cap) blocks = cap;
  int rc = WJ_OK;
  float* part = reinterpret_cast<float*>(det_ws(static_cast<size_t>(blocks) * sizeof(float), &rc));
  if (rc) return rc;
  masked_mse_kernel<<<blocks, 256, 0, WJ_STREAM(stream)>>>(reinterpret_cast<const bf16*>(pred_bf16), targets, tgt_rows,
                                                          Nt, D, loss, reinterpret_cast<bf16*>(dpred_bf16), part);
  rc = check_launch("masked_mse");
  if (rc == WJ_OK && part != nullptr) rc = det_reduce_f32(part, blocks, 1, 1, loss, 1, WJ_STREAM(stream));
  return rc;
}

extern "C" int wj_ema_update(float* teacher, const float* student, int64_t n, double decay, void* stream) {
  if (n <= 0) return WJ_OK;
  const float r = static_cast<float>(decay), q = static_cast<float>(1.0 - decay);
  ema_kernel<<<grid_for(n / 4 + 1), 256, 0, WJ_STREAM(stream)>>>(teacher, student, r, q, n / 4, n);
  return check_launch("ema_update");
}

extern "C" int wj_sumsq(const float* x, int64_t n, float scale, double* out, void* stream) {
  if (n <= 0) return WJ_OK;
  const int blocks = grid_for(n, 256, 8);
  int rc = WJ_OK;
  double* part = reinterpret_cast<double*>(det_ws(static_cast<size_t>(blocks) * sizeof(double), &rc));
  if (rc) return rc;
  sumsq_kernel<<<blocks, 256, 0, WJ_STREAM(stream)>>>(x, n, scale, out, part);
  rc = check_launch("sumsq");
  if (rc == WJ_OK && part != nullptr) rc = det_reduce_f64(part, blocks, 1, out, WJ_STREAM(stream));
  return rc;
}

extern "C" int wj_adamw_ema_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                                 float beta2, float eps, float weight_decay, int step, float grad_scale, float max_norm,
                                 const double* grad_sumsq, void* p_bf16, float* teacher, void* teacher_bf16,
                                 int64_t ema_lo, int64_t ema_hi, double ema_decay, void* stream) {
  if (n <= 0) return WJ_OK;
  if (teacher != nullptr && (ema_lo % 4 != 0 || ema_hi % 4 != 0 || ema_lo < 0 || ema_hi > n || ema_hi < ema_lo)) {
    set_error("wj_adamw_ema_step: the EMA range must be 4-aligned and inside [0, n) (n=%lld, [%lld, %lld))", (long long)n,
              (long long)ema_lo, (long long)ema_hi);
    return WJ_ERR_ARG;
  }
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), step);
  const double bc2 = 1.0 - pow(static_cast<double>(beta2), step);
  adamw_kernel<<<grid_for(n / 4 + 1), 256, 0, WJ_STREAM(stream)>>>(
      p, g, m, v, n / 4, lr, beta1, beta2, eps, weight_decay, static_cast<float>(bc1), static_cast<float>(sqrt(bc2)),
      grad_scale, max_norm, grad_sumsq, reinterpret_cast<bf16*>(p_bf16), teacher, reinterpret_cast<bf16*>(teacher_bf16),
      ema_lo / 4, ema_hi / 4, static_cast<float>(ema_decay), static_cast<float>(1.0 - ema_decay), n);
  return check_launch("adamw_step");
}

extern "C" int wj_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int step, float grad_scale, float max_norm,
                             const double* grad_sumsq, void* p_bf16, void* stream) {
  return wj_adamw_ema_step(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, step, grad_scale, max_norm, grad_sumsq,
                           p_bf16, nullptr, nullptr, 0, 0, 0.0, stream);
}

extern "C" int wj_add_bf16(float* a, const void* b_bf16, int64_t n, void* stream) {
  if (n <= 0) return WJ_OK;
  if (n % 4 != 0) { set_error("wj_add_bf16: n must be a multiple of 4"); return WJ_ERR_ARG; }
  add_bf16_kernel<<<grid_for(n / 4), 256, 0, WJ_STREAM(stream)>>>(a, reinterpret_cast<const bf16*>(b_bf16), n / 4);
  return check_launch("add_bf16");
}

extern "C" int wj_cast_bf16(const float* x, void* y_bf16, int64_t n, void* stream) {
  if (n <= 0) return WJ_OK;
  cast_kernel<<<grid_for(n / 4 + 1), 256, 0, WJ_STREAM(stream)>>>(x, reinterpret_cast<bf16*>(y_bf16), n);
  return check_launch("cast_bf16");
}

// y = x rounded to nearest tf32 (fp32 words with the low 13 mantissa bits zero): the working weights and the layer-0
// operand of the TF32 inference path.  y may alias x.
__global__ void tf32_round_kernel(const float* x, float* y, int64_t n) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    y[i] = tf32_round(x[i]);
}

extern "C" int wj_tf32_round(const float* x, float* y, int64_t n, void* stream) {
  if (n <= 0) return WJ_OK;
  tf32_round_kernel<<<grid_for(n), 256, 0, WJ_STREAM(stream)>>>(x, y, n);
  return check_launch("tf32_round");
}

extern "C" int wj_colsum(const void* x, int x_is_bf16, int64_t M, int N, int64_t ld, float* out, void* stream) {
  if (M <= 0) return WJ_OK;
  if (N % 2) { set_error("wj_colsum: N must be even"); return WJ_ERR_ARG; }
  const bool aligned = (reinterpret_cast<uintptr_t>(x) % 16 == 0) && (ld % 8 == 0);
  float* part = nullptr;
  int rc = WJ_OK, nb = 0;
  if (N % 8 == 0 && aligned) {
    const int bx = (N / 8 + 31) / 32;
    int by = (8 * sm_count() + bx - 1) / bx;
    if (by > (M + 31) / 32) by = static_cast<int>((M + 31) / 32);
    const int rows_per_block = static_cast<int>((M + by - 1) / by);
    by = static_cast<int>((M + rows_per_block - 1) / rows_per_block);
    part = reinterpret_cast<float*>(det_ws(static_cast<size_t>(by) * N * sizeof(float), &rc));
    if (rc) return rc;
    nb = by;
    colsum8_kernel<<<dim3(bx, by), dim3(32, 8), 0, WJ_STREAM(stream)>>>(x, x_is_bf16, M, N, ld, rows_per_block, out, part);
  } else {
    const int bx = (N / 2 + 255) / 256;
    int by = (2 * sm_count() + bx - 1) / bx;
    if (by > M) by = static_cast<int>(M);
    const int rows_per_block = static_cast<int>((M + by - 1) / by);
    by = static_cast<int>((M + rows_per_block - 1) / rows_per_block);
    part = reinterpret_cast<float*>(det_ws(static_cast<size_t>(by) * N * sizeof(float), &rc));
    if (rc) return rc;
    nb = by;
    colsum_kernel<<<dim3(bx, by), 256, 0, WJ_STREAM(stream)>>>(x, x_is_bf16, M, N, ld, rows_per_block, out, part);
  }
  rc = check_launch("colsum");
  if (rc == WJ_OK && part != nullptr) rc = det_reduce_f32(part, nb, 1, N, out, N, WJ_STREAM(stream));   // fixed order
  return rc;
}

extern "C" int wj_scale_bf16(void* x_bf16, const float* scale_dev, int64_t n, void* stream) {
  if (n <= 0) return WJ_OK;
  scale_kernel<<<grid_for(n), 256, 0, WJ_STREAM(stream)>>>(reinterpret_cast<bf16*>(x_bf16), scale_dev, n);
  return check_launch("scale_bf16");
}
