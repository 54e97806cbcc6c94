// Kernels of the WavJEPA-Nat denoiser stage (SURVEY.md 8(f)-4) that are not already covered by the encoder kernels:
//   * the two dense latent MSE losses of Denoiser.forward (wavjepa/denoiser.py:352-356) with their gradient,
//   * segmental-SNR mixing of a convolved source with aggregated noise (data_modules/scene_module/
//     generate_scenes_batch.py:107-146).
// Both are HBM-bound streaming passes (grid-stride, 16-byte accesses, warp-shuffle + one atomic per block).
#include "common.cuh"

namespace wj {

// pred [2, M] (clean half, generated half), target [M]:  sums[h] += sum (pred[h] - target)^2  (fp64 accumulators);
// dpred[h] = w[h] * (pred[h] - target), w = 2 * (alpha, 1 - alpha) / M
__global__ void __launch_bounds__(256) mse_pair_kernel(const float4* __restrict__ pred, const float4* __restrict__ target,
                                                       long long m4, float w0, float w1, double* __restrict__ sums,
                                                       float4* __restrict__ dpred) {
  float s0 = 0.f, s1 = 0.f;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < m4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 t = target[i], a = pred[i], b = pred[m4 + i];
    const float4 da = make_float4(a.x - t.x, a.y - t.y, a.z - t.z, a.w - t.w);
    const float4 db = make_float4(b.x - t.x, b.y - t.y, b.z - t.z, b.w - t.w);
    s0 += da.x * da.x + da.y * da.y + da.z * da.z + da.w * da.w;
    s1 += db.x * db.x + db.y * db.y + db.z * db.z + db.w * db.w;
    if (dpred != nullptr) {
      dpred[i] = make_float4(w0 * da.x, w0 * da.y, w0 * da.z, w0 * da.w);
      dpred[m4 + i] = make_float4(w1 * db.x, w1 * db.y, w1 * db.z, w1 * db.w);
    }
  }
  __shared__ float red[2][8];
  s0 = warp_sum(s0);
  s1 = warp_sum(s1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][warp] = s0; red[1][warp] = s1; }
  __syncthreads();
  if (warp == 0) {
    float a = lane < 8 ? red[0][lane] : 0.f, b = lane < 8 ? red[1][lane] : 0.f;
    a = warp_sum(a);
    b = warp_sum(b);
    if (lane == 0) {
      atomicAdd(sums, static_cast<double>(a));
      atomicAdd(sums + 1, static_cast<double>(b));
    }
  }
}

// dpred[h] = (2 / M) * w[h] * (pred[h] - target), w [2] on the device: the backward of the two losses of mse_pair_kernel
// under autograd.  The scale is formed in fp64 and rounded once, as wj_mse_pair does on the host, so w = (alpha,
// 1 - alpha) gives mse_pair_kernel's dpred bit for bit.  One writer per element: no reduction, no atomics.
__global__ void __launch_bounds__(256) mse_pair_bwd_kernel(const float4* __restrict__ pred,
                                                           const float4* __restrict__ target, long long m4,
                                                           const float* __restrict__ w, float4* __restrict__ dpred) {
  const double m = static_cast<double>(4 * m4);
  const float w0 = static_cast<float>(2.0 * static_cast<double>(w[0]) / m);
  const float w1 = static_cast<float>(2.0 * static_cast<double>(w[1]) / m);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < m4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 t = target[i], a = pred[i], b = pred[m4 + i];
    dpred[i] = make_float4(w0 * (a.x - t.x), w0 * (a.y - t.y), w0 * (a.z - t.z), w0 * (a.w - t.w));
    dpred[m4 + i] = make_float4(w1 * (b.x - t.x), w1 * (b.y - t.y), w1 * (b.z - t.z), w1 * (b.w - t.w));
  }
}

// energy[b] = (sum source^2, sum noise^2) over the active window [start_b, start_b + len_b) of row b
__global__ void __launch_bounds__(256) snr_energy_kernel(const float* __restrict__ source, const float* __restrict__ noise,
                                                         const int* __restrict__ start, const int* __restrict__ len,
                                                         long long T, double* __restrict__ energy) {
  const int b = blockIdx.y;
  long long lo = start[b], hi = lo + len[b];
  if (lo < 0) lo = 0;
  if (hi > T) hi = T;
  const float* s = source + b * T;
  const float* n = noise + b * T;
  float es = 0.f, en = 0.f;
  for (long long i = lo + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < hi;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float x = s[i], y = n[i];
    es = fmaf(x, x, es);
    en = fmaf(y, y, en);
  }
  __shared__ float red[2][8];
  es = warp_sum(es);
  en = warp_sum(en);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][warp] = es; red[1][warp] = en; }
  __syncthreads();
  if (warp == 0) {
    float a = lane < 8 ? red[0][lane] : 0.f, c = lane < 8 ? red[1][lane] : 0.f;
    a = warp_sum(a);
    c = warp_sum(c);
    if (lane == 0) {
      atomicAdd(energy + 2 * b, static_cast<double>(a));
      atomicAdd(energy + 2 * b + 1, static_cast<double>(c));
    }
  }
}

// out = source + a_b * noise,  a_b = sqrt(E_s / (E_n + 1e-9) * 10^(-snr_b / 10))
__global__ void __launch_bounds__(256) snr_mix_kernel(const float* __restrict__ source, const float* __restrict__ noise,
                                                      const double* __restrict__ energy, const float* __restrict__ snr,
                                                      long long T, float* __restrict__ out) {
  const int b = blockIdx.y;
  const float es = static_cast<float>(energy[2 * b]), en = static_cast<float>(energy[2 * b + 1]);
  const float a = sqrtf(es / (en + 1e-9f) * powf(10.0f, -snr[b] / 10.0f));
  const float* s = source + b * T;
  const float* n = noise + b * T;
  float* o = out + b * T;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < T;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    o[i] = fmaf(a, n[i], s[i]);
}

}  // namespace wj

using namespace wj;

extern "C" int wj_mse_pair(const float* pred, const float* target, int64_t M, float alpha, double* sums, float* dpred,
                           void* stream) {
  if (M <= 0) return WJ_OK;
  if (M % 4) { set_error("wj_mse_pair: M %% 4 != 0"); return WJ_ERR_ARG; }
  const long long m4 = M / 4;
  long long blocks = (m4 + 255) / 256;
  const long long cap = static_cast<long long>(sm_count()) * 8;
  if (blocks > cap) blocks = cap;
  const float w0 = static_cast<float>(2.0 * alpha / static_cast<double>(M));
  const float w1 = static_cast<float>(2.0 * (1.0 - alpha) / static_cast<double>(M));
  mse_pair_kernel<<<static_cast<unsigned>(blocks), 256, 0, WJ_STREAM(stream)>>>(
      reinterpret_cast<const float4*>(pred), reinterpret_cast<const float4*>(target), m4, w0, w1, sums,
      reinterpret_cast<float4*>(dpred));
  return check_launch("mse_pair");
}

extern "C" int wj_mse_pair_bwd(const float* pred, const float* target, int64_t M, const float* w, float* dpred,
                               void* stream) {
  if (M <= 0) return WJ_OK;
  if (M % 4) { set_error("wj_mse_pair_bwd: M %% 4 != 0"); return WJ_ERR_ARG; }
  const long long m4 = M / 4;
  long long blocks = (m4 + 255) / 256;
  const long long cap = static_cast<long long>(sm_count()) * 8;
  if (blocks > cap) blocks = cap;
  mse_pair_bwd_kernel<<<static_cast<unsigned>(blocks), 256, 0, WJ_STREAM(stream)>>>(
      reinterpret_cast<const float4*>(pred), reinterpret_cast<const float4*>(target), m4, w,
      reinterpret_cast<float4*>(dpred));
  return check_launch("mse_pair_bwd");
}

extern "C" int wj_snr_mix(const float* source, const float* noise, const int* start, const int* length, const float* snr,
                          int B, int64_t T, double* energy, float* out, void* stream) {
  if (B <= 0 || T <= 0) return WJ_OK;
  int bx = static_cast<int>((T + 256 * 8 - 1) / (256 * 8));
  const int cap = (sm_count() * 8 + B - 1) / B;
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  cudaError_t e = cudaMemsetAsync(energy, 0, sizeof(double) * 2 * B, WJ_STREAM(stream));
  if (e != cudaSuccess) { set_error("wj_snr_mix memset: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
  snr_energy_kernel<<<dim3(bx, B), 256, 0, WJ_STREAM(stream)>>>(source, noise, start, length, T, energy);
  int rc = check_launch("snr_energy");
  if (rc != WJ_OK) return rc;
  snr_mix_kernel<<<dim3(bx, B), 256, 0, WJ_STREAM(stream)>>>(source, noise, energy, snr, T, out);
  return check_launch("snr_mix");
}
