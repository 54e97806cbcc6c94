// Fused short-sequence multi-head attention over variable-length packed token sets (fwd + bwd).
//
// Reference op: F.multi_head_attention_forward -> scaled_dot_product_attention with a key-padding mask, as used by
// nn.TransformerEncoderLayer in the student / teacher / predictor stacks (built at wavjepa/jepa.py:126-130, called at
// :397, :438, :258-259).  Because the mask only hides KEYS and every other op is per token, running on the visible
// tokens alone reproduces the reference at those positions; sequences are given by cu_seqlens over a packed
// [tokens, 3*D] qkv buffer (q | k | v, head h = columns [h*DH, (h+1)*DH) of each part).
//
// Sequences are <= ~400 tokens with head dim 32/64, i.e. a few KB per (sequence, head): the kernels keep whole
// K/V (fwd) or Q/K/V/dO (bwd) in shared memory and use warp-level mma.sync.m16n8k16 bf16 tiles (the tiles are far
// below a 128-row tcgen05 atom; attention is ~4% of the step's FLOPs).  fp32 softmax, exp2 with pre-scaled logits.
#include "common.cuh"

namespace wj {

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ uint32_t lds32(const bf16* p) { return *reinterpret_cast<const uint32_t*>(p); }

__device__ __forceinline__ void ldsm_x4(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Asynchronously copies rows [0, n) x DH of one head from the packed qkv-like buffer into padded smem (cp.async, all
// requests in flight at once); rows [n, npad) are zero-filled with plain stores.
template <int DH>
__device__ __forceinline__ void load_rows_async(bf16* dst, const bf16* src, long long ld, int npad, int n) {
  constexpr int PITCH = DH + 8;
  constexpr int CH = DH / 8;  // 16-byte chunks per row
  for (int i = threadIdx.x; i < npad * CH; i += blockDim.x) {
    const int r = i / CH, c = i - r * CH;
    if (r < n) cp_async16(dst + r * PITCH + c * 8, src + static_cast<long long>(r) * ld + c * 8);
    else *reinterpret_cast<uint4*>(dst + r * PITCH + c * 8) = make_uint4(0u, 0u, 0u, 0u);
  }
}

// A-operand fragments (16 rows x DH) read straight from padded smem rows [row0, row0+16)
template <int DH>
__device__ __forceinline__ void load_a_frags(uint32_t (&f)[DH / 16][4], const bf16* s, int row0, int g, int tg) {
  constexpr int PITCH = DH + 8;
#pragma unroll
  for (int ks = 0; ks < DH / 16; ++ks) {
    const bf16* p = s + (row0 + g) * PITCH + ks * 16 + 2 * tg;
    f[ks][0] = lds32(p);
    f[ks][1] = lds32(p + 8 * PITCH);
    f[ks][2] = lds32(p + 8);
    f[ks][3] = lds32(p + 8 * PITCH + 8);
  }
}

// C[16 x 64] = A[16 x DH] * Bm[64 x DH]^T  with Bm rows in smem (row-major, padded).  Only the first `ntiles`
// 8-column tiles (rounded up to a pair) are computed; the others are zeroed.  B fragments come from ldmatrix.x4:
// one instruction feeds two n-tiles of one 16-deep k-step.
template <int DH, int NT = 8>
__device__ __forceinline__ void mm_abT(float (&c)[NT][4], const uint32_t (&a)[DH / 16][4], const bf16* sB, int brow0,
                                       int lane, int ntiles) {
  constexpr int PITCH = DH + 8;
  const bf16* base = sB + (brow0 + (lane & 7) + ((lane >> 4) << 3)) * PITCH + ((lane >> 3) & 1) * 8;
#pragma unroll
  for (int nt = 0; nt < NT; nt += 2) {
    c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
    c[nt + 1][0] = c[nt + 1][1] = c[nt + 1][2] = c[nt + 1][3] = 0.f;
    if (nt < ntiles) {
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4(b0, b1, b2, b3, base + nt * 8 * PITCH + ks * 16);
        mma16816(c[nt], a[ks], b0, b1);
        mma16816(c[nt + 1], a[ks], b2, b3);
      }
    }
  }
}

// acc[16 x DH] += P[16 x 64] * Bm[64 x DH]  (P given as C-fragments, packed on the fly; Bm rows in smem); only the
// first `kchunks` 16-row chunks of Bm contribute.
template <int DH, int NT = 8>
__device__ __forceinline__ void mm_pb(float (&acc)[DH / 8][4], const float (&pf)[NT][4], const bf16* sB, int brow0,
                                      int lane, int kchunks) {
  constexpr int PITCH = DH + 8;
#pragma unroll
  for (int kk = 0; kk < NT / 2; ++kk) {
    if (kk < kchunks) {
      uint32_t a[4];
      a[0] = pack_bf16x2(pf[2 * kk][0], pf[2 * kk][1]);
      a[1] = pack_bf16x2(pf[2 * kk][2], pf[2 * kk][3]);
      a[2] = pack_bf16x2(pf[2 * kk + 1][0], pf[2 * kk + 1][1]);
      a[3] = pack_bf16x2(pf[2 * kk + 1][2], pf[2 * kk + 1][3]);
#pragma unroll
      for (int dt = 0; dt < DH / 8; dt += 2) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4_trans(b0, b1, b2, b3, sB + (brow0 + kk * 16 + (lane & 15)) * PITCH + dt * 8 + ((lane >> 4) << 3));
        mma16816(acc[dt], a, b0, b1);
        mma16816(acc[dt + 1], a, b2, b3);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ forward
// One CTA per (sequence, head): Q, K, V of the whole sequence are brought into smem once (cp.async, one wait), then
// every warp walks its 16-query blocks over 64-key blocks with an online softmax; no block-level sync in the loop.
template <int DH>
__global__ void __launch_bounds__(256) attn_fwd_kernel(const bf16* __restrict__ qkv, const int* __restrict__ cu, int D,
                                                       int H, int NPAD, float scale_log2, bf16* __restrict__ out,
                                                       float* __restrict__ lse2) {
  constexpr int PITCH = DH + 8;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  bf16* sQ = reinterpret_cast<bf16*>(smem_attn);
  bf16* sK = sQ + NPAD * PITCH;
  bf16* sV = sK + NPAD * PITCH;
  const int s = blockIdx.y, h = blockIdx.x;
  const int start = cu[s], n = cu[s + 1] - start;
  if (n <= 0) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  const int nwarps = blockDim.x >> 5;
  const long long ld = 3LL * D;
  const bf16* base = qkv + static_cast<long long>(start) * ld + h * DH;
  const int npad = (n + 15) & ~15;
  load_rows_async<DH>(sQ, base, ld, npad, n);
  load_rows_async<DH>(sK, base + D, ld, npad, n);
  load_rows_async<DH>(sV, base + 2 * D, ld, npad, n);
  cp_async_wait_all();
  __syncthreads();
  for (int qb = warp; qb * 16 < n; qb += nwarps) {
    uint32_t qf[DH / 16][4];
    load_a_frags<DH>(qf, sQ, qb * 16, g, tg);
    float o[DH / 8][4];
#pragma unroll
    for (int i = 0; i < DH / 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    for (int kb = 0; kb * 64 < n; ++kb) {
      const int valid = min(64, n - kb * 64);
      float sc[8][4];
      mm_abT<DH>(sc, qf, sK, kb * 64, lane, (valid + 7) >> 3);
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int key = nt * 8 + 2 * tg;
        sc[nt][0] = key < valid ? sc[nt][0] * scale_log2 : -INFINITY;
        sc[nt][1] = key + 1 < valid ? sc[nt][1] * scale_log2 : -INFINITY;
        sc[nt][2] = key < valid ? sc[nt][2] * scale_log2 : -INFINITY;
        sc[nt][3] = key + 1 < valid ? sc[nt][3] * scale_log2 : -INFINITY;
        mx0 = fmaxf(mx0, fmaxf(sc[nt][0], sc[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(sc[nt][2], sc[nt][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);  // finite: key kb*64 < n is always valid
      const float al0 = ex2_approx(m0 - mn0), al1 = ex2_approx(m1 - mn1);
      m0 = mn0; m1 = mn1;
      float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        sc[nt][0] = ex2_approx(sc[nt][0] - mn0); sc[nt][1] = ex2_approx(sc[nt][1] - mn0);
        sc[nt][2] = ex2_approx(sc[nt][2] - mn1); sc[nt][3] = ex2_approx(sc[nt][3] - mn1);
        rs0 += sc[nt][0] + sc[nt][1];
        rs1 += sc[nt][2] + sc[nt][3];
      }
      l0 = l0 * al0 + rs0;
      l1 = l1 * al1 + rs1;
#pragma unroll
      for (int i = 0; i < DH / 8; ++i) { o[i][0] *= al0; o[i][1] *= al0; o[i][2] *= al1; o[i][3] *= al1; }
      mm_pb<DH>(o, sc, sV, kb * 64, lane, (valid + 15) >> 4);
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const int ra = qb * 16 + g, rb = ra + 8;
    const float i0 = 1.0f / l0, i1 = 1.0f / l1;
    if (ra < n) {
      bf16* op = out + static_cast<long long>(start + ra) * D + h * DH + 2 * tg;
#pragma unroll
      for (int dt = 0; dt < DH / 8; ++dt) *reinterpret_cast<uint32_t*>(op + dt * 8) = pack_bf16x2(o[dt][0] * i0, o[dt][1] * i0);
      if (lse2 != nullptr && tg == 0) lse2[static_cast<long long>(start + ra) * H + h] = m0 + log2f(l0);
    }
    if (rb < n) {
      bf16* op = out + static_cast<long long>(start + rb) * D + h * DH + 2 * tg;
#pragma unroll
      for (int dt = 0; dt < DH / 8; ++dt) *reinterpret_cast<uint32_t*>(op + dt * 8) = pack_bf16x2(o[dt][2] * i1, o[dt][3] * i1);
      if (lse2 != nullptr && tg == 0) lse2[static_cast<long long>(start + rb) * H + h] = m1 + log2f(l1);
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward
// One CTA per (sequence, head); Q, K, V, dO of the whole sequence live in smem (NPAD rows each).
//   phase A: warps own 16-query blocks -> dQ;  phase B: warps own 16-key blocks -> dK, dV.  No atomics.
// ROWSTATS: the per-query lse / delta live in the padding columns of the Q rows (floats at column DH, DH + 2) instead of
// two arrays after dO -- 3.5 KB less shared memory, which lets sequences of up to 400 tokens at head dim 64 (the dense
// WavJEPA-Nat student: two channels x 200 tokens) stay resident; rows past the Q block read as zeros.
template <int DH, bool ROWSTATS = false>
__global__ void __launch_bounds__(128, (DH == 32 ? 4 : 3)) attn_bwd_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ out,
                                                       const bf16* __restrict__ dout, const float* __restrict__ lse2,
                                                       const int* __restrict__ cu, int D, int H, int NPAD, float scale,
                                                       float scale_log2, bf16* __restrict__ dqkv) {
  constexpr int PITCH = DH + 8;
  constexpr int NT = 4;                    // 8-wide tiles per inner block: 32-wide blocks keep the DH=32 kernel at
  constexpr int KB = NT * 8;               // <= 128 registers (4 CTAs / SM); the lse / delta arrays stay padded to 64
  extern __shared__ __align__(16) uint8_t smem_attn[];
  bf16* sQ = reinterpret_cast<bf16*>(smem_attn);
  bf16* sK = sQ + NPAD * PITCH;
  bf16* sV = sK + NPAD * PITCH;
  bf16* sdO = sV + NPAD * PITCH;
  float* sLse = reinterpret_cast<float*>(sdO + NPAD * PITCH);
  float* sDl = sLse + ((NPAD + 63) & ~63);   // lse / delta rows are read in 64-query blocks: padded (zeros) to 64
  auto stat = [&](const float* arr, int i, int which) -> float {
    if constexpr (ROWSTATS) return i < NPAD ? reinterpret_cast<const float*>(sQ + i * PITCH + DH)[which] : 0.f;
    else return arr[i];
  };
  const int s = blockIdx.y, h = blockIdx.x;
  const int start = cu[s], n = cu[s + 1] - start;
  if (n <= 0) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  const int nwarps = blockDim.x >> 5;
  const long long ld = 3LL * D;
  const bf16* base = qkv + static_cast<long long>(start) * ld + h * DH;
  const int npad = (n + 15) & ~15;
  load_rows_async<DH>(sQ, base, ld, npad, n);
  load_rows_async<DH>(sK, base + D, ld, npad, n);
  load_rows_async<DH>(sV, base + 2 * D, ld, npad, n);
  load_rows_async<DH>(sdO, dout + static_cast<long long>(start) * D + h * DH, D, npad, n);
  for (int i = threadIdx.x; i < ((n + 63) & ~63); i += blockDim.x) {
    float dsum = 0.f, l = 0.f;
    if (i < n) {
      const bf16* op = out + static_cast<long long>(start + i) * D + h * DH;
      const bf16* dp = dout + static_cast<long long>(start + i) * D + h * DH;
#pragma unroll
      for (int c = 0; c < DH; c += 8) {
        const uint4 a = *reinterpret_cast<const uint4*>(op + c);
        const uint4 b = *reinterpret_cast<const uint4*>(dp + c);
        const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&a);
        const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&b);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 x = __bfloat1622float2(a2[t]), y = __bfloat1622float2(b2[t]);
          dsum += x.x * y.x + x.y * y.y;
        }
      }
      l = lse2[static_cast<long long>(start + i) * H + h];
    }
    if constexpr (ROWSTATS) {
      if (i < NPAD) {
        float* rp = reinterpret_cast<float*>(sQ + i * PITCH + DH);
        rp[0] = l;
        rp[1] = dsum;
      }
    } else {
      sLse[i] = l;
      sDl[i] = dsum;
    }
  }
  cp_async_wait_all();
  __syncthreads();

  // ---------------------------------------------------------------- phase A: dQ
  for (int rb = warp; rb * 16 < n; rb += nwarps) {
    uint32_t qf[DH / 16][4], dof[DH / 16][4];
    load_a_frags<DH>(qf, sQ, rb * 16, g, tg);
    load_a_frags<DH>(dof, sdO, rb * 16, g, tg);
    const float la = stat(sLse, rb * 16 + g, 0), lb = stat(sLse, rb * 16 + g + 8, 0);
    const float da = stat(sDl, rb * 16 + g, 1), db = stat(sDl, rb * 16 + g + 8, 1);
    float dq[DH / 8][4];
#pragma unroll
    for (int i = 0; i < DH / 8; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
    for (int kb = 0; kb * KB < n; ++kb) {
      float sc[NT][4], dp[NT][4];
      const int valid = min(KB, n - kb * KB);
      mm_abT<DH, NT>(sc, qf, sK, kb * KB, lane, (valid + 7) >> 3);
      mm_abT<DH, NT>(dp, dof, sV, kb * KB, lane, (valid + 7) >> 3);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const int key = kb * KB + nt * 8 + 2 * tg;
        const float p0 = key < n ? ex2_approx(sc[nt][0] * scale_log2 - la) : 0.f;
        const float p1 = key + 1 < n ? ex2_approx(sc[nt][1] * scale_log2 - la) : 0.f;
        const float p2 = key < n ? ex2_approx(sc[nt][2] * scale_log2 - lb) : 0.f;
        const float p3 = key + 1 < n ? ex2_approx(sc[nt][3] * scale_log2 - lb) : 0.f;
        sc[nt][0] = p0 * (dp[nt][0] - da); sc[nt][1] = p1 * (dp[nt][1] - da);
        sc[nt][2] = p2 * (dp[nt][2] - db); sc[nt][3] = p3 * (dp[nt][3] - db);
      }
      mm_pb<DH, NT>(dq, sc, sK, kb * KB, lane, (valid + 15) >> 4);
    }
    const int ra = rb * 16 + g, rbb = ra + 8;
    if (ra < n) {
      bf16* op = dqkv + static_cast<long long>(start + ra) * ld + h * DH + 2 * tg;
#pragma unroll
      for (int dt = 0; dt < DH / 8; ++dt) *reinterpret_cast<uint32_t*>(op + dt * 8) = pack_bf16x2(dq[dt][0] * scale, dq[dt][1] * scale);
    }
    if (rbb < n) {
      bf16* op = dqkv + static_cast<long long>(start + rbb) * ld + h * DH + 2 * tg;
#pragma unroll
      for (int dt = 0; dt < DH / 8; ++dt) *reinterpret_cast<uint32_t*>(op + dt * 8) = pack_bf16x2(dq[dt][2] * scale, dq[dt][3] * scale);
    }
  }

  // ---------------------------------------------------------------- phase B: dK, dV
  for (int cb = warp; cb * 16 < n; cb += nwarps) {
    uint32_t kf[DH / 16][4], vf[DH / 16][4];
    load_a_frags<DH>(kf, sK, cb * 16, g, tg);
    load_a_frags<DH>(vf, sV, cb * 16, g, tg);
    float dk[DH / 8][4], dv[DH / 8][4];
#pragma unroll
    for (int i = 0; i < DH / 8; ++i) {
      dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
      dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
    }
    const bool ka = cb * 16 + g < n, kbv = cb * 16 + g + 8 < n;
    for (int qb = 0; qb * KB < n; ++qb) {
      float st[NT][4], dpt[NT][4];
      const int valid = min(KB, n - qb * KB);
      mm_abT<DH, NT>(st, kf, sQ, qb * KB, lane, (valid + 7) >> 3);     // S^T tile: rows = keys, cols = queries
      mm_abT<DH, NT>(dpt, vf, sdO, qb * KB, lane, (valid + 7) >> 3);   // dP^T tile
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const int q = qb * KB + nt * 8 + 2 * tg;
        const float l0 = stat(sLse, q, 0), l1 = stat(sLse, q + 1, 0), d0 = stat(sDl, q, 1), d1 = stat(sDl, q + 1, 1);
        const bool q0 = q < n, q1 = q + 1 < n;
        const float p0 = (ka && q0) ? ex2_approx(st[nt][0] * scale_log2 - l0) : 0.f;
        const float p1 = (ka && q1) ? ex2_approx(st[nt][1] * scale_log2 - l1) : 0.f;
        const float p2 = (kbv && q0) ? ex2_approx(st[nt][2] * scale_log2 - l0) : 0.f;
        const float p3 = (kbv && q1) ? ex2_approx(st[nt][3] * scale_log2 - l1) : 0.f;
        st[nt][0] = p0; st[nt][1] = p1; st[nt][2] = p2; st[nt][3] = p3;
        dpt[nt][0] = p0 * (dpt[nt][0] - d0); dpt[nt][1] = p1 * (dpt[nt][1] - d1);
        dpt[nt][2] = p2 * (dpt[nt][2] - d0); dpt[nt][3] = p3 * (dpt[nt][3] - d1);
      }
      mm_pb<DH, NT>(dv, st, sdO, qb * KB, lane, (valid + 15) >> 4);
      mm_pb<DH, NT>(dk, dpt, sQ, qb * KB, lane, (valid + 15) >> 4);
    }
    const int ra = cb * 16 + g, rbb = ra + 8;
    if (ra < n) {
      bf16* kp = dqkv + static_cast<long long>(start + ra) * ld + D + h * DH + 2 * tg;
      bf16* vp = kp + D;
#pragma unroll
      for (int dt = 0; dt < DH / 8; ++dt) {
        *reinterpret_cast<uint32_t*>(kp + dt * 8) = pack_bf16x2(dk[dt][0] * scale, dk[dt][1] * scale);
        *reinterpret_cast<uint32_t*>(vp + dt * 8) = pack_bf16x2(dv[dt][0], dv[dt][1]);
      }
    }
    if (rbb < n) {
      bf16* kp = dqkv + static_cast<long long>(start + rbb) * ld + D + h * DH + 2 * tg;
      bf16* vp = kp + D;
#pragma unroll
      for (int dt = 0; dt < DH / 8; ++dt) {
        *reinterpret_cast<uint32_t*>(kp + dt * 8) = pack_bf16x2(dk[dt][2] * scale, dk[dt][3] * scale);
        *reinterpret_cast<uint32_t*>(vp + dt * 8) = pack_bf16x2(dv[dt][2], dv[dt][3]);
      }
    }
  }
}

}  // namespace wj

using namespace wj;

namespace wj {
int attn_fwd_tc_launch(const void* qkv, const int* cu, int n_seqs, int max_len, long long total_tokens, int D, int H,
                       void* out, float* lse2, cudaStream_t st, float* out_f32 = nullptr);
}

// Forward of the TF32 inference path: the same tcgen05 kernels (bf16 Q/K/V and P), O written as fp32 rounded to nearest
// tf32.  Built for head dim 64 and sequences of <= 512 tokens; other shapes are refused (there is no bf16 fallback).
extern "C" int wj_attn_varlen_fwd_f32out(const void* qkv_bf16, const int* cu_seqlens, int n_seqs, int max_len,
                                         int64_t total_tokens, int D, int H, float* out_f32, void* stream) {
  if (n_seqs <= 0 || max_len <= 0) return WJ_OK;
  if (D % H != 0 || D / H != 64 || D % 64 != 0 || max_len > 512 || total_tokens <= 0) {
    set_error("wj_attn_varlen_fwd_f32out: built for head dim 64 and <= 512 tokens (D=%d H=%d max_len=%d)", D, H, max_len);
    return WJ_ERR_ARG;
  }
  const int rc = wj::attn_fwd_tc_launch(qkv_bf16, cu_seqlens, n_seqs, max_len, total_tokens, D, H, nullptr, nullptr,
                                        WJ_STREAM(stream), out_f32);
  if (rc == 1) { set_error("wj_attn_varlen_fwd_f32out: tensor-map encoding unavailable"); return WJ_ERR_RUNTIME; }
  return rc;
}

extern "C" int wj_attn_varlen_fwd(const void* qkv_bf16, const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens,
                                  int D, int H, void* out_bf16, float* lse2, void* stream) {
  if (n_seqs <= 0 || max_len <= 0) return WJ_OK;
  const int dh = D / H;
  if (D % H != 0 || (dh != 32 && dh != 64)) { set_error("wj_attn_varlen_fwd: head dim must be 32 or 64 (D=%d H=%d)", D, H); return WJ_ERR_ARG; }
  {
    // sequences of <= 512 tokens: tcgen05 kernels (attention_tc.cu); longer ones: the mma.sync kernel below
    const int rc = wj::attn_fwd_tc_launch(qkv_bf16, cu_seqlens, n_seqs, max_len, total_tokens, D, H, out_bf16, lse2, WJ_STREAM(stream));
    if (rc <= 0) return rc;
  }
  const int npad = (max_len + 15) & ~15;
  const size_t smem = static_cast<size_t>(3) * npad * (dh + 8) * 2;
  if (smem > 227 * 1024) { set_error("wj_attn_varlen_fwd: sequence of %d tokens (head dim %d) exceeds the shared-memory resident design", max_len, dh); return WJ_ERR_ARG; }
  const float scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(dh));
  dim3 grid(H, n_seqs);
  const int threads = max_len > 144 ? 256 : 128;   // long sequences (teacher / inference: 200 tokens): 8 warps share K/V
  const bf16* q = reinterpret_cast<const bf16*>(qkv_bf16);
  bf16* o = reinterpret_cast<bf16*>(out_bf16);
  cudaError_t e;
  if (dh == 64) {
    e = cudaFuncSetAttribute(attn_fwd_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) { set_error("attn_fwd attr: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    attn_fwd_kernel<64><<<grid, threads, smem, WJ_STREAM(stream)>>>(q, cu_seqlens, D, H, npad, scale_log2, o, lse2);
  } else {
    e = cudaFuncSetAttribute(attn_fwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) { set_error("attn_fwd attr: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    attn_fwd_kernel<32><<<grid, threads, smem, WJ_STREAM(stream)>>>(q, cu_seqlens, D, H, npad, scale_log2, o, lse2);
  }
  return check_launch("attn_varlen_fwd");
}

namespace wj {
int attn_bwd_tc_launch(const void* qkv, const void* out, const void* dout, const float* lse2, const int* cu, int n_seqs,
                       int max_len, long long total_tokens, int D, int H, void* dqkv, float* dbias, cudaStream_t st);
}

extern "C" int wj_attn_varlen_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16, const float* lse2,
                                  const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens, int D, int H,
                                  void* dqkv_bf16, void* stream) {
  return wj_attn_varlen_bwd_bias(qkv_bf16, out_bf16, dout_bf16, lse2, cu_seqlens, n_seqs, max_len, total_tokens, D, H,
                                 dqkv_bf16, nullptr, stream);
}

static int attn_bwd_bias(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16, const float* lse2,
                         const int* cu_seqlens, int n_seqs, int max_len, int64_t total_tokens, int D, int H,
                         void* dqkv_bf16, float* dbias, void* stream, bool allow_rowstats) {
  if (n_seqs <= 0 || max_len <= 0) return WJ_OK;
  const int dh = D / H;
  if (D % H != 0 || (dh != 32 && dh != 64)) { set_error("wj_attn_varlen_bwd: head dim must be 32 or 64"); return WJ_ERR_ARG; }
  {
    // head dim 32, <= 128 tokens: tcgen05 kernel (attention_tc.cu); everything else: the mma.sync kernel below
    // (deterministic mode: the fused column sums end in shared / global atomics, so the bias gradient is taken from the
    // stored dqkv by the ordered wj_colsum instead)
    const bool det = wj::det_on();
    const int rc = wj::attn_bwd_tc_launch(qkv_bf16, out_bf16, dout_bf16, lse2, cu_seqlens, n_seqs, max_len, total_tokens, D, H,
                                          dqkv_bf16, det ? nullptr : dbias, WJ_STREAM(stream));
    if (rc < 0) return rc;
    if (rc == 0 && det) {
      if (dbias != nullptr) return wj_colsum(dqkv_bf16, 1, total_tokens, 3 * D, 3 * D, dbias, stream);
      return WJ_OK;
    }
    if (rc == 0) {
      // the tcgen05 kernel added the query third in its epilogue; the value third of the bias gradient is the column sum
      // of dO (softmax rows sum to one), the key third is identically zero (softmax ignores a constant key shift)
      if (dbias != nullptr) return wj_colsum(dout_bf16, 1, total_tokens, D, D, dbias + 2 * D, stream);
      return WJ_OK;
    }
  }
  const int npad = (max_len + 15) & ~15;
  size_t smem = static_cast<size_t>(4) * npad * (dh + 8) * 2 + static_cast<size_t>(2) * ((npad + 63) & ~63) * 4;
  const bool rowstats = allow_rowstats && dh == 64 && smem > 227 * 1024;   // lse / delta in the Q rows' padding
  if (rowstats) smem = static_cast<size_t>(4) * npad * (dh + 8) * 2;
  if (smem > 227 * 1024) { set_error("wj_attn_varlen_bwd: sequence of %d tokens (head dim %d) exceeds the shared-memory resident design", max_len, dh); return WJ_ERR_ARG; }
  const float scale = 1.0f / sqrtf(static_cast<float>(dh));
  const float scale_log2 = scale * 1.4426950408889634f;
  dim3 grid(H, n_seqs);
  const bf16* q = reinterpret_cast<const bf16*>(qkv_bf16);
  const bf16* o = reinterpret_cast<const bf16*>(out_bf16);
  const bf16* d_o = reinterpret_cast<const bf16*>(dout_bf16);
  bf16* dq = reinterpret_cast<bf16*>(dqkv_bf16);
  cudaError_t e;
  if (rowstats) {
    e = cudaFuncSetAttribute(attn_bwd_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) { set_error("attn_bwd attr: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    attn_bwd_kernel<64, true><<<grid, 128, smem, WJ_STREAM(stream)>>>(q, o, d_o, lse2, cu_seqlens, D, H, npad, scale, scale_log2, dq);
  } else if (dh == 64) {
    e = cudaFuncSetAttribute(attn_bwd_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) { set_error("attn_bwd attr: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    attn_bwd_kernel<64><<<grid, 128, smem, WJ_STREAM(stream)>>>(q, o, d_o, lse2, cu_seqlens, D, H, npad, scale, scale_log2, dq);
  } else {
    e = cudaFuncSetAttribute(attn_bwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) { set_error("attn_bwd attr: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    attn_bwd_kernel<32><<<grid, 128, smem, WJ_STREAM(stream)>>>(q, o, d_o, lse2, cu_seqlens, D, H, npad, scale, scale_log2, dq);
  }
  const int rc = check_launch("attn_varlen_bwd");
  if (rc != WJ_OK || dbias == nullptr) return rc;
  return wj_colsum(dqkv_bf16, 1, total_tokens, 3 * D, 3 * D, dbias, stream);
}

extern "C" int wj_attn_varlen_bwd_bias(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                                       const float* lse2, const int* cu_seqlens, int n_seqs, int max_len,
                                       int64_t total_tokens, int D, int H, void* dqkv_bf16, float* dbias, void* stream) {
  return attn_bwd_bias(qkv_bf16, out_bf16, dout_bf16, lse2, cu_seqlens, n_seqs, max_len, total_tokens, D, H, dqkv_bf16,
                       dbias, stream, false);
}

// The same backward for head-dim-64 sequences of up to 400 tokens (the dense two-channel WavJEPA-Nat student): past 384
// tokens the per-query lse / delta move into the padding columns of the shared-memory Q rows (attn_bwd_kernel<64, true>).
extern "C" int wj_attn_varlen_bwd_bias_long(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                                            const float* lse2, const int* cu_seqlens, int n_seqs, int max_len,
                                            int64_t total_tokens, int D, int H, void* dqkv_bf16, float* dbias,
                                            void* stream) {
  return attn_bwd_bias(qkv_bf16, out_bf16, dout_bf16, lse2, cu_seqlens, n_seqs, max_len, total_tokens, D, H, dqkv_bf16,
                       dbias, stream, true);
}
