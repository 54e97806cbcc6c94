// tcgen05 forward attention for short packed sequences (<= 128 tokens: the student's visible context sets and the
// predictor's context + target sets of wavjepa/jepa.py:397,438).  One work item = one (sequence, head):
//
//   TMA      Q, K, V tiles [128 tokens x dh] (128B swizzle for dh 64, 64B for dh 32) straight out of qkv [tokens, 3D],
//            double-buffered for dh 32 so that the next item's tiles land while this item's softmax runs
//   UMMA #1  S = Q K^T        128 x n16 x dh    (tcgen05.mma, fp32 accumulator in TMEM columns [0, 128))
//   softmax  4 warps, one query row per thread: tcgen05.ld of its S row in 32-column chunks, masked max, then
//            exp2 / sum; P (bf16 pairs) goes straight back to TMEM with tcgen05.st over the S columns already consumed
//            (P chunk c lands on columns [16c, 16c+16), S chunk c lives on [32c, 32c+32))
//   UMMA #2  O = P V          128 x dh x n16    (A = P from TMEM, B = V MN-major from smem; TMEM columns [64, 64+dh))
//   epilogue O row / sum -> bf16 -> out[token, head*dh ...], lse2[token, head]
//
// 128 TMEM columns and 48 KB of smem per CTA: four CTAs (160 threads each) share an SM and fill each other's latency
// gaps; the single-KV-block structure needs no online softmax.  Rows / keys past the end of the sequence are other
// sequences' (finite) tokens or TMA zero fill: keys >= n are masked, query rows >= n are never stored.
#include "common.cuh"

namespace wj {

constexpr int kAtQ = 128;   // query rows per tile = TMEM lanes
constexpr int kAtK = 128;   // keys per tile

struct AttnTcParams {
  const int* cu;
  int n_seqs, D, H, items;
  float scale_log2;
  bf16* out;
  float* lse2;
  float* out_f32;   // F32OUT kernels: O as fp32 rounded to nearest tf32 (the operand of the tf32 out_proj GEMM)
};

// KT = keys per item (128, 256 or 512 = TMEM columns of S); sequences of 129..512 tokens run as 2..4 query tiles.  With
// KT > 128 the keys are split into 128-key blocks ("halves": 2 or 4), each with its own 4 softmax warps (own max / sum,
// own P and O blocks in TMEM); the epilogue merges the partial results (flash-decoding style) from (max, sum) pairs in
// smem.  KT = 512 (the 400-token binaural sequences) takes all of TMEM and 192 KB of smem: one CTA per SM.
template <int DH, int KT> struct AttnTcCfg {
  static constexpr int TILE = kAtQ * DH * 2;                 // bytes of one [128 x DH] bf16 tile
  static constexpr int HALVES = KT / 128;
  static constexpr int NW = 4 * HALVES;                      // softmax warps; warp NW = control
  static constexpr int THREADS = (NW + 1) * 32;
  static constexpr int STAGE = 3 * HALVES * TILE;            // Q tile(s) | K | V of one (sequence, head)
  static constexpr int STAGES = DH == 32 ? 2 : 1;            // 48 KB (KT 128) / 96 KB (KT 256) either way
  static constexpr int BAR_OFF = STAGES * STAGE;
  static constexpr int ML_OFF = BAR_OFF + 128;               // (max, sum) [2 item parities][HALVES][128 rows] float2
  static constexpr int SMEM = ML_OFF + (HALVES >= 2 ? 2 * HALVES * kAtQ * 8 : 0) + 1024;   // + alignment slack
  static constexpr int CTAS = 512 / KT;                      // per SM, by TMEM columns
  static constexpr uint32_t SWZ = DH == 64 ? 2u : 4u;        // UMMA layout type: 128B / 64B swizzle
  static constexpr uint32_t SBO = DH == 64 ? 1024u : 512u;   // 8 rows x row pitch
  static constexpr uint32_t O_COL = 64;                      // inside a half's 128-column block: P at [0,64), O at [64,64+DH)
};

__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout) << 61;
  return d;
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand (bf16, row = lane, two K elements per 32-bit column) read from TMEM
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32_x16(uint32_t taddr, const uint32_t (&w)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
               ::"r"(taddr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]), "r"(w[8]),
               "r"(w[9]), "r"(w[10]), "r"(w[11]), "r"(w[12]), "r"(w[13]), "r"(w[14]), "r"(w[15])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
// EC (8 / 16 / 32 / 64) consecutive fp32 columns of this thread's TMEM lane
template <int EC> __device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t* v) {
  if constexpr (EC == 8) {
    tmem_ld_32x8(taddr, v);
  } else if constexpr (EC == 16) {
    tmem_ld_32x16(taddr, v);
  } else {
#pragma unroll
    for (int c = 0; c < EC / 32; ++c) tmem_ld_32x32(taddr + c * 32, *reinterpret_cast<uint32_t(*)[32]>(v + c * 32));
  }
}

// (F32OUT at 128 keys: 3 CTAs per SM instead of 4 -- its fp32 epilogue does not fit in 96 registers without spilling)
template <int DH, int KT, bool F32OUT = false>
__global__ void __launch_bounds__(AttnTcCfg<DH, KT>::THREADS, (F32OUT && KT == 128) ? 3 : 512 / KT)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const AttnTcParams p) {
  using Cfg = AttnTcCfg<DH, KT>;
  constexpr int STAGES = Cfg::STAGES, HALVES = Cfg::HALVES, NW = Cfg::NW;
  constexpr int QT = HALVES;                        // query tiles per unit = (sequence, head); K / V are loaded once per unit
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar_load = reinterpret_cast<uint64_t*>(smem + Cfg::BAR_OFF);   // [STAGES]
  uint64_t* bar_s = bar_load + 2;                 // S accumulator complete (MMA commit)
  uint64_t* bar_p = bar_load + 3;                 // P written by the softmax warps (S fully read)
  uint64_t* bar_o = bar_load + 4;                 // O accumulator(s) complete (MMA commit)
  uint64_t* bar_done = bar_load + 5;              // O read by the epilogue warps: TMEM (and this stage's smem) reusable
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_load + 6);
  float2* sML = reinterpret_cast<float2*>(smem + Cfg::ML_OFF);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == NW) {
    if (lane == 0) {
      tma_prefetch_desc(&tmQ);
      mbar_init(bar_load, 1);
      mbar_init(bar_load + 1, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_p, NW);
      mbar_init(bar_o, 1);
      mbar_init(bar_done, NW);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, KT);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == NW) {
    // ================================================================================ control: TMA + MMA issue
    if (lane == 0) {
      constexpr uint32_t idesc_o = umma_idesc_bf16(kAtQ, DH, false, true);
      auto issue_loads = [&](int unit, int stage) {
        const int s = unit / p.H, head = unit - s * p.H;
        const int start = p.cu[s];
        const int halves = min(QT, (p.cu[s + 1] - start + 127) >> 7);   // 128-token tiles that hold valid tokens (>= 1)
        uint8_t* base = smem + stage * Cfg::STAGE;
        mbar_arrive_expect_tx(bar_load + stage, 3 * halves * Cfg::TILE);
        for (int h = 0; h < halves; ++h) {
          tma_load_2d(base + h * Cfg::TILE, &tmQ, bar_load + stage, head * DH, start + h * 128);
          tma_load_2d(base + (QT + h) * Cfg::TILE, &tmQ, bar_load + stage, p.D + head * DH, start + h * 128);
          tma_load_2d(base + (2 * QT + h) * Cfg::TILE, &tmQ, bar_load + stage, 2 * p.D + head * DH, start + h * 128);
        }
      };
      uint32_t ph_load[2] = {0, 0}, ph_p = 0, ph_done = 0;
      int iu = 0, it = 0;
      if (STAGES == 2 && blockIdx.x < p.items) issue_loads(blockIdx.x, 0);
      for (int unit = blockIdx.x; unit < p.items; unit += gridDim.x, ++iu) {
        const int stage = STAGES == 2 ? (iu & 1) : 0;
        const int s = unit / p.H;
        const int n = p.cu[s + 1] - p.cu[s];
        const int n16 = (n + 15) & ~15;
        // S = Q K^T over the n16 valid keys: one UMMA group of N <= 256 per 256-key chunk
        const int nc0 = n16 > 256 ? 256 : (n16 > 0 ? n16 : 16);
        const uint32_t idesc_s = umma_idesc_bf16(kAtQ, nc0, false, false);
        const uint32_t idesc_s1 = umma_idesc_bf16(kAtQ, n16 > 256 ? n16 - 256 : 16, false, false);
        const uint32_t sQ = smem_u32(smem + stage * Cfg::STAGE), sK = sQ + QT * Cfg::TILE, sV = sK + QT * Cfg::TILE;
        const uint64_t vdesc = umma_smem_desc(sV, Cfg::TILE, Cfg::SBO, Cfg::SWZ);
#pragma unroll 1
        for (int qt = 0; qt < QT; ++qt) {
          if (qt > 0 && qt * 128 >= n) break;     // no valid query row in this tile (every warp skips it alike)
          if (it > 0) {   // the previous tile's O has been read: its MMAs are complete, TMEM (and its smem stage) are free
            mbar_wait(bar_done, ph_done);
            ph_done ^= 1;
          }
          if (qt == 0) {
            if (STAGES == 1) issue_loads(unit, 0);
            mbar_wait(bar_load + stage, ph_load[stage]);
            ph_load[stage] ^= 1;
          }
          tc_fence_after();
#pragma unroll
          for (int ks = 0; ks < DH / 16; ++ks)
            umma_bf16(tmem_base, umma_smem_desc(sQ + qt * Cfg::TILE + ks * 32, 0, Cfg::SBO, Cfg::SWZ),
                      umma_smem_desc(sK + ks * 32, 0, Cfg::SBO, Cfg::SWZ), idesc_s, ks > 0 ? 1u : 0u);
          if constexpr (HALVES == 4) {
            if (n16 > 256) {
#pragma unroll
              for (int ks = 0; ks < DH / 16; ++ks)
                umma_bf16(tmem_base + 256, umma_smem_desc(sQ + qt * Cfg::TILE + ks * 32, 0, Cfg::SBO, Cfg::SWZ),
                          umma_smem_desc(sK + 2 * Cfg::TILE + ks * 32, 0, Cfg::SBO, Cfg::SWZ), idesc_s1, ks > 0 ? 1u : 0u);
            }
          }
          umma_commit(bar_s);
          if (STAGES == 2 && qt == 0 && unit + gridDim.x < p.items) issue_loads(unit + gridDim.x, stage ^ 1);   // lands during the softmax
          mbar_wait(bar_p, ph_p);
          ph_p ^= 1;
          tc_fence_after();
          // O_h = P_h V_h per 128-key half, over the 16-key steps that hold valid keys (at least one step of half 0,
          // so that bar_o always completes)
#pragma unroll
          for (int h = 0; h < HALVES; ++h) {
            int steps = (min(n16, 128 * (h + 1)) - 128 * h) / 16;
            if (h == 0 && steps < 1) steps = 1;
            const uint32_t tPh = tmem_base + h * 128, tOh = tPh + Cfg::O_COL;
            for (int kk = 0; kk < steps; ++kk)
              umma_bf16_ts(tOh, tPh + kk * 8, vdesc + static_cast<uint64_t>(((h * 128 + kk * 16) * DH * 2) >> 4), idesc_o, kk > 0 ? 1u : 0u);
          }
          umma_commit(bar_o);
          ++it;
        }
      }
    }
  } else {
    // ================================================================================ softmax + epilogue warps
    const int quad = warp & 3, half = warp >> 2;
    const int row = quad * 32 + lane;                       // query row of the tile = TMEM lane
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t tSh = tmem_base + half * 128 + lane_addr;   // this half's S block (P over its first 64 columns)
    uint32_t ph_s = 0, ph_o = 0;
    int nstart = 0, nn = 0, it = 0;
    if (blockIdx.x < p.items) {
      const int s = blockIdx.x / p.H;
      nstart = p.cu[s];
      nn = p.cu[s + 1] - nstart;
    }
    for (int unit = blockIdx.x; unit < p.items; unit += gridDim.x) {
      const int head = unit % p.H;
      const int ustart = nstart, n = nn;            // tokens (= keys) of this sequence
      if (unit + gridDim.x < p.items) {   // next unit's bounds: the load latency hides behind this unit
        const int s = (unit + gridDim.x) / p.H;
        nstart = p.cu[s];
        nn = p.cu[s + 1] - nstart;
      }
      const int nk = min(n - half * 128, 128);      // keys of this warp's half (<= 0: none)
#pragma unroll 1
      for (int qt = 0; qt < QT; ++qt, ++it) {
      if (qt > 0 && qt * 128 >= n) break;           // (same rule as the control warp)
      const int start = ustart + qt * 128;          // first token of this query tile
      const int nq = n - qt * 128;                  // valid query rows of the tile (<= 0: none)
      mbar_wait(bar_s, ph_s);
      ph_s ^= 1;
      tc_fence_after();
      // pass 1: row maximum over the valid keys
      float m = -INFINITY;
#pragma unroll 1
      for (int c0 = 0; c0 < nk; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(tSh + c0, v);
        tmem_ld_wait();
        if (c0 + 32 <= nk) {
#pragma unroll
          for (int j = 0; j < 32; ++j) m = fmaxf(m, __uint_as_float(v[j]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (c0 + j < nk) m = fmaxf(m, __uint_as_float(v[j]));
        }
      }
      const float ms = m * p.scale_log2;
      // pass 2: p = exp2(s * scale - m * scale), row sum; P (bf16 pairs) -> TMEM columns [16 c, 16 c + 16) of the block
      float l = 0.f;
#pragma unroll 1
      for (int c0 = 0; c0 < nk; c0 += 32) {
        uint32_t v[32], w[16];
        tmem_ld_32x32(tSh + c0, v);
        tmem_ld_wait();
        if (c0 + 32 <= nk) {
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float p0 = ex2_approx(fmaf(__uint_as_float(v[j]), p.scale_log2, -ms));
            const float p1 = ex2_approx(fmaf(__uint_as_float(v[j + 1]), p.scale_log2, -ms));
            l += p0 + p1;
            w[j >> 1] = pack_bf16x2(p0, p1);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float p0 = c0 + j < nk ? ex2_approx(fmaf(__uint_as_float(v[j]), p.scale_log2, -ms)) : 0.f;
            const float p1 = c0 + j + 1 < nk ? ex2_approx(fmaf(__uint_as_float(v[j + 1]), p.scale_log2, -ms)) : 0.f;
            l += p0 + p1;
            w[j >> 1] = pack_bf16x2(p0, p1);
          }
        }
        tmem_st_32x32_x16(tSh + (c0 >> 1), w);
      }
      if constexpr (HALVES >= 2) sML[((it & 1) * HALVES + half) * kAtQ + row] = make_float2(ms, l);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_p);
      // epilogue: this warp's EC output columns of its rows
      mbar_wait(bar_o, ph_o);
      ph_o ^= 1;
      tc_fence_after();
      constexpr int EC = DH / HALVES;
      uint32_t o[EC];
      float fa = 1.f, lsum = l, mtot = ms;
      if constexpr (HALVES == 1) {
        tmem_ld_cols<EC>(tmem_base + lane_addr + Cfg::O_COL, o);
        tmem_ld_wait();
      } else if constexpr (HALVES == 2) {
        const float2 a = sML[((it & 1) * 2 + 0) * kAtQ + row], b = sML[((it & 1) * 2 + 1) * kAtQ + row];
        const bool hasb = n > 128;                   // warp-uniform
        mtot = hasb ? fmaxf(a.x, b.x) : a.x;
        fa = ex2_approx(a.x - mtot);
        const float fb = hasb ? ex2_approx(b.x - mtot) : 0.f;
        lsum = a.y * fa + (hasb ? b.y * fb : 0.f);
        tmem_ld_cols<EC>(tmem_base + lane_addr + Cfg::O_COL + half * EC, o);
        if (hasb) {
          uint32_t ob[EC];
          tmem_ld_cols<EC>(tmem_base + 128 + lane_addr + Cfg::O_COL + half * EC, ob);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < EC; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) * fa + __uint_as_float(ob[j]) * fb);
          fa = 1.f;
        } else {
          tmem_ld_wait();
        }
      } else {
        // merge the partial results of the key blocks that hold valid keys (nb is warp-uniform)
        const int nb = min(HALVES, (n + 127) >> 7);
        const float2* ml = sML + (it & 1) * HALVES * kAtQ + row;
        float mb[HALVES], fb[HALVES];
        mtot = ml[0].x;
#pragma unroll
        for (int b = 0; b < HALVES; ++b) {
          mb[b] = b < nb ? ml[b * kAtQ].x : -INFINITY;
          mtot = fmaxf(mtot, mb[b]);
        }
        lsum = 0.f;
#pragma unroll
        for (int b = 0; b < HALVES; ++b) {
          fb[b] = b < nb ? ex2_approx(mb[b] - mtot) : 0.f;
          if (b < nb) lsum += ml[b * kAtQ].y * fb[b];
        }
        tmem_ld_cols<EC>(tmem_base + lane_addr + Cfg::O_COL + half * EC, o);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < EC; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) * fb[0]);
#pragma unroll
        for (int b = 1; b < HALVES; ++b) {
          if (b < nb) {
            uint32_t ob[EC];
            tmem_ld_cols<EC>(tmem_base + b * 128 + lane_addr + Cfg::O_COL + half * EC, ob);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < EC; ++j) o[j] = __float_as_uint(fmaf(__uint_as_float(ob[j]), fb[b], __uint_as_float(o[j])));
          }
        }
        fa = 1.f;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_done);
      if (row < nq) {
        const float inv = fa / lsum;
        if constexpr (F32OUT) {
          float* of = p.out_f32 + static_cast<long long>(start + row) * p.D + head * DH + (HALVES >= 2 ? half * EC : 0);
#pragma unroll
          for (int j = 0; j < EC; j += 4)
            *reinterpret_cast<float4*>(of + j) = make_float4(
                tf32_round(__uint_as_float(o[j]) * inv), tf32_round(__uint_as_float(o[j + 1]) * inv),
                tf32_round(__uint_as_float(o[j + 2]) * inv), tf32_round(__uint_as_float(o[j + 3]) * inv));
        }
        bf16* op = p.out + static_cast<long long>(start + row) * p.D + head * DH + (HALVES >= 2 ? half * EC : 0);
#pragma unroll
        for (int j = 0; j < EC && !F32OUT; j += 8) {
          uint4 w;
          w.x = pack_bf16x2(__uint_as_float(o[j]) * inv, __uint_as_float(o[j + 1]) * inv);
          w.y = pack_bf16x2(__uint_as_float(o[j + 2]) * inv, __uint_as_float(o[j + 3]) * inv);
          w.z = pack_bf16x2(__uint_as_float(o[j + 4]) * inv, __uint_as_float(o[j + 5]) * inv);
          w.w = pack_bf16x2(__uint_as_float(o[j + 6]) * inv, __uint_as_float(o[j + 7]) * inv);
          *reinterpret_cast<uint4*>(op + j) = w;
        }
        if (p.lse2 != nullptr && half == 0) p.lse2[static_cast<long long>(start + row) * p.H + head] = mtot + log2f(lsum);
      }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NW) {
    tc_fence_after();
    tmem_dealloc(tmem_base, KT);
  }
}

// ------------------------------------------------------------------------------------------------------- backward
// One work item = one (sequence, head) of <= 128 tokens, head dim 32 (the predictor; the student's dim-64 heads stay
// on the mma.sync kernel).  All five products of the attention backward are UMMAs:
//
//   S  = Q K^T, dP = dO V^T        TMEM columns [0,128) and [128,256)
//   gradient warps (8: two per TMEM lane quadrant, splitting the key chunks; one query row per thread):
//        P = exp2(S*scale - lse), dS = P * (dP - delta), both bf16 -> smem [128 queries][128 keys], 128B swizzle
//   dV = P^T dO, dK = dS^T Q       A = the smem tiles read MN-major (M = keys), B = dO / Q read MN-major
//   dQ = dS K                      A = the dS tile read K-major, B = K read MN-major
//        (TMEM columns [0,32), [32,64), [64,96) over the consumed S block)
//   epilogue: rows < n of dQ*scale, dK*scale, dV -> dqkv[token, {0, D, 2D} + head*32 ...], transposed through the
//        warp's own (consumed) corner of the P tile so that four lanes store one 64-byte row
//        optionally the column sums of the stored dQ rows (the query third of the in_proj bias gradient, which autograd
//        takes over the bf16 dqkv): 5-step reduce-scatter across the warp's 32 rows, shared-memory accumulators [D] per
//        CTA, one global atomic per column per CTA at the end; with the value third = column sums of dO and the key
//        third = 0 this replaces a separate pass over dqkv (398 MB per layer)
//   delta: the O tile rides along with the TMA loads; every gradient thread reduces its own row of O * dO out of
//        smem while the S / dP products run.  lse is fetched one item ahead into a register.
//
// Query rows >= n are written as zeros into P / dS (they are K-dimension rows of the dV / dK products); key columns
// >= n are masked to zero.  104 KB smem + 256 TMEM columns: two CTAs per SM.
struct AttnBwdParams {
  const int* cu;
  int D, H, items;
  float scale, scale_log2;
  const bf16* out;
  const bf16* dout;
  const float* lse2;
  bf16* dqkv;
  float* dbias;   // optional [3 D]: [0, D) += column sums of the stored dQ rows (query third of the in_proj bias gradient)
};

constexpr int kBwdTile = kAtQ * 32 * 2;                  // 8 KB: [128 x 32] bf16, 64B swizzle
constexpr int kBwdPs = 2 * kAtQ * 128;                   // 32 KB: [2 key blocks][128 queries][64 keys] bf16, 128B swizzle
constexpr int kBwdBarOff = 5 * kBwdTile + 2 * kBwdPs;    // Q | K | V | dO | O | P | dS | barriers
constexpr int kBwdCsOff = kBwdBarOff + 128;             // fp32 [D] column sums of this CTA's dQ rows (D <= kBwdCsMaxD)
constexpr int kBwdCsMaxD = 1024;
constexpr int kBwdSmem = kBwdCsOff + kBwdCsMaxD * 4 + 1024;

__global__ void __launch_bounds__(288, 2) attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ,
                                                             const __grid_constant__ CUtensorMap tmDO,
                                                             const __grid_constant__ CUtensorMap tmO, const AttnBwdParams p) {
  constexpr int DH = 32;
  constexpr uint32_t SWZ = 4u, SBO = 512u;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sP = smem + 5 * kBwdTile;
  uint8_t* sDS = sP + kBwdPs;
  uint64_t* bar_load = reinterpret_cast<uint64_t*>(smem + kBwdBarOff);
  uint64_t* bar_s = bar_load + 1;      // S and dP complete
  uint64_t* bar_p = bar_load + 2;      // P / dS written (8 warps)
  uint64_t* bar_g = bar_load + 3;      // dV, dK, dQ complete
  uint64_t* bar_done = bar_load + 4;   // gradients read out of TMEM (8 warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_load + 5);
  float* s_cs = reinterpret_cast<float*>(smem + kBwdCsOff);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (p.dbias != nullptr)
    for (int i = threadIdx.x; i < p.D; i += blockDim.x) s_cs[i] = 0.f;

  if (warp == 8) {
    if (lane == 0) {
      tma_prefetch_desc(&tmQ);
      tma_prefetch_desc(&tmDO);
      tma_prefetch_desc(&tmO);
      mbar_init(bar_load, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_p, 8);
      mbar_init(bar_g, 1);
      mbar_init(bar_done, 8);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, 256);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tS = tmem_base, tDP = tmem_base + 128, tDV = tmem_base, tDK = tmem_base + 32, tDQ = tmem_base + 64;

  if (warp == 8) {
    if (lane == 0) {
      constexpr uint32_t idesc_g = umma_idesc_bf16(kAtQ, DH, true, true);    // dV, dK: A and B MN-major
      constexpr uint32_t idesc_q = umma_idesc_bf16(kAtQ, DH, false, true);   // dQ: A K-major, B MN-major
      const uint32_t sQ = smem_u32(smem), sK = sQ + kBwdTile, sV = sK + kBwdTile, sDO = sV + kBwdTile;
      uint32_t ph_load = 0, ph_p = 0, ph_g = 0, ph_done = 0;
      int it = 0;
      for (int item = blockIdx.x; item < p.items; item += gridDim.x, ++it) {
        const int s = item / p.H, head = item - s * p.H;
        const int start = p.cu[s], n = p.cu[s + 1] - start;
        const int n16 = n > 0 ? (n + 15) & ~15 : 16;
        const uint32_t idesc_s = umma_idesc_bf16(kAtQ, n16, false, false);
        if (it > 0) {   // the previous item's last MMAs are complete: every smem tile may be overwritten
          mbar_wait(bar_g, ph_g);
          ph_g ^= 1;
        }
        mbar_arrive_expect_tx(bar_load, 5 * kBwdTile);
        tma_load_2d(smem, &tmQ, bar_load, head * DH, start);
        tma_load_2d(smem + kBwdTile, &tmQ, bar_load, p.D + head * DH, start);
        tma_load_2d(smem + 2 * kBwdTile, &tmQ, bar_load, 2 * p.D + head * DH, start);
        tma_load_2d(smem + 3 * kBwdTile, &tmDO, bar_load, head * DH, start);
        tma_load_2d(smem + 4 * kBwdTile, &tmO, bar_load, head * DH, start);
        mbar_wait(bar_load, ph_load);
        ph_load ^= 1;
        if (it > 0) {   // the previous item's gradients have been read out of TMEM
          mbar_wait(bar_done, ph_done);
          ph_done ^= 1;
        }
        tc_fence_after();
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          umma_bf16(tS, umma_smem_desc(sQ + ks * 32, 0, SBO, SWZ), umma_smem_desc(sK + ks * 32, 0, SBO, SWZ), idesc_s, ks > 0 ? 1u : 0u);
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks)
          umma_bf16(tDP, umma_smem_desc(sDO + ks * 32, 0, SBO, SWZ), umma_smem_desc(sV + ks * 32, 0, SBO, SWZ), idesc_s, ks > 0 ? 1u : 0u);
        umma_commit(bar_s);
        if (item + gridDim.x < p.items) {
          // the next item's five tiles cannot land in shared memory before this item's last MMAs have read it (one
          // stage: 104 KB per CTA buys the second CTA per SM), but they can be pulled into L2 now, so that the TMA loads
          // at the top of the next iteration cost an L2 hit instead of a DRAM round trip on this CTA's critical path
          const int nitem = item + gridDim.x, ns = nitem / p.H, nh = nitem - ns * p.H, nst = p.cu[ns];
          tma_prefetch_2d(&tmQ, nh * DH, nst);
          tma_prefetch_2d(&tmQ, p.D + nh * DH, nst);
          tma_prefetch_2d(&tmQ, 2 * p.D + nh * DH, nst);
          tma_prefetch_2d(&tmDO, nh * DH, nst);
          tma_prefetch_2d(&tmO, nh * DH, nst);
        }
        mbar_wait(bar_p, ph_p);
        ph_p ^= 1;
        tc_fence_after();
        const int steps = n16 / 16;
        const uint64_t dP_mn = umma_smem_desc(smem_u32(sP), kAtQ * 128, 1024, 2u);     // A = P^T  (M = keys, K = queries)
        const uint64_t dS_mn = umma_smem_desc(smem_u32(sDS), kAtQ * 128, 1024, 2u);    // A = dS^T
        const uint64_t bDO = umma_smem_desc(sDO, kBwdTile, SBO, SWZ), bQ = umma_smem_desc(sQ, kBwdTile, SBO, SWZ),
                       bK = umma_smem_desc(sK, kBwdTile, SBO, SWZ);
        for (int kk = 0; kk < steps; ++kk)    // 16 queries per step: 16 rows of the P tile (2 KB) and of dO (1 KB)
          umma_bf16(tDV, dP_mn + static_cast<uint64_t>((kk * 2048) >> 4), bDO + static_cast<uint64_t>((kk * 1024) >> 4), idesc_g, kk > 0 ? 1u : 0u);
        for (int kk = 0; kk < steps; ++kk)
          umma_bf16(tDK, dS_mn + static_cast<uint64_t>((kk * 2048) >> 4), bQ + static_cast<uint64_t>((kk * 1024) >> 4), idesc_g, kk > 0 ? 1u : 0u);
        for (int kk = 0; kk < steps; ++kk) {  // 16 keys per step
          const uint32_t a = smem_u32(sDS) + (kk >> 2) * (kAtQ * 128) + (kk & 3) * 32;
          umma_bf16(tDQ, umma_smem_desc(a, 0, 1024, 2u), bK + static_cast<uint64_t>((kk * 1024) >> 4), idesc_q, kk > 0 ? 1u : 0u);
        }
        umma_commit(bar_g);
      }
    }
  } else {
    // ================================================================================ gradient warps
    const int quad = warp & 3, half = warp >> 2;
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    // this warp's private 4 KB of the P tile (its 32 query rows x its 64 keys): staging for the coalesced stores
    uint8_t* stage = sP + half * (kAtQ * 128) + quad * 32 * 128;
    uint32_t ph_s = 0, ph_g = 0, ph_l = 0;
    // software pipeline of the per-item scalars: sequence bounds two items ahead, this row's lse one item ahead
    int nstart = 0, nn = 0, n2start = 0, n2n = 0;
    float nlse = 0.f;
    if (blockIdx.x < p.items) {
      const int s = blockIdx.x / p.H;
      nstart = p.cu[s];
      nn = p.cu[s + 1] - nstart;
      if (row < nn) nlse = p.lse2[static_cast<long long>(nstart + row) * p.H + blockIdx.x % p.H];
    }
    if (blockIdx.x + gridDim.x < p.items) {
      const int s = (blockIdx.x + gridDim.x) / p.H;
      n2start = p.cu[s];
      n2n = p.cu[s + 1] - n2start;
    }
    const uint8_t* sOrow = smem + 4 * kBwdTile + row * 64;
    const uint8_t* sDOrow = smem + 3 * kBwdTile + row * 64;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
      const int head = item % p.H;
      const int start = nstart, n = nn;
      const float lse = nlse;
      nstart = n2start;
      nn = n2n;
      if (item + gridDim.x < p.items)     // (addresses known: the loads' latency hides behind this item)
        nlse = row < nn ? p.lse2[static_cast<long long>(nstart + row) * p.H + (item + gridDim.x) % p.H] : 0.f;
      if (item + 2 * gridDim.x < p.items) {
        const int s = (item + 2 * gridDim.x) / p.H;
        n2start = p.cu[s];
        n2n = p.cu[s + 1] - n2start;
      }
      const bool live = row < n;
      // delta = sum(O * dO) of this thread's row out of the TMA tiles (64B swizzle), while the S / dP products run
      mbar_wait(bar_load, ph_l);
      ph_l ^= 1;
      float delta = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int o = (c ^ ((row >> 1) & 3)) << 4;
        const uint4 a = *reinterpret_cast<const uint4*>(sOrow + o);
        const uint4 b = *reinterpret_cast<const uint4*>(sDOrow + o);
        const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&a);
        const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&b);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 x = __bfloat1622float2(a2[t]), y = __bfloat1622float2(b2[t]);
          delta += x.x * y.x + x.y * y.y;
        }
      }
      mbar_wait(bar_s, ph_s);
      ph_s ^= 1;
      tc_fence_after();
#pragma unroll 1
      for (int c0 = half * 64; c0 < half * 64 + 64 && c0 < n; c0 += 32) {
        uint32_t sv[32], dv[32];
        tmem_ld_32x32(tS + lane_addr + c0, sv);
        tmem_ld_32x32(tDP + lane_addr + c0, dv);
        tmem_ld_wait();
        const int off = (c0 >> 6) * (kAtQ * 128) + row * 128;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t wp[4], wd[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int j = q * 8 + 2 * t;
            // selects, not multiplies: TMEM columns >= n16 and rows >= n hold stale bits
            const bool k0 = live && c0 + j < n, k1 = live && c0 + j + 1 < n;
            const float p0 = k0 ? ex2_approx(fmaf(__uint_as_float(sv[j]), p.scale_log2, -lse)) : 0.f;
            const float p1 = k1 ? ex2_approx(fmaf(__uint_as_float(sv[j + 1]), p.scale_log2, -lse)) : 0.f;
            wp[t] = pack_bf16x2(p0, p1);
            wd[t] = pack_bf16x2(k0 ? p0 * (__uint_as_float(dv[j]) - delta) : 0.f, k1 ? p1 * (__uint_as_float(dv[j + 1]) - delta) : 0.f);
          }
          const int chunk = ((c0 & 63) >> 3) + q;
          const int o = off + ((chunk ^ (row & 7)) << 4);
          *reinterpret_cast<uint4*>(sP + o) = make_uint4(wp[0], wp[1], wp[2], wp[3]);
          *reinterpret_cast<uint4*>(sDS + o) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_p);
      mbar_wait(bar_g, ph_g);
      ph_g ^= 1;
      tc_fence_after();
      // warps 0-3: dQ and dV rows; warps 4-7: dK rows.  TMEM -> registers -> bf16 rows in this warp's staging corner
      // (16-byte pieces XOR-swizzled by the row pair) -> four lanes per 64-byte row to global memory
      const int ntile = half == 0 ? 2 : 1;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        if (t < ntile) {
          uint32_t g[32];
          tmem_ld_32x32((half == 0 ? (t == 0 ? tDQ : tDV) : tDK) + lane_addr, g);
          tmem_ld_wait();
          const float sc = (half == 0 && t == 1) ? 1.0f : p.scale;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 w;
            w.x = pack_bf16x2(__uint_as_float(g[8 * q]) * sc, __uint_as_float(g[8 * q + 1]) * sc);
            w.y = pack_bf16x2(__uint_as_float(g[8 * q + 2]) * sc, __uint_as_float(g[8 * q + 3]) * sc);
            w.z = pack_bf16x2(__uint_as_float(g[8 * q + 4]) * sc, __uint_as_float(g[8 * q + 5]) * sc);
            w.w = pack_bf16x2(__uint_as_float(g[8 * q + 6]) * sc, __uint_as_float(g[8 * q + 7]) * sc);
            *reinterpret_cast<uint4*>(stage + t * 2048 + lane * 64 + ((q ^ ((lane >> 1) & 3)) << 4)) = w;
          }
        }
      }
      if (p.dbias != nullptr && half == 1) {
        // Bias gradient of the query projection = column sums of the stored (bf16) dQ rows of this warp's lane quadrant:
        // 5-step reduce-scatter over the warp's 32 rows (lane l ends with column l), one shared-memory atomic per lane.
        // Done by the dK warps, which stage one tile where the dQ / dV warps stage two.  (The key third of the bias
        // gradient is exactly zero -- softmax is invariant to a constant added to every key's logit -- and the value
        // third equals the column sums of dO because softmax rows sum to one: the host side adds that with one pass over
        // dO instead of a reduction here.)
        uint32_t g[32];
        tmem_ld_32x32(tDQ + lane_addr, g);
        tmem_ld_wait();
        float c32[32];
#pragma unroll
        for (int j = 0; j < 32; j += 2) {   // rows >= n hold stale bits: select, do not multiply
          const uint32_t w = pack_bf16x2(__uint_as_float(g[j]) * p.scale, __uint_as_float(g[j + 1]) * p.scale);
          c32[j] = live ? __uint_as_float(w << 16) : 0.f;
          c32[j + 1] = live ? __uint_as_float(w & 0xffff0000u) : 0.f;
        }
#pragma unroll
        for (int sft = 16; sft >= 1; sft >>= 1) {
          const bool up = (lane & sft) != 0;
#pragma unroll
          for (int i = 0; i < sft; ++i) {
            const float mine = up ? c32[sft + i] : c32[i];
            const float other = up ? c32[i] : c32[sft + i];
            c32[i] = mine + __shfl_xor_sync(0xffffffffu, other, sft);
          }
        }
        atomicAdd(s_cs + head * DH + lane, c32[0]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_done);
      {
        const int rsub = lane >> 2, piece = lane & 3;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          if (t < ntile) {
            const int col = half == 0 ? (t == 0 ? 0 : 2 * p.D) : p.D;
#pragma unroll
            for (int r0 = 0; r0 < 32; r0 += 8) {
              const int lr = r0 + rsub, r = quad * 32 + lr;
              if (r < n) {
                const uint4 w = *reinterpret_cast<const uint4*>(stage + t * 2048 + lr * 64 + ((piece ^ ((lr >> 1) & 3)) << 4));
                *reinterpret_cast<uint4*>(p.dqkv + static_cast<long long>(start + r) * (3LL * p.D) + col + head * DH + piece * 8) = w;
              }
            }
          }
        }
      }
      __syncwarp();   // the staging corner is rewritten by this warp's next P / dS chunk
    }
  }
  tc_fence_before();
  __syncthreads();
  if (p.dbias != nullptr)
    for (int i = threadIdx.x; i < p.D; i += blockDim.x) atomicAdd(p.dbias + i, s_cs[i]);
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

typedef CUresult (*PFN_encodeTiledA)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Returns WJ_OK and launches when the problem fits this kernel; 1 when the caller should use the mma.sync kernel.
int attn_fwd_tc_launch(const void* qkv, const int* cu, int n_seqs, int max_len, long long total_tokens, int D, int H,
                       void* out, float* lse2, cudaStream_t st, float* out_f32) {
  const int dh = D / H;
  if (max_len > 512 || D % 64 != 0 || (dh != 32 && dh != 64) || total_tokens <= 0) return 1;
  static PFN_encodeTiledA enc = nullptr;
  if (enc == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return 1;
    enc = reinterpret_cast<PFN_encodeTiledA>(sym);
  }
  CUtensorMap tm;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(3) * D, static_cast<cuuint64_t>(total_tokens)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(3) * D * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(dh), kAtQ}, es[2] = {1, 1};
  if (enc(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(qkv), dims, strides, box, es,
          CU_TENSOR_MAP_INTERLEAVE_NONE, dh == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return 1;
  AttnTcParams p;
  const int qt = max_len > 256 ? 4 : (max_len > 128 ? 2 : 1);
  p.cu = cu; p.n_seqs = n_seqs; p.D = D; p.H = H; p.items = n_seqs * H;   // units = (sequence, head)
  p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(dh));
  p.out = reinterpret_cast<bf16*>(out); p.lse2 = lse2; p.out_f32 = out_f32;
  auto go = [&](auto kernel, int smem, int ctas, int threads) -> int {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { set_error("attn_fwd_tc attr: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    int grid = ctas * sm_count();
    if (grid > p.items) grid = p.items;
    kernel<<<grid, threads, smem, st>>>(tm, p);
    return check_launch("attn_fwd_tc");
  };
  if (out_f32 != nullptr) {   // fp32 output: head dim 64 (the encoder), 128 / 256 / 512 keys
    if (dh != 64) { set_error("attn_fwd_tc: the fp32-output kernels are built for head dim 64 (got %d)", dh); return WJ_ERR_ARG; }
    if (qt == 4) return go(attn_fwd_tc_kernel<64, 512, true>, AttnTcCfg<64, 512>::SMEM, AttnTcCfg<64, 512>::CTAS, AttnTcCfg<64, 512>::THREADS);
    if (qt == 2) return go(attn_fwd_tc_kernel<64, 256, true>, AttnTcCfg<64, 256>::SMEM, AttnTcCfg<64, 256>::CTAS, AttnTcCfg<64, 256>::THREADS);
    return go(attn_fwd_tc_kernel<64, 128, true>, AttnTcCfg<64, 128>::SMEM, AttnTcCfg<64, 128>::CTAS, AttnTcCfg<64, 128>::THREADS);
  }
  if (dh == 64 && qt == 4) return go(attn_fwd_tc_kernel<64, 512>, AttnTcCfg<64, 512>::SMEM, AttnTcCfg<64, 512>::CTAS, AttnTcCfg<64, 512>::THREADS);
  if (qt == 4) return go(attn_fwd_tc_kernel<32, 512>, AttnTcCfg<32, 512>::SMEM, AttnTcCfg<32, 512>::CTAS, AttnTcCfg<32, 512>::THREADS);
  if (dh == 64 && qt == 1) return go(attn_fwd_tc_kernel<64, 128>, AttnTcCfg<64, 128>::SMEM, AttnTcCfg<64, 128>::CTAS, AttnTcCfg<64, 128>::THREADS);
  if (dh == 64) return go(attn_fwd_tc_kernel<64, 256>, AttnTcCfg<64, 256>::SMEM, AttnTcCfg<64, 256>::CTAS, AttnTcCfg<64, 256>::THREADS);
  if (qt == 1) return go(attn_fwd_tc_kernel<32, 128>, AttnTcCfg<32, 128>::SMEM, AttnTcCfg<32, 128>::CTAS, AttnTcCfg<32, 128>::THREADS);
  return go(attn_fwd_tc_kernel<32, 256>, AttnTcCfg<32, 256>::SMEM, AttnTcCfg<32, 256>::CTAS, AttnTcCfg<32, 256>::THREADS);
}


// Returns WJ_OK and launches when the problem fits (head dim 32, <= 128 tokens); 1 -> caller uses the mma.sync kernel.
int attn_bwd_tc_launch(const void* qkv, const void* out, const void* dout, const float* lse2, const int* cu, int n_seqs,
                       int max_len, long long total_tokens, int D, int H, void* dqkv, float* dbias, cudaStream_t st) {
  const int dh = D / H;
  if (max_len > 128 || dh != 32 || D % 8 != 0 || total_tokens <= 0) return 1;
  if (dbias != nullptr && D > kBwdCsMaxD) return 1;   // (no room for the column-sum accumulators: the caller sums separately)
  static PFN_encodeTiledA enc = nullptr;
  if (enc == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return 1;
    enc = reinterpret_cast<PFN_encodeTiledA>(sym);
  }
  CUtensorMap tq, tdo, to;
  cuuint32_t box[2] = {32, kAtQ}, es[2] = {1, 1};
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(3) * D, static_cast<cuuint64_t>(total_tokens)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(3) * D * 2};
    if (enc(&tq, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(qkv), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return 1;
  }
  {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(total_tokens)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(D) * 2};
    if (enc(&tdo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(dout), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return 1;
    if (enc(&to, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(out), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return 1;
  }
  AttnBwdParams p;
  p.cu = cu; p.D = D; p.H = H; p.items = n_seqs * H;
  p.scale = 1.0f / sqrtf(static_cast<float>(dh));
  p.scale_log2 = p.scale * 1.4426950408889634f;
  p.out = reinterpret_cast<const bf16*>(out); p.dout = reinterpret_cast<const bf16*>(dout); p.lse2 = lse2;
  p.dqkv = reinterpret_cast<bf16*>(dqkv);
  p.dbias = dbias;
  cudaError_t e = cudaFuncSetAttribute(attn_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBwdSmem);
  if (e != cudaSuccess) { set_error("attn_bwd_tc attr: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
  int grid = 2 * sm_count();
  if (grid > p.items) grid = p.items;
  attn_bwd_tc_kernel<<<grid, 288, kBwdSmem, st>>>(tq, tdo, to, p);
  return check_launch("attn_bwd_tc");
}

}  // namespace wj
