// tcgen05 / TMEM / TMA GEMM core for the WavJEPA hot path (sm_100a only).
//
// One persistent, warp-specialised kernel body (gemm_body) serves every GEMM-shaped op of the path:
//   * Linear layers fwd / dgrad            (reference: torch.nn.Linear inside nn.TransformerEncoderLayer,
//                                            wavjepa/jepa.py:126-132; MHA in/out-proj, MLP, the three mappers)
//   * Conv1d 512->512 (k3 s2, k2 s2) fwd / dgrad as implicit GEMM over channels-last activations
//                                           (reference: nn.Conv1d, wavjepa/extractors/audio_feature_extractor.py:70)
//   * weight gradients (WGRAD mode: both operands MN-major, split over the token dimension, fp32 reduce-add)
//
// Layout of a CTA (640 threads, 1 CTA / SM, grid = min(#tiles, #SMs), static round-robin tile schedule):
//   warp 0      : TMA producer (one elected lane)   global -> 128B-swizzled smem ring (STAGES deep)
//   warp 1      : MMA issuer   (one elected lane)   tcgen05.mma.cta_group::1.kind::f16, D in TMEM (2 accumulators)
//   warp 2      : TMEM allocator / deallocator
//   warp 3      : idle
//   warps 4..19 : epilogue: tcgen05.ld -> registers -> fused bias / GELU / GELU' / residual -> global
//
// The body has two entry points: gemm_kernel runs it on single CTAs (128-row tiles), gemm_pair_kernel on CTA pairs
// (__cluster_dims__(2, 1, 1), 256-row tiles, tcgen05.mma.cta_group::2, grid = 2 * min(#tiles, #SMs / 2)); every
// pair-specific step is an `if constexpr (CTAS == 2)` inside the one body.
//
// Operand addressing is "virtual column" based so that the same kernel covers implicit-GEMM convolutions: the
// reduction (normal mode) or output-column (WGRAD mode) index vc is split into segments of `seg.width` columns;
// segment s reads the 4-D tensor map at (vc % width, seg.q[s], row + seg.p[s], batch).  A plain matrix is the
// single-segment case.
#include "ptx.cuh"
#include "common.cuh"

#include <stdio.h>
#include <string.h>

namespace wj {

struct SegInfo {
  int width;
  int q[4];
  int p[4];
};

struct GemmParams {
  int L;             // rows per batch entry (normal: output rows; wgrad: reduction rows)
  int batch;
  int N;             // normal: output columns.  wgrad: output columns (= virtual columns of operand B)
  int K;             // normal: reduction length (virtual columns of A).  wgrad: unused
  int M;             // wgrad: output rows (columns of operand A)
  int mb_per_batch;  // normal: ceil(L / 128)
  int m_blocks;      // normal: batch * mb_per_batch; wgrad: M / 128
  int n_blocks;
  int total_tiles;
  int splits;        // wgrad: split of the reduction
  int b_single;      // wgrad: the BN columns of a B tile lie in one segment -> one TMA per k-block
  long long split_stride;   // wgrad, deterministic mode: elements between the output slabs of consecutive token splits
  int kb_per_batch;  // wgrad: ceil(L / 64)
  SegInfo seg;       // normal/dgrad: segments of A's K;  wgrad: segments of B's N
  int segB_col[4];   // dgrad: column offset into W for each reduction segment
  // epilogue
  void* out;
  long long ld_out;
  int out_f32;
  int accumulate;    // out (fp32) += result with red.global.add
  bf16* out2;        // optional second output (pre-activation, bf16)
  long long ld_out2;
  const float* bias;
  const void* resid;
  int resid_f32;
  long long ld_resid;
  int resid_mod;     // residual row = row % resid_mod when > 0 (positional table broadcast)
  const bf16* aux;   // GELU'(pre-activation) saved by an act == 1 forward, for act == 2
  long long ld_aux;
  int act;           // 0 none; 1: h = bf16(acc + bias), out2 = gelu'(h), v = gelu(h); 2: v = acc * aux; 3: v = bf16(v)
  const int* out_rows;  // optional row indirection for the output / residual / aux rows (scatter), -1 = skip
  float* colsum;        // optional: colsum[n] += sum over rows of the stored output (bias gradients)
  int tma_store;        // bf16 outputs without residual / aux / scatter: staged in smem and written by TMA stores
  int transpose_out;    // wgrad: the tile holds out^T (operands swapped so that the wide dimension is BN = 256)
  long long* dbg;       // optional per-CTA cycle counters (wj_gemm_debug): [0] MMA thread waiting for operands, [1] for a free
                        // accumulator, [2] its total, [3] producer waiting for a free stage, [4] epilogue warp 4 waiting for
                        // an accumulator, [5] its total, [6] tiles, [7] unused
  int round_tf32;       // tf32 kernel: fp32 outputs are rounded to nearest tf32 (they are the next GEMM's operand)
};

struct OutMaps {
  CUtensorMap o;    // out  as {N, L, batch} bf16, box {32, 32, 1}, 64-byte swizzle
  CUtensorMap o2;   // out2 (saved GELU')
};

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kThreads = 640;
constexpr int kEpiWarp0 = 4;
constexpr int kEpiWarps = 16;
// setmaxnreg targets.  The pool a CTA re-distributes is its LAUNCH allocation (640 threads x 96 registers), not the
// SM's register file: 128 * ctrl + 512 * epi must stay <= 61440 or setmaxnreg.inc waits forever.
constexpr int kLaunchRegs = 96;
template <bool WIDE>
struct RegSplit {   // WIDE: the two-output GELU epilogue holds 64 accumulator + 32 result registers
  static constexpr int EPI = WIDE ? 112 : 104;
  static constexpr int CTRL = WIDE ? 24 : 40;
  static_assert(128 * CTRL + 512 * EPI <= kThreads * kLaunchRegs, "setmaxnreg split exceeds the CTA's register pool");
};

// AUX: the GELU-backward dgrad (MODE 2, HEAVY): every epilogue warp owns TWO 2 KB tiles (one per 32-column chunk of its
// tile) that first receive the saved GELU' factors by TMA -- a whole tile ahead of their use -- and then stage the
// output; the extra 32 KB come out of the operand ring (3 stages on single CTAs, 5 on pairs: that kernel is
// epilogue-bound, not operand-bound).  CTAS = 2: each CTA of a pair stages its 128 rows of A and HALF of the B tile.
template <int BN, bool AUX, int CTAS>
struct Cfg {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = (BN / CTAS) * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = CTAS == 2 ? (AUX ? 5 : ((BN == 256) ? 6 : 8))
                                          : AUX ? ((BN == 256) ? 3 : 4) : ((BN == 256) ? 4 : ((BN == 192) ? 4 : ((BN == 128) ? 6 : 8)));
  static constexpr int STAGING_OFF = STAGES * STAGE_BYTES + 1024;   // barriers live in the 1 KB before it
  static constexpr int WARP_STAGING = AUX ? 4096 : 2048;
  static constexpr int SMEM_BYTES = STAGING_OFF + 1024 /*align slack*/ + kEpiWarps * WARP_STAGING /*TMA-store staging*/;
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
};

__device__ __forceinline__ void seg_coords(const SegInfo& s, int vc, int& c0, int& q, int& p) {
  if (s.width > 0) {
    const int si = vc / s.width;
    c0 = vc - si * s.width;
    q = s.q[si];
    p = s.p[si];
  } else {
    c0 = vc;
    q = 0;
    p = 0;
  }
}

// Tile decode.  normal: tile -> (m_blk, n_blk), n fastest (CTAs running together share the A rows through L2), then
// m_blk -> (batch entry b, row0 = this CTA's first row inside it).  wgrad: tile -> (split, m_blk, n_blk), row0 = this
// CTA's first output row.  tile_rows: rows of an m-block (BM, or 2 * BM for a CTA pair); row_off: this CTA's offset in it.
struct TileCoords {
  int split, m_blk, n_blk, b, row0;
};

template <bool WGRAD>
__device__ __forceinline__ TileCoords tile_coords(const GemmParams& p, int tile, int tile_rows, int row_off) {
  TileCoords t;
  t.split = 0;
  t.b = 0;
  if constexpr (WGRAD) {
    const int mn = p.m_blocks * p.n_blocks;
    t.split = tile / mn;
    tile -= t.split * mn;
  }
  t.m_blk = tile / p.n_blocks;
  t.n_blk = tile - t.m_blk * p.n_blocks;
  if constexpr (!WGRAD) {
    t.b = t.m_blk / p.mb_per_batch;
    t.row0 = (t.m_blk - t.b * p.mb_per_batch) * tile_rows + row_off;
  } else {
    t.row0 = t.m_blk * tile_rows + row_off;
  }
  return t;
}

// wgrad: the k-blocks [lo, hi) of the (batch, 64-token block) reduction that token split `split` covers (may be empty)
__device__ __forceinline__ void wgrad_kb_range(const GemmParams& p, int split, int& lo, int& hi) {
  const int kb_total = p.batch * p.kb_per_batch;
  const int per = (kb_total + p.splits - 1) / p.splits;
  lo = split * per;
  hi = min(lo + per, kb_total);
}

// One TMA load into a stage of the operand ring.  Its bytes are counted on the stage's full barrier: this CTA's own
// (`bar`), or on CTA pairs the leader's (`fb`, a shared::cluster address).
template <int CTAS>
__device__ __forceinline__ void stage_load(void* dst, const CUtensorMap* tm, uint64_t* bar, uint32_t fb, int c0, int c1) {
  if constexpr (CTAS == 1) tma_load_2d(dst, tm, bar, c0, c1);
  else tma_load_2d_pair(dst, tm, fb, c0, c1);
}
template <int CTAS>
__device__ __forceinline__ void stage_load(void* dst, const CUtensorMap* tm, uint64_t* bar, uint32_t fb, int c0, int c1,
                                           int c2) {
  if constexpr (CTAS == 1) tma_load_3d(dst, tm, bar, c0, c1, c2);
  else tma_load_3d_pair(dst, tm, fb, c0, c1, c2);
}
template <int CTAS>
__device__ __forceinline__ void stage_load(void* dst, const CUtensorMap* tm, uint64_t* bar, uint32_t fb, int c0, int c1,
                                           int c2, int c3) {
  if constexpr (CTAS == 1) tma_load_4d(dst, tm, bar, c0, c1, c2, c3);
  else tma_load_4d_pair(dst, tm, fb, c0, c1, c2, c3);
}
template <int CTAS>
__device__ __forceinline__ void stage_load(void* dst, const CUtensorMap* tm, uint64_t* bar, uint32_t fb, int c0, int c1,
                                           int c2, int c3, int c4) {
  if constexpr (CTAS == 1) tma_load_5d(dst, tm, bar, c0, c1, c2, c3, c4);
  else tma_load_5d_pair(dst, tm, fb, c0, c1, c2, c3, c4);
}

// One accumulator tile (this warp's 32 TMEM lanes x BN/4 columns) -> fused epilogue -> global memory.
// Shared-memory bandwidth belongs to the MMA (a 128x256x16 UMMA reads 12 KB of operands per 128 cycles = 96 of the
// 128 B/cycle), so the epilogue never touches smem: tcgen05.ld.16x256b hands every quad of lanes 8 consecutive
// columns of a row (2 per lane), a 4x4 quad transpose through warp shuffles gives each lane 8 CONSECUTIVE columns
// (32 B fp32 / 16 B bf16) of rows g and g+8, and all global traffic (bias, residual, saved GELU', outputs) is
// 16-byte vectors with 64-128 contiguous bytes per row per instruction.  Work unit = 16 TMEM lanes x 32 columns;
// the next unit's TMEM load is in flight during the math of the current one.  `arrive()` hands the accumulator back
// to the MMA warp as soon as this warp's last tcgen05.ld has completed.
// TF32: the reference-precision inference GEMM (act 4 = exact erf GELU in fp32, no bf16 rounding anywhere).
template <int BN, bool WGRAD, bool TF32 = false, typename Arrive>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, uint32_t t_base, int lane, int lane_grp, int col_q,
                                              int n_blk, int b, int row_in_batch0, long long wgrad_row0, bool have_k,
                                              Arrive arrive, long long out_off = 0) {
  // out_off: wgrad in deterministic mode writes every token split to its own [M, N] slab (p.split_stride elements apart)
  // work units of 16 TMEM lanes x 32 columns: 2 * BN / 32 per lane group, BN / 64 consecutive ones per warp (the four
  // warps of a lane group split them by col_q); t_base addresses column 0 of the accumulator for this lane group
  constexpr int UNITS = BN / 64;
  const int g = lane >> 2, tg = lane & 3;
  uint32_t v[16];
  tmem_ld_16x256b_x4(t_base + (static_cast<uint32_t>(((col_q * UNITS) & 1) * 16) << 16) + ((col_q * UNITS) >> 1) * 32, v);
#pragma unroll 1
  for (int u = 0; u < UNITS; ++u) {
    const int ug = col_q * UNITS + u;
    const int ch = ug >> 1, half = ug & 1;
    const int n0 = n_blk * BN + ch * 32 + tg * 8;
    const bool col_ok = n0 < p.N;   // N is a multiple of 8: groups of 8 columns are all-or-nothing
    // physical output rows of tile rows (lane_grp*32 + 16*half + 8*hr + g); -1 = nothing to write
    long long orow2[2];
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {
      const int r_local = lane_grp * 32 + half * 16 + hr * 8 + g;
      long long orow;
      bool ok;
      if constexpr (!WGRAD) {
        const int rib = row_in_batch0 + r_local;
        ok = rib < p.L;
        orow = static_cast<long long>(b) * p.L + rib;
      } else {
        orow = wgrad_row0 + r_local;
        ok = orow < p.M && have_k;
      }
      if (ok && p.out_rows != nullptr) orow = p.out_rows[orow];
      orow2[hr] = (ok && col_ok) ? orow : -1;
    }
    // the global inputs of this unit (fp32/bf16 residual or the saved GELU') are requested BEFORE waiting for TMEM
    uint4 pre[2][2];
    const bool pre_resid = p.resid != nullptr;
    const bool pre_aux = !pre_resid && p.act == 2;
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {
      pre[hr][0] = make_uint4(0u, 0u, 0u, 0u);
      pre[hr][1] = make_uint4(0u, 0u, 0u, 0u);
      if (orow2[hr] >= 0) {
        if (pre_resid) {
          const long long rrow = p.resid_mod > 0 ? (orow2[hr] % p.resid_mod) : orow2[hr];
          if (p.resid_f32) {
            const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.resid) + rrow * p.ld_resid + n0);
            pre[hr][0] = rp[0];
            pre[hr][1] = rp[1];
          } else {
            pre[hr][0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(p.resid) + rrow * p.ld_resid + n0);
          }
        } else if (pre_aux) {
          pre[hr][0] = *reinterpret_cast<const uint4*>(p.aux + orow2[hr] * p.ld_aux + n0);
        }
      }
    }
    tmem_ld_wait();
    // v[4*j + 2*hr + {0,1}] = (row g + 8*hr + 16*half, columns 8*j + 2*tg + {0,1}) of this warp's 32 x 32 chunk
    float f[2][8];
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {
      uint32_t a[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) { a[2 * j] = v[4 * j + 2 * hr]; a[2 * j + 1] = v[4 * j + 2 * hr + 1]; }
      quad_transpose(a, tg);   // -> a[0..7] = columns 8*tg .. 8*tg+7 of that row
#pragma unroll
      for (int c = 0; c < 8; ++c) f[hr][c] = __uint_as_float(a[c]);
    }
    if (u + 1 < UNITS) {
      const int nu = ug + 1;
      tmem_ld_16x256b_x4(t_base + (static_cast<uint32_t>((nu & 1) * 16) << 16) + (nu >> 1) * 32, v);
    } else {
      // every lane has executed tcgen05.wait::ld for its last unit -> hand the accumulator back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) arrive();
    }

    float bias8[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) bias8[c] = 0.f;
    if (p.bias != nullptr && col_ok) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + n0));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + 4));
      bias8[0] = b0.x; bias8[1] = b0.y; bias8[2] = b0.z; bias8[3] = b0.w;
      bias8[4] = b1.x; bias8[5] = b1.y; bias8[6] = b1.z; bias8[7] = b1.w;
    }
    float cs[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) cs[c] = 0.f;
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {
      const long long orow = orow2[hr];
      if (orow < 0) continue;
      float* x = f[hr];
      if (p.bias != nullptr) {
#pragma unroll
        for (int c = 0; c < 8; ++c) x[c] += bias8[c];
      }
      if constexpr (TF32) {
        if (p.act == 4) {
#pragma unroll
          for (int c = 0; c < 8; ++c) x[c] = gelu_erf(x[c]);
        }
      } else if (p.act == 3) {
        // the Linear output is bf16 under autocast before it meets the fp32 residual / positional table
#pragma unroll
        for (int c = 0; c < 8; c += 2) bf16_round2(x[c], x[c + 1]);
      } else if (p.act == 1) {
        // autocast semantics: the linear/conv output is bf16 and GELU is evaluated on that bf16 value; out2
        // receives GELU'(h) (bf16), which is all the backward needs of the pre-activation
#pragma unroll
        for (int c = 0; c < 8; c += 2) bf16_round2(x[c], x[c + 1]);
        if (p.out2 != nullptr) {
          float d[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) gelu_fast2(x[c], x[c], d[c]);
          uint4 w;
          w.x = pack_bf16x2(d[0], d[1]); w.y = pack_bf16x2(d[2], d[3]);
          w.z = pack_bf16x2(d[4], d[5]); w.w = pack_bf16x2(d[6], d[7]);
          *reinterpret_cast<uint4*>(p.out2 + orow * p.ld_out2 + n0) = w;
        } else {
#pragma unroll
          for (int c = 0; c < 8; ++c) x[c] = gelu_fast(x[c]);
        }
      } else if (p.act == 2) {
        const uint4 w = pre_aux ? pre[hr][0] : *reinterpret_cast<const uint4*>(p.aux + orow * p.ld_aux + n0);
        x[0] *= __uint_as_float(w.x << 16); x[1] *= __uint_as_float(w.x & 0xffff0000u);
        x[2] *= __uint_as_float(w.y << 16); x[3] *= __uint_as_float(w.y & 0xffff0000u);
        x[4] *= __uint_as_float(w.z << 16); x[5] *= __uint_as_float(w.z & 0xffff0000u);
        x[6] *= __uint_as_float(w.w << 16); x[7] *= __uint_as_float(w.w & 0xffff0000u);
      }
      if (p.resid != nullptr) {
        if (p.resid_f32) {
          const float4 r0 = *reinterpret_cast<const float4*>(&pre[hr][0]);
          const float4 r1 = *reinterpret_cast<const float4*>(&pre[hr][1]);
          x[0] += r0.x; x[1] += r0.y; x[2] += r0.z; x[3] += r0.w;
          x[4] += r1.x; x[5] += r1.y; x[6] += r1.z; x[7] += r1.w;
        } else {
          const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&pre[hr][0]);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 hh = __bfloat1622float2(h2[t]);
            x[2 * t] += hh.x; x[2 * t + 1] += hh.y;
          }
        }
      }
      if (WGRAD && p.transpose_out) {
        // element (orow, n0 + c) of the computed tile is out[n0 + c][orow]: 8 lanes (g) cover 8 consecutive floats
        float* op = reinterpret_cast<float*>(p.out) + static_cast<long long>(n0) * p.ld_out + orow;
#pragma unroll
        for (int c = 0; c < 8; ++c) atomicAdd(op + c * p.ld_out, x[c]);
      } else if (p.out_f32) {
        if constexpr (TF32) {
          if (p.round_tf32) {
#pragma unroll
            for (int c = 0; c < 8; ++c) x[c] = tf32_round(x[c]);
          }
        }
        float* op = reinterpret_cast<float*>(p.out) + out_off + orow * p.ld_out + n0;
        if (p.accumulate) {
          red_add_v4(op, x[0], x[1], x[2], x[3]);
          red_add_v4(op + 4, x[4], x[5], x[6], x[7]);
        } else {
          *reinterpret_cast<float4*>(op) = make_float4(x[0], x[1], x[2], x[3]);
          *reinterpret_cast<float4*>(op + 4) = make_float4(x[4], x[5], x[6], x[7]);
        }
      } else {
        const uint32_t w0 = pack_bf16x2(x[0], x[1]), w1 = pack_bf16x2(x[2], x[3]), w2 = pack_bf16x2(x[4], x[5]),
                       w3 = pack_bf16x2(x[6], x[7]);
        *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(p.out) + orow * p.ld_out + n0) = make_uint4(w0, w1, w2, w3);
        if (p.colsum != nullptr) {   // sums of the values as stored (bf16), like autograd's bias gradient
          x[0] = __uint_as_float(w0 << 16); x[1] = __uint_as_float(w0 & 0xffff0000u);
          x[2] = __uint_as_float(w1 << 16); x[3] = __uint_as_float(w1 & 0xffff0000u);
          x[4] = __uint_as_float(w2 << 16); x[5] = __uint_as_float(w2 & 0xffff0000u);
          x[6] = __uint_as_float(w3 << 16); x[7] = __uint_as_float(w3 & 0xffff0000u);
        }
      }
      if (p.colsum != nullptr) {
#pragma unroll
        for (int c = 0; c < 8; ++c) cs[c] += x[c];
      }
    }
    if (p.colsum != nullptr) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        cs[c] += __shfl_xor_sync(0xffffffffu, cs[c], 4);
        cs[c] += __shfl_xor_sync(0xffffffffu, cs[c], 8);
        cs[c] += __shfl_xor_sync(0xffffffffu, cs[c], 16);
      }
      if (g == 0 && col_ok) {
        red_add_v4(p.colsum + n0, cs[0], cs[1], cs[2], cs[3]);
        red_add_v4(p.colsum + n0 + 4, cs[4], cs[5], cs[6], cs[7]);
      }
    }
  }
}

// bf16 outputs with nothing but bias / GELU in the epilogue (QKV projections, MLP fc1 fwd, conv fwd, plain dgrads) skip
// the per-element addressing, transposes and predicates of the generic path: tcgen05.ld.32x32b (row per lane) -> math
// -> 4 x st.shared.v4 into a 64B-swizzled 32 x 32 staging tile (2 KB per warp) -> ONE TMA store per 32 x 32 chunk
// (the hardware clips rows >= L and columns >= N).  ~5x fewer issued instructions per element than the generic path.
// (Measured alternatives, all slower on B200: reading the staged tile back transposed and writing it with coalesced
// st.global.v4 instead of the TMA store -- 0.247 vs 0.209 ms on the 172k x 1536 x 384 GEMM; draining both 32-column
// chunks from TMEM and releasing the accumulator before any math -- 0.353 vs 0.302 ms with the two-output GELU.)
__device__ __forceinline__ void stage_rows(uint8_t* stg, int lane, const uint32_t (&w)[16]) {
  uint8_t* srow = stg + lane * 64;          // staging row = lane (64 B); 16-byte chunk c lives at c ^ ((row >> 1) & 3)
  const int sw = (lane >> 1) & 3;           // (CU_TENSOR_MAP_SWIZZLE_64B)
#pragma unroll
  for (int c = 0; c < 4; ++c)
    *reinterpret_cast<uint4*>(srow + ((c ^ sw) << 4)) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
}

// staged 32 x 32 bf16 chunk -> global memory through one TMA store
__device__ __forceinline__ void chunk_to_global(const CUtensorMap* map, uint8_t* stg, int lane, const uint32_t (&w)[16],
                                                int n0, int row0, int b) {
  if (lane == 0) bulk_wait_read0();   // the previous TMA store of this warp has finished reading the staging tile
  __syncwarp();
  stage_rows(stg, lane, w);
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    tma_store_3d(map, stg, n0, row0, b);
    bulk_commit();
  }
}

template <int BN, bool HEAVY, typename Arrive>
__device__ __forceinline__ void epilogue_tile_tma(const GemmParams& p, const OutMaps& om, uint32_t t_base, uint8_t* stg,
                                                  int lane, int lane_grp, int col_q, int n_blk, int b, int row_in_batch0,
                                                  Arrive arrive) {
  // 32-column chunks per warp: BN/128, except BN = 192 (6 chunks per lane group): the warps of column quarters 0..2
  // take two each and quarter 3 only hands the accumulator back
  constexpr int CHUNKS = (BN / 32 + 3) / 4;
  const int n_ch = (BN / 32 - col_q * CHUNKS) < CHUNKS ? (BN / 32 - col_q * CHUNKS) : CHUNKS;
  if (n_ch <= 0) {
    __syncwarp();
    if (lane == 0) arrive();
    return;
  }
  const int row0 = row_in_batch0 + lane_grp * 32;
  uint32_t v[32];
  tmem_ld_32x32(t_base, v);
#pragma unroll 1
  for (int ch = 0; ch < n_ch; ++ch) {
    const int n0 = n_blk * BN + (col_q * CHUNKS + ch) * 32;
    const bool live = n0 < p.N && row0 < p.L;   // warp-uniform
    tmem_ld_wait();
    float f[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
    if (ch + 1 < n_ch) {
      tmem_ld_32x32(t_base + (ch + 1) * 32, v);   // in flight during the math of this chunk
    } else {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) arrive();
    }
    if (!live) continue;
    if (p.bias != nullptr) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        if (n0 + j < p.N) {
          const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + j));
          f[j] += bb.x; f[j + 1] += bb.y; f[j + 2] += bb.z; f[j + 3] += bb.w;
        }
      }
    }
    uint32_t w[16];
    uint32_t w2[HEAVY ? 16 : 1];
    if constexpr (!HEAVY) {
      if (p.act == 1) {   // GELU of the Linear / conv output, two values per instruction (see ptx.cuh: gelu_h2)
#pragma unroll
        for (int j = 0; j < 32; j += 2) w[j >> 1] = gelu_h2(f[j], f[j + 1]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 2) w[j >> 1] = pack_bf16x2(f[j], f[j + 1]);
      }
    } else {
      if (p.act == 1) {
#pragma unroll
        for (int j = 0; j < 32; j += 2) gelu_h2_save(f[j], f[j + 1], w[j >> 1], w2[j >> 1]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 2) w[j >> 1] = pack_bf16x2(f[j], f[j + 1]);
      }
    }
    chunk_to_global(&om.o, stg, lane, w, n0, row0, b);
    if constexpr (HEAVY) {
      if (p.act == 1 && p.out2 != nullptr) {
        __syncwarp();
        chunk_to_global(&om.o2, stg, lane, w2, n0, row0, b);
      }
    }
  }
}

// Backward of GELU on the TMA-store path (dgrad only): out (bf16) = acc * saved GELU'(h), optional fused column sums
// (the bias gradient of the Linear whose output was h).
//
// clock64 counters of the three roles (profiles/r02_gemm_cycle_counters.txt) showed this epilogue to be what the K = 384
// dgrad waits for: 9700 cycles per tile with the MMA thread idle 5200 of them, because every 32 x 32 chunk began with
// a DRAM round trip for its factors (row-per-lane global loads, consumed ~3000 cycles later); registers for a deeper
// software pipeline do not exist (64 accumulator + 16 factor + 16 result registers per chunk).  So the factors now come
// the way the operands do: ONE TMA box per chunk ([32 rows x 32 columns], 64B swizzle = the staging layout) into a
// shared-memory tile owned by the warp, completion on the warp's own mbarrier, issued a whole tile before use:
//
//   tile t, chunk c (tile X_c of this warp):  wait barrier_c -> each lane reads its row's 64 B of factors -> multiply,
//   pack -> the SAME tile X_c stages the output -> TMA store -> (column sums from registers) -> once the store has read
//   X_c: TMA load of the factors of (tile t + gridDim, chunk c) into X_c.
//
// Two tiles per warp (64 KB per CTA) are paid for with one operand stage (3 instead of 4).
struct AuxPipe {
  uint8_t* buf;        // this warp's two 2 KB tiles
  uint64_t* bar;       // [2] mbarriers, one per tile
  uint32_t phase[2];
};

template <int BN>
__device__ __forceinline__ bool aux_issue(const GemmParams& p, const OutMaps& om, AuxPipe& ap, int lane, int lane_grp,
                                          int col_q, int tile, int ch, int tile_rows, int row_off) {
  // tile_rows / row_off: rows of an m-block and this CTA's offset inside it (see tile_coords)
  constexpr int CHUNKS = BN / 32 / 4;
  if (tile >= p.total_tiles) return false;
  const TileCoords tc = tile_coords<false>(p, tile, tile_rows, row_off);
  const int row0 = tc.row0 + lane_grp * 32;
  const int n0 = tc.n_blk * BN + (col_q * CHUNKS + ch) * 32;
  const bool live = n0 < p.N && row0 < p.L;   // warp-uniform; the same predicate gates the consumer
  if (live && lane == 0) {
    mbar_arrive_expect_tx(&ap.bar[ch], 2048);   // (TMA always delivers the whole box: out-of-range parts are zero-filled)
    tma_load_3d(ap.buf + ch * 2048, &om.o2, &ap.bar[ch], n0, row0, tc.b);
  }
  return live;
}

template <int BN, typename Arrive>
__device__ __forceinline__ void epilogue_tile_tma_aux(const GemmParams& p, const OutMaps& om, uint32_t t_base, AuxPipe& ap,
                                                      int lane, int lane_grp, int col_q, int n_blk, int b,
                                                      int row_in_batch0, int next_tile, Arrive arrive, int tile_rows,
                                                      int row_off) {
  constexpr int CHUNKS = BN / 32 / 4;
  const int row0 = row_in_batch0 + lane_grp * 32;
  const int sw = (lane >> 1) & 3;
  uint32_t v[32];
  tmem_ld_32x32(t_base, v);
#pragma unroll 1
  for (int ch = 0; ch < CHUNKS; ++ch) {
    const int n0 = n_blk * BN + (col_q * CHUNKS + ch) * 32;
    const bool live = n0 < p.N && row0 < p.L;   // warp-uniform
    uint8_t* stg = ap.buf + ch * 2048;
    uint8_t* srow = stg + lane * 64;
    tmem_ld_wait();
    float f[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
    if (ch + 1 < CHUNKS) {
      tmem_ld_32x32(t_base + (ch + 1) * 32, v);
    } else {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) arrive();
    }
    if (live) {
      mbar_wait(&ap.bar[ch], ap.phase[ch]);     // the factors of this chunk have landed (issued one tile ago)
      ap.phase[ch] ^= 1;
      uint4 a[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) a[c] = *reinterpret_cast<const uint4*>(srow + ((c ^ sw) << 4));
      uint32_t w[16];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint32_t aw[4] = {a[c].x, a[c].y, a[c].z, a[c].w};
#pragma unroll
        for (int t = 0; t < 4; ++t)
          w[4 * c + t] = pack_bf16x2(f[8 * c + 2 * t] * __uint_as_float(aw[t] << 16),
                                     f[8 * c + 2 * t + 1] * __uint_as_float(aw[t] & 0xffff0000u));
      }
      __syncwarp();                           // every lane has read its factors: the tile now stages the output
#pragma unroll
      for (int c = 0; c < 4; ++c)
        *reinterpret_cast<uint4*>(srow + ((c ^ sw) << 4)) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_3d(&om.o, stg, n0, row0, b);
        bulk_commit();
      }
      if (p.colsum != nullptr) {
        // sums of the values as stored (bf16), like autograd's bias gradient: reduce-scatter over the 32 rows of the warp
        float c32[32];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          c32[2 * j] = __uint_as_float(w[j] << 16);
          c32[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
        }
#pragma unroll
        for (int s = 16; s >= 1; s >>= 1) {
          const bool up = (lane & s) != 0;
#pragma unroll
          for (int i = 0; i < s; ++i) {
            const float mine = up ? c32[s + i] : c32[i];
            const float other = up ? c32[i] : c32[s + i];
            c32[i] = mine + __shfl_xor_sync(0xffffffffu, other, s);
          }
        }
        if (n0 + lane < p.N) atomicAdd(p.colsum + n0 + lane, c32[0]);
      }
      if (lane == 0) bulk_wait_read0();       // the store has read the tile: it may receive the next tile's factors
    }
    __syncwarp();
    aux_issue<BN>(p, om, ap, lane, lane_grp, col_q, next_tile, ch, tile_rows, row_off);
  }
}

// MODE 0: A K-major, B K-major (fwd)   MODE 1: A, B MN-major (wgrad)   MODE 2: A K-major, B MN-major (dgrad)
// TF32 (MODE 0 only): fp32 operands, tcgen05.mma.kind::tf32.  A 128-byte swizzle row holds 64 bf16 or 32 fp32, and one
// UMMA consumes 32 bytes of K either way, so the shared-memory ring, descriptors and barriers are byte-identical; only
// the element count of a k-block (KB), the instruction kind and the descriptor's operand formats change.
//
// CTAS = 2: two CTAs of a cluster (one TPC) work on one 256 x BN tile with tcgen05.mma.cta_group::2: each CTA stages
// its own 128 rows of A and its own HALF of B (BN/2 columns), the leader's single MMA thread drives both tensor cores,
// and each CTA's TMEM receives its 128 accumulator rows.  Per SM that is 32 KB of operands per 128 x 256 x 64 of MMA
// work instead of 48 KB (less L2 -> SM traffic, 6 pipeline stages instead of 4 in the same shared memory, and only 2/3
// of the shared-memory read bandwidth), which is what a single CTA runs out of.  Barrier protocol: both producers
// signal the LEADER's full barriers (TMA .cta_group::2), the leader's commits are multicast to the empty /
// accumulator-full barriers of both CTAs, the epilogue warps of both CTAs arrive on the leader's accumulator-empty
// barrier.
// `tid` is threadIdx.x as read by the __global__ entry point, where __launch_bounds__ tells the compiler it is below
// kThreads (a read in this inlined body would not carry that range, which costs registers in the control warps).
template <int BN, int MODE, bool HEAVY, bool TF32, int CTAS>
__device__ __forceinline__ void gemm_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmB1,
                                          const OutMaps& om, const GemmParams& p, uint32_t tid) {
  static_assert(!TF32 || (MODE == 0 && !HEAVY && CTAS == 1), "the tf32 kernel is the plain single-CTA forward");
  constexpr bool AUXQ = (MODE == 2 && HEAVY);   // GELU-backward dgrad: TMA-fed factor tiles (see epilogue_tile_tma_aux)
  using C = Cfg<BN, AUXQ, CTAS>;
  constexpr bool WGRAD = (MODE == 1);
  constexpr bool B_MN = (MODE != 0);
  constexpr bool DBG = (CTAS == 1);   // wj_gemm_debug cycle counters: single-CTA launches
  constexpr int STAGES = C::STAGES;
  constexpr int KB = TF32 ? BK / 2 : BK;   // elements of K per k-block (128 bytes of each operand row)
  constexpr int TILE_ROWS = CTAS * BM;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  uint64_t* aux_bar = full_bar + 64;            // [kEpiWarps][2], 512 bytes into the barrier KB

  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int rank = CTAS == 2 ? static_cast<int>(cluster_ctarank()) : 0;   // this CTA's rows of a pair tile: rank * BM
  const bool leader = rank == 0;
  // static round-robin tile schedule over CTAs (CTA pairs); read where used rather than kept live through all roles
  auto first_tile = [] { return static_cast<int>(blockIdx.x / CTAS); };
  auto tile_step = [] { return static_cast<int>(gridDim.x / CTAS); };
  // single CTAs sleep between probes of the empty / accumulator-empty barriers (see mbar_wait_relaxed)
  auto wait_free = [](uint64_t* bar, uint32_t parity) {
    if constexpr (CTAS == 1) mbar_wait_relaxed(bar, parity);
    else mbar_wait(bar, parity);
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], CTAS * kEpiWarps);
    }
    if constexpr (AUXQ) {
      for (int i = 0; i < 2 * kEpiWarps; ++i) mbar_init(&aux_bar[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    if constexpr (CTAS == 1) tmem_alloc(tmem_slot, 512);
    else tmem_alloc_pair(tmem_slot, 512);
  }
  tc_fence_before();
  if constexpr (CTAS == 1) __syncthreads();
  else cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto num_kb = [&](int tile) -> int {
    if constexpr (!WGRAD) {
      return p.K / KB;
    } else {
      int lo, hi;
      wgrad_kb_range(p, tile_coords<true>(p, tile, TILE_ROWS, rank * BM).split, lo, hi);
      return hi > lo ? hi - lo : 0;
    }
  };

  using RS = RegSplit<(MODE == 0 && HEAVY)>;
  if (warp < kEpiWarp0) reg_dealloc<RS::CTRL>();
  if (warp == 0) {
    // ======================================================================================= TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      long long dbg_prod = 0;
      for (int tile = first_tile(); tile < p.total_tiles; tile += tile_step()) {
        const TileCoords tc = tile_coords<WGRAD>(p, tile, TILE_ROWS, rank * BM);
        // this CTA's B columns: the whole tile, or its half of a pair tile
        const int nb0 = tc.n_blk * BN + rank * (BN / CTAS);
        if constexpr (!WGRAD) {
          const int nkb = p.K / KB;
          for (int kb = 0; kb < nkb; ++kb) {
            const long long tw = (DBG && p.dbg) ? clock64() : 0;
            wait_free(&empty_bar[stage], phase ^ 1);
            if (DBG && p.dbg) dbg_prod += clock64() - tw;
            uint8_t* sa = smem + stage * C::STAGE_BYTES;
            uint8_t* sb = sa + C::A_BYTES;
            const uint32_t fb = CTAS == 2 ? mapa_shared(smem_u32(&full_bar[stage]), 0) : 0u;
            int c0, q, po;
            seg_coords(p.seg, kb * KB, c0, q, po);
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], CTAS * C::STAGE_BYTES);
            stage_load<CTAS>(sa, &tmA, &full_bar[stage], fb, c0, q, tc.row0 + po, tc.b);
            if constexpr (!B_MN) {
              stage_load<CTAS>(sb, &tmB, &full_bar[stage], fb, kb * KB, nb0);
            } else {
              // dgrad: W is [reduction rows, output cols] row-major -> BN/CTAS/64 MN-major atoms of 64 reduction rows,
              // all fetched by ONE TMA instruction through a 3-D view {64 cols, rows, column atoms} (the TMA unit is
              // instruction-rate limited: 5-6 small boxes per k-block held these modes at ~600-900 TFLOP/s)
              const int si = p.seg.width > 0 ? (kb * BK) / p.seg.width : 0;
              const int r0 = kb * BK - si * (p.seg.width > 0 ? p.seg.width : 0);
              stage_load<CTAS>(sb, &tmB, &full_bar[stage], fb, 0, r0, (p.segB_col[si] + nb0) >> 6);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        } else {
          int lo, hi;
          wgrad_kb_range(p, tc.split, lo, hi);
          for (int kb = lo; kb < hi; ++kb) {
            const int b = kb / p.kb_per_batch;
            const int row0 = (kb - b * p.kb_per_batch) * BK;
            wait_free(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * C::STAGE_BYTES;
            uint8_t* sb = sa + C::A_BYTES;
            const uint32_t fb = CTAS == 2 ? mapa_shared(smem_u32(&full_bar[stage]), 0) : 0u;
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], CTAS * C::STAGE_BYTES);
            // A operand: dY[b, row, m] (m contiguous): this CTA's BM/64 MN atoms of 64 reduction rows, one 5-D TMA
            // {64 cols, rows, column atoms, q, batch}
            stage_load<CTAS>(sa, &tmA, &full_bar[stage], fb, 0, row0, tc.row0 >> 6, 0, b);
            // B operand: X[b, row + p, (q), n]: BN/CTAS/64 atoms; one TMA when they lie inside one segment (the host
            // routes pairs here only then), else one per atom
            if (CTAS == 2 || p.b_single) {
              int c0, q, po;
              seg_coords(p.seg, nb0, c0, q, po);
              stage_load<CTAS>(sb, &tmB, &full_bar[stage], fb, 0, row0 + po, c0 >> 6, q, b);
            } else {
#pragma unroll
              for (int a = 0; a < BN / 64; ++a) {
                int c0, q, po;
                seg_coords(p.seg, nb0 + a * 64, c0, q, po);
                stage_load<CTAS>(sb + a * (BK * 128), &tmB1, &full_bar[stage], fb, 0, row0 + po, c0 >> 6, q, b);
              }
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
      if (DBG && p.dbg) p.dbg[blockIdx.x * 8 + 3] = dbg_prod;
    }
  } else if (warp == 1) {
    // ======================================================================================= MMA issuer (leader CTA)
    if (leader && lane == 0) {
      constexpr uint32_t idesc = TF32 ? umma_idesc_tf32(TILE_ROWS, BN) : umma_idesc_bf16(TILE_ROWS, BN, WGRAD, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      long long dbg_full = 0, dbg_empty = 0;
      const long long dbg_t0 = (DBG && p.dbg) ? clock64() : 0;
      for (int tile = first_tile(); tile < p.total_tiles; tile += tile_step(), ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        const int nkb = num_kb(tile);
        long long tw = (DBG && p.dbg) ? clock64() : 0;
        wait_free(&tempty_bar[acc], acc_phase ^ 1);
        if (DBG && p.dbg) dbg_empty += clock64() - tw;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < nkb; ++kb) {
          tw = (DBG && p.dbg) ? clock64() : 0;
          mbar_wait(&full_bar[stage], phase);
          if (DBG && p.dbg) dbg_full += clock64() - tw;
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t sb = sa + C::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            uint64_t da, db;
            // K-major, 128B swizzle: rows of 128 B, 8-row groups 1024 B apart; advance 16 elements = 32 B
            // MN-major, 128B swizzle: atom = 64 (MN) x 8 (K) = 1024 B; K groups 1024 B apart (SBO),
            // MN atoms BK*128 B apart (LBO); advance 16 reduction rows = 2048 B
            if constexpr (!WGRAD) da = umma_smem_desc_sw128(sa + k * 32, 0, 1024);
            else da = umma_smem_desc_sw128(sa + k * 2048, BK * 128, 1024);
            if constexpr (!B_MN) db = umma_smem_desc_sw128(sb + k * 32, 0, 1024);
            else db = umma_smem_desc_sw128(sb + k * 2048, BK * 128, 1024);
            const uint32_t accum = (kb > 0 || k > 0) ? 1u : 0u;
            if constexpr (CTAS == 2) umma_bf16_pair(d_tmem, da, db, idesc, accum);
            else if constexpr (TF32) umma_tf32(d_tmem, da, db, idesc, accum);
            else umma_bf16(d_tmem, da, db, idesc, accum);
          }
          // frees the smem slot (of both CTAs) when these MMAs retire
          if constexpr (CTAS == 1) umma_commit(&empty_bar[stage]);
          else umma_commit_pair(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        // accumulator complete -> epilogue (of both CTAs)
        if constexpr (CTAS == 1) umma_commit(&tfull_bar[acc]);
        else umma_commit_pair(&tfull_bar[acc]);
      }
      if (DBG && p.dbg) {
        p.dbg[blockIdx.x * 8 + 0] = dbg_full;
        p.dbg[blockIdx.x * 8 + 1] = dbg_empty;
        p.dbg[blockIdx.x * 8 + 2] = clock64() - dbg_t0;
        p.dbg[blockIdx.x * 8 + 6] = it;
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ======================================================================================= epilogue (16 warps)
    // Shared-memory bandwidth belongs to the MMA (a 128x256x16 UMMA reads 12 KB of operands per 128 cycles = 96 of the
    // 128 B/cycle), so the epilogue never touches smem: tcgen05.ld.16x256b hands every quad of lanes 8 consecutive
    // columns of a row (2 per lane), a 4x4 quad transpose through warp shuffles gives each lane 8 CONSECUTIVE columns
    // (32 B fp32 / 16 B bf16) of rows g and g+8, and all global traffic (bias, residual, saved GELU', outputs) is
    // 16-byte vectors with 64-128 contiguous bytes per row per instruction.  Work unit = 16 TMEM lanes x 32 columns;
    // the next unit's TMEM load is in flight during the math of the current one.  16 warps (4 per scheduler) hide the
    // shuffle / global-load latencies; registers come from the producer/MMA warpgroup via setmaxnreg.
    reg_alloc<RS::EPI>();
    const int ew = warp - kEpiWarp0;
    const int lane_grp = warp & 3;            // TMEM lanes [32*lane_grp, +32) are accessible to this warp
    const int col_q = ew >> 2;                // which quarter of the BN columns this warp handles
    constexpr int CHUNKS = (BN / 32 + 3) / 4; // 32-column chunks per warp (TMA-store paths)
    int it = 0;
    long long dbg_epi = 0;
    const long long dbg_e0 = (DBG && p.dbg) ? clock64() : 0;
    AuxPipe ap;
    ap.buf = smem + C::STAGING_OFF + ew * C::WARP_STAGING;
    ap.bar = aux_bar + ew * 2;
    ap.phase[0] = ap.phase[1] = 0;
    if constexpr (AUXQ) {
      if (p.tma_store) {   // factors of this CTA's first tile
#pragma unroll
        for (int ch = 0; ch < BN / 128; ++ch) aux_issue<BN>(p, om, ap, lane, lane_grp, col_q, first_tile(), ch, TILE_ROWS, rank * BM);
      }
    }
    for (int tile = first_tile(); tile < p.total_tiles; tile += tile_step(), ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const TileCoords tc = tile_coords<WGRAD>(p, tile, TILE_ROWS, rank * BM);
      const bool have_k = !WGRAD || num_kb(tile) > 0;
      const long long tw = (DBG && p.dbg && warp == kEpiWarp0) ? clock64() : 0;
      mbar_wait(&tfull_bar[acc], acc_phase);
      if (DBG && p.dbg && warp == kEpiWarp0) dbg_epi += clock64() - tw;
      tc_fence_after();
      const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(lane_grp * 32) << 16) + acc * BN;
      const uint32_t t_base = t_acc + col_q * (CHUNKS * 32);   // (TMA-store paths: CHUNKS consecutive chunks per warp)
      // the accumulator goes back to the MMA warp through the (leader's) accumulator-empty barrier
      const uint32_t te = CTAS == 2 ? mapa_shared(smem_u32(&tempty_bar[acc]), 0) : 0u;
      auto arrive = [&]() {
        if constexpr (CTAS == 1) mbar_arrive(&tempty_bar[acc]);
        else mbar_arrive_cluster(te);
      };
      if constexpr (!WGRAD && !TF32) {
        if (p.tma_store) {
          if constexpr (AUXQ) {   // (for dgrad the second instantiation is the GELU-backward path)
            epilogue_tile_tma_aux<BN>(p, om, t_base, ap, lane, lane_grp, col_q, tc.n_blk, tc.b, tc.row0,
                                      tile + tile_step(), arrive, TILE_ROWS, rank * BM);
          } else {
            epilogue_tile_tma<BN, HEAVY>(p, om, t_base, ap.buf, lane, lane_grp, col_q, tc.n_blk, tc.b, tc.row0, arrive);
          }
          continue;
        }
      }
      long long out_off = 0;
      if constexpr (WGRAD) out_off = static_cast<long long>(tc.split) * p.split_stride;
      epilogue_tile<BN, WGRAD, TF32>(p, t_acc, lane, lane_grp, col_q, tc.n_blk, tc.b, tc.row0, tc.row0, have_k, arrive,
                                     out_off);
    }
    if (p.tma_store && lane == 0) bulk_wait0();   // all TMA stores of this warp are complete before smem goes away
    if (DBG && p.dbg && warp == kEpiWarp0 && lane == 0) {
      p.dbg[blockIdx.x * 8 + 4] = dbg_epi;
      p.dbg[blockIdx.x * 8 + 5] = clock64() - dbg_e0;
    }
  }

  tc_fence_before();
  if constexpr (CTAS == 1) __syncthreads();
  else cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CTAS == 1) tmem_dealloc(tmem_base, 512);
    else tmem_dealloc_pair(tmem_base, 512);
  }
}

template <int BN, int MODE, bool HEAVY, bool TF32 = false>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmB1, const __grid_constant__ OutMaps om, const GemmParams p) {
  gemm_body<BN, MODE, HEAVY, TF32, 1>(tmA, tmB, tmB1, om, p, threadIdx.x);
}

template <int BN, int MODE, bool HEAVY>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ OutMaps om, const GemmParams p) {
  gemm_body<BN, MODE, HEAVY, false, 2>(tmA, tmB, tmB, om, p, threadIdx.x);
}

// =================================================================================================== host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(sym);
  }
  return fn;
}


static int encode_map(CUtensorMap* tm, const wj_operand_t* op, const uint32_t box[4],
                      CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)"); return WJ_ERR_RUNTIME; }
  cuuint64_t dims[4];
  cuuint64_t strides[3];
  cuuint32_t bx[4], es[4] = {1, 1, 1, 1};
  for (int i = 0; i < 4; ++i) { dims[i] = static_cast<cuuint64_t>(op->dim[i]); bx[i] = box[i]; }
  for (int i = 0; i < 3; ++i) strides[i] = static_cast<cuuint64_t>(op->stride_bytes[i]);
  CUresult r = enc(tm, dt, 4, const_cast<void*>(op->ptr), dims, strides, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: %d (dims %llu %llu %llu %llu strides %llu %llu %llu box %u %u %u %u)",
              (int)r, dims[0], dims[1], dims[2], dims[3], strides[0], strides[1], strides[2], bx[0], bx[1], bx[2],
              bx[3]);
    return WJ_ERR_RUNTIME;
  }
  return WJ_OK;
}

static int encode_map_2d(CUtensorMap* tm, const void* ptr, uint64_t inner, uint64_t outer, uint64_t stride_bytes,
                         uint32_t box_inner, uint32_t box_outer,
                         CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)"); return WJ_ERR_RUNTIME; }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {stride_bytes};
  cuuint32_t bx[2] = {box_inner, box_outer}, es[2] = {1, 1};
  CUresult r = enc(tm, dt, 2, const_cast<void*>(ptr), dims, strides, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(2d) failed: %d (dims %llu %llu stride %llu box %u %u)", (int)r, dims[0], dims[1],
              strides[0], bx[0], bx[1]);
    return WJ_ERR_RUNTIME;
  }
  return WJ_OK;
}

// MN-major operand view {64 contiguous columns, rows, column atoms (stride 128 B), q, batch}: a box {64, 64, atoms, 1, 1}
// lands in smem as [atom][64 rows][128 B] = the UMMA MN-major 128B-swizzle layout, with ONE TMA instruction.
static int encode_map_mn5(CUtensorMap* tm, const wj_operand_t* op, uint32_t atoms_box) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)"); return WJ_ERR_RUNTIME; }
  if (op->dim[0] % 64 != 0) { set_error("MN-major operand: column count %lld is not a multiple of 64", (long long)op->dim[0]); return WJ_ERR_ARG; }
  cuuint64_t dims[5] = {64, (cuuint64_t)op->dim[2], (cuuint64_t)(op->dim[0] / 64), (cuuint64_t)op->dim[1], (cuuint64_t)op->dim[3]};
  cuuint64_t strides[4] = {(cuuint64_t)op->stride_bytes[1], 128, (cuuint64_t)op->stride_bytes[0], (cuuint64_t)op->stride_bytes[2]};
  cuuint32_t bx[5] = {64, 64, atoms_box, 1, 1}, es[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(op->ptr), dims, strides, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(mn5) failed: %d (dims %llu %llu %llu %llu %llu strides %llu %llu %llu %llu)", (int)r,
              dims[0], dims[1], dims[2], dims[3], dims[4], strides[0], strides[1], strides[2], strides[3]);
    return WJ_ERR_RUNTIME;
  }
  return WJ_OK;
}
static int encode_map_mn3(CUtensorMap* tm, const void* ptr, uint64_t rows, uint64_t cols, uint64_t stride_bytes,
                          uint32_t atoms_box) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)"); return WJ_ERR_RUNTIME; }
  cuuint64_t dims[3] = {64, rows, (cols + 63) / 64};
  cuuint64_t strides[2] = {stride_bytes, 128};
  cuuint32_t bx[3] = {64, 64, atoms_box}, es[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(mn3) failed: %d (dims %llu %llu %llu strides %llu %llu)", (int)r, dims[0], dims[1],
              dims[2], strides[0], strides[1]);
    return WJ_ERR_RUNTIME;
  }
  return WJ_OK;
}

// bf16 output viewed as {N, L, batch} for the TMA-store epilogue (box 32 x 32, 64-byte swizzle)
static int encode_out_map(CUtensorMap* tm, const void* ptr, int N, int L, int batch, int64_t ld) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)"); return WJ_ERR_RUNTIME; }
  cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)L, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)L * (cuuint64_t)ld * 2};
  cuuint32_t bx[3] = {32, 32, 1}, es[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(out) failed: %d (dims %llu %llu %llu strides %llu %llu)", (int)r, dims[0], dims[1],
              dims[2], strides[0], strides[1]);
    return WJ_ERR_RUNTIME;
  }
  return WJ_OK;
}

// Whether the epilogue can take the TMA-store path: bf16 outputs with bias / GELU (optionally saving GELU'), and in
// dgrads also the GELU-backward form out = acc * aux (+ fused column sums), no bias.  Everything else (fp32 outputs,
// reduce-add, residual, row scatter) takes the generic epilogue.
static bool tma_store_ok(const wj_epilogue_t* e, int N, bool dgrad) {
  if (e == nullptr) return false;
  const bool gelu_bwd = dgrad && e->act == 2 && e->aux != nullptr && e->bias == nullptr && e->out2 == nullptr &&
                        e->ld_aux % 8 == 0 && reinterpret_cast<uintptr_t>(e->aux) % 16 == 0 && N % 8 == 0;
  return !e->out_f32 && !e->accumulate && e->resid == nullptr && e->out_rows == nullptr &&
         (gelu_bwd || (e->colsum == nullptr && (e->act == 0 || e->act == 1))) && e->ld_out % 8 == 0 &&
         reinterpret_cast<uintptr_t>(e->out) % 16 == 0 &&
         (e->out2 == nullptr || (e->ld_out2 % 8 == 0 && reinterpret_cast<uintptr_t>(e->out2) % 16 == 0));
}

// Decides whether the epilogue takes the TMA-store path and builds its maps.
static int setup_out_maps(GemmParams& p, OutMaps& om, const wj_epilogue_t* e, int N, int L, int batch, bool dgrad) {
  memset(&om, 0, sizeof(om));
  p.tma_store = 0;
  if (!tma_store_ok(e, N, dgrad)) return WJ_OK;
  int rc = encode_out_map(&om.o, p.out, N, L, batch, p.ld_out);
  if (rc) return rc;
  if (p.out2 != nullptr) {
    rc = encode_out_map(&om.o2, p.out2, N, L, batch, p.ld_out2);
    if (rc) return rc;
  }
  if (p.act == 2) {   // GELU backward: the saved factors have the output's shape, read by TMA loads (OutMaps::o2)
    rc = encode_out_map(&om.o2, p.aux, N, L, batch, p.ld_aux);
    if (rc) return rc;
  }
  p.tma_store = 1;
  return WJ_OK;
}

static int num_sms() { return sm_count(); }

// 192-column tiles exist for the generic (fp32-output) epilogue and for the plain bf16 TMA-store epilogue
static bool tile192_ok(const wj_epilogue_t* e, int N) {
  return e != nullptr && N % 192 == 0 && (e->out_f32 || (tma_store_ok(e, N, false) && e->out2 == nullptr));
}

// Grid: one CTA (CTA pair) per tile, at most one per SM (pair of SMs); the kernels loop over the remaining tiles.
template <int BN, int MODE, bool HEAVY, bool TF32, int CTAS>
static int launch_variant(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmB1, const OutMaps& om,
                          const GemmParams& p, cudaStream_t st) {
  static bool attr_set = false;
  constexpr int kSmem = Cfg<BN, (MODE == 2 && HEAVY), CTAS>::SMEM_BYTES;
  if (!attr_set) {
    cudaError_t e;
    if constexpr (CTAS == 1) e = cudaFuncSetAttribute(gemm_kernel<BN, MODE, HEAVY, TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    else e = cudaFuncSetAttribute(gemm_pair_kernel<BN, MODE, HEAVY>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    attr_set = true;
  }
  const int units = p.total_tiles < num_sms() / CTAS ? p.total_tiles : num_sms() / CTAS;
  if constexpr (CTAS == 1) gemm_kernel<BN, MODE, HEAVY, TF32><<<units, kThreads, kSmem, st>>>(tmA, tmB, tmB1, om, p);
  else gemm_pair_kernel<BN, MODE, HEAVY><<<CTAS * units, kThreads, kSmem, st>>>(tmA, tmB, om, p);
  return check_launch(CTAS == 1 ? "gemm_tcgen05 launch" : "gemm_tcgen05 pair launch");
}

// The two-output epilogue (GELU + saved GELU') and the GELU-backward dgrad (TMA-fed factor tiles) are their own
// instantiations of the TMA-store path (HEAVY: register budget, shared-memory layout).  192-column tiles (N = 384-like
// shapes) have the generic epilogue and the plain bf16 TMA-store epilogue (bias / GELU) only.
template <int BN, int MODE, int CTAS>
static int launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmB1, const OutMaps& om,
                  const GemmParams& p, cudaStream_t st) {
  const bool heavy = p.tma_store && (p.out2 != nullptr || p.act == 2);
  if constexpr (BN == 192) {
    if (heavy) { set_error("gemm: BN = 192 has only the plain TMA-store epilogue"); return WJ_ERR_ARG; }
  } else if constexpr (MODE != 1) {
    if (heavy) return launch_variant<BN, MODE, true, false, CTAS>(tmA, tmB, tmB1, om, p, st);
  }
  return launch_variant<BN, MODE, false, false, CTAS>(tmA, tmB, tmB1, om, p, st);
}

static void fill_seg(SegInfo& s, const wj_operand_t* op) {
  s.width = op->seg_width;
  for (int i = 0; i < 4; ++i) { s.q[i] = op->seg_q[i]; s.p[i] = op->seg_p[i]; }
}

static long long* g_gemm_dbg = nullptr;   // wj_gemm_debug(): per-CTA cycle counters of the NEXT single-CTA GEMM launches

static void fill_epilogue(GemmParams& p, const wj_epilogue_t* e) {
  p.dbg = g_gemm_dbg;
  p.out = e->out; p.ld_out = e->ld_out; p.out_f32 = e->out_f32; p.accumulate = e->accumulate;
  p.out2 = reinterpret_cast<bf16*>(e->out2); p.ld_out2 = e->ld_out2;
  p.bias = e->bias; p.resid = e->resid; p.resid_f32 = e->resid_f32; p.ld_resid = e->ld_resid;
  p.resid_mod = e->resid_mod; p.aux = reinterpret_cast<const bf16*>(e->aux); p.ld_aux = e->ld_aux;
  p.act = e->act; p.out_rows = e->out_rows; p.colsum = e->colsum;
}

// Parameters of the row-tiled modes (forward, dgrad, tf32): m-blocks of tile_rows rows (BM, or 2 * BM for CTA pairs)
// per batch entry, BN-column n-blocks.
static void row_tiled_params(GemmParams& p, const wj_operand_t* A, const wj_epilogue_t* epi, int L, int batch, int N,
                             int K, int block_n, int tile_rows) {
  memset(&p, 0, sizeof(p));
  p.L = L; p.batch = batch; p.N = N; p.K = K;
  p.mb_per_batch = (L + tile_rows - 1) / tile_rows;
  p.m_blocks = batch * p.mb_per_batch;
  p.n_blocks = (N + block_n - 1) / block_n;
  p.total_tiles = p.m_blocks * p.n_blocks;
  fill_seg(p.seg, A);
  fill_epilogue(p, epi);
}

}  // namespace wj

using namespace wj;

// Routing switches (A/B measurements and tests): WJ_GEMM_OPT_PAIR_WGRAD / WJ_GEMM_OPT_PAIR_DGRAD = 1 (default) lets the
// weight- / data-gradient GEMMs use the CTA-pair kernel where the shape allows, 0 keeps them on single CTAs.
static int g_pair_wgrad = 1, g_pair_dgrad = 1;
extern "C" int wj_gemm_option(int key, int value) {
  if (key == 1) g_pair_wgrad = value;
  else if (key == 2) g_pair_dgrad = value;
  else { set_error("wj_gemm_option: unknown key %d", key); return WJ_ERR_ARG; }
  return WJ_OK;
}

// Development aid: device buffer of 8 int64 per CTA (>= 8 * #SMs) that the single-CTA GEMM kernels fill with cycle
// counters (see GemmParams::dbg); NULL switches the counters off (the default).
extern "C" int wj_gemm_debug(void* counters) {
  g_gemm_dbg = reinterpret_cast<long long*>(counters);
  return WJ_OK;
}

// out[b*L + t, n] = epilogue( sum_vc A(vc; t, b) * W[n, vc] )        W is [N, K] row-major (K contiguous), bf16.
extern "C" int wj_gemm_bf16(const wj_operand_t* A, const void* W, int64_t ldw, int L, int batch, int N, int K,
                            const wj_epilogue_t* epi, int block_n, void* stream) {
  if (L <= 0 || batch <= 0) return WJ_OK;
  if (epi != nullptr && epi->colsum != nullptr && det_on()) {
    // deterministic mode: the fused column sums end in atomics; sum the stored output in a fixed order instead
    if (epi->out_rows != nullptr || epi->accumulate) { set_error("wj_gemm_bf16: deterministic column sums need a plain output"); return WJ_ERR_ARG; }
    wj_epilogue_t e2 = *epi;
    e2.colsum = nullptr;
    const int rc0 = wj_gemm_bf16(A, W, ldw, L, batch, N, K, &e2, block_n, stream);
    if (rc0) return rc0;
    return wj_colsum(epi->out, epi->out_f32 ? 0 : 1, static_cast<int64_t>(L) * batch, N, epi->ld_out, epi->colsum, stream);
  }
  if (K % BK != 0 || N % 8 != 0) { set_error("wj_gemm_bf16: K must be a multiple of 64 and N of 8 (K=%d N=%d)", K, N); return WJ_ERR_ARG; }
  if (A->seg_width > 0 && (A->seg_width % BK != 0 || K > 4 * A->seg_width)) { set_error("wj_gemm_bf16: bad segment width"); return WJ_ERR_ARG; }
  bool pair = block_n < 0;   // -128 / -256: CTA-pair kernel (256-row tiles, tcgen05 cta_group::2)
  if (pair) block_n = -block_n;
  // automatic choice: CTA pairs (each SM stages its own 128 rows of A and HALF of the 256 B columns) for bf16 outputs
  // on the TMA-store epilogue with K >= 768 -- measured +5..11 % on the teacher / student / conv forward shapes
  // (1257 vs 1170, 1275 vs 1190, 1360 vs 1271, 1377 vs 1235 TFLOP/s); the K = 384 shapes and the generic fp32 epilogue
  // are faster on single CTAs (607 vs 696 TFLOP/s on the predictor's fc1)
  if (block_n == 0 && K >= 768 && N % 256 == 0 && static_cast<long long>(L) * batch >= 4096 && tma_store_ok(epi, N, false)) {
    pair = true;
    block_n = 256;
  }
  // N = 384-like fp32-output GEMMs: 192-column tiles (a 128-column B tile leaves the main loop smem-bandwidth bound)
  const bool ok192 = !pair && tile192_ok(epi, N);
  if (block_n == 0) block_n = (ok192 && N % 256 != 0 && N <= 768) ? 192 : ((N % 256 == 0 || N > 1024) ? 256 : 128);
  if (block_n != 128 && block_n != 256 && !(block_n == 192 && ok192)) { set_error("wj_gemm_bf16: block_n must be 128 or 256 (192: N %% 192 == 0 with an fp32 or plain bf16 output)"); return WJ_ERR_ARG; }
  CUtensorMap tmA, tmB;
  const uint32_t boxA[4] = {BK, 1, BM, 1};
  int rc = encode_map(&tmA, A, boxA);
  if (rc) return rc;
  rc = encode_map_2d(&tmB, W, (uint64_t)K, (uint64_t)N, (uint64_t)ldw * 2, BK, (uint32_t)(pair ? block_n / 2 : block_n));
  if (rc) return rc;
  GemmParams p;
  row_tiled_params(p, A, epi, L, batch, N, K, block_n, pair ? 2 * BM : BM);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  OutMaps om;
  rc = setup_out_maps(p, om, epi, N, L, batch, /*dgrad=*/false);
  if (rc) return rc;
  if (pair) return block_n == 256 ? launch<256, 0, 2>(tmA, tmB, tmB, om, p, st) : launch<128, 0, 2>(tmA, tmB, tmB, om, p, st);
  if (block_n == 256) return launch<256, 0, 1>(tmA, tmB, tmB, om, p, st);
  if (block_n == 192) return launch<192, 0, 1>(tmA, tmB, tmB, om, p, st);
  return launch<128, 0, 1>(tmA, tmB, tmB, om, p, st);
}

// dW[m, vc] (+)= sum_{b, t} dY(b, t; m) * X(vc; t, b)      fp32 output, reduce-add when splits > 1 or accumulate.
extern "C" int wj_gemm_wgrad_bf16(const wj_operand_t* dY, const wj_operand_t* X, int L, int batch, int M, int N,
                                  float* out, int64_t ld_out, int accumulate, int splits, void* stream) {
  if (L <= 0 || batch <= 0) return WJ_OK;
  if (M % BM != 0 || N % 64 != 0) { set_error("wj_gemm_wgrad_bf16: M must be a multiple of 128 and N of 64 (M=%d N=%d)", M, N); return WJ_ERR_ARG; }
  bool transposed = false;
  const bool det = det_on();   // deterministic mode: no operand swap (its epilogue scatters with atomics), split slabs below
  // A 128-column B tile makes the main loop shared-memory-bandwidth bound (two 16 KB operand tiles per 128x128x64
  // block of MMAs); when the OTHER dimension allows 256-wide tiles, compute out^T = X^T dY instead and let the
  // (once-per-CTA) epilogue scatter the transposed tile.
  // (A partial last 256-column tile is fine: TMA zero-fills the missing column atoms, the epilogue masks them.)
  if (!det && N % 256 != 0 && N % 128 == 0 && M > N && dY->seg_width == 0 && X->seg_width == 0) {
    const wj_operand_t* t = dY; dY = X; X = t;
    const int tm = M; M = N; N = tm;
    transposed = true;
  }
  const int block_n = (N % 256 == 0 || (transposed && N > 512)) ? 256 : ((N % 128 == 0) ? 128 : 0);
  if (block_n == 0) { set_error("wj_gemm_wgrad_bf16: N must be a multiple of 128"); return WJ_ERR_ARG; }
  if (X->seg_width > 0 && X->seg_width % 64 != 0) { set_error("wj_gemm_wgrad_bf16: bad segment width"); return WJ_ERR_ARG; }
  // CTA pairs (256 x 256 tiles, each SM stages 128 dY columns and 128 X columns per k-block = 32 KB instead of 48 KB):
  // whole 256-row / 256-column tiles only, and a CTA's half of the B tile inside one segment
  const bool pair = g_pair_wgrad && !transposed && M % 256 == 0 && N % 256 == 0 &&
                    (X->seg_width == 0 || X->seg_width % 128 == 0);
  CUtensorMap tmA, tmB, tmB1;
  int rc = encode_map_mn5(&tmA, dY, BM / 64);
  if (rc) return rc;
  rc = encode_map_mn5(&tmB, X, (uint32_t)((pair ? block_n / 2 : block_n) / 64));
  if (rc) return rc;
  rc = encode_map_mn5(&tmB1, X, 1);
  if (rc) return rc;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.L = L; p.batch = batch; p.N = N; p.M = M;
  p.m_blocks = pair ? M / (2 * BM) : M / BM;
  p.n_blocks = (N + block_n - 1) / block_n;
  p.kb_per_batch = (L + BK - 1) / BK;
  const int kb_total = batch * p.kb_per_batch;
  if (splits <= 0) {
    // (m, n) tiles x splits should fill whole rounds of the persistent grid: pick the split count with the best
    // occupancy over 1..4 rounds (ties: fewer rounds = fewer fp32 reduce-adds)
    const int mn = p.m_blocks * p.n_blocks;
    const int sms = pair ? num_sms() / 2 : num_sms();
    double best = -1.0;
    splits = 1;
    for (int r = 1; r <= 4; ++r) {
      int sp = (r * sms) / mn;
      if (sp < 1) sp = 1;
      if (sp > kb_total) sp = kb_total;
      const int tiles = sp * mn;
      const double eff = static_cast<double>(tiles) / (static_cast<double>((tiles + sms - 1) / sms) * sms);
      if (eff > best + 0.02) { best = eff; splits = sp; }
    }
  }
  // make every split non-empty
  const int per = (kb_total + splits - 1) / splits;
  splits = (kb_total + per - 1) / per;
  p.splits = splits;
  p.total_tiles = p.m_blocks * p.n_blocks * splits;
  fill_seg(p.seg, X);
  p.b_single = (X->seg_width == 0 || X->seg_width % block_n == 0) ? 1 : 0;
  p.out = out; p.ld_out = ld_out; p.out_f32 = 1;
  p.dbg = g_gemm_dbg;
  p.accumulate = (accumulate || splits > 1 || transposed) ? 1 : 0;
  p.transpose_out = transposed ? 1 : 0;
  float* det_slabs = nullptr;
  if (det && p.accumulate) {
    // every token split stores its own [M, N] tile set (plain stores); det_reduce_f32 then adds the slabs in split order
    int rc2 = WJ_OK;
    det_slabs = reinterpret_cast<float*>(det_ws(static_cast<size_t>(splits) * M * N * sizeof(float), &rc2));
    if (rc2) return rc2;
    p.out = det_slabs; p.ld_out = N; p.accumulate = 0;
    p.split_stride = static_cast<long long>(M) * N;
    if (!accumulate) {
      cudaError_t e = cudaMemset2DAsync(out, ld_out * sizeof(float), 0, (size_t)N * sizeof(float), (size_t)M,
                                        reinterpret_cast<cudaStream_t>(stream));
      if (e != cudaSuccess) { set_error("memset2d: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
    }
  } else if ((splits > 1 || transposed) && !accumulate) {
    // caller asked for overwrite semantics but we reduce with atomics: clear the destination first
    // (rows x columns of the caller's matrix: M x N, or N x M when the operands were swapped)
    cudaError_t e = cudaMemset2DAsync(out, ld_out * sizeof(float), 0, (size_t)(transposed ? M : N) * sizeof(float),
                                      (size_t)(transposed ? N : M), reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) { set_error("memset2d: %s", cudaGetErrorString(e)); return WJ_ERR_RUNTIME; }
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  OutMaps om;
  memset(&om, 0, sizeof(om));
  if (pair) rc = launch<256, 1, 2>(tmA, tmB, tmB, om, p, st);
  else if (block_n == 256) rc = launch<256, 1, 1>(tmA, tmB, tmB1, om, p, st);
  else rc = launch<128, 1, 1>(tmA, tmB, tmB1, om, p, st);
  if (rc == WJ_OK && det_slabs != nullptr) rc = det_reduce_f32(det_slabs, splits, M, N, out, ld_out, st);
  return rc;
}

// out[b*L + t, n] = epilogue( sum_{s, r} A(s*width + r; t, b) * W[r, col_off[s] + n] ),  W bf16 row-major [R, ldw]:
// the reduction runs over ROWS of W (B operand read MN-major), i.e. dX = dY * W for y = x W^T without a transposed copy.
extern "C" int wj_gemm_dgrad_bf16(const wj_operand_t* A, const void* W, int64_t ldw, int w_rows, int w_cols,
                                  const int32_t* seg_col_off, int L, int batch, int N, int K, const wj_epilogue_t* epi,
                                  int block_n, void* stream) {
  if (L <= 0 || batch <= 0) return WJ_OK;
  if (epi != nullptr && epi->colsum != nullptr && det_on()) {   // (see wj_gemm_bf16)
    if (epi->out_rows != nullptr || epi->accumulate) { set_error("wj_gemm_dgrad_bf16: deterministic column sums need a plain output"); return WJ_ERR_ARG; }
    wj_epilogue_t e2 = *epi;
    e2.colsum = nullptr;
    const int rc0 = wj_gemm_dgrad_bf16(A, W, ldw, w_rows, w_cols, seg_col_off, L, batch, N, K, &e2, block_n, stream);
    if (rc0) return rc0;
    return wj_colsum(epi->out, epi->out_f32 ? 0 : 1, static_cast<int64_t>(L) * batch, N, epi->ld_out, epi->colsum, stream);
  }
  if (K % BK != 0 || N % 64 != 0) { set_error("wj_gemm_dgrad_bf16: K must be a multiple of 64 and N of 64 (K=%d N=%d)", K, N); return WJ_ERR_ARG; }
  if (A->seg_width > 0 && (A->seg_width % BK != 0 || K > 4 * A->seg_width)) { set_error("wj_gemm_dgrad_bf16: bad segment width"); return WJ_ERR_ARG; }
  const bool auto_bn = block_n == 0;
  bool pair = block_n < 0;   // -256: CTA-pair kernel requested explicitly (tests)
  if (pair) block_n = -block_n;
  const bool ok192 = !pair && tile192_ok(epi, N) && (epi->out_f32 || epi->act == 0);
  if (block_n == 0) block_n = (ok192 && N % 256 != 0 && N <= 768) ? 192 : ((N % 256 == 0 || N > 1024) ? 256 : 128);
  if (block_n != 128 && block_n != 256 && !(block_n == 192 && ok192)) { set_error("wj_gemm_dgrad_bf16: block_n must be 128 or 256 (192: N %% 192 == 0 with an fp32 or plain bf16 output)"); return WJ_ERR_ARG; }
  // CTA pairs for the plain bf16-output data gradients (TMA-store epilogue) with K >= 768 and whole 256-column tiles: the
  // same rule as the forward GEMMs (wj_gemm_bf16)
  // (plain bf16 outputs, or the GELU-backward form out = acc * saved factor with optional fused column sums)
  const bool pair_ok = tma_store_ok(epi, N, /*dgrad=*/true) && epi->out2 == nullptr && epi->act != 1 && N % 256 == 0;
  if (pair && !(pair_ok && block_n == 256)) { set_error("wj_gemm_dgrad_bf16: the CTA-pair kernel takes plain bf16 outputs with N %% 256 == 0"); return WJ_ERR_ARG; }
  // (K >= 512 for plain outputs: +4 % on the K = 512 conv data gradient; the GELU-backward form loses there, 645 vs 738)
  if (auto_bn && g_pair_dgrad && pair_ok && K >= (epi->act == 2 ? 768 : 512) && static_cast<long long>(L) * batch >= 4096) {
    pair = true;
    block_n = 256;
  }
  CUtensorMap tmA, tmB;
  const uint32_t boxA[4] = {BK, 1, BM, 1};
  int rc = encode_map(&tmA, A, boxA);
  if (rc) return rc;
  rc = encode_map_mn3(&tmB, W, (uint64_t)w_rows, (uint64_t)w_cols, (uint64_t)ldw * 2, (uint32_t)((pair ? block_n / 2 : block_n) / 64));
  if (rc) return rc;
  GemmParams p;
  row_tiled_params(p, A, epi, L, batch, N, K, block_n, pair ? 2 * BM : BM);
  for (int i = 0; i < 4; ++i) p.segB_col[i] = seg_col_off ? seg_col_off[i] : 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  OutMaps om;
  rc = setup_out_maps(p, om, epi, N, L, batch, /*dgrad=*/true);
  if (rc) return rc;
  if (pair) {
    if (!p.tma_store) { set_error("wj_gemm_dgrad_bf16: pair kernel without a TMA-store epilogue"); return WJ_ERR_ARG; }
    return launch<256, 2, 2>(tmA, tmB, tmB, om, p, st);
  }
  if (block_n == 192) return launch<192, 2, 1>(tmA, tmB, tmB, om, p, st);
  if (block_n == 256) return launch<256, 2, 1>(tmA, tmB, tmB, om, p, st);
  return launch<128, 2, 1>(tmA, tmB, tmB, om, p, st);
}

// Reference-precision (TF32) inference GEMM: out[b*L + t, n] = epilogue( sum_vc A(vc; t, b) * W[n, vc] ) with A and W fp32
// (the caller rounds them to nearest tf32: the tensor core would truncate), K-major, tcgen05.mma.kind::tf32, fp32
// accumulation.  Epilogue: v = acc + bias; act 4: v = exact erf GELU(v); v += resid; out = v as bf16, or fp32 rounded
// to nearest tf32 when round_out (an output that is the next GEMM's operand).
extern "C" int wj_gemm_tf32(const wj_operand_t* A, const float* W, int64_t ldw, int L, int batch, int N, int K,
                            const wj_epilogue_t* epi, int round_out, void* stream) {
  if (L <= 0 || batch <= 0) return WJ_OK;
  constexpr int KB = BK / 2;
  if (epi == nullptr) { set_error("wj_gemm_tf32: no epilogue"); return WJ_ERR_ARG; }
  if (K % KB != 0 || N % 128 != 0) { set_error("wj_gemm_tf32: K must be a multiple of 32 and N of 128 (K=%d N=%d)", K, N); return WJ_ERR_ARG; }
  if (A->seg_width > 0 && (A->seg_width % KB != 0 || K > 4 * A->seg_width)) { set_error("wj_gemm_tf32: bad segment width"); return WJ_ERR_ARG; }
  if (epi->accumulate || epi->out2 != nullptr || epi->aux != nullptr || epi->out_rows != nullptr || epi->colsum != nullptr ||
      (epi->act != 0 && epi->act != 4)) {
    set_error("wj_gemm_tf32: the epilogue takes bias, act 0 / 4 (exact GELU), a residual and a plain output");
    return WJ_ERR_ARG;
  }
  if (round_out && !epi->out_f32) { set_error("wj_gemm_tf32: tf32 rounding needs an fp32 output"); return WJ_ERR_ARG; }
  if (epi->ld_out % 8 != 0 || reinterpret_cast<uintptr_t>(epi->out) % 16 != 0 ||
      (epi->resid != nullptr && (epi->ld_resid % 8 != 0 || reinterpret_cast<uintptr_t>(epi->resid) % 16 != 0))) {
    set_error("wj_gemm_tf32: outputs / residual need 16-byte aligned rows");
    return WJ_ERR_ARG;
  }
  const int block_n = N % 256 == 0 ? 256 : 128;
  CUtensorMap tmA, tmB;
  const uint32_t boxA[4] = {KB, 1, BM, 1};
  int rc = encode_map(&tmA, A, boxA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
  if (rc) return rc;
  rc = encode_map_2d(&tmB, W, (uint64_t)K, (uint64_t)N, (uint64_t)ldw * 4, KB, (uint32_t)block_n, CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
  if (rc) return rc;
  GemmParams p;
  row_tiled_params(p, A, epi, L, batch, N, K, block_n, BM);
  p.round_tf32 = round_out ? 1 : 0;
  OutMaps om;
  memset(&om, 0, sizeof(om));   // (generic epilogue: no TMA stores)
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (block_n == 256) return launch_variant<256, 0, false, true, 1>(tmA, tmB, tmB, om, p, st);
  return launch_variant<128, 0, false, true, 1>(tmA, tmB, tmB, om, p, st);
}
