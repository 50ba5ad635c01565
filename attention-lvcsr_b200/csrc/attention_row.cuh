// take_glimpses for ONE decoder row, executed by a thread-block cluster of `cs` CTAs that
// split the attention window along time.  Shared by the stand-alone attention step kernel
// (attention.cu: beam-search state functions) and the persistent teacher-forced decoder
// (dec_scan.cu).  Math follows lvsr/bricks/attention.py:98-114,120-183,191-213 and
// libs/blocks/blocks/bricks/attention.py:235-256.
//
// r1d -> r1e (profiles/): the first version spent 8.7 us in the conv, 13 us in the energies
// (issue/latency bound: ~17 instructions per (t,m) element) and 4.5 us in the context pass.
// Now:
//   * conv: each thread owns one position and a quarter of the taps for ALL filters
//     (2.5 FMA per shared-memory load instead of 1.4), quarters meet by two shuffles;
//   * energies: match = P + q + F.Wh runs on the tensor cores -- mma.sync m16n8k16 bf16 with
//     fp32 accumulate, P (+q) is the accumulator init (so P and q stay exact fp32), and the
//     K<=16 handler product uses a 3-term hi/lo bf16 split of both operands (error ~2^-17 of
//     the location term only).  tcgen05 does not apply: K = 10, the accumulator is consumed
//     immediately by tanh in registers, and each warp owns a private 16x32 strip;
//   * tanh = 1 - 2/(1+2^(2x log2e)): 2 MUFU + 3 FP32 instructions, |err| ~ 2e-7;
//   * context: 8 independent 16-byte loads in flight per thread, 512 threads.
#pragma once
#include <cuda_bf16.h>

#include "kernels.h"
#include "lvsr_b200.h"

namespace lvsr {

constexpr int ATT_NT = 512;          // threads per CTA in every kernel that runs attention_row
constexpr int ATT_NW = ATT_NT / 32;

__host__ __device__ inline int att_filter_row(int K) { return K <= 12 ? 12 : 16; }

// sred holds the 8 column groups of the partial context and, earlier in the step, the 16 warps'
// partial energies.  No shared-memory float atomics: they compile to contended CAS loops AND make
// the summation order (hence the last bits of every output) vary from run to run.
__host__ __device__ inline size_t att_red_floats(int E, int tc_cap) {
  const size_t a = (size_t)8 * E, b = (size_t)ATT_NW * (tc_cap + 16);
  return a > b ? a : b;
}

// Shared-memory footprint (floats) of attention_row for a chunk capacity of tc_cap positions.
// wh_rows: rows of the handler copy in shared memory: 16 (zero-padded to the MMA depth, unpredicated fragment loads: the
// fast default) or K (compact; the planner falls back to it when the padded copy does not fit, e.g. 16 rows x T' = 2000)
__host__ __device__ inline size_t att_smem_floats(int M, int E, int K, int n, int tc_cap, int cs, int wh_rows = 16) {
  size_t f = 0;
  f += M;                                         // sq
  f += M;                                         // sv
  f += (size_t)wh_rows * M;                       // sWh (rows >= K are zero, or supplied by predicates in the compact layout)
  f += (size_t)(2 * n + 1) * att_filter_row(K);   // sfiltT [tap][filter]
  f += tc_cap + 2 * n + 8;                        // salpha
  f += (size_t)(tc_cap + 16) * 16;                // sF: packed bf16 pairs, 8 hi + 8 lo words per position
  f += tc_cap + 16;                               // se
  f += tc_cap + 16;                               // su
  f += 96;                                        // block reduction scratch
  f += att_red_floats(E, tc_cap);                 // sred: partial context / per-warp partial energies
  f += (size_t)cs * 4;                            // xs: per-rank scalars (lmax, lsum, anyone, lpos)
  f += (size_t)cs * E;                            // xctx: per-rank partial context (meaningful on rank 0)
  return f + 32;
}

struct AttRowIO {
  const float* P;        // [Tp, U, M]
  const float* H;        // [Tp, U, E]
  const float* maskH;    // [Tp, U]
  const float* q_row;    // [M]   states . W_state for this row
  const float* w_prev;   // [Tp]  previous alignment of this row
  const float* filt;     // [K, 2n+1]
  const float* Wh;       // [K, M]
  const float* v;        // [M]
  float v_bias;
  float* w_out;          // [Tp]
  float* e_out;          // [Tp]
  float* ctx_out;        // [E]
  int u;                 // utterance column of this row in P/H/maskH
  int U, Tp, M, E, K, n, normalizer;
  int wh_rows = 16;      // handler rows held in shared memory (att_smem_floats)
  int b0, b1;            // global window cut
  float lo, hi;          // strict per-row bounds (additional mask)
  // optional: position statistic of the NEW alignment for the next step's window prior
  // (LVSR_PRIOR_WINDOW_MEAN / _MEDIAN, lvsr/bricks/attention.py:134-144); nullptr to skip
  float* rowpos_out = nullptr;
  int rowpos_mode = 0;
  unsigned long long* trace = nullptr;   // optional [8] globaltimer stamps (debug)
  // P of this CTA's positions is resident in tensor memory (att_stage_p_tmem): the energies read it from
  // there instead of L2.  p_taddr = this thread's TMEM address of tile 0 (att_p_taddr).
  int p_tmem = 0;
  uint32_t p_taddr = 0;
};

__device__ __forceinline__ unsigned long long att_global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
  return t;
}
#define ATT_STAMP(j) do { if (a.trace && threadIdx.x == 0) a.trace[j] = att_global_ns(); } while (0)

// -DLVSR_DEC_DEBUG: record the first NaN sightings (stage, step, CTA, thread, index) of a launch.
#ifdef LVSR_DEC_DEBUG
__device__ unsigned long long g_dbg_events[64];
__device__ unsigned int g_dbg_count = 0;
__device__ int g_dbg_step = 0;
__device__ __forceinline__ void dbg_nan(int stage, float v, int idx) {
  if (v != v) {
    const unsigned k = atomicAdd(&g_dbg_count, 1u);
    if (k < 64)
      g_dbg_events[k] = ((unsigned long long)stage << 56) | ((unsigned long long)(g_dbg_step & 0xff) << 48) |
                        ((unsigned long long)(blockIdx.x & 0xffff) << 32) | ((unsigned long long)(threadIdx.x & 0xffff) << 16) |
                        (unsigned long long)(idx & 0xffff);
  }
}
#define DBG_NAN(stage, v, idx) dbg_nan(stage, v, idx)
#else
#define DBG_NAN(stage, v, idx) do { } while (0)
#endif

struct AttSmem {
  float *sq, *sv, *sWh, *sfiltT, *salpha, *se, *su, *sblk, *sred, *xs, *xctx;
  uint32_t* sF;          // [(tc_cap+16)][16]: words 0..7 = hi pairs, 8..15 = lo pairs
};

__device__ __forceinline__ AttSmem att_carve(float* smem, int M, int E, int K, int n, int tc_cap, int cs, int wh_rows = 16) {
  AttSmem s;
  float* p = smem;
  s.sq = p; p += M;
  s.sv = p; p += M;
  s.sWh = p; p += (size_t)wh_rows * M;
  s.sfiltT = p; p += (size_t)(2 * n + 1) * att_filter_row(K);
  p += (4 - ((p - smem) & 3)) & 3;
  s.salpha = p; p += tc_cap + 2 * n + 8;
  p += (4 - ((p - smem) & 3)) & 3;
  s.sF = reinterpret_cast<uint32_t*>(p); p += (size_t)(tc_cap + 16) * 16;
  s.se = p; p += tc_cap + 16;
  s.su = p; p += tc_cap + 16;
  s.sblk = p; p += 96;
  p += (4 - ((p - smem) & 3)) & 3;
  s.sred = p; p += att_red_floats(E, tc_cap);
  s.xs = p; p += (size_t)cs * 4;
  s.xctx = p; p += (size_t)cs * E;
  return s;
}

// Constants that never change during a sequence: energy vector, handler (zero-padded to 16
// rows), transposed + zero-padded filter bank.  Persistent callers stage them once.
__device__ __forceinline__ void att_stage_constants(const AttSmem& s, const float* v, const float* Wh,
                                                    const float* filt, int M, int K, int n, int wh_rows = 16) {
  const int tid = threadIdx.x, w = 2 * n + 1, fw = att_filter_row(K);
  for (int i = tid; i < M; i += ATT_NT) s.sv[i] = v[i];
  for (int i = tid; i < wh_rows * M; i += ATT_NT) s.sWh[i] = (i / M < K) ? Wh[i] : 0.f;
  for (int i = tid; i < w * fw; i += ATT_NT) {
    const int j = i / fw, k = i % fw;
    s.sfiltT[i] = (k < K) ? filt[(size_t)k * w + j] : 0.f;
  }
}

__device__ __forceinline__ uint32_t pack_bf16(float lo_col, float hi_col) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo_col, hi_col);   // .x (low half) = first argument
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// ---- P resident in tensor memory ---------------------------------------------------------
// When a persistent caller's window is the whole utterance on every step, each CTA reads the same P
// slice on every step.  It can instead keep that slice in its 512 TMEM columns: thread-private, in
// exactly the order of the mma.sync accumulator fragments the energy loop initialises from P.  Warp w
// may address TMEM lanes 32*(w%4)..+31 only, so the four warps of a lane quarter take 128 columns
// each; a thread's tile k holds its 4*NTW accumulator values at columns [k*4*NTW, +4*NTW):
//   column j*4 + {0, 1, 2, 3} = P[row g][n0 + 2tig], P[row g][n0 + 2tig + 1], P[row g+8][...], P[row g+8][... + 1]
// of the 16-position tile (n0 = first column of the warp's j-th 8-column tile).  Fits when
// ceil(tc_cap / 16) * 4 * NTW <= 128 (the planner checks it).
__host__ __device__ inline bool att_p_fits_tmem(int M, int tc_cap) { return ((tc_cap + 15) / 16) * (M / 128) <= 32; }

__device__ __forceinline__ uint32_t att_p_taddr(uint32_t tmem_base) {
  const int warp = threadIdx.x >> 5;
  return tmem_base + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)((warp >> 2) * 128);
}

template <int N>
__device__ __forceinline__ void tmem_st_32x32b(uint32_t taddr, const uint32_t (&v)[N]) {
  static_assert(N == 4 || N == 8 || N == 16, "4, 8 or 16 columns");
  if constexpr (N == 4) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};\n"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
  } else if constexpr (N == 8) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
  } else {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
                 "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
                 : "memory");
  }
}

// load + wait: the destination registers are complete when this returns
template <int N>
__device__ __forceinline__ void tmem_ld_32x32b(uint32_t taddr, uint32_t (&v)[N]) {
  static_assert(N == 4 || N == 8 || N == 16, "4, 8 or 16 columns");
  if constexpr (N == 4) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr));
  } else if constexpr (N == 8) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
  } else {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
  }
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

// One-time copy of P rows [t0, t0 + nt) of utterance column u into this thread's TMEM columns (layout above).
// Tail rows >= nt are clamped to nt - 1 exactly as the L2 path of att_energies does.  All ATT_NT threads.
template <int NTW>
__device__ __forceinline__ void att_stage_p_tmem_t(const float* P, int U, int M, int u, int t0, int nt, uint32_t taddr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, tig = lane & 3;
  const float* pbase = P + ((long long)t0 * U + u) * M + warp * NTW * 8 + 2 * tig;
  const long long prow = (long long)U * M;
  const int ntile = (nt + 15) / 16;
  for (int tile = 0; tile < ntile; ++tile) {
    const int r0 = min(tile * 16 + g, nt - 1), r1 = min(tile * 16 + g + 8, nt - 1);
    uint32_t v[4 * NTW];
#pragma unroll
    for (int j = 0; j < NTW; ++j) {
      const float2 x0 = __ldg(reinterpret_cast<const float2*>(pbase + r0 * prow + j * 8));
      const float2 x1 = __ldg(reinterpret_cast<const float2*>(pbase + r1 * prow + j * 8));
      v[j * 4 + 0] = __float_as_uint(x0.x); v[j * 4 + 1] = __float_as_uint(x0.y);
      v[j * 4 + 2] = __float_as_uint(x1.x); v[j * 4 + 3] = __float_as_uint(x1.y);
    }
    tmem_st_32x32b<4 * NTW>(taddr + (uint32_t)(tile * 4 * NTW), v);
  }
  asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
}

__device__ __forceinline__ void att_stage_p_tmem(const float* P, int U, int M, int u, int t0, int nt, uint32_t taddr) {
  if (M == 512) att_stage_p_tmem_t<4>(P, U, M, u, t0, nt, taddr);
  else if (M == 256) att_stage_p_tmem_t<2>(P, U, M, u, t0, nt, taddr);
  else att_stage_p_tmem_t<1>(P, U, M, u, t0, nt, taddr);
}

// NTW: 8-column tiles of the matcher dimension per warp (M = 128 * NTW).
// P_TMEM: P comes from tensor memory (a.p_taddr, staged once by att_stage_p_tmem) instead of L2.
template <int NTW, bool COMPACT, bool P_TMEM = false>
__device__ __forceinline__ void att_energies(const AttRowIO& a, const AttSmem& s, int nt, int t0, int tc_cap) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, tig = lane & 3;
  const int M = a.M;
  // B fragments (handler, hi/lo split), energy vector and query for this warp's columns
  uint32_t bh[NTW][2], bl[NTW][2];
  float vv[NTW][2], qq[NTW][2];
#pragma unroll
  for (int j = 0; j < NTW; ++j) {
    const int n0 = (warp * NTW + j) * 8;
    const int colb = n0 + g;                       // B fragment column
    // B fragment rows 2tig, 2tig+1, 2tig+8, 2tig+9 of the 16-deep product; only K rows exist (K <= 16)
    auto wh = [&](int row) -> float { return (!COMPACT || row < a.K) ? s.sWh[(size_t)row * M + colb] : 0.f; };
    const float w00 = wh(2 * tig), w01 = wh(2 * tig + 1), w10 = wh(2 * tig + 8), w11 = wh(2 * tig + 9);
    const float h00 = bf16_round(w00), h01 = bf16_round(w01), h10 = bf16_round(w10), h11 = bf16_round(w11);
    bh[j][0] = pack_bf16(h00, h01);
    bh[j][1] = pack_bf16(h10, h11);
    bl[j][0] = pack_bf16(w00 - h00, w01 - h01);
    bl[j][1] = pack_bf16(w10 - h10, w11 - h11);
    const int colc = n0 + 2 * tig;                 // accumulator columns
    vv[j][0] = s.sv[colc]; vv[j][1] = s.sv[colc + 1];
    qq[j][0] = s.sq[colc]; qq[j][1] = s.sq[colc + 1];
  }
  float* part = s.sred + (size_t)warp * (tc_cap + 16);
  const int ntile = (nt + 15) / 16;
  const float* pbase = a.P + ((long long)(a.b0 + t0) * a.U + a.u) * M + warp * NTW * 8 + 2 * tig;
  const long long prow = (long long)a.U * M;
  float2 pc[NTW][2], pn[NTW][2];
  auto load_p = [&](float2 (&dst)[NTW][2], int tile) {
    const int r0 = min(tile * 16 + g, nt - 1), r1 = min(tile * 16 + g + 8, nt - 1);   // clamp: tail rows are discarded
#pragma unroll
    for (int j = 0; j < NTW; ++j) {
      dst[j][0] = __ldg(reinterpret_cast<const float2*>(pbase + r0 * prow + j * 8));
      dst[j][1] = __ldg(reinterpret_cast<const float2*>(pbase + r1 * prow + j * 8));
    }
  };
  if (!P_TMEM && ntile > 0) load_p(pc, 0);
  for (int tile = 0; tile < ntile; ++tile) {
    if constexpr (P_TMEM) {
      uint32_t r[4 * NTW];
      tmem_ld_32x32b<4 * NTW>(a.p_taddr + (uint32_t)(tile * 4 * NTW), r);
#pragma unroll
      for (int j = 0; j < NTW; ++j) {
        pc[j][0] = make_float2(__uint_as_float(r[j * 4 + 0]), __uint_as_float(r[j * 4 + 1]));
        pc[j][1] = make_float2(__uint_as_float(r[j * 4 + 2]), __uint_as_float(r[j * 4 + 3]));
      }
    } else if (tile + 1 < ntile) {
      load_p(pn, tile + 1);
    }
    const int ta = tile * 16 + g, tb = ta + 8;
    uint32_t ah[4], al[4];
    ah[0] = s.sF[(size_t)ta * 16 + tig];     ah[1] = s.sF[(size_t)tb * 16 + tig];
    ah[2] = s.sF[(size_t)ta * 16 + tig + 4]; ah[3] = s.sF[(size_t)tb * 16 + tig + 4];
    al[0] = s.sF[(size_t)ta * 16 + 8 + tig];     al[1] = s.sF[(size_t)tb * 16 + 8 + tig];
    al[2] = s.sF[(size_t)ta * 16 + 8 + tig + 4]; al[3] = s.sF[(size_t)tb * 16 + 8 + tig + 4];
    float ea = 0.f, eb = 0.f;
#pragma unroll
    for (int j = 0; j < NTW; ++j) {
      float d[4];
      d[0] = pc[j][0].x + qq[j][0]; d[1] = pc[j][0].y + qq[j][1];
      d[2] = pc[j][1].x + qq[j][0]; d[3] = pc[j][1].y + qq[j][1];
      DBG_NAN(4, pc[j][0].x + pc[j][0].y + pc[j][1].x + pc[j][1].y, tile * 16 + g);
      DBG_NAN(5, qq[j][0] + qq[j][1], j);
      mma_bf16_16816(d, al, bh[j][0], bh[j][1]);     // small terms first
      mma_bf16_16816(d, ah, bl[j][0], bl[j][1]);
      mma_bf16_16816(d, ah, bh[j][0], bh[j][1]);
      DBG_NAN(6, d[0] + d[1] + d[2] + d[3], tile * 16 + g);
      ea = fmaf(vv[j][0], fast_tanh(d[0]), ea);
      ea = fmaf(vv[j][1], fast_tanh(d[1]), ea);
      eb = fmaf(vv[j][0], fast_tanh(d[2]), eb);
      eb = fmaf(vv[j][1], fast_tanh(d[3]), eb);
    }
    ea += __shfl_xor_sync(0xffffffffu, ea, 1); ea += __shfl_xor_sync(0xffffffffu, ea, 2);
    eb += __shfl_xor_sync(0xffffffffu, eb, 1); eb += __shfl_xor_sync(0xffffffffu, eb, 2);
    DBG_NAN(7, ea + eb, tile * 16 + g);
    if (tig == 0) {
      part[ta] = ea;       // this warp's private partial sums; rows >= nt land in the 16-row padding
      part[tb] = eb;
    }
    if constexpr (!P_TMEM) {
#pragma unroll
      for (int j = 0; j < NTW; ++j) { pc[j][0] = pn[j][0]; pc[j][1] = pn[j][1]; }
    }
  }
}

__device__ __forceinline__ float gmax_of(const float* xs, int cs) {
  float g = -INFINITY;
  for (int r = 0; r < cs; ++r) g = fmaxf(g, xs[r * 4 + 0]);
  return g;
}

// ATT_NT threads.  `constants_staged`: a persistent caller already ran att_stage_constants.
// `flow`: q and the previous alignment are produced by other CTAs of the same launch into
// sentinel-initialised buffers (common.cuh, "the data is the flag"): they are read with polling
// loads and the outputs other CTAs consume are written with gpu-scope stores.
// `entry_wait_pending`: the caller issued barrier.cluster.arrive at kernel entry.
// P_TMEM_OK: compile the energy loop that reads P from tensor memory (taken when a.p_tmem is set).
template <bool COMPACT = false, bool P_TMEM_OK = false>
__device__ __forceinline__ void attention_row(const AttRowIO& a, float* smem, int tc_cap, int rank, int cs,
                                              bool constants_staged, bool flow,
                                              bool entry_wait_pending) {
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NT = ATT_NT, NW = ATT_NW;
  const int M = a.M, E = a.E, K = a.K, n = a.n, w = 2 * n + 1, Tp = a.Tp, U = a.U, u = a.u;
  const AttSmem s = att_carve(smem, M, E, K, n, tc_cap, cs, a.wh_rows);

  const int b0 = a.b0;
  const int Tw = max(0, a.b1 - a.b0);
  const int tc = (Tw + cs - 1) / cs;
  const int t0 = min(Tw, rank * tc), t1 = min(Tw, t0 + tc);
  const int nt = t1 - t0;             // positions owned by this CTA (window-relative t0..t1)

  ATT_STAMP(0);
  // ---- stage the row's query, the slice of the previous alignment, zero the energies ----
  if (!constants_staged) att_stage_constants(s, a.v, a.Wh, a.filt, M, K, n, a.wh_rows);
  {
    const int len = nt + 2 * n + 8;
    for (int i = tid; i < len; i += NT) {
      const int prel = t0 - n + i;            // window-relative position; zero padding is
      float val = 0.f;                        // relative to the CUT (SURVEY quirk 10)
      if (prel >= 0 && prel < Tw) val = flow ? ld_flow_f32(a.w_prev + b0 + prel) : a.w_prev[b0 + prel];
      DBG_NAN(1, val, i);
      s.salpha[i] = val;
    }
  }
  // attended mask of the owned positions: requested now, consumed after the energies
  float mreg[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int t = tid + r * NT;
    mreg[r] = (t < nt) ? __ldg(a.maskH + (long long)(b0 + t0 + t) * U + u) : 0.f;
  }
  __syncthreads();
  ATT_STAMP(1);

  // ---- location features F[t][k] = sum_j alpha_cut[t + 2n - j] * filt[k][j], written as the
  //      bf16 hi/lo A-fragments of the handler product ----------------------------------
  {
    const int fw = att_filter_row(K);
    const int qtr = lane >> 3;                         // tap quarter 0..3
    const int seg = (w + 3) / 4;
    const int j0 = qtr * seg, j1 = min(w, j0 + seg);
    const int npass = (nt + 16 + 127) / 128;           // also clears the padding rows up to nt+15
    for (int pass = 0; pass < npass; ++pass) {
      const int t = pass * 128 + warp * 8 + (lane & 7);
      float acc[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) acc[k] = 0.f;
      if (t < nt) {
        if (fw == 12) {
          for (int j = j0; j < j1; ++j) {
            const float av = s.salpha[t + 2 * n - j];
            const float* fr = s.sfiltT + (size_t)j * 12;
            const float4 f0 = *reinterpret_cast<const float4*>(fr);
            const float4 f1 = *reinterpret_cast<const float4*>(fr + 4);
            const float4 f2 = *reinterpret_cast<const float4*>(fr + 8);
            acc[0] = fmaf(av, f0.x, acc[0]); acc[1] = fmaf(av, f0.y, acc[1]);
            acc[2] = fmaf(av, f0.z, acc[2]); acc[3] = fmaf(av, f0.w, acc[3]);
            acc[4] = fmaf(av, f1.x, acc[4]); acc[5] = fmaf(av, f1.y, acc[5]);
            acc[6] = fmaf(av, f1.z, acc[6]); acc[7] = fmaf(av, f1.w, acc[7]);
            acc[8] = fmaf(av, f2.x, acc[8]); acc[9] = fmaf(av, f2.y, acc[9]);
            acc[10] = fmaf(av, f2.z, acc[10]); acc[11] = fmaf(av, f2.w, acc[11]);
          }
        } else {
          for (int j = j0; j < j1; ++j) {
            const float av = s.salpha[t + 2 * n - j];
            const float* fr = s.sfiltT + (size_t)j * 16;
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const float4 f = *reinterpret_cast<const float4*>(fr + q4 * 4);
              acc[q4 * 4 + 0] = fmaf(av, f.x, acc[q4 * 4 + 0]); acc[q4 * 4 + 1] = fmaf(av, f.y, acc[q4 * 4 + 1]);
              acc[q4 * 4 + 2] = fmaf(av, f.z, acc[q4 * 4 + 2]); acc[q4 * 4 + 3] = fmaf(av, f.w, acc[q4 * 4 + 3]);
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 8);
        acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], 16);
      }
      if (qtr == 0 && t < nt + 16 && t < tc_cap + 16) {
        uint32_t* row = s.sF + (size_t)t * 16;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float x0 = (t < nt) ? acc[2 * c] : 0.f, x1 = (t < nt) ? acc[2 * c + 1] : 0.f;
          DBG_NAN(2, x0 + x1, t);
          const float h0 = bf16_round(x0), h1 = bf16_round(x1);
          row[c] = pack_bf16(h0, h1);
          row[8 + c] = pack_bf16(x0 - h0, x1 - h1);
        }
      }
    }
  }
  // the query is consumed only now: in flow mode its producers ran concurrently with the conv
  for (int i = tid; i < M; i += NT) {
    s.sq[i] = flow ? ld_flow_f32(a.q_row + i) : a.q_row[i];
    DBG_NAN(3, s.sq[i], i);
  }
  __syncthreads();
  ATT_STAMP(2);

  // ---- energies: e[t] = v . tanh(P[t] + q + F[t] . Wh) on the tensor cores -------------
  if (P_TMEM_OK && a.p_tmem) {
    if (M == 512) att_energies<4, COMPACT, P_TMEM_OK>(a, s, nt, t0, tc_cap);
    else if (M == 256) att_energies<2, COMPACT, P_TMEM_OK>(a, s, nt, t0, tc_cap);
    else att_energies<1, COMPACT, P_TMEM_OK>(a, s, nt, t0, tc_cap);
  } else {
    if (M == 512) att_energies<4, COMPACT>(a, s, nt, t0, tc_cap);
    else if (M == 256) att_energies<2, COMPACT>(a, s, nt, t0, tc_cap);
    else att_energies<1, COMPACT>(a, s, nt, t0, tc_cap);
  }
  __syncthreads();
  {
    // e[t] = the 16 warps' partial sums, added in a fixed order
    const int stride = tc_cap + 16;
    for (int t = tid; t < nt; t += NT) {
      float e = 0.f;
#pragma unroll
      for (int w = 0; w < NW; ++w) e += s.sred[(size_t)w * stride + t];
      DBG_NAN(8, e, t);
      s.se[t] = e;
    }
  }
  __syncthreads();
  ATT_STAMP(3);

  // ---- local normaliser statistics ---------------------------------------------------
  float* sblk_max = s.sblk;
  float* sblk_sum = s.sblk + 32;
  float* sblk_any = s.sblk + 64;
  float lmax = -INFINITY;
  if (a.normalizer == LVSR_NORM_SOFTMAX) {
    for (int t = tid; t < nt; t += NT) lmax = fmaxf(lmax, s.se[t]);   // max over masked positions too
    lmax = warp_max(lmax);
    if (lane == 0) sblk_max[warp] = lmax;
    __syncthreads();
    lmax = sblk_max[0];
#pragma unroll
    for (int i = 1; i < NW; ++i) lmax = fmaxf(lmax, sblk_max[i]);
  } else {
    lmax = 0.f;
  }
  float lsum = 0.f, anyone = 0.f;
  for (int t = tid, r = 0; t < nt; t += NT, ++r) {
    const int tabs = b0 + t0 + t;
    const float pos = (float)tabs;
    float mval = (r < 4) ? mreg[r < 4 ? r : 0] : __ldg(a.maskH + (long long)tabs * U + u);
    mval *= (pos > a.lo && pos < a.hi) ? 1.f : 0.f;          // strict inequalities, attention.py:156-157
    float uv;
    const float e = s.se[t] + a.v_bias;                       // v_bias is 0 for the softmax normaliser
    s.se[t] = e;
    if (a.normalizer == LVSR_NORM_SOFTMAX) uv = __expf(e - lmax);
    else if (a.normalizer == LVSR_NORM_LOGISTIC) uv = fast_sigmoid(e);
    else uv = fmaxf(e / 1000.f, 0.f);
    uv *= mval;
    s.su[t] = uv;
    lsum += uv;
    if (mval == 1.f) anyone = 1.f;
  }
  lsum = warp_sum(lsum);
  anyone = warp_max(anyone);
  if (lane == 0) { sblk_sum[warp] = lsum; sblk_any[warp] = anyone; }
  __syncthreads();
  lsum = 0.f; anyone = 0.f;
#pragma unroll
  for (int i = 0; i < NW; ++i) { lsum += sblk_sum[i]; anyone = fmaxf(anyone, sblk_any[i]); }

  ATT_STAMP(4);
  // ---- partial weighted average with the LOCAL weights ------------------------------
  const int ncol4 = E / 4;
  const int ng = max(1, min(8, NT / ncol4));
  {
    const int c4 = tid % ncol4, g = tid / ncol4;
    if (g < ng) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      const float* hbase = a.H + ((long long)(b0 + t0) * U + u) * E + c4 * 4;
      const long long hstride = (long long)U * E;
      int t = g;
      for (; t + 7 * ng < nt; t += 8 * ng) {
        float4 h[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) h[q] = __ldg(reinterpret_cast<const float4*>(hbase + (long long)(t + q * ng) * hstride));
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float wq = s.su[t + q * ng];
          acc.x = fmaf(wq, h[q].x, acc.x); acc.y = fmaf(wq, h[q].y, acc.y);
          acc.z = fmaf(wq, h[q].z, acc.z); acc.w = fmaf(wq, h[q].w, acc.w);
        }
      }
      for (; t < nt; t += ng) {
        const float4 h0 = __ldg(reinterpret_cast<const float4*>(hbase + (long long)t * hstride));
        const float w0 = s.su[t];
        acc.x = fmaf(w0, h0.x, acc.x); acc.y = fmaf(w0, h0.y, acc.y); acc.z = fmaf(w0, h0.z, acc.z); acc.w = fmaf(w0, h0.w, acc.w);
      }
      *reinterpret_cast<float4*>(s.sred + (size_t)g * E + c4 * 4) = acc;
    }
  }
  __syncthreads();
  ATT_STAMP(5);

  // ---- first moment of the local weights (only for the window_around_mean prior) -------
  float lpos = 0.f;
  if (a.rowpos_out != nullptr && a.rowpos_mode == LVSR_PRIOR_WINDOW_MEAN) {
    for (int t = tid; t < nt; t += NT) lpos += (float)(b0 + t0 + t) * s.su[t];
    lpos = warp_sum(lpos);
    if (lane == 0) sblk_max[warp] = lpos;     // sblk_max is free again
    __syncthreads();
    lpos = 0.f;
#pragma unroll
    for (int i = 0; i < NW; ++i) lpos += sblk_max[i];
  }

  // ---- exchange through distributed shared memory ------------------------------------
  if (entry_wait_pending)   // pairs with the caller's early barrier.cluster.arrive: peers are resident
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
  float* xs = s.xs;
  float* xctx = s.xctx;
  if (tid < cs) {
    float* dst = cluster.map_shared_rank(xs, tid);
    dst[rank * 4 + 0] = lmax;
    dst[rank * 4 + 1] = lsum;
    dst[rank * 4 + 2] = anyone;
    dst[rank * 4 + 3] = lpos;
  }
  {
    float* dst0 = cluster.map_shared_rank(xctx, 0);
    for (int e = tid; e < E; e += NT) {
      float acc = 0.f;
      for (int g = 0; g < ng; ++g) acc += s.sred[(size_t)g * E + e];
      dst0[(size_t)rank * E + e] = acc;
    }
  }
  cluster.sync();
  ATT_STAMP(6);

  // ---- combine ---------------------------------------------------------------------
  // Everything this step still needs from the exchange buffers is read into registers first; a CTA
  // barrier then separates those reads from the stores that let other CTAs run ahead (a peer's NEXT
  // exchange overwrites xs / xctx, and it can only get there through values stored below).
  const float gmax = gmax_of(xs, cs);
  auto scale_of = [&](int r) -> float {
    if (a.normalizer != LVSR_NORM_SOFTMAX) return 1.f;
    return (xs[r * 4 + 1] > 0.f) ? __expf(xs[r * 4 + 0] - gmax) : 0.f;
  };
  float gsum = 0.f, gany = 0.f, myscale = 0.f;
  for (int r = 0; r < cs; ++r) {
    const float ls = xs[r * 4 + 1];
    float sc = 0.f;
    if (a.normalizer == LVSR_NORM_SOFTMAX) sc = (ls > 0.f) ? __expf(xs[r * 4 + 0] - gmax) : 0.f;
    else sc = 1.f;
    gsum += sc * ls;
    gany = fmaxf(gany, xs[r * 4 + 2]);
    if (r == rank) myscale = sc;
  }
  const float norm = gsum + (gany > 0.f ? 0.f : 1.f);     // +1 when no position has mask == 1, attention.py:211-212
  const float inv = 1.f / norm;

  // position statistic of the new alignment (next step's window): who reports it is decided by ONE
  // rule evaluated identically by every thread of every rank from the exchanged masses (same
  // instruction sequence on the same xs values), so exactly one thread in the cluster writes
  // rowpos_out for any input.
  //   mean:   rank 0.
  //   median: the first rank whose inclusive prefix of alignment mass reaches 0.5 and that owns at
  //           least one position; rank 0 reports 0 when no prefix does (all positions masked:
  //           cumsum never crosses, argmax of zeros = 0, attention.py:138-144).
  float mean_pos = 0.f, owner_prefix = 0.f;
  int owner = -1;
  if (a.rowpos_out != nullptr) {
    if (a.rowpos_mode == LVSR_PRIOR_WINDOW_MEAN) {
      for (int r = 0; r < cs; ++r) mean_pos = fmaf(scale_of(r), xs[r * 4 + 3], mean_pos);
      mean_pos *= inv;
    } else {
      float prefix = 0.f;
      for (int r = 0; r < cs; ++r) {
        const float mass = scale_of(r) * xs[r * 4 + 1] * inv;
        const int nt_r = min(Tw, r * tc + tc) - min(Tw, r * tc);
        if (owner < 0 && nt_r > 0 && prefix + mass >= 0.5f) { owner = r; owner_prefix = prefix; }
        prefix += mass;
      }
    }
  }
  float ctx_reg[4] = {0.f, 0.f, 0.f, 0.f};     // E <= 4 * NT (checked by the planners)
  if (rank == 0) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + q * NT;
      if (e < E) {
        float acc = 0.f;
        for (int r = 0; r < cs; ++r) acc = fmaf(scale_of(r), xctx[(size_t)r * E + e], acc);
        ctx_reg[q] = acc * inv;
      }
    }
  }
  __syncthreads();

  for (int t = tid; t < nt; t += NT) {
    const float wv = s.su[t] * myscale * inv;
    if (flow) st_flow_f32(a.w_out + b0 + t0 + t, wv); else a.w_out[b0 + t0 + t] = wv;
    a.e_out[b0 + t0 + t] = s.se[t];
  }
  // zero outside the window (paste into zeros, attention.py:177-181); ranks interleave the work
  for (int pidx = rank * NT + tid; pidx < Tp; pidx += cs * NT) {
    if (pidx < b0 || pidx >= b0 + Tw) {
      if (flow) st_flow_f32(a.w_out + pidx, 0.f); else a.w_out[pidx] = 0.f;
      a.e_out[pidx] = 0.f;
    }
  }
  if (rank == 0) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = tid + q * NT;
      if (e < E) {
        if (flow) st_flow_f32(a.ctx_out + e, ctx_reg[q]); else a.ctx_out[e] = ctx_reg[q];
      }
    }
  }

  ATT_STAMP(7);
  if (a.rowpos_out != nullptr && warp == 0) {
    if (a.rowpos_mode == LVSR_PRIOR_WINDOW_MEAN) {
      if (rank == 0 && lane == 0) st_flow_f32(a.rowpos_out, mean_pos);
    } else if (owner < 0) {
      if (rank == 0 && lane == 0) st_flow_f32(a.rowpos_out, 0.f);
    } else if (owner == rank) {
      // median: first index j with cumsum(alpha) >= 0.5 -> j - 1 (0 when j == 0)
      const int chunk = (nt + 31) / 32;
      const int i0 = min(nt, lane * chunk), i1 = min(nt, i0 + chunk);
      const double sc = (double)(myscale * inv);
      double part = 0.0;
      for (int t = i0; t < i1; ++t) part += (double)s.su[t] * sc;
      double incl = part;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double nb = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += nb;
      }
      double run = (double)owner_prefix + (incl - part);
      int cross = 0x7fffffff;
      for (int t = i0; t < i1; ++t) {
        run += (double)s.su[t] * sc;
        if (run - 0.5 >= 0.0) { cross = t; break; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cross = min(cross, __shfl_xor_sync(0xffffffffu, cross, o));
      if (cross == 0x7fffffff) cross = nt - 1;            // the fp32 prefix said "here", the fp64 rescan fell one ulp short
      const int j = b0 + t0 + cross;
      if (lane == 0) st_flow_f32(a.rowpos_out, (j == 0) ? 0.f : (float)(j - 1));
    }
  }
}

}  // namespace lvsr
