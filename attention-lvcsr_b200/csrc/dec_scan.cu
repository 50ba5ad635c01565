// Persistent teacher-forced decoder: ONE cooperative kernel runs all L steps of
// AttentionRecurrent.do_apply (libs/blocks/blocks/bricks/attention.py:668-707) for the
// whole batch -- take_glimpses -> Distribute -> GatedRecurrent step -- i.e. the scan inside
// BaseSequenceGenerator.evaluate (libs/blocks/blocks/bricks/sequence_generators.py:254-311).
//
// B200 mapping
//   * one CTA per SM, resident for the whole sequence; the GRU / state-transform weight
//     slices of each CTA stay in SHARED MEMORY across all steps (2.75 MB spread over the
//     grid), as do the attention constants (conv filters, handler, energy vector).
//   * phase A (attention) is row-parallel: a cluster of `cs` CTAs per decoder row streams the
//     row's P and H slices once and merges (max, sum, partial context) through DSMEM.  When the
//     window is the whole utterance on every step (expanding prior that never cuts) and the CTA's
//     P fragments fit its 512 TMEM columns, P is staged into tensor memory once per launch and the
//     energies read it from there instead of from L2 (a.p_in_tmem, attention_row.cuh).
//   * phases B1..B3 (gates, candidate, next query) are 2-D tiled skinny products:
//     16-row x nc-column tiles, K split over the 16 warps of the CTA, fused GRU epilogues.  A CTA's
//     gate tile and candidate tile cover the same units of the same rows, so update gate,
//     candidate input and the state never leave its shared memory.
//   * the batch is cut into independent islands of <= 16 rows (rows' attention clusters own the
//     island's dense tiles); there are NO barriers or flags between CTAs: every cross-CTA value
//     (query, context, h*r, next state, alignment, position statistic) lives in a per-step
//     buffer the host fills with 0xFF bytes and is polled by its consumers until it is no longer
//     the sentinel (common.cuh: ld_flow / st_flow).  One store + one load per hand-over.
//   * the window statistics of the next step (mean / median position) ride on the attention
//     exchange, so the windowing priors need no extra pass and no host round trip.
#include "attention_row.cuh"

namespace lvsr {

namespace {

constexpr int DS_THREADS = ATT_NT;
constexpr int DS_WARPS = DS_THREADS / 32;
constexpr int DS_ROWS = 16;          // rows per dense tile

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
  return t;
}

enum { EP_GATES = 0, EP_CAND = 1, EP_QUERY = 2 };

struct DenseIO {
  const float* X1; int K1;      // rows of width K1
  const float* X2; int K2;      // appended columns (may be null)
  int R;                        // valid rows
  int N;                        // total output columns
  int mode;
  int C;
  const float* add;             // [*, N] addend
  const long long* arow;        // row index into add (or null: identity)
  long long add_rows;           // rows of the addend table (labels are clamped into it)
  float* hr;                    // EP_GATES: reset-gated state [R, C], consumed by every candidate tile
  float* loc;                   // smem [3][DS_ROWS][ncu]: update gate, candidate input, state of this tile's units
  int ncu;                      // units per tile (EP_GATES / EP_CAND)
  const float* rmask;           // [R] or null
  float* out;                   // EP_CAND: next state [R, C]; EP_QUERY: q [R, N]
  unsigned long long* tr;       // LVSR_DEC_TRACE: [x arrived, products done, cross-warp sums done] or null
};

// One 16-row x (8*NQ)-column tile.  lane = ks*16 + rq*2 + cq: rows {2rq, 2rq+1}, columns
// [cq*4NQ, +4NQ); warp w and k-half ks own the contiguous k range [(2w+ks)*Ktot/32, +Ktot/32).
// All of a lane's x values (2 rows x Ktot/32) are requested from L2 before the first FMA:
// one exposed L2 round trip per phase instead of one per k-block.
template <int NQ, int KPER>
__device__ __noinline__ void dense_tile(const DenseIO& d, const float* ws, int wstride, int r0, int c0,
                                           float* red) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ks = lane >> 4, rq = (lane >> 1) & 7, cq = lane & 1;
  constexpr int NCL = 4 * NQ;
  constexpr int NC = 2 * NCL;
  const int kbeg = (warp * 2 + ks) * KPER;
  float acc[2][NCL];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < NCL; ++j) acc[i][j] = 0.f;
  // Operand of this thread's epilogue (the tile has at most one output per thread): the label's
  // row of the feedback table / the label mask.  Requested first -- two dependent global loads
  // that would otherwise sit at the very end of the phase, on the decoder's critical path.
  static_assert(DS_ROWS * NC <= DS_THREADS, "one output per thread");
  float ep_pref = 0.f;
  {
    // volatile asm keeps the two dependent loads here, in front of the polling loads (plain loads
    // may be sunk to their use at the end of the phase, where they would be exposed)
    const int rl = tid / NC, cl = tid % NC, r = r0 + rl;
    if (tid < DS_ROWS * NC && r < d.R) {
      if (d.mode == EP_GATES) {
        const int ncu = d.ncu, gate = cl / ncu, u = c0 + (cl - gate * ncu);
        if (gate < 3 && u < d.C) {
          long long lab;
          asm volatile("ld.global.nc.s64 %0, [%1];\n" : "=l"(lab) : "l"(d.arow + r));
          lab = lab < 0 ? 0 : (lab > d.add_rows - 1 ? d.add_rows - 1 : lab);     // device labels are not range-checked by the API: never index outside the table
          asm volatile("ld.global.nc.f32 %0, [%1];\n" : "=f"(ep_pref) : "l"(d.add + lab * 3 * d.C + gate * d.C + u));
        }
      } else if (d.mode == EP_CAND) {
        ep_pref = 1.f;
        if (d.rmask) asm volatile("ld.global.nc.f32 %0, [%1];\n" : "=f"(ep_pref) : "l"(d.rmask + r));
      }
    }
  }
  float4 xv[2][KPER / 4];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int row = min(r0 + rq * 2 + i, d.R - 1);
#pragma unroll
    for (int kb = 0; kb < KPER / 4; ++kb) {
      const int k = kbeg + kb * 4;
      const float* src = (k < d.K1) ? (d.X1 + (long long)row * d.K1 + k) : (d.X2 + (long long)row * d.K2 + (k - d.K1));
      xv[i][kb] = ld_relaxed_f4(src);     // all requests in flight before the first check
    }
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int row = min(r0 + rq * 2 + i, d.R - 1);
#pragma unroll
    for (int kb = 0; kb < KPER / 4; ++kb) {
      if (!flow_ready(xv[i][kb])) {
        const int k = kbeg + kb * 4;
        const float* src = (k < d.K1) ? (d.X1 + (long long)row * d.K1 + k) : (d.X2 + (long long)row * d.K2 + (k - d.K1));
        xv[i][kb] = ld_flow_f4(src);
      }
    }
  }
  if (d.tr && tid == 0) d.tr[0] = global_ns();
#pragma unroll
  for (int kb = 0; kb < KPER / 4; ++kb) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float* wr = ws + (size_t)(kbeg + kb * 4 + kk) * wstride + cq * NCL;
      float wv[NCL];
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const float4 w4 = *reinterpret_cast<const float4*>(wr + q * 4);
        wv[q * 4 + 0] = w4.x; wv[q * 4 + 1] = w4.y; wv[q * 4 + 2] = w4.z; wv[q * 4 + 3] = w4.w;
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float4 x4 = xv[i][kb];
        const float x = kk == 0 ? x4.x : kk == 1 ? x4.y : kk == 2 ? x4.z : x4.w;
#pragma unroll
        for (int j = 0; j < NCL; ++j) acc[i][j] = fmaf(x, wv[j], acc[i][j]);
      }
    }
  }
  if (d.tr && tid == 0) d.tr[1] = global_ns();
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < NCL; ++j) {
      float v = acc[i][j];
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      if (ks == 0) red[(size_t)warp * (DS_ROWS * NC) + (rq * 2 + i) * NC + cq * NCL + j] = v;
    }
  __syncthreads();
  if (d.tr && tid == 0) d.tr[2] = global_ns();
  const int C = d.C;
  for (int o = tid; o < DS_ROWS * NC; o += DS_THREADS) {     // at most one iteration
    const int rl = o / NC, cl = o % NC;
    const int r = r0 + rl;
    if (r >= d.R) continue;
    float v = 0.f;
#pragma unroll
    for (int wq = 0; wq < DS_WARPS; ++wq) v += red[(size_t)wq * (DS_ROWS * NC) + o];
    if (d.mode == EP_GATES) {
      // tile columns are [update | reset | candidate input] of the SAME ncu units (c0 = first unit)
      const int ncu = d.ncu, gate = cl / ncu, ul = cl - gate * ncu, u = c0 + ul;
      if (gate >= 3 || u >= C) continue;
      v += ep_pref;
      float* lz = d.loc, *lai = d.loc + DS_ROWS * ncu, *ls = d.loc + 2 * DS_ROWS * ncu;
      if (gate == 0) lz[rl * ncu + ul] = fast_sigmoid(v);
      else if (gate == 1) st_flow_f32(d.hr + (long long)r * C + u, ls[rl * ncu + ul] * fast_sigmoid(v));
      else lai[rl * ncu + ul] = v;
    } else if (d.mode == EP_CAND) {
      const int ncu = d.ncu, u = c0 + cl;
      if (cl >= ncu || u >= C) continue;
      float* lz = d.loc, *lai = d.loc + DS_ROWS * ncu, *ls = d.loc + 2 * DS_ROWS * ncu;
      const float cand = fast_tanh(v + lai[rl * ncu + cl]);
      const float zz = lz[rl * ncu + cl];
      const float sold = ls[rl * ncu + cl];
      float sn = cand * zz + sold * (1.f - zz);
      sn = ep_pref * sn + (1.f - ep_pref) * sold;     // label mask (1 when there is none)
      ls[rl * ncu + cl] = sn;
      st_flow_f32(d.out + (long long)r * C + u, sn);
    } else {
      const int c = c0 + cl;
      if (c < d.N) st_flow_f32(d.out + (long long)r * d.N + c, v);
    }
  }
  __syncthreads();
}

// nq = (columns per CTA) / 8 in {1,2,3}; kper = Ktot / 32 in {4, 8, 12, 16, 24}
__device__ __forceinline__ void dense_dispatch(int nq, const DenseIO& d, const float* ws, int wstride, int r0,
                                               int c0, float* red) {
  const int kper = (d.K1 + d.K2) / 32;
#define DS_CASE(NQ_, KP_) \
  if (nq == NQ_ && kper == KP_) { dense_tile<NQ_, KP_>(d, ws, wstride, r0, c0, red); return; }
  DS_CASE(1, 4) DS_CASE(2, 4) DS_CASE(3, 4)
  DS_CASE(1, 8) DS_CASE(2, 8) DS_CASE(3, 8)
  DS_CASE(1, 12) DS_CASE(2, 12) DS_CASE(3, 12)
  DS_CASE(1, 16) DS_CASE(2, 16) DS_CASE(3, 16)
  DS_CASE(1, 24) DS_CASE(2, 24) DS_CASE(3, 24)
#undef DS_CASE
  __trap();   // plan() only admits the shapes above
}

// COMPACT: the handler copy in shared memory holds only its K rows (a.wh_rows == K); a separate instantiation so that
// the default kernel's energy loop stays exactly the unpredicated code (it is sensitive to every extra register)
template <bool COMPACT>
__global__ void __launch_bounds__(DS_THREADS, 1) dec_scan_kernel(DecScanArgs a) {
  extern __shared__ __align__(16) float smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const int cs = (int)cluster.num_blocks();
  const int rank = (int)cluster.block_rank();
  const int bid = blockIdx.x, G = gridDim.x;
  const int cluster_id = bid / cs;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int R = a.B, C = a.C, E = a.E, M = a.M;
  // The whole plan (chunk capacity, shared-memory carve-up, who owns which row) assumes clusters of
  // a.cs CTAs.  A launch path that loses the cluster attribute (seen under Nsight Compute when the
  // launch also carried the cooperative attribute: the kernel ran with 1-CTA clusters, overran its
  // shared-memory chunks and produced NaNs) must not compute anything: every CTA sees the same
  // mismatch and leaves before the first barrier.
  if (cs != a.cs) {
    if (bid == 0 && tid == 0 && a.status) atomicCAS(a.status, 0u, (unsigned)LVSR_FLOW_BAD_CLUSTER);
    return;
  }

  // ---- tensor memory for the resident P slice (a.p_in_tmem) ---------------------------------
  // All 512 columns: the kernel runs one CTA per SM (its shared memory admits no second CTA of this or
  // any other kernel that allocates tensor memory), so the allocation never waits for another owner.
  // From here on every path reaches the dealloc at the end of the kernel.
  uint32_t tmem_base = 0;
  if (!COMPACT && a.p_in_tmem) {
    uint32_t* slot = reinterpret_cast<uint32_t*>(smem + att_smem_floats(M, E, a.K, a.n, a.tc_cap, cs, a.wh_rows) - 16);
    if (warp == 0) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n"
                   ::"r"((uint32_t)__cvta_generic_to_shared(slot)), "r"(512u) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    tmem_base = *slot;
  }

  // ---- who synchronises with whom --------------------------------------------------------
  // island mode: the batch is cut into islands of <= 16 rows; an island's CTAs (its rows'
  // attention clusters) also own the island's dense tiles, so islands never wait for each other.
  // global mode (small batches): one island made of every CTA, rows tiled over nrg row groups.
  int isl_cta0 = 0, isl_n = G, r0 = 0, Rlim = R, cgi = 0;
  if (a.nisl > 0) {
    const int base = R / a.nisl, rem = R % a.nisl;
    const int row = min(cluster_id, R - 1);
    int k = 0, start = 0;
    for (; k < a.nisl; ++k) {
      const int cnt = base + (k < rem ? 1 : 0);
      if (row < start + cnt) { isl_n = cnt * cs; break; }
      start += cnt;
    }
    isl_cta0 = start * cs;
    r0 = start;
    Rlim = start + isl_n / cs;
    cgi = bid - isl_cta0;
  } else {
    r0 = (bid % a.nrg) * DS_ROWS;
    cgi = bid / a.nrg;
  }
  // a CTA's gate tile (B1) and candidate tile (B2) cover the same nc2 units of the same rows, so
  // the update gate, the candidate input and the state itself never leave its shared memory
  const bool in2 = cgi < a.ncg && cgi * a.nc2 < C, in1 = in2, in3 = cgi < a.ncg && cgi * a.nc3 < M;

  // ---- shared memory: [attention region][w1][w2][w3][red] -----------------------------
  float* att = smem;
  size_t off = att_smem_floats(M, E, a.K, a.n, a.tc_cap, cs, a.wh_rows);
  off = (off + 3) & ~(size_t)3;
  const int ws1 = a.nc1 + 4, ws2 = a.nc2 + 4, ws3 = a.nc3 + 4;
  float* w1s = smem + off; off += (size_t)(E + C) * ws1;
  float* w2s = smem + off; off += (size_t)C * ws2;
  float* w3s = smem + off; off += (size_t)C * ws3;
  float* loc = smem + off; off += (size_t)3 * DS_ROWS * a.nc2;
  off = (off + 3) & ~(size_t)3;
  // the cross-warp scratch of the dense tiles may live in the attention phase's reduction scratch: a CTA runs its
  // phases one after the other (CTA barriers in between), so the two never hold live data at the same time
  float* red = a.red_alias ? att_carve(att, M, E, a.K, a.n, a.tc_cap, cs, a.wh_rows).sred : smem + off;

  // ---- one-time staging: weight slices + attention constants -----------------------------
  for (int i = tid; i < (E + C) * a.nc1; i += DS_THREADS) {
    const int k = i / a.nc1, c = i % a.nc1, gate = c / a.nc2, u = cgi * a.nc2 + c % a.nc2;
    w1s[(size_t)k * ws1 + c] = (in1 && u < C) ? a.Wb1[(long long)k * 3 * C + gate * C + u] : 0.f;
  }
  for (int i = tid; i < DS_ROWS * a.nc2; i += DS_THREADS) {
    const int rl = i / a.nc2, r = r0 + rl, u = cgi * a.nc2 + i % a.nc2;
    loc[2 * DS_ROWS * a.nc2 + i] = (in2 && r < Rlim && u < C) ? a.s_all[(long long)r * C + u] : 0.f;
  }
  for (int i = tid; i < C * a.nc2; i += DS_THREADS) {
    const int k = i / a.nc2, c = i % a.nc2, col = cgi * a.nc2 + c;
    w2s[(size_t)k * ws2 + c] = (in2 && col < C) ? a.Wstate[(long long)k * C + col] : 0.f;
  }
  for (int i = tid; i < C * a.nc3; i += DS_THREADS) {
    const int k = i / a.nc3, c = i % a.nc3, col = cgi * a.nc3 + c;
    w3s[(size_t)k * ws3 + c] = (in3 && col < M) ? a.Ws[(long long)k * M + col] : 0.f;
  }
  att_stage_constants(att_carve(att, M, E, a.K, a.n, a.tc_cap, cs, a.wh_rows), a.v, a.Wh, a.filt, M, a.K, a.n, a.wh_rows);
  // the window is [0, T') on every step (planner): this CTA's positions are the same on every step
  const uint32_t p_taddr = att_p_taddr(tmem_base);
  if (!COMPACT && a.p_in_tmem && cluster_id < R) {
    const int tc = (a.Tp + cs - 1) / cs, t0 = min(a.Tp, rank * tc), nt = min(a.Tp, t0 + tc) - t0;
    att_stage_p_tmem(a.P, R, M, cluster_id, t0, nt, p_taddr);
  }
  __syncthreads();

  // query of the first step: q = s_0 . W_state
  if (in3) {
    DenseIO dq = {};
    dq.X1 = a.s_all; dq.K1 = C; dq.X2 = nullptr; dq.K2 = 0; dq.R = Rlim; dq.N = M; dq.mode = EP_QUERY; dq.C = C;
    dq.out = a.q_all;
    dense_dispatch(a.nc3 / 8, dq, w3s, ws3, r0, cgi * a.nc3, red);
  }
  cluster.sync();     // every CTA of the cluster is resident before the first DSMEM write

  const int trace_slot = (bid == 0) ? 0 : (bid == G - 1 ? 1 : -1);
#define DS_STAMP(j)                                                                         \
  do {                                                                                      \
    if (a.trace && trace_slot >= 0 && tid == 0)                                             \
      a.trace[((size_t)trace_slot * a.L + i) * 9 + (j)] = global_ns();                      \
  } while (0)
  for (int i = 0; i < a.L; ++i) {
#ifdef LVSR_DEC_DEBUG
    if (bid == 0 && tid == 0) g_dbg_step = i;     // approximate (CTA 0's step)
#endif
    DS_STAMP(0);
    // No barriers or flags below: every cross-CTA value lives in a per-step, sentinel-filled
    // buffer and is polled by its consumers (common.cuh).  Phases of different rows / tiles
    // overlap freely; the only ordering is true data dependence.
    const float* w_prev = (i == 0) ? a.w0 : a.w_all + (size_t)(i - 1) * R * a.Tp;
    float* w_cur = a.w_all + (size_t)i * R * a.Tp;
    float* e_cur = a.e_seq ? a.e_seq + (size_t)i * R * a.Tp : a.e_scratch;
    float* hr_cur = a.hr_all + (size_t)i * R * C;
    float* ctx_cur = a.ctx_all + (size_t)i * R * E;
    const float* s_cur = a.s_all + (size_t)i * R * C;
    float* s_next = a.s_all + (size_t)(i + 1) * R * C;

    // ================= phase A: take_glimpses, one cluster per row =====================
    const float* rowpos_rd = a.rowpos_all + (size_t)i * R;
    float* rowpos_wr = a.rowpos_all + (size_t)(i + 1) * R;
    if (cluster_id < R) {
      const int row = cluster_id;
      // window (lvsr/bricks/attention.py:123-163)
      int b0, b1;
      float lo = -1e30f, hi = 1e30f;
      if (a.prior.type == LVSR_PRIOR_EXPANDING) {
        const double st = (double)i;                     // step[0] == i under teacher forcing
        double bb = a.prior.initial_begin + st * a.prior.min_speed;
        double ee = a.prior.initial_end + st * a.prior.max_speed;
        bb = fmax(0.0, fmin((double)(a.Tp - 1), bb));
        ee = fmax(0.0, fmin((double)a.Tp, ee));
        b0 = (int)floor(bb);
        b1 = (int)ceil(ee);
      } else {
        // the batch-global cut needs the position statistic of EVERY row of the previous step
        float* wsh = att + att_smem_floats(M, E, a.K, a.n, a.tc_cap, cs, a.wh_rows) - 8;   // spare floats at the tail
        if (warp == 0) {
          float mn = 1e30f, mx = -1e30f;
          for (int r = lane; r < R; r += 32) {
            const double pos = (double)ld_flow_f32(rowpos_rd + r);
            mn = fminf(mn, (float)floor(pos - a.prior.before));
            mx = fmaxf(mx, (float)ceil(pos + a.prior.after));
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          }
          if (lane == 0) { wsh[0] = mn; wsh[1] = mx; }
        }
        __syncthreads();
        b0 = (int)fmaxf(0.f, wsh[0]);
        b1 = (int)fminf((float)a.Tp, wsh[1]);
        const double pos = (double)ld_flow_f32(rowpos_rd + row);
        lo = (float)floor(pos - a.prior.before);
        hi = (float)ceil(pos + a.prior.after);
        __syncthreads();
      }
      AttRowIO io;
      io.P = a.P; io.H = a.H; io.maskH = a.maskH;
      io.q_row = a.q_all + ((size_t)i * R + row) * M;
      io.w_prev = w_prev + (long long)row * a.Tp;
      io.filt = a.filt; io.Wh = a.Wh; io.v = a.v; io.v_bias = a.v_bias;
      io.w_out = w_cur + (long long)row * a.Tp;
      io.e_out = e_cur + (long long)row * a.Tp;
      io.ctx_out = ctx_cur + (long long)row * E;
      io.u = row; io.U = R; io.Tp = a.Tp; io.M = M; io.E = E; io.K = a.K; io.n = a.n;
      io.normalizer = a.normalizer;
      io.wh_rows = a.wh_rows;
      io.b0 = b0; io.b1 = b1; io.lo = lo; io.hi = hi;
      io.rowpos_out = (a.prior.type == LVSR_PRIOR_EXPANDING) ? nullptr : (rowpos_wr + row);
      io.rowpos_mode = a.prior.type;
      io.trace = (a.trace && bid == 0) ? a.trace + (size_t)2 * a.L * 9 + (size_t)i * 8 : nullptr;
      io.p_tmem = a.p_in_tmem;
      io.p_taddr = p_taddr;
      attention_row<COMPACT, !COMPACT>(io, att, a.tc_cap, rank, cs, true, true, false);
    }
    DS_STAMP(1);
    if (a.trace && rank == 0 && tid == 0 && cluster_id < R)
      a.trace[(size_t)2 * a.L * 9 + (size_t)a.L * 12 + (size_t)i * R + cluster_id] = global_ns();
    DS_STAMP(2);

    // ================= phase B1: gates + candidate inputs ==============================
    if (in1) {
      DenseIO d = {};
      d.X1 = ctx_cur; d.K1 = E; d.X2 = s_cur; d.K2 = C; d.R = Rlim; d.N = 3 * C; d.mode = EP_GATES; d.C = C;
      d.add = a.FF; d.arow = a.labels + (size_t)i * R; d.add_rows = a.V + 1; d.hr = hr_cur; d.loc = loc; d.ncu = a.nc2;
      d.tr = (a.trace && bid == 0) ? a.trace + (size_t)2 * a.L * 9 + (size_t)a.L * 8 + (size_t)i * 4 : nullptr;
      dense_dispatch(a.nc1 / 8, d, w1s, ws1, r0, cgi * a.nc2, red);
    }
    DS_STAMP(3);
    DS_STAMP(4);

    // ================= phase B2: candidate, blend, label mask ===========================
    if (in2) {
      DenseIO d = {};
      d.X1 = hr_cur; d.K1 = C; d.X2 = nullptr; d.K2 = 0; d.R = Rlim; d.N = C; d.mode = EP_CAND; d.C = C;
      d.loc = loc; d.ncu = a.nc2;
      d.rmask = a.lmask ? a.lmask + (size_t)i * R : nullptr;
      d.out = s_next;
      dense_dispatch(a.nc2 / 8, d, w2s, ws2, r0, cgi * a.nc2, red);
    }
    DS_STAMP(5);
    DS_STAMP(6);

    // ================= phase B3: query of the next step ================================
    if (i + 1 < a.L) {
      if (in3) {
        DenseIO d = {};
        d.X1 = s_next; d.K1 = C; d.X2 = nullptr; d.K2 = 0; d.R = Rlim; d.N = M; d.mode = EP_QUERY; d.C = C;
        d.out = a.q_all + (size_t)(i + 1) * R * M;
        dense_dispatch(a.nc3 / 8, d, w3s, ws3, r0, cgi * a.nc3, red);
      }
      DS_STAMP(7);
      DS_STAMP(8);
    }
  }
  if (!COMPACT && a.p_in_tmem) asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  cluster.sync();   // no CTA exits while a peer may still address its shared memory
  if (!COMPACT && a.p_in_tmem && warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

int sm_count() { return device_sm_count(); }

int round_up8(int x) { return (x + 7) & ~7; }
bool kper_ok(int ktot) {
  const int kp = ktot / 32;
  return ktot % 128 == 0 && (kp == 4 || kp == 8 || kp == 12 || kp == 16 || kp == 24);
}

// Fill the derived fields for a grid of G CTAs; returns the dynamic shared memory in bytes (0 = unsupported).
// want_islands: cut the batch into independent islands of <= 16 rows (grid = R*cs exactly).
size_t derive(DecScanArgs& a, int cs, int G, bool want_islands) {
  const int R = a.B, C = a.C, E = a.E, M = a.M;
  a.cs = cs;
  a.tc_cap = ceil_div(a.Tp, cs);
  if (want_islands) {
    a.nisl = ceil_div(R, DS_ROWS);
    a.ncg = (R / a.nisl) * cs;           // the smallest island's CTA count
    a.nrg = 1;
  } else {
    a.nisl = 0;
    a.nrg = ceil_div(R, DS_ROWS);
    a.ncg = G / a.nrg;
  }
  if (a.ncg < 1) return 0;
  a.nc2 = round_up8(ceil_div(C, a.ncg));
  a.nc1 = 3 * a.nc2;
  a.nc3 = round_up8(ceil_div(M, a.ncg));
  if (a.nc1 > 24 || a.nc2 > 24 || a.nc3 > 24) return 0;
  const size_t red_f = (size_t)DS_WARPS * DS_ROWS * std::max(a.nc1, std::max(a.nc2, a.nc3));
  a.red_alias = att_red_floats(E, a.tc_cap) >= red_f ? 1 : 0;
  // handler copy: zero-padded to 16 rows (fast path) if it fits, else only its K rows (long utterances)
  for (int rows : {16, a.K}) {
    a.wh_rows = rows;
    size_t f = att_smem_floats(M, E, a.K, a.n, a.tc_cap, cs, a.wh_rows);
    f = (f + 3) & ~(size_t)3;
    f += (size_t)(E + C) * (a.nc1 + 4) + (size_t)C * (a.nc2 + 4) + (size_t)C * (a.nc3 + 4);
    f = (f + 3) & ~(size_t)3;
    f += (size_t)3 * DS_ROWS * a.nc2 + 4;
    if (!a.red_alias) f += red_f;
    const size_t bytes = f * sizeof(float) + 64;
    if (bytes <= 227 * 1024) return bytes;
  }
  return 0;
}

// Does the attention window cover the whole utterance on every step?  Only the expanding prior can say so
// before the launch (b0 = 0 and b1 = T' for every i < L).  The bounds keep a margin of one position to the
// device's rounding: a window that only just reaches an end takes the L2 path, which is always correct.
bool window_is_whole_utterance(const DecScanArgs& a) {
  if (a.prior.type != LVSR_PRIOR_EXPANDING) return false;
  for (int i = 0; i < a.L; ++i) {
    const double bb = a.prior.initial_begin + (double)i * a.prior.min_speed;
    const double ee = a.prior.initial_end + (double)i * a.prior.max_speed;
    if (!(bb < 1.0 - 1e-6) || !(ee > (double)(a.Tp - 1) + 1e-6)) return false;   // false on NaN too
  }
  return true;
}

// plan of the last plan_and_launch (lvsr_dec_scan_plan); cs = 0: the persistent decoder did not run
struct DecScanPlan { int cs, islands, p_in_tmem; };
DecScanPlan g_last_plan = {0, 0, 0};

int plan_and_launch(DecScanArgs& a, int* supported, cudaStream_t stream) {
  *supported = 0;
  g_last_plan = {0, 0, 0};
  const int sms = sm_count();
  const int R = a.B, C = a.C, E = a.E, M = a.M;
  if (!kper_ok(E + C) || !kper_ok(C) || !(M == 128 || M == 256 || M == 512) || E % 4 != 0 || E / 4 > DS_THREADS) return 0;
  if (a.K < 1 || a.K > 16 || R < 1) return 0;
  int cs = 1;
  while (cs < 8 && R * cs * 2 <= sms && ceil_div(a.Tp, cs * 2) >= 16) cs *= 2;
  LVSR_CUDA_OK(cudaFuncSetAttribute(dec_scan_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  LVSR_CUDA_OK(cudaFuncSetAttribute(dec_scan_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  for (; cs >= 1; cs >>= 1) {
    // prefer islands (grid = one cluster per row); fall back to one global island on all SMs
    bool islands = R >= DS_ROWS;
    int G = islands ? R * cs : (sms / cs) * cs;
    size_t smem = derive(a, cs, G, islands);
    if (smem == 0 && islands) {
      islands = false;
      G = (sms / cs) * cs;
      smem = derive(a, cs, G, false);
    }
    if (smem == 0) continue;
    // every cluster must be co-resident (consumers poll producers): ask the driver how many fit.  GPCs of
    // 16-20 SMs hold only two 8-CTA clusters each, so large clusters cannot cover all SMs.
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G);
    cfg.blockDim = dim3(DS_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    // Co-residency of the whole grid comes from the occupancy query below (one CTA per SM, grid <=
    // max active clusters), NOT from the cooperative-launch attribute: combined with a cluster
    // dimension that attribute made profilers drop the cluster shape (round-1 NaN under ncu).
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int max_clusters = 0;
    const bool compact = a.wh_rows != 16;
    if ((compact ? cudaOccupancyMaxActiveClusters(&max_clusters, dec_scan_kernel<true>, &cfg)
                 : cudaOccupancyMaxActiveClusters(&max_clusters, dec_scan_kernel<false>, &cfg)) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    if (max_clusters * cs < G) {
      if (islands) continue;          // islands need exactly one cluster per row
      G = max_clusters * cs;
      if (G < cs) continue;
      smem = derive(a, cs, G, false);
      if (smem == 0) continue;
      cfg.gridDim = dim3(G);
      cfg.dynamicSmemBytes = smem;
    }
    if (R * cs > G) continue;        // not enough clusters for one per row: try a smaller cluster
    {
      // P in tensor memory: each CTA re-reads the same P slice on every step when the window is the whole
      // utterance; keep it on chip if its fragments fit.  LVSR_DEC_TMEM_P=0 forces the L2 path (A/B runs).
      const char* tp = getenv("LVSR_DEC_TMEM_P");
      const bool allow = !(tp && strcmp(tp, "0") == 0);
      a.p_in_tmem = (allow && !compact && att_p_fits_tmem(M, a.tc_cap) && window_is_whole_utterance(a)) ? 1 : 0;
    }
    {
      // profilers slow the kernel down by orders of magnitude: let them raise the hang guard
      const char* sl = getenv("LVSR_FLOW_SPIN_LIMIT");
      const unsigned lim = sl ? (unsigned)strtoul(sl, nullptr, 10) : LVSR_SPIN_LIMIT;
      LVSR_CUDA_OK(cudaMemcpyToSymbolAsync(g_flow_spin_limit, &lim, sizeof(lim), 0, cudaMemcpyHostToDevice, stream));
      LVSR_CUDA_OK(cudaMemcpyToSymbolAsync(g_flow_status, &a.status, sizeof(a.status), 0, cudaMemcpyHostToDevice, stream));
    }
    cudaError_t e = (a.wh_rows != 16) ? cudaLaunchKernelEx(&cfg, dec_scan_kernel<true>, a)
                                      : cudaLaunchKernelEx(&cfg, dec_scan_kernel<false>, a);
    if (e != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    g_launch_count++;
    *supported = 1;
    g_last_plan = {cs, islands ? 1 : 0, a.p_in_tmem};
#ifdef LVSR_DEC_DEBUG
    {
      LVSR_CUDA_OK(cudaStreamSynchronize(stream));
      unsigned long long ev[64]; unsigned int cnt = 0;
      LVSR_CUDA_OK(cudaMemcpyFromSymbol(&cnt, g_dbg_count, sizeof(cnt)));
      LVSR_CUDA_OK(cudaMemcpyFromSymbol(ev, g_dbg_events, sizeof(ev)));
      fprintf(stderr, "[dec debug] G=%d cs=%d NaN sightings: %u\n", G, cs, cnt);
      for (unsigned k = 0; k < cnt && k < 64; ++k)
        fprintf(stderr, "   stage %llu step~%llu cta %llu tid %llu idx %llu\n", ev[k] >> 56, (ev[k] >> 48) & 0xff,
                (ev[k] >> 32) & 0xffff, (ev[k] >> 16) & 0xffff, ev[k] & 0xffff);
      cnt = 0;
      LVSR_CUDA_OK(cudaMemcpyToSymbol(g_dbg_count, &cnt, sizeof(cnt)));
    }
#endif
    return 0;
  }
  return 0;
}

}  // namespace

// Runs the persistent decoder if the shapes fit (*supported = 1); otherwise leaves everything
// untouched (*supported = 0) and the caller falls back to the per-step kernels.
int dec_scan_try(DecScanArgs& a, int* supported, cudaStream_t stream) {
  ProfScope prof("dec_scan", stream);
  return plan_and_launch(a, supported, stream);
}

}  // namespace lvsr

extern "C" int lvsr_dec_scan_plan(int* cs, int* islands, int* p_in_tmem) {
  if (cs) *cs = lvsr::g_last_plan.cs;
  if (islands) *islands = lvsr::g_last_plan.islands;
  if (p_in_tmem) *p_in_tmem = lvsr::g_last_plan.p_in_tmem;
  return 0;
}
