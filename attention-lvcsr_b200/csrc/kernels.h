// Internal (C++) launch interfaces of the kernels behind the C ABI in include/lvsr_b200.h.
#pragma once
#include "common.cuh"

namespace lvsr {

// ---- gemm.cu ------------------------------------------------------------------------
struct GemmArgs {
  const float* A;          // row r lives at A + (r / rows_per_block) * block_stride + (r % rows_per_block) * lda
  int M, K;
  int rows_per_block;
  long long block_stride;
  int lda;
  const float* W;          // [K, N] row-major, leading dimension ldw
  int N, ldw;
  const float* bias;       // [N] or nullptr
  float* C;                // [M, N], leading dimension ldc
  int ldc;
  int accumulate;          // C += ... instead of C = ...
};
int gemm_bias(const GemmArgs& g, cudaStream_t stream);

inline GemmArgs make_gemm(const float* A, int M, int K, const float* W, int N, const float* bias,
                          float* C, bool accumulate = false) {
  GemmArgs g;
  g.A = A; g.M = M; g.K = K; g.rows_per_block = M > 0 ? M : 1; g.block_stride = 0; g.lda = K;
  g.W = W; g.N = N; g.ldw = N; g.bias = bias; g.C = C; g.ldc = N; g.accumulate = accumulate ? 1 : 0;
  return g;
}

// ---- gemm_tc.cu: tcgen05 / TMEM / TMA path (3xTF32 split) ------------------------------
bool gemm_tc_supported(int M, int N, int K);
int gemm_tc_kpad(int K);                 // contraction dimension as stored in the hi/lo operands (multiple of 32)
int split_weight_tf32(const float* W, int K, int N, float* Wt_hi, float* Wt_lo, cudaStream_t stream);
int transpose_split_tf32(const float* W, int K, int N, int ldw, float* hi, float* lo, cudaStream_t stream);
int split_tf32(const float* x, float* hi, float* lo, long long n, cudaStream_t stream);
int gemm_tc_presplit(const float* A_hi, const float* A_lo, int M, const float* B_hi, const float* B_lo, int N, int Kpad,
                     const float* bias, float* C, int ldc, int splits, long long split_stride, cudaStream_t stream);
int gemm_tc_splits_launched(int Kpad, int splits);   // how many partial outputs gemm_tc_presplit writes
// fp16 head/tail variant (kind::f16): half the operand bytes and tensor time of the tf32 split; inputs of bounded range only
bool gemm_tc_h16_supported(int M, int N, int K);
int gemm_tc_kpad_h16(int K);             // contraction dimension as stored in the fp16 operands (multiple of 64)
int split_weight_h16(const float* W, int K, int N, void* head, void* tail, float* scale2, cudaStream_t stream);
int gemm_tc_h16(const float* A, void* A_head, void* A_tail, int M, int K, const void* Wt_head, const void* Wt_tail,
                const float* scale2, int N, const float* bias, float* C, int ldc, cudaStream_t stream);
int gemm_tc(const float* A, float* A_hi, float* A_lo, int M, int K, const float* Wt_hi, const float* Wt_lo, int N,
            const float* bias, float* C, int ldc, cudaStream_t stream);

// ---- bigru.cu -----------------------------------------------------------------------
struct BiGruArgs {
  const float* pre;        // [T*B, 6D]: per direction [inputs D | update-gate D | reset-gate D], fwd then bwd
  const float* mask;       // [T, B] view (time stride mask_tstride) or nullptr
  long long mask_tstride;
  const float *Wg_f, *Ws_f, *h0_f;   // forward  state_to_gates [D,2D], state_to_state [D,D], initial_state [D]
  const float *Wg_b, *Ws_b, *h0_b;   // backward
  float* out;              // [ceil(T/subsample), B, 2D] (forward units first)
  int T, B, D, subsample;
  // training only (both null for inference): the tape the backward scan reads
  float* tape;             // = pre, written in place: candidate c over the inputs slot, z / r over the gate slots
  float* hext;             // [(T+2), B, 2D]: slot t+1 = states after time t; slot 0 (forward half) and slot T+1
                           // (backward half) = the broadcast initial states
};
bool bigru_supported(int D);
int bigru_layer(const BiGruArgs& a, cudaStream_t stream);

// ---- bigru_bwd.cu: reverse-time scan of one layer (training) ------------------------------
struct BiGruBwdArgs {
  float* tape;             // [T*B, 6D] in: c | z | r per direction (forward's tape); out: dA | dGz | dGr
  const float* hext;       // [(T+2), B, 2D] (see BiGruArgs)
  const float* mask;       // [T, B] view or nullptr
  long long mask_tstride;
  const float* dout;       // [ceil(T/subsample), B, 2D] gradient of the layer's (subsampled) output
  const float *Wg_f, *Ws_f, *Wg_b, *Ws_b;
  float* hr_out;           // [T, B, 2D]: h_prev * r (operand of the state_to_state gradient)
  float* dh0;              // [2, B, D]: gradient of the broadcast initial state, per direction and row
  int T, B, D, subsample;
};
int bigru_layer_backward(const BiGruBwdArgs& a, cudaStream_t stream);

// ---- attention.cu -------------------------------------------------------------------
struct PriorParams {
  int type;                // LVSR_PRIOR_*
  double initial_begin, initial_end, min_speed, max_speed, before, after;
};

// Window of take_glimpses (lvsr/bricks/attention.py:123-163), computed on device.
//   win[0] = begin, win[1] = end (global cut); lohi[2r], lohi[2r+1] = per-row strict bounds
struct WindowArgs {
  const float* weights;    // [R, Tp] previous alignment
  const long long* step;   // [R] (only step[0] is used, by the expanding prior); may be nullptr (= 0)
  long long step_offset;   // added to step[0] (teacher forcing: the step index)
  int R, Tp;
  PriorParams prior;
  int* win;                // [2] (or [2 * nseg])
  float* lohi;             // [2R]
  // optional segmentation (batched beam search: one segment = the hypotheses of one utterance, which is the
  // reference's "batch" for the batch-global cut): rows [seg_start[s], seg_start[s+1]) -> win[2s], win[2s+1]
  const int* seg_start;    // [nseg + 1] or nullptr (one segment = all rows)
  int nseg;
  const int* seg_len;      // [nseg] valid encoded frames of the segment's utterance (<= Tp) or nullptr (= Tp)
};
int attention_window(const WindowArgs& a, cudaStream_t stream);

struct AttStepArgs {
  const float* P;          // [Tp, U, M] preprocessed attended
  const float* H;          // [Tp, U, E] attended
  const float* maskH;      // [Tp, U]
  const int* row_utt;      // [R] or nullptr (identity)
  const float* q;          // [R, M]  states . W_state
  const float* w_prev;     // [R, Tp]
  const int* win;          // [2] from attention_window ([2 * nseg] with row_seg)
  const int* row_seg;      // [R] segment of each row or nullptr (all rows share win[0..1])
  const float* lohi;       // [2R]
  const float* filt;       // [K, 2n+1]
  const float* Wh;         // [K, M]
  const float* v;          // [M]
  float v_bias;            // energy bias (only when normalizer != softmax)
  float* w_out;            // [R, Tp]
  float* e_out;            // [R, Tp]
  float* ctx;              // [R, E]
  int R, U, Tp, M, E, K, n, normalizer;
};
int attention_step(const AttStepArgs& a, cudaStream_t stream);
int attention_max_cluster();

// ---- decoder.cu ---------------------------------------------------------------------
// out[R,N] = epilogue( X1[R,K1].W1[K1,N] (+ X2[R,K2].W2[K2,N2], columns < N2 only) + add[arow[r]] )
enum { DENSE_PLAIN = 0, DENSE_GATES = 1, DENSE_CAND = 2 };
struct DenseArgs {
  const float* X1; int K1; const float* W1;        // W1 [K1, N]
  const float* X2; int K2; const float* W2; int N2; // W2 [K2, N2], may be null
  const float* add;        // [*, N] addend rows or nullptr
  const long long* arow;   // [R] row index into add (labels) or nullptr (identity)
  long long add_rows;      // rows of `add` when arow is given (0 = unknown): indices are clamped into the table
  int R, N, mode;
  // DENSE_PLAIN: out[R,N]
  float* out;
  // DENSE_GATES (N = 3C): cols [0,C) update -> z[R,C]; [C,2C) reset -> hr[R,C] = s*r; [2C,3C) -> ai[R,C]
  // DENSE_CAND  (N = C):  c = tanh(acc + ai); s' = c*z + s*(1-z); optional row mask blend -> out[R,C]
  const float* s;          // [R, C] current states
  float* z; float* hr; float* ai;
  const float* rmask;      // [R] or nullptr
  int C;
};
int dense_step(const DenseArgs& a, cudaStream_t stream);

// readouts -> -log softmax.  merged [R, Cpm] (already merge + nothing else): adds bias, maxout/relu,
// Linear(Cpm/pieces -> V), log-softmax; writes either all V costs or the cost of labels[r].
struct ReadoutArgs {
  const float* merged;     // [R, Cpm]
  const float* b_pm;       // [Cpm]
  const float* Wo;         // [Cpm/pieces, V]
  const float* bo;         // [V]
  int R, Cpm, pieces, V, act;   // act: LVSR_ACT_*
  const long long* labels; // [R] or nullptr
  const float* lmask;      // [R] or nullptr (multiplies the picked cost)
  float* costs_all;        // [R, V] or nullptr
  float* costs_picked;     // [R] or nullptr
  const unsigned* poison;  // optional launch-status word of the producer: non-zero -> every cost is NaN
};
int readout_costs(const ReadoutArgs& a, cudaStream_t stream);

// ---- dec_scan.cu: persistent teacher-forced decoder -----------------------------------
struct DecScanArgs {
  const float *P, *H, *maskH;          // [Tp,B,M], [Tp,B,E], [Tp,B]
  const float *filt, *Wh, *v;          // attention constants
  float v_bias;
  PriorParams prior;
  const float* Wb1;                    // [E+C, 3C]: rows <E = distribute [gates|inputs], rows >=E = [state_to_gates | 0]
  const float* Wstate;                 // [C, C]
  const float* Ws;                     // [C, M]
  const float* FF;                     // [(V+1), 3C] fork(feedback(y)), gate columns first
  const long long* labels;             // [L, B]
  const float* lmask;                  // [L, B] or nullptr
  // Every buffer another CTA reads is per-step and pre-filled with the sentinel (0xFF bytes) by
  // the host, except step 0 (s_all[0], rowpos_all[0], w0): written once, polled by consumers.
  float* s_all;                        // [(L+1), B, C]; s_all[0] = initial states on entry
  float* ctx_all;                      // [L, B, E]
  const float* w0;                     // [B, Tp] initial alignment
  float* w_all;                        // [L, B, Tp] alignments (the caller's weights output or scratch)
  float* e_seq;                        // [L, B, Tp] or nullptr
  float* e_scratch;                    // [B, Tp]
  float* q_all;                        // [L, B, M]
  float* hr_all;                       // [L, B, C] reset-gated states (the only gate value that crosses CTAs)
  float* rowpos_all;                   // [L+1, B]; rowpos_all[0] = 0
  unsigned long long* trace;           // optional debug stamps, or nullptr
  unsigned* status;                    // launch status word (common.cuh: LVSR_FLOW_*), zeroed by the caller
  int Tp, B, L, M, E, C, K, n, normalizer;
  int V;                               // num_phonemes: the feedback table FF has V + 1 rows
  // derived by the planner
  int cs, tc_cap, nrg, nc1, nc2, nc3;
  int nisl, ncg;                       // nisl > 0: islands of <= 16 rows whose CTAs own their dense tiles
  int wh_rows;                         // handler rows in shared memory: 16 (fast) or K (compact, long utterances)
  int red_alias;                       // dense-tile scratch shares the attention reduction scratch (long utterances)
  int p_in_tmem;                       // each CTA's P slice is staged once into tensor memory (whole-utterance window)
};
int dec_scan_try(DecScanArgs& a, int* supported, cudaStream_t stream);

// small utility kernels
int fill_f32(float* p, long long n, float v, cudaStream_t stream);
int fill_i64(long long* p, long long n, long long v, cudaStream_t stream);
int broadcast_rows(float* dst, const float* src, int R, int N, cudaStream_t stream);   // dst[r,:] = src[:]
int onehot_rows(float* dst, int R, int N, cudaStream_t stream);                         // dst[r,:] = e_0
int count_sentinels(const float* p, long long n, long long* host_count, cudaStream_t stream);   // synchronises
int gather_rows(float* dst, const float* src, const int* idx, int Rn, int N, cudaStream_t stream);   // dst[r,:] = src[idx[r],:]
int gather_i64(long long* dst, const long long* src, const int* idx, int Rn, long long inc, cudaStream_t stream);
// k smallest of cost_so_far[r] + neglogp[r, v] over the rows of each segment (B/search.py:341-344)
int segment_topk(const float* neglogp, const float* cost_so_far, const int* seg_start, int nseg, int V, int k,
                 int* top_parent, int* top_symbol, float* top_cost, int* top_count, cudaStream_t stream);
int add_bias_rows(float* dst, const float* src, const float* bias, int R, int N, cudaStream_t stream);   // dst[r,:] = src[r,:] + bias
int add_i64(long long* dst, const long long* src, int n, long long inc, cudaStream_t stream);
int gather_time_subsample(float* dst, const float* src, int Tout, int k, long long row_elems,
                          cudaStream_t stream);                                         // dst[t] = src[t*k]

}  // namespace lvsr
