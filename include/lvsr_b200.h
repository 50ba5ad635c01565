/*
 * lvsr_b200.h -- C ABI of the B200-native attention-lvcsr hot path.
 *
 * The reference (rizar/attention-lvcsr) has no FFI of its own on this path: Theano
 * generates and compiles C at run time and the "operator ABI" is the set of compiled
 * theano.function objects that Blocks/lvsr call.  Each entry point below replaces one
 * of those compiled functions 1:1 (SURVEY.md section 8b, tier b3); the reference-side
 * binding a maintainer would add is a ctypes stub, shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C: opaque handle, raw pointers, sizes.  No torch / C++ types.
 *   - all tensors are TIME-MAJOR and contiguous, float32 unless noted, exactly the
 *     layouts the reference feeds its compiled functions
 *     (lvsr/datasets/__init__.py:22-29,308; lvsr/bricks/recognizer.py:129-133,353-361).
 *   - `*_dev` pointers are device pointers on the model's GPU, `*_host` are host pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are
 *     stream-ordered and never synchronise, except the `*_host` convenience calls,
 *     which copy H2D, compute, copy D2H and synchronise the stream before returning.
 *   - every call returns 0 on success, non-zero on error; lvsr_last_error() then
 *     describes the failure (thread-local).
 *   - one model handle per GPU; a handle is not thread-safe.
 */
#ifndef LVSR_B200_H
#define LVSR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lvsr_model lvsr_model;

enum { LVSR_MAX_LAYERS = 8 };
enum { LVSR_NORM_SOFTMAX = 0, LVSR_NORM_LOGISTIC = 1, LVSR_NORM_RELU = 2 };
enum { LVSR_ACT_MAXOUT = 0, LVSR_ACT_RELU = 1, LVSR_ACT_TANH = 2, LVSR_ACT_IDENTITY = 3 };
enum { LVSR_PRIOR_EXPANDING = 0, LVSR_PRIOR_WINDOW_MEAN = 1, LVSR_PRIOR_WINDOW_MEDIAN = 2 };

/* The subset of config['net'] the path depends on
 * (SpeechRecognizer.__init__, lvsr/bricks/recognizer.py:176-204). */
typedef struct {
  int32_t num_features;            /* F: input_dims['recordings']                     */
  int32_t num_layers;              /* len(dims_bidir)                                  */
  int32_t dims_bidir[LVSR_MAX_LAYERS];
  int32_t subsample[LVSR_MAX_LAYERS];
  int32_t dim_dec;                 /* C                                                */
  int32_t dim_matcher;             /* M (defaults to dim_dec, recognizer.py:225-226)   */
  int32_t conv_n;                  /* n, filter length 2n+1                            */
  int32_t conv_num_filters;        /* K                                                */
  int32_t num_phonemes;            /* V; the lookup table has V+1 rows                 */
  int32_t dim_feedback;            /* Cfb (dim_dec unless dim_output_embedding)        */
  int32_t post_merge_dim;          /* post_merge_dims[0]                               */
  int32_t maxout_pieces;           /* num_pieces of Maxout, 1 otherwise                */
  int32_t post_merge_activation;   /* LVSR_ACT_* (reference default: Tanh)             */
  int32_t use_states_for_readout;
  int32_t energy_normalizer;       /* LVSR_NORM_*                                      */
  int32_t prior_type;              /* LVSR_PRIOR_*                                     */
  double prior_initial_begin, prior_initial_end, prior_min_speed, prior_max_speed;
  double prior_before, prior_after;
  int32_t one_of_n_feedback;       /* 0: LookupFeedback(V+1, dim_feedback) (embed_outputs=True, the default);
                                      1: OneOfNFeedback(V+1) (embed_outputs=False, lvsr/bricks/__init__.py:86-109;
                                      exp/wsj/configs/wsj_jan_new.yaml:46): feedback = one-hot, dim_feedback = V+1  */
  int32_t reserved;
} lvsr_config;

const char* lvsr_last_error(void);
int lvsr_version(void);

/* ---- model life cycle ----------------------------------------------------------- */
/* SpeechRecognizer(**config['net']) + allocate(): lvsr/main.py:213-221. Uses the
 * CUDA device current on the calling thread. */
int lvsr_model_create(const lvsr_config* cfg, lvsr_model** out);
int lvsr_model_destroy(lvsr_model* m);

/* Parameter table in Blocks order/names ("/recognizer/encoder/bidir0/forward/fork/fork_inputs.W"
 * ...): Selector.get_parameters, libs/blocks/blocks/select.py:160-220. */
int lvsr_model_num_params(const lvsr_model* m);
const char* lvsr_model_param_name(const lvsr_model* m, int index);
int lvsr_model_param_shape(const lvsr_model* m, int index, int64_t shape[2], int32_t* ndim);
/* Model.set_parameter_values / get_parameter_values (lvsr/bricks/recognizer.py:408-412). */
int lvsr_model_set_param(lvsr_model* m, const char* name, const float* values_host, int64_t count);
int lvsr_model_get_param(const lvsr_model* m, const char* name, float* values_host, int64_t count);
/* All parameters live in ONE device allocation ("flat" layout: parameter i at float offset
 * lvsr_model_param_offset, 256-byte aligned, padding zero).  Gradients, optimizer state and the
 * gradient all-reduce of the training step use buffers of the same layout and size. */
int64_t lvsr_model_flat_size(const lvsr_model* m);
int lvsr_model_param_offset(const lvsr_model* m, int index, int64_t* offset, int64_t* count);
float* lvsr_model_flat_params(lvsr_model* m);     /* device pointer; call lvsr_model_finalize after writing through it */
/* Re-derive the packed kernel-side weights after parameters changed. */
int lvsr_model_finalize(lvsr_model* m);
/* Launch status of the persistent teacher-forced decoder of the LAST lvsr_cost_matrix call on this
 * handle (synchronises with the device): 0 = ok, 2 = a hand-over value never arrived within the
 * polling limit, 3 = the launch lost its cluster shape.  On a non-zero status the costs of that call
 * are NaN (never plausible garbage); lvsr_recognizer_cost_host re-runs such a call on the step-wise
 * kernels by itself and counts it in *stepwise_fallbacks (may be NULL).  No reference counterpart:
 * Theano raises from inside the compiled function instead. */
int lvsr_model_status(lvsr_model* m, int32_t* launch_status, int64_t* stepwise_fallbacks);
/* Plan of the persistent decoder's last planning call in this process (any handle): cluster size
 * (0 = the step-wise kernels ran instead), island mode, and whether each CTA kept its slice of the
 * preprocessed context in tensor memory (whole-utterance windows only; LVSR_DEC_TMEM_P=0 turns it off).
 * Any pointer may be NULL.  Host-only, does not synchronise. */
int lvsr_dec_scan_plan(int* cs, int* islands, int* p_in_tmem);

/* ---- encoder: BeamSearch.context_computer / Encoder.apply -------------------------
 * (libs/blocks/blocks/search.py:97-99; lvsr/bricks/__init__.py:71-78).
 * recordings [T,B,F], mask [T,B] (NULL = no mask) -> attended [T',B,E], attended_mask [T',B]
 * with T' = lvsr_encoded_length(T), E = 2*dims_bidir[last]. */
int lvsr_encoded_length(const lvsr_model* m, int32_t T);
int lvsr_encoded_dim(const lvsr_model* m);
int lvsr_encoder_forward(lvsr_model* m, const float* recordings_dev, const float* mask_dev,
                         int32_t T, int32_t B, float* attended_dev, float* attended_mask_dev,
                         void* stream);

/* attention.preprocess: lvsr/bricks/attention.py:228-230. attended [T',U,E] -> [T',U,M]. */
int lvsr_preprocess(lvsr_model* m, const float* attended_dev, int32_t Tp, int32_t U,
                    float* preprocessed_dev, void* stream);

/* ---- teacher-forced decoder: generator.cost_matrix --------------------------------
 * (libs/blocks/blocks/bricks/sequence_generators.py:254-326).
 * labels int64 [L,B], every entry in [0, num_phonemes) -- device memory, NOT range-checked here
 * (lvsr_recognizer_cost_host checks its host copy); labels_mask [L,B] or NULL.  Outputs: costs [L,B]; optional (NULL to
 * skip) weights [L,B,T'], energies [L,B,T'], states [L,B,C] (= s_{i-1}),
 * weighted_averages [L,B,E]. */
int lvsr_cost_matrix(lvsr_model* m, const float* attended_dev, const float* attended_mask_dev,
                     int32_t Tp, int32_t B, const int64_t* labels_dev, const float* labels_mask_dev,
                     int32_t L, float* costs_dev, float* weights_dev, float* energies_dev,
                     float* states_dev, float* weighted_averages_dev, void* stream);

/* ---- the BeamSearch state functions (libs/blocks/blocks/search.py:101-142) ---------
 * R rows (beam hypotheses); row r attends utterance row_utt[r] of `attended` [T',U,E]
 * (row_utt NULL = identity, U == R: the reference's replicated-context call).
 * `preprocessed` may be NULL: it is then recomputed, as the reference does on every call. */
int lvsr_initial_states(lvsr_model* m, int32_t Tp, int32_t R, float* states_dev, int64_t* outputs_dev,
                        float* weighted_averages_dev, float* weights_dev, float* energies_dev,
                        int64_t* step_dev, void* stream);
int lvsr_logprobs(lvsr_model* m, const float* attended_dev, const float* preprocessed_dev,
                  const float* attended_mask_dev, int32_t Tp, int32_t U, const int32_t* row_utt_dev,
                  int32_t R, const float* states_dev, const float* weights_dev, const int64_t* step_dev,
                  float* neg_logprobs_dev, void* stream);
int lvsr_next_states(lvsr_model* m, const float* attended_dev, const float* preprocessed_dev,
                     const float* attended_mask_dev, int32_t Tp, int32_t U, const int32_t* row_utt_dev,
                     int32_t R, const float* states_dev, const float* weights_dev, const int64_t* step_dev,
                     const int64_t* outputs_dev, float* next_states_dev, float* next_weighted_averages_dev,
                     float* next_weights_dev, float* next_energies_dev, int64_t* next_step_dev,
                     void* stream);

/* ---- batched beam search: one step for MANY utterances --------------------------------------------
 * The hypotheses (rows) of utterance s are the contiguous rows [seg_start[s], seg_start[s+1]) -- one segment is
 * what the reference calls the batch inside BeamSearch.search (libs/blocks/blocks/search.py:244-399), so the
 * batch-global window cut of take_glimpses is taken per segment.  row_utt[r] = column of the row's utterance in
 * attended / preprocessed / attended_mask [T',U,.]; row_seg[r] = its segment; utt_len[s] = valid encoded frames of
 * the segment's utterance (NULL: T').  All hypothesis state stays on the device:
 *
 *   lvsr_search_expand  = logprobs_computer + BeamSearch._smallest (:109-117,220-242,341-344): take_glimpses once per
 *     row (kept in wavg / new_weights / new_energies for lvsr_search_advance), readout, -log softmax, and per
 *     segment the k smallest cost_so_far + (-logp) in increasing order: top_parent (row index), top_symbol,
 *     top_cost [nseg * k], top_count [nseg] (= min(k, width * V); -1 if a log-probability was not finite).
 *     Only these k triples per utterance have to reach the host.
 *   lvsr_search_advance = next_state_computer (:119-142) for the Rn selected children (parent rows + symbols):
 *     gathers the parents' state and -- reuse_glimpses != 0 -- their glimpses (exact when the window does not
 *     depend on which rows are in the batch: the expanding prior), else recomputes take_glimpses over the selected
 *     rows as the reference does (window_around_* priors); then Distribute + GRU step; step + 1. */
int lvsr_search_expand(lvsr_model* m, const float* attended_dev, const float* preprocessed_dev,
                       const float* attended_mask_dev, int32_t Tp, int32_t U, const int32_t* utt_len_dev,
                       const int32_t* row_utt_dev, const int32_t* row_seg_dev, const int32_t* seg_start_dev,
                       int32_t nseg, int32_t R, const float* states_dev, const float* weights_dev,
                       const int64_t* step_dev, const float* cost_so_far_dev, int32_t k, float* wavg_dev,
                       float* new_weights_dev, float* new_energies_dev, int32_t* top_parent_dev,
                       int32_t* top_symbol_dev, float* top_cost_dev, int32_t* top_count_dev, void* stream);
int lvsr_search_advance(lvsr_model* m, const float* attended_dev, const float* preprocessed_dev,
                        const float* attended_mask_dev, int32_t Tp, int32_t U, const int32_t* utt_len_dev, int32_t Rn,
                        const int32_t* parent_dev, const int64_t* symbols_dev, const int32_t* row_utt_dev,
                        const int32_t* row_seg_dev, const int32_t* seg_start_dev, int32_t nseg, const float* states_dev,
                        const float* weights_dev, const int64_t* step_dev, const float* wavg_dev,
                        const float* new_weights_dev, const float* new_energies_dev, int32_t reuse_glimpses,
                        float* next_states_dev, float* next_wavg_dev, float* next_weights_dev,
                        float* next_energies_dev, int64_t* next_step_dev, void* stream);

/* The whole search loop of BeamSearch.search (libs/blocks/blocks/search.py:244-399) for U utterances decoded in
 * lock-step: the reference's bookkeeping (histories, `done`, both stopping criteria, final ranking) in C++ around
 * lvsr_search_expand / lvsr_search_advance; per step one small H2D, one small D2H, one synchronisation for ALL
 * utterances.  utt_len_host[u] = valid encoded frames, max_length_host[u] = int(T_u / max_decoded_length_scale)
 * (lvsr/bricks/recognizer.py:519-520).  stop_on_optimistic: 0 = 'patience', 1 = 'optimistic_future_cost'.
 * Result: per utterance the finished hypotheses ranked by cost - char_discount * length, each as its full token
 * and cumulative-cost history INCLUDING the initial symbol (what BeamSearch keeps in `done`).  A
 * validate_solution_function callback is not available here (the Python mirror runs its own loop for that). */
typedef struct lvsr_search_result lvsr_search_result;
int lvsr_beam_search_many(lvsr_model* m, const float* attended_dev, const float* preprocessed_dev,
                          const float* attended_mask_dev, int32_t Tp, int32_t U, const int32_t* utt_len_host,
                          const int32_t* max_length_host, int32_t beam_size, int32_t eol_symbol,
                          int32_t ignore_first_eol, double char_discount, double round_to_inf,
                          int32_t stop_on_optimistic, lvsr_search_result** result, void* stream);
int lvsr_search_result_count(const lvsr_search_result* r, int32_t utt);                     /* finished hypotheses */
int lvsr_search_result_length(const lvsr_search_result* r, int32_t utt, int32_t j);         /* history length     */
int lvsr_search_result_get(const lvsr_search_result* r, int32_t utt, int32_t j, int64_t* tokens, float* costs);
int lvsr_search_result_destroy(lvsr_search_result* r);

/* ---- host-buffer entry points (the call a user of the reference makes) -------------
 * SpeechRecognizer.cost on a batch (lvsr/bricks/recognizer.py:375-390): H2D copies,
 * encoder, cost_matrix, D2H of costs [L,B]; synchronises.  Buffers should be pinned. */
int lvsr_recognizer_cost_host(lvsr_model* m, const float* recordings_host, const float* mask_host,
                              const int64_t* labels_host, const float* labels_mask_host,
                              int32_t T, int32_t B, int32_t L, float* costs_host, void* stream);

/* ---- training step: GradientDescent._function -------------------------------------------------
 * (libs/blocks/blocks/algorithms/__init__.py:244-256,284-287 as assembled by lvsr/main.py:340-345,480-519).
 * Split in two so a data-parallel caller can all-reduce the gradient buffer in between:
 *
 *   lvsr_train_cost_and_grads: forward + backward of one batch (device pointers, layouts as lvsr_encoder_forward /
 *     lvsr_cost_matrix).  cost_dev[0] = gscale * sum(cost_matrix); grads_dev (lvsr_model_flat_size floats, flat
 *     parameter layout) = gscale * d sum(cost_matrix) / d parameter.  Single GPU: gscale = 1/B gives the reference's
 *     cost = sum / batch_size.  N GPUs: pass gscale = 1, all-reduce(sum) grads_dev, then apply with
 *     gscale = 1 / global batch (SURVEY.md 8e).  Softmax energy normaliser only.
 *   lvsr_train_apply_updates: grads_dev *= gscale (+ 2 decay W on WEIGHT parameters), then the CompositeRule of
 *     lvsr/main.py:509-516: StepClipping(gradient_threshold) -> Momentum(scale, momentum) -> AdaDelta(decay_rate,
 *     epsilon) -> Restrict(VariableClipping(max_norm, axis=0), WEIGHT parameters) -> RemoveNotFinite(0.0) -> BurnIn,
 *     parameter -= step, and the kernel-side weights are re-packed.  grads_dev holds the steps afterwards.
 *     Optimizer state lives in the handle (lvsr_train_reset clears it). */
typedef struct {
  float gradient_threshold;        /* StepClipping threshold, 0 = off (B/algorithms/__init__.py:610-643)        */
  int32_t use_momentum;            /* 'momentum' in config['training']['rules'] (lvsr/main.py:483-486)          */
  float scale, momentum;           /* Momentum(learning_rate=scale, momentum)                                   */
  int32_t use_adadelta;            /* 'adadelta' in rules                                                        */
  float decay_rate, epsilon;       /* AdaDelta(decay_rate, epsilon), :464-516                                    */
  float max_norm;                  /* regularization.max_norm, 0 = off (lvsr/main.py:490-505)                    */
  int32_t burn_in_steps;           /* BurnIn(num_steps), lvsr/algorithms.py:19-43                                */
  float decay;                     /* regularization.decay: + decay * ||WEIGHT parameters||^2 (lvsr/main.py:419-421) */
} lvsr_train_config;
int lvsr_train_cost_and_grads(lvsr_model* m, const float* recordings_dev, const float* mask_dev,
                              const int64_t* labels_dev, const float* labels_mask_dev, int32_t T, int32_t B,
                              int32_t L, float gscale, float* cost_dev, float* grads_dev, void* stream);
int lvsr_train_apply_updates(lvsr_model* m, float* grads_dev, float gscale, const lvsr_train_config* tc,
                             void* stream);
int lvsr_train_gradient_norm(lvsr_model* m, float* norm_host);   /* total_gradient_norm of the last update (synchronises) */
int lvsr_train_reset(lvsr_model* m);

/* Counters for bench.py: number of kernels this library launched since the last reset. */
int64_t lvsr_launch_count(int reset);

/* Per-kernel-class device timing (CUDA events recorded on the launching stream around every
 * launch of that class) -- the analogue of the reference's Theano ProfileStats
 * (libs/Theano/theano/compile/profiling.py:97).  Classes: "gemm", "bigru", "attention",
 * "window", "dense", "readout".  lvsr_profile_read synchronises the device, returns the
 * summed milliseconds and launch count recorded since the last read of that class. */
int lvsr_profile_enable(int on);
int lvsr_profile_read(const char* kernel_class, double* total_ms, int64_t* count);

#ifdef __cplusplus
}
#endif
#endif /* LVSR_B200_H */
