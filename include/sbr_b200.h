/* sbr_b200.h -- C ABI of libsbr_b200.so: the B200-native replacement for the three callables
 * that theano.function compiles on the reference's RNN training hot path.
 *
 * Reference interface replaced (paths relative to rdevooght/sequence-based-recommendations):
 *   train_function(*theano_inputs) -> cost, in-place parameter/optimizer update
 *       built at neural_networks/rnn_base.py:175-186, called at rnn_base.py:290
 *       inputs: OneHot   [X, mask, Y, pop, exclude]           rnn_one_hot.py:61
 *               Sampling [X, mask, Y, samples, pop, exclude]  rnn_sampling.py:128
 *               Margin   [X, mask, Ymat, weight, exclude]     rnn_margin.py:100
 *   test_function(theano_inputs, k) -> ids[k]     rnn_base.py:196-213, rnn_sampling.py:140-157
 *   predict_function(X, mask) -> scores[1,N]      rnn_base.py:188-194
 *   lasagne.layers.get/set_all_param_values       rnn_base.py:476,515
 *
 * Conventions
 *   - plain C, no C++/torch types; every pointer argument is a HOST pointer, borrowed for the
 *     duration of the call (C-contiguous, caller-owned, e.g. a numpy buffer);
 *   - every function returns 0 on success, a negative sbr_status otherwise; the message is read
 *     with sbr_last_error(); errors coming from CUDA/NCCL are sticky on the handle;
 *   - a handle is NOT thread-safe: one handle per GPU rank, one caller thread per handle;
 *   - X is int32 [B, max_length, ids_per_step], left-aligned; mask is float32 [B, max_length]
 *     with mask[b, :len_b] = 1 exactly as _prepare_input builds it (rnn_one_hot.py:100-101).
 *     A mask that is not a left-aligned run of ones is rejected with SBR_E_MASK;
 *   - `exclude` of the reference's train inputs is not part of the ABI: the train cost never reads
 *     it (on_unused_input='ignore', rnn_base.py:185); at test time the excluded ids are passed
 *     as a ragged list (sbr_topk);
 *   - parameters are addressed by their index in the reference checkpoint order
 *     (lasagne get_all_param_values order, rnn_base.py:476), per-gate matrices, row-major.
 */
#ifndef SBR_B200_H
#define SBR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SBR_API __attribute__((visibility("default")))
#else
#define SBR_API
#endif

#define SBR_ABI_VERSION 2
#define SBR_MAX_LAYERS 8
#define SBR_NCCL_ID_BYTES 128

typedef struct sbr_model sbr_model;

typedef enum sbr_status {
  SBR_OK = 0,
  SBR_E_ARG = -1,       /* bad argument / unsupported configuration        */
  SBR_E_CUDA = -2,      /* CUDA runtime or driver error (sticky)           */
  SBR_E_NCCL = -3,      /* NCCL error or libnccl not loadable (sticky)     */
  SBR_E_MASK = -4,      /* mask is not a left-aligned run of ones          */
  SBR_E_RANGE = -5,     /* an id is outside [0, n_items + n_extra_ids)     */
  SBR_E_NOGPU = -6      /* no CUDA device: there is no CPU fallback        */
} sbr_status;

enum { SBR_CELL_LSTM = 0, SBR_CELL_GRU = 1, SBR_CELL_VANILLA = 2 };          /* --r_t, recurrent_layers.py:9 */
enum { SBR_LOSS_CCE = 0, SBR_LOSS_BPR = 1, SBR_LOSS_BPRI = 2, SBR_LOSS_TOP1 = 3,
       SBR_LOSS_BLACKOUT = 4, SBR_LOSS_HINGE = 5, SBR_LOSS_LOGIT = 6, SBR_LOSS_LOGSIG = 7 }; /* --loss */
enum { SBR_UPD_ADAM = 0, SBR_UPD_ADAGRAD = 1, SBR_UPD_ADADELTA = 2, SBR_UPD_RMSPROP = 3,
       SBR_UPD_NESTEROV = 4 };                                               /* --u_m, update_manager.py:4 */
/* arithmetic of the GEMM-shaped stages; both keep fp32 storage and fp32 accumulation */
enum { SBR_MATH_FP32 = 0,   /* fp32-accurate: CUDA-core FFMA or 3xTF32 split on tcgen05 */
       SBR_MATH_TF32 = 1 }; /* single-pass TF32 on tcgen05 (10-bit mantissa inputs)       */

typedef struct sbr_config {
  int32_t struct_size;              /* = sizeof(sbr_config), ABI guard                         */
  int32_t cell;                     /* SBR_CELL_*                                              */
  int32_t n_layers;                 /* --r_l "a-b-c"                                           */
  int32_t layers[SBR_MAX_LAYERS];
  int32_t n_items;                  /* dataset.n_items (rnn_base.py:109)                       */
  int32_t n_extra_ids;              /* optional-feature id rows appended after the items (10 with --rf) */
  int32_t ids_per_step;             /* K = RNNBase._input_size() (rnn_base.py:615-622)         */
  int32_t embedding;                /* --r_emb, 0 = gather-sum layer 0                         */
  int32_t max_length;               /* T, --max_length                                         */
  int32_t batch_size;               /* rows per call on THIS rank (local batch)                */
  int32_t loss;                     /* SBR_LOSS_*                                              */
  int32_t n_samples;                /* S of RNNSampling (rnn_sampling.py:105-108)              */
  int32_t last_layer_tanh;          /* rnn_sampling.py:19                                      */
  int32_t updater;                  /* SBR_UPD_*                                               */
  float lr, rho, beta1, beta2;      /* update_manager.py:5-8                                   */
  float grad_clip;                  /* always 100 in the reference (recurrent_layers.py:19)    */
  float regularization;             /* output-bias L2 (>0) / L1 (<0), rnn_one_hot.py:73-77      */
  int32_t math_mode;                /* SBR_MATH_*                                              */
  int32_t device;                   /* CUDA ordinal                                            */
  int32_t n_ranks;                  /* data-parallel world size (1 = no NCCL)                  */
  int32_t rank;
  int32_t global_batch;             /* rows over all ranks; 0 -> batch_size * n_ranks          */
  int32_t n_slots;                  /* device-resident batch slots (>=1), see sbr_stage_*      */
  int32_t bidirectional;            /* --r_bi: every depth = forward + backwards layer, concatenated (recurrent_layers.py:72-78) */
  uint8_t nccl_id[SBR_NCCL_ID_BYTES]; /* from sbr_nccl_unique_id on rank 0, shared by the host */
} sbr_config;

/* ---- life cycle ------------------------------------------------------------------------- */
SBR_API int sbr_abi_version(void);
SBR_API int sbr_device_count(void);                       /* 0 when no CUDA device is visible          */
SBR_API int sbr_nccl_unique_id(uint8_t out[SBR_NCCL_ID_BYTES]);
SBR_API int sbr_create(const sbr_config* cfg, sbr_model** out);   /* replaces _prepare_networks + _compile_* */
SBR_API void sbr_destroy(sbr_model* m);
SBR_API const char* sbr_last_error(const sbr_model* m);   /* m == NULL: error of the last failed sbr_create */

/* ---- parameters: lasagne get/set_all_param_values (rnn_base.py:476,515) ------------------ */
SBR_API int sbr_param_count(const sbr_model* m);
SBR_API int sbr_param_info(const sbr_model* m, int idx, char* name, int name_cap, int* ndim, int64_t shape[4]);
SBR_API int sbr_get_param(sbr_model* m, int idx, float* host);
SBR_API int sbr_set_param(sbr_model* m, int idx, const float* host);
SBR_API int sbr_get_grad(sbr_model* m, int idx, float* host);     /* gradient left by the last step when skip_update=1 */
SBR_API int64_t sbr_total_params(const sbr_model* m);
SBR_API int sbr_reset_optimizer(sbr_model* m);                    /* zero the updater state and its step counter */
SBR_API int sbr_set_skip_update(sbr_model* m, int flag);          /* 1: steps compute cost+gradients only (tests) */

/* ---- train_function --------------------------------------------------------------------- */
/* RNNOneHot: cost = mean_b(-log softmax(h W + b)[Y_b] / pop_b) (+ bias reg), rnn_one_hot.py:65-77.
 * On a single rank the call returns as soon as the cost is on the host; the backward pass and the update may still
 * be running on the handle's stream (every later call on the handle is ordered behind them). */
SBR_API int sbr_train_step_cce(sbr_model* m, const int32_t* X, const float* mask, const int32_t* Y,
                       const float* pop, int B, float* cost);
/* RNNSampling: cells = [Y_all; samples], rnn_sampling.py:68-91,137 and sparse_lstm.py:41-54.
 * Y_all holds the targets of the WHOLE global batch (n_all of them); this rank's rows are
 * Y_all[row_offset : row_offset+B].  Single rank: Y_all = Y, n_all = B, row_offset = 0. */
SBR_API int sbr_train_step_sampled(sbr_model* m, const int32_t* X, const float* mask, const int32_t* Y_all,
                           int n_all, int row_offset, const int32_t* samples, int S,
                           const float* pop, int B, float* cost);
/* RNNMargin with the reference's dense inputs Ymat/weight [B, n_items], rnn_margin.py:100,109 */
SBR_API int sbr_train_step_margin_dense(sbr_model* m, const int32_t* X, const float* mask, const float* Ymat,
                                const float* weight, int B, float* cost);
/* RNNMargin, ragged form of the same inputs: the device rebuilds what rnn_margin.py:121-149
 * fills -- weight = w_neg[b] everywhere, -1 on the row's targets, 0 on the items of X (when
 * exclude_seen); Y = default_target (NULL = 0) everywhere, 1 on targets, 0 on seen items. */
SBR_API int sbr_train_step_margin(sbr_model* m, const int32_t* X, const float* mask,
                          const int32_t* target_offsets /* [B+1] */, const int32_t* target_ids,
                          const float* w_neg /* [B] */, const float* default_target /* [n_items] or NULL */,
                          int exclude_seen, int B, float* cost);

/* Device-side batch assembly (SURVEY.md §8 f1; replaces the per-item python loop of rnn_one_hot.py:90-101 /
 * rnn_base.py:396-415): upload the training sequences ONCE as a CSR of ids ([total, ids_per_step] int32, offsets
 * [n_seqs+1]); a mini-batch is then B (sequence, start, length) triples -- row b reads
 * ids[offsets[seq_b] + start_b : + len_b] -- and the padded X / lengths are built on the device.  Same arithmetic and
 * same results as sbr_train_step_cce on the equivalent X / mask. */
SBR_API int sbr_dataset_upload(sbr_model* m, int n_seqs, const int32_t* offsets, const int32_t* ids);
SBR_API int sbr_train_step_cce_rows(sbr_model* m, const int32_t* seq, const int32_t* start, const int32_t* len,
                                    const int32_t* Y, const float* pop, int B, float* cost);

/* Device-resident batches (bench `value`, prefetch): stage a batch into slot s once, then step on
 * it any number of times with no host->device traffic.  cost may be NULL (no sync, no D2H). */
SBR_API int sbr_stage_cce(sbr_model* m, int slot, const int32_t* X, const float* mask, const int32_t* Y,
                  const float* pop, int B);
SBR_API int sbr_train_step_staged(sbr_model* m, int slot, float* cost);
SBR_API int sbr_synchronize(sbr_model* m, float* last_cost /* may be NULL */);

/* ---- predict_function / test_function --------------------------------------------------- */
/* scores[B, n_items]: softmax probabilities for CCE, raw linear scores otherwise; softmax != 0
 * forces a softmax (RNNSampling test function, rnn_sampling.py:143). */
SBR_API int sbr_scores(sbr_model* m, const int32_t* X, const float* mask, int B, int softmax, float* scores);
/* Fused exclude + sorted top-k on the device.  excl_* is a ragged list of ids per row (may be
 * NULL).  mode bit0: softmax first; bit1: 0 = excluded scores are multiplied by 0 (test_function,
 * rnn_base.py:201-202), 1 = set to -inf (top_k_recommendations, rnn_base.py:154-156).
 * ids_out [B, k], best first (np.argpartition(-out, range(k))[:k], rnn_base.py:159,207). */
SBR_API int sbr_topk(sbr_model* m, const int32_t* X, const float* mask, int B, const int32_t* excl_offsets,
             const int32_t* excl_ids, int k, int mode, int32_t* ids_out);

/* ---- RNNCluster (neural_networks/rnn_cluster.py) ------------------------------------------ */
/* A sampled-output RNN (BlackoutLayer, no /pop, no tanh) trained together with a soft assignment of the items to
 * clusters: selection q = h Wc (Wc [H_last, C], no bias), P = softmax(s (q + noise)); membership rows R [N, C];
 * cluster scores P act(s R[cells_c])^T with the same loss as the recommendation branch (rnn_cluster.py:222-251).
 * cluster.R and cluster.W follow out.b in the parameter, gradient and optimizer arenas, so sbr_param_*, sbr_get_grad,
 * sbr_reset_optimizer, the fused update and the one all-reduce per step cover them.  The cluster cost reaches only
 * Wc and R, the recommendation cost only the stack and out.*: one fused update over both is exactly the reference's
 * two updater instances (disjoint parameters, elementwise rules, equal step counters). */
enum { SBR_CLUSTER_SOFTMAX = 0, SBR_CLUSTER_MIX = 1, SBR_CLUSTER_SIGMOID = 2 };            /* --cluster_type */
enum { SBR_CLOSS_BLACKOUT = 0, SBR_CLOSS_CCE = 1, SBR_CLOSS_BPR = 2, SBR_CLOSS_TOP1 = 3,
       SBR_CLOSS_BPRELU = 4, SBR_CLOSS_LIN = 5 };                                          /* --loss with --clusters */
typedef struct sbr_cluster_config {
  int32_t struct_size;              /* = sizeof(sbr_cluster_config), ABI guard                 */
  int32_t n_clusters;               /* C = --clusters (>= 1)                                    */
  int32_t cluster_type;             /* SBR_CLUSTER_*                                            */
  int32_t loss;                     /* SBR_CLOSS_*, both branches (rnn_cluster.py:85-98)        */
  int32_t n_cluster_samples;        /* capacity of the separate cluster samples (--c_sampling), 0 = none */
} sbr_cluster_config;
/* cfg->loss is ignored: the model scores its outputs linearly like the sampled models (sbr_scores / sbr_topk) */
SBR_API int sbr_create_cluster(const sbr_config* cfg, const sbr_cluster_config* ccfg, sbr_model** out);
/* One step of both branches.  cells = [Y_all; samples], cluster cells = [Y_all; cluster_samples] (NULL: the samples);
 * noise [B, C] (this rank's rows) or NULL; scale = the current s.  cost and cluster_cost (may be NULL) are global means
 * over the whole batch (the cluster cost is all-reduced with the cost). */
SBR_API int sbr_train_step_cluster(sbr_model* m, const int32_t* X, const float* mask, const int32_t* Y_all, int n_all,
                                   int row_offset, const int32_t* samples, int S, const int32_t* cluster_samples, int Sc,
                                   const float* noise, float scale, int B, float* cost, float* cluster_cost);
/* Validation test function (rnn_cluster.py:327-355): score1 = softmax(h W + b) with the excluded ids multiplied by 0,
 * c = argmax(h Wc), score2 = score1 * hard[:, c] (hard = softmax / clip(softmax + sigmoid) / sigmoid of 100 R);
 * per row the top-k of both scores, c, and n_used = sum_n hard[n, c].  k <= 64. */
SBR_API int sbr_cluster_test_topk(sbr_model* m, const int32_t* X, const float* mask, int B, const int32_t* excl_offsets,
                                  const int32_t* excl_ids, int k, int32_t* ids_full, int32_t* ids_cluster,
                                  int32_t* selected, float* n_used);
/* prepare_tests (rnn_cluster.py:461-487): item n belongs to every cluster j with R[n, j] > 0, an item without a
 * positive entry to the first arg-max of its row; clusters list their items in ascending id.  Built on the device and
 * kept there; sizes [C] (may be NULL) receives the cluster sizes. */
SBR_API int sbr_cluster_build(sbr_model* m, int32_t* sizes);
/* top_k_recommendations (rnn_cluster.py:293-322).  use_clusters: c = argmax(h Wc), only the items of cluster c are
 * scored (h W[:, items] + b[items]), excluded ids are -inf, ids_out[b, :min(k, |c|)] best first (-1 beyond),
 * n_out[b] = |c|, selected_out[b] = c (may be NULL).  use_clusters = 0: the whole catalog, n_out[b] = n_items.  The
 * work scales with sum_b |cluster(b)| * H_last.  Needs sbr_cluster_build after the last parameter change. */
SBR_API int sbr_cluster_topk(sbr_model* m, const int32_t* X, const float* mask, int B, const int32_t* excl_offsets,
                             const int32_t* excl_ids, int k, int32_t* ids_out, int32_t* n_out, int32_t* selected_out,
                             int use_clusters);

/* ---- measurement ------------------------------------------------------------------------ */
#define SBR_N_STAGES 9
SBR_API const char* sbr_stage_name(int i);            /* "h2d","gather","rnn_fwd","output","rnn_bwd","wgrad","scatter","allreduce","optimizer" */
SBR_API int sbr_set_profiling(sbr_model* m, int on);  /* record a cudaEvent pair around every stage */
SBR_API int sbr_stage_times(sbr_model* m, float ms[SBR_N_STAGES]);   /* of the last profiled step   */
SBR_API int64_t sbr_kernel_launches(const sbr_model* m);             /* kernels launched since create */
/* Host-only: how the tcgen05 scan launchers would tile a batch with these lengths on `slots` co-resident 8-CTA
 * clusters (rnn_tc.cu::plan_tiles): tile height of the main launch (8 / 16 rows), its tiles in launch order (longest
 * first, order64 has room for 64), and the 16-row group that runs as a second launch in the mixed tiling (-1: none).
 * `lens` may be NULL (static rule).  Touches no device; used by the CPU tests. */
SBR_API int sbr_plan_scan_tiles(const int32_t* lens, int B, int t_max, int slots, float ratio8,
                                int* tile_rows, int* n_tiles, int* extra16, unsigned char* order64);
/* Which recurrent-scan kernel variant one layer (cell, H) runs for a batch of B rows (lengths `lens`, may be NULL) in
 * one direction, as launch_rnn_forward / launch_rnn_backward decide it.  Families, in the order they are tried: */
enum { SBR_SCAN_TC_CLUSTER = 0,   /* tcgen05 cluster scans (rnn_tc.cu): <G, BT> forward, <G, MT, BT> backward        */
       SBR_SCAN_PERSISTENT = 1,   /* persistent tensor-core scans (tc_scan.cu), sliced into co-resident launches     */
       SBR_SCAN_STEP = 2,         /* one tensor-core kernel per time step (tc_gemm.cu)                               */
       SBR_SCAN_FFMA = 3 };       /* FFMA cluster scans (rnn_cluster.cu): <G, BT, JU, WSMEM>                         */
typedef struct sbr_scan_plan {
  int32_t family;            /* SBR_SCAN_*                                                                         */
  int32_t G;                 /* gate blocks: 4 LSTM, 3 GRU, 1 Vanilla                                              */
  int32_t BT;                /* batch rows per tile of the main launch: tcgen05 8|16, FFMA 8|16|32, persistent 128
                                forward / 32 backward, 0 for the step scans                                        */
  int32_t MT;                /* tcgen05 backward: 128-unit hidden tiles, else 0                                    */
  int32_t JU;                /* FFMA: hidden units per lane (1|2), else 0                                          */
  int32_t wsmem;             /* FFMA: W_hid slice resident in shared memory                                        */
  int32_t splitk;            /* persistent backward: split-K clusters of 4 CTAs                                    */
  int32_t C, Hs;             /* hidden-unit ownership: slice r < C holds units [r*Hs, min(H, (r+1)*Hs))            */
  int32_t launches;          /* scan kernel launches of this layer and direction                                  */
  int32_t tiles_per_launch;  /* persistent: batch tiles per launch, else 0                                        */
} sbr_scan_plan;
/* m != NULL: the handle's switches, SM count and co-resident cluster counts (queried on its device); n_sm, tc_slots
 * and splitk_slots are ignored.  m == NULL: touches no device; the switches are read from the environment
 * (SBR_DISABLE_TC, SBR_DISABLE_TC_BWD, SBR_DISABLE_STEP_SCAN, SBR_DISABLE_PERSISTENT_SCAN, SBR_DISABLE_SPLITK_SCAN,
 * SBR_DISABLE_TC_GEMM, SBR_DISABLE_TMA_GEMM, SBR_TC_BT, ...) and the device is described by n_sm, tc_slots[i] =
 * co-resident tcgen05 scan clusters of 2^i CTAs (i = 0..3) and splitk_slots = co-resident split-K clusters.
 * Returns SBR_E_ARG for a layer no scan takes and under SBR_SCAN_MULTICAST.  sbr_scan_launches counts the scan
 * kernel launches of a handle (part of sbr_kernel_launches). */
SBR_API int sbr_plan_layer_scan(const sbr_model* m, int cell, int H, int B, const int32_t* lens, int t_max, int backward,
                                int n_sm, const int32_t* tc_slots, int splitk_slots, sbr_scan_plan* out);
SBR_API int64_t sbr_scan_launches(const sbr_model* m);
/* Diagnostics: C[M,N] = alpha * op(A) * op(B) (+ bias[n]) (+ beta * C) on the device the handle lives on, host buffers
 * in and out (row-major; ta: A stored [K,lda]; tb: B stored [N,ldb]; beta in {0,1}; bias may be NULL).  engine 0 = the
 * fp32 FFMA kernels (gemm.cu), 1 = the tcgen05 3xTF32 kernel (tc_gemm.cu), which is what every GEMM-shaped stage of
 * the path runs on.  Used by the GPU tests to check the tensor-core kernel against float64 in isolation; `ms` (may be
 * NULL) receives the device time of `reps` back-to-back launches. */
SBR_API int sbr_debug_gemm(sbr_model* m, int engine, int ta, int tb, int M, int N, int K, const float* A, int lda,
                           const float* B, int ldb, float* C, int ldc, float alpha, float beta, const float* bias,
                           int reps, float* ms);
/* device-side stopwatch on the handle's stream (cudaEvent pair): start synchronises the stream
 * first, stop blocks until the stop event has completed and returns the elapsed milliseconds */
SBR_API int sbr_timer_start(sbr_model* m);
SBR_API int sbr_timer_stop(sbr_model* m, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* SBR_B200_H */
