// common.cuh -- shared declarations of libsbr_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <algorithm>

#include "../../include/sbr_b200.h"

#define SBR_WARP 32
#define SBR_NSM 148  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

// ---- error plumbing -------------------------------------------------------------------------
struct sbr_model;
void sbr_set_error(sbr_model* m, int code, const char* fmt, ...);

#define CU_TRY(m, expr)                                                                 \
  do {                                                                                  \
    cudaError_t e__ = (expr);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      sbr_set_error((m), SBR_E_CUDA, "%s failed: %s (%s:%d)", #expr,                    \
                    cudaGetErrorString(e__), __FILE__, __LINE__);                       \
      return SBR_E_CUDA;                                                                \
    }                                                                                   \
  } while (0)

#define KERNEL_CHECK(m)                                                                 \
  do {                                                                                  \
    cudaError_t e__ = cudaGetLastError();                                               \
    if (e__ != cudaSuccess) {                                                           \
      sbr_set_error((m), SBR_E_CUDA, "kernel launch failed: %s (%s:%d)",                \
                    cudaGetErrorString(e__), __FILE__, __LINE__);                       \
      return SBR_E_CUDA;                                                                \
    }                                                                                   \
    (m)->launches++;                                                                    \
  } while (0)

static inline int64_t round_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }
static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- model description ----------------------------------------------------------------------
struct LayerDesc {
  int level = 0;       // depth in the stack
  int relu = 0;        // Vanilla cell fed by a dense input (Lasagne RecurrentLayer): rectifier instead of tanh
  int dir = 0;         // 0 forward layer, 1 backwards layer of a bidirectional stack (runs on row-reversed inputs)
  int H = 0;           // hidden units
  int G = 0;           // stacked gate blocks: LSTM 4 [in,forget,cell,out], GRU 3 [reset,update,hidden], Vanilla 1
  int I = 0;           // dense input width; 0 = id gather-sum layer (layer 0 without embedding)
  int in_rows = 0;     // rows of W_in (n_items + n_extra_ids for the gather layer, I otherwise)
  int64_t W_in = 0;    // arena offsets (floats)            [in_rows, G*H]
  int64_t W_hid = 0;   //                                   [H, G*H]
  int64_t b = 0;       //                                   [G*H]
  int64_t peep = 0;    // LSTM only: w_ci, w_cf, w_co       [3, H]
  int64_t c_init = 0;  // LSTM only                         [H]
  int64_t h_init = 0;  //                                   [H]
  // per-layer workspaces (time-major, row = t*B + b)
  float* Xg = nullptr;    // [T*B, G*H]  input pre-activations (gather / input GEMM + bias)
  float* act = nullptr;   // [T*B, 4*H]  saved activations (LSTM i,f,g,o | GRU r,u,cand,a_c)
  float* hs = nullptr;    // [(T+1)*B, H] hs[0] = init broadcast, hs[t+1] = state after step t
  float* cs = nullptr;    // LSTM: same for the cell state
  float* dXg = nullptr;   // [T*B, G*H]  gradient wrt Xg (zero on masked steps)
  float* dac = nullptr;   // GRU: [T*B, H] gradient wrt the candidate's hidden pre-activation (da_c)
  float* dhs = nullptr;   // [T*B, H]   gradient arriving from the layer above (nullptr for the top layer)
  // K-major, pre-split (hi | lo) copies written by the tcgen05 scans for the tensor-core weight-gradient GEMM:
  //   hT[part][h/128][row/4][h%128][row%4]  (state before each step),  aT[part][col/128][row/4][col%128][row%4]  (da)
  float* hT = nullptr;
  float* aT = nullptr;
  int64_t hT_part = 0, hT_tile = 0, aT_part = 0, aT_tile = 0;   // strides in floats
  bool kmajor_valid = false;   // set by the tc backward scan of the current step
};

struct ParamView {       // one entry of the reference checkpoint list
  std::string name;
  int ndim = 1;
  int64_t shape[4] = {1, 1, 1, 1};
  int64_t off = 0;       // arena offset of element (0,0)
  int64_t rows = 1, cols = 1;
  int64_t ld = 1;        // arena row stride
  bool transposed = false;  // arena holds the transpose ([cols, rows] with stride ld)
};

struct BatchSlot {       // device-resident inputs of one mini-batch
  int32_t* X = nullptr;       // [B, T, K]
  int32_t* len = nullptr;     // [B]
  int32_t* Y = nullptr;       // [n_all] targets (CCE: B)
  float* pop = nullptr;       // [B]
  int B = 0, t_max = 0, n_all = 0, row_offset = 0;
  std::vector<int32_t> hlen;  // host copy of len (the scan launchers schedule their cluster tiles from it)
};

struct sbr_model {
  sbr_config cfg{};
  int dev = 0;
  int n_sm = SBR_NSM;
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;        // off-critical-path work (see side_fork / side_join in model.cu)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaStream_t aux = nullptr;         // second scan launch of a mixed 8-/16-row tiling (rnn_tc.cu), concurrent with the first
  cudaEvent_t ev_aux_fork = nullptr, ev_aux_join = nullptr;
  cudaEvent_t ev_staged = nullptr;    // the H2D copies out of the pinned staging buffers have completed
  cudaEvent_t ev_cost = nullptr;      // the step's cost has landed in h_cost (recorded right after the loss kernels)
  bool cost_early = false;            // this step's cost was copied out early: finish_step() waits on ev_cost only
  bool side_pending = false;
  int deferred_out_B = 0;             // >0: output-layer weight gradients still to be launched on the side stream
  bool staging_in_flight = false;     // pinned staging buffers still feed an H2D copy
  std::string err;
  int err_code = 0;
  int64_t launches = 0;
  int64_t scan_launches = 0;          // of these, launches of a recurrent-scan kernel (all four families)

  // geometry
  int B = 0, T = 0, K = 1, N = 0, n_in = 0, E = 0, L = 0, H_last = 0;
  int nd = 1;              // directional layers per depth (2 with --r_bi); layers[level * nd + dir]
  int global_batch = 0;
  std::vector<LayerDesc> layers;
  std::vector<ParamView> views;

  // flat arenas (one allocation each => one all-reduce, one fused optimizer launch)
  int64_t P = 0;           // number of parameters
  int64_t P_pad = 0;       // arena length (16B-aligned blocks + cost slot)
  int64_t cost_slot = 0;   // index of the cost scalar inside the gradient arena
  float* params = nullptr;
  float* grads = nullptr;
  float* opt_a = nullptr;
  float* opt_b = nullptr;
  int64_t opt_t = 0;
  int64_t emb_W = 0, out_WT = 0, out_b = 0;   // arena offsets; out_WT is [N, H_last] (item-major)

  // workspaces
  std::vector<BatchSlot> slots;
  float* emb_out = nullptr;   // [T*B, K*E]
  float* demb = nullptr;
  // bidirectional stacks: the backwards layers run the forward-only scan kernels on rows whose valid prefix is reversed
  bool on_side = false;     // launchers are currently enqueuing on the side stream (work that overlaps a cluster scan)
  int* wg_list = nullptr; int wg_list_rows = 0;   // wgrad_tc: [1 + T*B/32] stages of the contraction holding valid rows (this batch)
  int32_t* X_rev = nullptr;   // [B, T, K] ids with every row's valid prefix reversed
  float* emb_out_rv = nullptr; float* demb_rv = nullptr;       // embedding path in reversed coordinates
  float* cat_al = nullptr;    // [T*B, 2*maxH] level output [forward | backward] aligned with the input positions
  float* cat_rv = nullptr;    // [T*B, 2*maxH] the same in reversed coordinates (input of the backwards layers)
  float* dcat_al = nullptr; float* dcat_rv = nullptr;          // their gradients
  float* h_last_dir = nullptr; float* dh_last_dir = nullptr;   // [2][B, H_top] per-direction final states / gradients
  float* h_last = nullptr;    // [B, H_last]
  float* dh_last = nullptr;   // [B, H_last]
  float* logits = nullptr;    // [B, max(N, n_all+S)]
  float* row_loss = nullptr;  // [B]
  float* WhidT = nullptr;     // scratch transpose of the largest W_hid (global-memory fallback of the bwd kernel)
  // margin / sampled
  float* mY = nullptr;        // [B, N]
  float* mW = nullptr;        // [B, N]
  int32_t* cells = nullptr;   // [n_all + S]
  float* Wc = nullptr;        // [n_all+S, H_last] gathered output rows
  float* dWc = nullptr;
  float* bc = nullptr;        // gathered output bias [n_all+S]
  int32_t* tgt_off = nullptr; // ragged margin targets
  int32_t* tgt_ids = nullptr;
  float* w_neg = nullptr;
  float* def_tgt = nullptr;
  int tgt_cap = 0;
  // RNNCluster (sbr_create_cluster): cluster.R [N, C] and cluster.W [H_last, C] follow out.b in the arenas
  int n_clusters = 0;         // 0: not a cluster model
  int cluster_type = 0;       // SBR_CLUSTER_*
  int cluster_loss = 0;       // sampling_loss_kernel code of the SBR_CLOSS_* of both branches
  int n_csamples = 0;         // capacity of the cluster-sample vector
  int64_t cl_R = 0, cl_W = 0; // arena offsets
  int32_t* ccells = nullptr;  // [n_all + Sc] cluster cells = [Y_all; cluster samples]
  float* cq = nullptr;        // [B, C] h Wc
  float* cnoise = nullptr;    // [B, C] selection noise of this rank's rows
  float* cP = nullptr;        // [B, C] scaled selection softmax
  float* cdP = nullptr;       // [B, C]
  float* cdq = nullptr;       // [B, C]
  float* cM = nullptr;        // [n_all + Sc, C] membership rows
  float* cdM = nullptr;
  float* cS = nullptr;        // [B, n_all + Sc] cluster scores, then their gradient
  float* crow_loss = nullptr; // [B]
  int32_t* csel = nullptr;    // [B] selected cluster per row
  float* cnused = nullptr;    // [B] items of the hard column per row
  int32_t* cperm = nullptr;   // [B] rows grouped by selected cluster
  float* ch_sorted = nullptr; // [B, H_last] final states in that order
  float* clse = nullptr;      // [N] logsumexp of 100 R per item
  float* logits2 = nullptr;   // [B, N] cluster-weighted test scores (allocated on first use)
  // item CSR of the hard clusters (sbr_cluster_build), device resident
  int32_t* cl_off = nullptr;  // [C + 1]
  int32_t* cl_items = nullptr;
  int32_t* cl_fb = nullptr;   // [N] fallback cluster of an item without a positive entry (-1: has one)
  int32_t* cl_cnt = nullptr;  // [chunks, C] counts, then offsets inside the cluster
  float* cl_Wg = nullptr;     // [max cluster size, H_last] gathered output rows of one cluster
  std::vector<int32_t> cl_hoff;   // host copy of cl_off (empty: not built)
  int64_t cl_cap_items = 0;   // allocated lengths of cl_items / rows of cl_Wg
  int cl_cap_rows = 0;
  // top-k
  int32_t* excl_off = nullptr;
  int32_t* excl_ids = nullptr;
  int excl_cap = 0;
  int32_t* topk_ids = nullptr;
  // device-side batch assembly: the training sequences as a CSR of ids
  int32_t* ds_off = nullptr;          // [ds_n + 1]
  int32_t* ds_ids = nullptr;          // [total, K]
  int32_t* ds_rows = nullptr;         // [3, B] (sequence, start, length) triples of the current batch
  int ds_n = 0;
  std::vector<int32_t> ds_hoff;       // host copy of the offsets (argument validation)
  // host staging (pinned)
  int32_t* h_len = nullptr;
  const int32_t* cur_hlen = nullptr;  // host lengths of the batch being processed (BatchSlot::hlen), may be null
  float* h_cost = nullptr;
  void* h_stage = nullptr;
  size_t h_stage_bytes = 0;

  // per-step tensor-core scans (tc_gemm.cu): carried gradient state of the BPTT steps
  float* step_carry = nullptr;   // [B, maxH]
  float* step_dcs = nullptr;     // [B, maxH]
  float* step_dpe = nullptr;     // [3][B, maxH]
  unsigned int* scan_sync = nullptr;   // persistent scans (tc_scan.cu): one release/acquire counter per batch tile
  bool bwd_did_bias = false;     // the last BPTT launcher accumulated the bias gradient itself (else: column sum of dXg)
  // switches read once from the environment at sbr_create (diagnostics / A-B tests)
  bool use_tc_gemm = true;       // SBR_DISABLE_TC_GEMM: FFMA GEMMs everywhere
  bool use_step_scan = true;
  bool use_persistent_scan = true;   // SBR_DISABLE_PERSISTENT_SCAN: one launch per time step instead of the cooperative scans
  bool use_scan_multicast = false; // SBR_SCAN_MULTICAST=1: clusters of 4 forward-scan CTAs share the h tile through TMA multicast (measured: no faster, the loads are not the limiter)
  bool use_splitk_scan = true;   // SBR_DISABLE_SPLITK_SCAN: one CTA per BPTT tile instead of a split-K cluster of 4
  int scan_fence_mode = 3;       // SBR_SCAN_FENCE: how the persistent scans publish a step (tc_scan.cu::publish_step)
  bool use_tma_gemm = true;      // SBR_DISABLE_TMA_GEMM: cp.async loaders in tc_gemm.cu even where a tensor map is possible
  bool no_side_stream = false, no_early_cost = false, disable_tc = false, disable_tc_bwd = false;   // SBR_NO_SIDE_STREAM, SBR_NO_EARLY_COST, SBR_DISABLE_TC, SBR_DISABLE_TC_BWD     // SBR_DISABLE_STEP_SCAN: FFMA cluster scans for hidden sizes beyond the tcgen05 cluster kernels

  // nccl
  void* nccl_comm = nullptr;
  bool grads_from_nccl = false;       // gradient arena allocated by ncclMemAlloc and registered with the communicator
  void* nccl_reg_handle = nullptr;

  // profiling
  bool profiling = false;
  bool skip_update = false;
  bool grads_dirty = false;            // the arena holds gradients of an inspection step (skip_update just went 1 -> 0)
  cudaEvent_t ev[SBR_N_STAGES + 1] = {};
  cudaEvent_t timer[2] = {};
  float stage_ms[SBR_N_STAGES] = {};
};

// ---- kernel launchers (defined in the .cu files) ---------------------------------------------
// gather_scatter.cu
int launch_gather_rows(sbr_model* m, const int32_t* X, const int32_t* len, const float* W, const float* bias,
                       float* out, int B, int T, int K, int ncols, int t_max, int n_rows_table);
int launch_scatter_add_rows(sbr_model* m, const int32_t* X, const int32_t* len, const float* dOut, float* dW,
                            int B, int T, int K, int ncols, int t_max);
int launch_colsum(sbr_model* m, const float* A, int rows, int cols, int ld, float* out /* += */);
int launch_gather_table_rows(sbr_model* m, const float* table, const float* bias, const int32_t* ids, int n_ids,
                             int ncols, float* out_rows, float* out_bias);
int launch_scatter_table_rows(sbr_model* m, const float* rows, const float* brow, const int32_t* ids, int n_ids,
                              int ncols, float* table_grad, float* bias_grad);
// bidirectional plumbing (gather_scatter.cu)
int launch_reverse_ids(sbr_model* m, const int32_t* X, const int32_t* len, int32_t* X_rev, int B, int T, int K);
int launch_bi_concat(sbr_model* m, const float* hs_f, const float* hs_b, const int32_t* len, float* cat_al, float* cat_rv,
                     int B, int t_max, int H);
int launch_bi_split(sbr_model* m, const float* dcat_al, const float* dcat_rv, const int32_t* len, float* dhs_f, float* dhs_b,
                    int B, int t_max, int H);
int launch_transpose(sbr_model* m, const float* in, int rows, int cols, int ld_in, float* out);
int launch_embed_gather(sbr_model* m, const int32_t* X, const int32_t* len, const float* table, float* out,
                        int B, int T, int K, int E, int t_max);
int launch_embed_scatter(sbr_model* m, const int32_t* X, const int32_t* len, const float* dOut, float* dTable,
                         int B, int T, int K, int E, int t_max);

// rnn_cluster.cu
int launch_rnn_forward(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last);
int launch_rnn_backward(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max,
                        const float* dh_last /* top layer, else nullptr */);

// Scan dispatch switches of one handle (sbr_create reads them from the environment); sbr_plan_layer_scan without a
// handle reads the same variables when it is called.
struct ScanSwitches {
  bool tc_gemm = true, step = true, persistent = true, tma_gemm = true, splitk = true, multicast = false;
  bool disable_tc_bwd = false;
};
ScanSwitches scan_switches(const sbr_model* m);
ScanSwitches scan_switches_from_env();

// rnn_tc.cu (returns 1 when the tcgen05 path does not apply)
int launch_rnn_forward_tc(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last);
int launch_rnn_backward_tc(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, const float* dh_last);
int tc_scan_applies(int G, int H);   // 1 when both tcgen05 scans handle this layer shape
// The decisions of the two tcgen05 launchers, for sbr_plan_layer_scan: the cluster shape of a layer (ok = false when
// tc_plan rejects it; bwd_ok: the backward fits TMEM too), the co-resident clusters of that shape on the current device,
// and the tile schedule of a batch.
struct TcShape { bool ok, bwd_ok; int C, Hs, MT; };
TcShape tc_scan_shape(int G, int H);
int tc_scan_slots(int G, int H);
void tc_scan_schedule(const int32_t* hl, int B, int t_max, int slots, bool backward, int* tile_rows, int* n_launches);

// wgrad_tc.cu : dW_hid[H, G*H] += sum_rows h_prev[row]^T da[row] on tcgen05 (3xTF32) from the K-major copies
int launch_wgrad_stage_list(sbr_model* m, const int32_t* len, int B, int rows);
int launch_wgrad_tc(sbr_model* m, const LayerDesc& L, int rows, float* dW, int ldw);

// tc_gemm.cu : the same product on tcgen05 (3xTF32, operands split on the fly); returns 1 when it does not apply
int launch_gemm_tc(sbr_model* m, bool ta, bool tb, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                   float* C, int ldc, float alpha, float beta, const float* bias);
// per-step tensor-core scans for hidden sizes the cluster-resident kernels do not hold
int step_scan_applies(const sbr_model* m, int G, int H);
int step_scan_applies(const ScanSwitches& s, int H);
int launch_rnn_forward_steps(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last);
int launch_rnn_backward_steps(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, const float* dh_last);
// tc_scan.cu : the same scans as ONE cooperative launch per layer (return 1 when they do not apply)
int persistent_scan_applies(const sbr_model* m, int G, int H);
int persistent_scan_applies(const ScanSwitches& s, int H);
// How the persistent launchers slice a batch: tiles of `tile_rows` rows (128 forward, 32 backward), at most
// `tiles_per_launch` of them per launch so that every CTA of a launch is co-resident; owner = hidden units per CTA slice
// (8 forward, 128 backward).  splitk_slots = co-resident 4-CTA split-K clusters (persistent_splitk_slots()).
struct PersistentSlicing { int tile_rows, n_tiles, tiles_per_launch, owner; bool splitk; };
PersistentSlicing persistent_fwd_slicing(int n_sm, int H, int B);
PersistentSlicing persistent_bwd_slicing(int n_sm, int H, int B, bool use_splitk, int splitk_slots);
int persistent_splitk_slots();
int launch_rnn_forward_persistent(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last);
int launch_rnn_backward_persistent(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, const float* dh_last);

// gemm.cu : C[M,N] = alpha * op(A)[M,K] * op(B)[K,N] + beta * C   (row-major, beta in {0,1})
int launch_gemm(sbr_model* m, bool ta, bool tb, int M, int N, int K, const float* A, int lda, const float* B,
                int ldb, float* C, int ldc, float alpha, float beta);
// C = A * op(B) + bias[n] broadcast over the rows (input GEMMs: Xg = in W_in + b)
int launch_gemm_bias(sbr_model* m, bool tb, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                     float* C, int ldc, const float* bias);

// loss.cu
int launch_cce(sbr_model* m, float* logits, int ld, const float* bias, const int32_t* Y, const float* pop, int B,
               int N, float inv_global_batch, float* row_loss);
int launch_softmax_rows(sbr_model* m, float* logits, int ld, const float* bias, int B, int N);
int launch_add_bias_rows(sbr_model* m, float* logits, int ld, const float* bias, int B, int N);
int launch_sampling_loss(sbr_model* m, int loss, bool tanh_out, float* A, int ld, const float* bias_cells,
                         const float* pop, int B, int n_all, int row_offset, int S, float inv_global_batch,
                         float* row_loss);
int launch_margin_loss(sbr_model* m, int loss, float* pred, int ld, const float* bias, const float* Y,
                       const float* W, int B, int N, float inv_global_batch, float* row_loss);
int launch_margin_loss_ragged(sbr_model* m, int loss, float* pred, int ld, const float* bias, const int32_t* toff,
                              const int32_t* tids, const int32_t* X, const int32_t* len, const float* w_neg,
                              const float* def_tgt, int exclude_seen, int B, int T, int K, int N, int max_special,
                              float inv_gb, float* row_loss);
int launch_margin_fill(sbr_model* m, float* Y, float* W, const int32_t* X, const int32_t* len, const int32_t* toff,
                       const int32_t* tids, const float* w_neg, const float* def_tgt, int exclude_seen, int B,
                       int T, int K, int N);
int launch_bias_reg(sbr_model* m, const float* b, float* db, int N, float reg, float* cost_acc);
int launch_reduce_cost(sbr_model* m, const float* row_loss, int B, float* cost_acc);
int launch_topk(sbr_model* m, float* scores, int ld, int B, int N, const int32_t* excl_off, const int32_t* excl_ids,
                int k, int neg_inf, int32_t* ids_out);

// optim.cu
int launch_optimizer(sbr_model* m);

// sampling_loss_kernel codes used only by the cluster model (never accepted by sbr_create): the sampled softmax
// cross-entropy, the leaky-rectified BPR and the linear loss of rnn_cluster.py:158-175
enum { SBR_LK_SCCE = 100, SBR_LK_BPRELU = 101, SBR_LK_LIN = 102 };

// cluster.cu : the cluster branch of RNNCluster (rnn_cluster.py:232-251) and its test paths
int launch_cluster_select(sbr_model* m, const float* q, const float* noise, int B, int C, float scale, float* P);
int launch_cluster_members(sbr_model* m, const float* R, const int32_t* cells, int n, int C, int type, float scale, float* M);
int launch_cluster_dq(sbr_model* m, const float* P, const float* dP, int B, int C, float scale, float* dq);
int launch_cluster_dR(sbr_model* m, const float* R, const int32_t* cells, int n, int C, int type, float scale,
                      const float* dM, float* gR);
int launch_cluster_hard(sbr_model* m, const float* scores, int ld, const float* q, const float* R, int B, int N, int C,
                        int type, float* scores2, int32_t* sel, float* n_used);
int launch_cluster_argmax(sbr_model* m, const float* q, int B, int C, int32_t* sel);
int launch_cluster_csr(sbr_model* m, const float* R, int N, int C);    // fallback, counts, m->cl_off
int launch_cluster_fill(sbr_model* m, const float* R, int N, int C);   // m->cl_items (sized from m->cl_off[C])
int launch_cluster_row_topk(sbr_model* m, float* scores, int ld, int B, const int32_t* perm, const int32_t* sel,
                            const float* bias, const int32_t* excl_off, const int32_t* excl_ids, int k, int32_t* ids_out);
