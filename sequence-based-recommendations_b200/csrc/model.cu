// model.cu -- the C ABI of libsbr_b200.so (include/sbr_b200.h): handle life cycle, the flat
// parameter / gradient arenas, batch staging, and the orchestration of one training step
//
//     gather -> recurrent scan -> catalog projection + loss -> BPTT -> scatter -> all-reduce -> update
//
// which replaces the single `cost = self.train_function(*batch)` call of the reference
// (neural_networks/rnn_base.py:290; graph built at rnn_one_hot.py:37-77, rnn_sampling.py:93-137,
// rnn_margin.py:70-109, compiled at rnn_base.py:175-186).
#include <dlfcn.h>
#include <nccl.h>
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_create_error;

void sbr_set_error(sbr_model* m, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (m) {
    // CUDA / NCCL errors are sticky: keep the first one
    if (m->err_code == SBR_E_CUDA || m->err_code == SBR_E_NCCL) return;
    m->err = buf;
    m->err_code = code;
  } else {
    g_create_error = buf;
  }
}

#define CHECK_STICKY(m)                                                     \
  do {                                                                      \
    if (!(m)) return SBR_E_ARG;                                             \
    if ((m)->err_code == SBR_E_CUDA || (m)->err_code == SBR_E_NCCL) return (m)->err_code; \
  } while (0)

// ------------------------------------------------------------------------------------------------
// NCCL through dlopen: the library is only needed when n_ranks > 1
// ------------------------------------------------------------------------------------------------
namespace {
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  // optional (NCCL >= 2.19): user-buffer registration, so that the gradient arena is all-reduced in place through
  // NVLink SHARP / NVLS instead of being staged through NCCL's internal buffers
  ncclResult_t (*MemAlloc)(void**, size_t) = nullptr;
  ncclResult_t (*MemFree)(void*) = nullptr;
  ncclResult_t (*CommRegister)(const ncclComm_t, void*, size_t, void**) = nullptr;
  ncclResult_t (*CommDeregister)(const ncclComm_t, void*) = nullptr;
};
NcclApi g_nccl;

bool load_nccl(std::string* why) {
  if (g_nccl.lib) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) {
    *why = std::string("cannot dlopen libnccl.so.2: ") + dlerror();
    return false;
  }
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(g_nccl.lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(g_nccl.lib, "ncclCommInitRank");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(g_nccl.lib, "ncclAllReduce");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(g_nccl.lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(g_nccl.lib, "ncclGetErrorString");
  g_nccl.MemAlloc = (decltype(g_nccl.MemAlloc))dlsym(g_nccl.lib, "ncclMemAlloc");
  g_nccl.MemFree = (decltype(g_nccl.MemFree))dlsym(g_nccl.lib, "ncclMemFree");
  g_nccl.CommRegister = (decltype(g_nccl.CommRegister))dlsym(g_nccl.lib, "ncclCommRegister");
  g_nccl.CommDeregister = (decltype(g_nccl.CommDeregister))dlsym(g_nccl.lib, "ncclCommDeregister");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy) {
    *why = "libnccl.so.2 lacks a required symbol";
    g_nccl.lib = nullptr;
    return false;
  }
  return true;
}

const char* kStageNames[SBR_N_STAGES] = {"h2d", "gather", "rnn_fwd", "output", "rnn_bwd", "wgrad", "scatter", "allreduce", "optimizer"};

// X[b, t, :] = ids[(off[seq_b] + start_b + t), :] for t < len_b (0 beyond), lengths alongside
__global__ void assemble_rows_kernel(const int32_t* __restrict__ off, const int32_t* __restrict__ ids, const int32_t* __restrict__ rows,
                                     int32_t* __restrict__ X, int32_t* __restrict__ len, int B, int T, int K) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * T * K) return;
  const int k = (int)(i % K), t = (int)((i / K) % T), b = (int)(i / ((int64_t)K * T));
  const int s = rows[b], st = rows[B + b], l = rows[2 * B + b];
  X[i] = t < l ? ids[((int64_t)off[s] + st + t) * K + k] : 0;
  if (t == 0 && k == 0) len[b] = l;
}

__global__ void fill_rows_kernel(float* __restrict__ out, const float* __restrict__ bias, int64_t rows, int cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  out[i] = bias[i % cols];
}

template <typename T>
int dev_alloc(sbr_model* m, T** p, size_t n, bool zero = true) {
  if (n == 0) n = 1;
  CU_TRY(m, cudaMalloc((void**)p, n * sizeof(T)));
  if (zero) CU_TRY(m, cudaMemset(*p, 0, n * sizeof(T)));
  return 0;
}

void stage_mark(sbr_model* m, int i) {
  if (m->profiling) cudaEventRecord(m->ev[i], m->stream);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// life cycle
// ------------------------------------------------------------------------------------------------
extern "C" int sbr_abi_version(void) { return SBR_ABI_VERSION; }

extern "C" int sbr_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" int sbr_nccl_unique_id(uint8_t out[SBR_NCCL_ID_BYTES]) {
  std::string why;
  if (!load_nccl(&why)) {
    sbr_set_error(nullptr, SBR_E_NCCL, "%s", why.c_str());
    return SBR_E_NCCL;
  }
  ncclUniqueId id;
  static_assert(sizeof(ncclUniqueId) == SBR_NCCL_ID_BYTES, "nccl id size");
  ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) {
    sbr_set_error(nullptr, SBR_E_NCCL, "ncclGetUniqueId: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
    return SBR_E_NCCL;
  }
  memcpy(out, &id, SBR_NCCL_ID_BYTES);
  return 0;
}

extern "C" const char* sbr_last_error(const sbr_model* m) { return m ? m->err.c_str() : g_create_error.c_str(); }

static int64_t take(int64_t& off, int64_t n) {
  const int64_t o = off;
  off = round_up(off + n, 4);
  return o;
}

static void add_view(sbr_model* m, const std::string& name, int ndim, int64_t s0, int64_t s1, int64_t off,
                     int64_t rows, int64_t cols, int64_t ld, bool transposed = false) {
  ParamView v;
  v.name = name; v.ndim = ndim; v.shape[0] = s0; v.shape[1] = s1;
  v.off = off; v.rows = rows; v.cols = cols; v.ld = ld; v.transposed = transposed;
  m->views.push_back(v);
}

static int build_layout(sbr_model* m) {
  const sbr_config& c = m->cfg;
  int64_t off = 0;
  m->P = 0;
  if (m->E > 0) {
    m->emb_W = take(off, (int64_t)m->n_in * m->E);
    m->P += (int64_t)m->n_in * m->E;
    add_view(m, "emb.W", 2, m->n_in, m->E, m->emb_W, m->n_in, m->E, m->E);
  }
  int n_inputs = m->E > 0 ? m->E * m->K : m->n_in;
  for (int li = 0; li < m->L; ++li) {
   for (int dir = 0; dir < m->nd; ++dir) {       // bidirectional: the forward layer's parameters, then the backwards layer's
    LayerDesc L;
    L.level = li; L.dir = dir;
    L.H = c.layers[li];
    L.G = c.cell == SBR_CELL_LSTM ? 4 : (c.cell == SBR_CELL_GRU ? 3 : 1);
    L.I = (li == 0 && m->E == 0) ? 0 : n_inputs;
    L.in_rows = n_inputs;
    const int H = L.H, GH = L.G * L.H;
    const std::string pre = "l" + std::to_string(li) + (dir ? "b." : ".");
    // A Vanilla layer with a dense input is Lasagne's own RecurrentLayer (recurrent_layers.py:98-99), not the in-tree
    // sparse copy: rectifier instead of tanh, parameters listed hid_init, W_in_to_hid, b, W_hid_to_hid.
    L.relu = (c.cell == SBR_CELL_VANILLA && L.I > 0) ? 1 : 0;
    if (L.relu) {
      L.h_init = take(off, H);
      add_view(m, pre + "hid_init", 2, 1, H, L.h_init, 1, H, H);
    }
    L.W_in = take(off, (int64_t)n_inputs * GH);
    if (L.relu) {
      L.b = take(off, GH);
      L.W_hid = take(off, (int64_t)H * GH);
      add_view(m, pre + "W_in_to_hid", 2, n_inputs, H, L.W_in, n_inputs, H, GH);
      add_view(m, pre + "b", 1, H, 1, L.b, 1, H, H);
      add_view(m, pre + "W_hid_to_hid", 2, H, H, L.W_hid, H, H, GH);
      m->P += (int64_t)n_inputs * GH + (int64_t)H * GH + GH + H;
      m->layers.push_back(L);
      continue;
    }
    L.W_hid = take(off, (int64_t)H * GH);
    L.b = take(off, GH);
    m->P += (int64_t)n_inputs * GH + (int64_t)H * GH + GH;
    if (c.cell == SBR_CELL_LSTM) {
      L.peep = take(off, 3 * H);
      L.c_init = take(off, H);
      m->P += 4 * H;
    }
    L.h_init = take(off, H);
    m->P += H;
    // creation order of the gates in the reference vs. position in the stacked matrices
    struct GateRef { const char* name; int sidx; };
    std::vector<GateRef> gates;
    if (c.cell == SBR_CELL_LSTM) gates = {{"ingate", 0}, {"forgetgate", 1}, {"cell", 2}, {"outgate", 3}};
    else if (c.cell == SBR_CELL_GRU) gates = {{"updategate", 1}, {"resetgate", 0}, {"hidden_update", 2}};
    else gates = {{"hidden_update", 0}};
    for (const GateRef& g : gates) {
      add_view(m, pre + "W_in_to_" + g.name, 2, n_inputs, H, L.W_in + (int64_t)g.sidx * H, n_inputs, H, GH);
      add_view(m, pre + "W_hid_to_" + g.name, 2, H, H, L.W_hid + (int64_t)g.sidx * H, H, H, GH);
      add_view(m, pre + "b_" + g.name, 1, H, 1, L.b + (int64_t)g.sidx * H, 1, H, H);
    }
    if (c.cell == SBR_CELL_LSTM) {
      add_view(m, pre + "W_cell_to_ingate", 1, H, 1, L.peep, 1, H, H);
      add_view(m, pre + "W_cell_to_forgetgate", 1, H, 1, L.peep + H, 1, H, H);
      add_view(m, pre + "W_cell_to_outgate", 1, H, 1, L.peep + 2 * H, 1, H, H);
      add_view(m, pre + "cell_init", 2, 1, H, L.c_init, 1, H, H);
    }
    add_view(m, pre + "hid_init", 2, 1, H, L.h_init, 1, H, H);
    m->layers.push_back(L);
   }
    n_inputs = c.layers[li] * m->nd;
  }
  m->H_last = m->layers.back().H * m->nd;
  m->out_WT = take(off, (int64_t)m->N * m->H_last);
  m->out_b = take(off, m->N);
  m->P += (int64_t)m->N * m->H_last + m->N;
  add_view(m, "out.W", 2, m->H_last, m->N, m->out_WT, m->H_last, m->N, m->H_last, /*transposed=*/true);
  add_view(m, "out.b", 1, m->N, 1, m->out_b, 1, m->N, m->N);
  if (m->n_clusters > 0) {   // RNNCluster: membership rows, then the selection layer (rnn_cluster.py:235,241)
    const int C = m->n_clusters;
    m->cl_R = take(off, (int64_t)m->N * C);
    m->cl_W = take(off, (int64_t)m->H_last * C);
    m->P += (int64_t)m->N * C + (int64_t)m->H_last * C;
    add_view(m, "cluster.R", 2, m->N, C, m->cl_R, m->N, C, C);
    add_view(m, "cluster.W", 2, m->H_last, C, m->cl_W, m->H_last, C, C);
  }
  m->P_pad = round_up(off, 4);
  m->cost_slot = m->P_pad;   // just past the optimised range, still inside the all-reduced range
  return 0;
}

extern "C" void sbr_destroy(sbr_model* m) {
  if (!m) return;
  cudaSetDevice(m->dev);
  if (m->stream) cudaStreamSynchronize(m->stream);
  if (m->nccl_comm && m->nccl_reg_handle && g_nccl.CommDeregister) g_nccl.CommDeregister((ncclComm_t)m->nccl_comm, m->nccl_reg_handle);
  if (m->nccl_comm && g_nccl.CommDestroy) g_nccl.CommDestroy((ncclComm_t)m->nccl_comm);
  auto F = [](void* p) { if (p) cudaFree(p); };
  if (m->grads_from_nccl && g_nccl.MemFree) { g_nccl.MemFree(m->grads); m->grads = nullptr; }
  F(m->params); F(m->grads); F(m->opt_a); F(m->opt_b);
  for (LayerDesc& L : m->layers) { F(L.Xg); F(L.act); F(L.hs); F(L.cs); F(L.dXg); F(L.dac); F(L.dhs); F(L.hT); F(L.aT); }
  for (BatchSlot& s : m->slots) { F(s.X); F(s.len); F(s.Y); F(s.pop); }
  F(m->emb_out); F(m->demb); F(m->h_last); F(m->dh_last); F(m->logits); F(m->row_loss); F(m->WhidT); F(m->step_carry); F(m->step_dcs); F(m->step_dpe); F(m->scan_sync); F(m->ds_off); F(m->ds_ids); F(m->ds_rows); F(m->wg_list); F(m->X_rev); F(m->emb_out_rv); F(m->demb_rv); F(m->cat_al); F(m->cat_rv); F(m->dcat_al); F(m->dcat_rv); F(m->h_last_dir); F(m->dh_last_dir);
  F(m->mY); F(m->mW); F(m->cells); F(m->Wc); F(m->dWc); F(m->bc);
  F(m->ccells); F(m->cq); F(m->cnoise); F(m->cP); F(m->cdP); F(m->cdq); F(m->cM); F(m->cdM); F(m->cS); F(m->crow_loss);
  F(m->csel); F(m->cnused); F(m->cperm); F(m->ch_sorted); F(m->clse); F(m->logits2);
  F(m->cl_off); F(m->cl_items); F(m->cl_fb); F(m->cl_cnt); F(m->cl_Wg);
  F(m->tgt_off); F(m->tgt_ids); F(m->w_neg); F(m->def_tgt); F(m->excl_off); F(m->excl_ids); F(m->topk_ids);
  if (m->h_len) cudaFreeHost(m->h_len);
  if (m->h_cost) cudaFreeHost(m->h_cost);
  if (m->h_stage) cudaFreeHost(m->h_stage);
  for (auto& e : m->timer) if (e) cudaEventDestroy(e);
  for (auto& e : m->ev) if (e) cudaEventDestroy(e);
  if (m->side) { cudaStreamSynchronize(m->side); cudaStreamDestroy(m->side); }
  if (m->ev_fork) cudaEventDestroy(m->ev_fork);
  if (m->ev_join) cudaEventDestroy(m->ev_join);
  if (m->ev_staged) cudaEventDestroy(m->ev_staged);
  if (m->ev_aux_fork) cudaEventDestroy(m->ev_aux_fork);
  if (m->ev_aux_join) cudaEventDestroy(m->ev_aux_join);
  if (m->aux) cudaStreamDestroy(m->aux);
  if (m->ev_cost) cudaEventDestroy(m->ev_cost);
  if (m->stream) cudaStreamDestroy(m->stream);
  delete m;
}

ScanSwitches scan_switches_from_env() {
  ScanSwitches s;
  s.tc_gemm = getenv("SBR_DISABLE_TC_GEMM") == nullptr;
  s.step = getenv("SBR_DISABLE_STEP_SCAN") == nullptr;
  s.tma_gemm = getenv("SBR_DISABLE_TMA_GEMM") == nullptr;
  s.persistent = getenv("SBR_DISABLE_PERSISTENT_SCAN") == nullptr;
  s.splitk = getenv("SBR_DISABLE_SPLITK_SCAN") == nullptr;
  s.multicast = getenv("SBR_SCAN_MULTICAST") != nullptr;
  s.disable_tc_bwd = getenv("SBR_DISABLE_TC_BWD") != nullptr;
  return s;
}
ScanSwitches scan_switches(const sbr_model* m) {
  ScanSwitches s;
  s.tc_gemm = m->use_tc_gemm; s.step = m->use_step_scan; s.tma_gemm = m->use_tma_gemm; s.persistent = m->use_persistent_scan;
  s.splitk = m->use_splitk_scan; s.multicast = m->use_scan_multicast; s.disable_tc_bwd = m->disable_tc_bwd;
  return s;
}

static int create_impl(sbr_model* m) {
  const sbr_config& c = m->cfg;
  CU_TRY(m, cudaSetDevice(m->dev));
  cudaDeviceProp prop;
  CU_TRY(m, cudaGetDeviceProperties(&prop, m->dev));
  if (prop.major < 10) {
    sbr_set_error(m, SBR_E_NOGPU, "device %d is sm_%d%d; libsbr_b200 is built for sm_100a only", m->dev, prop.major, prop.minor);
    return SBR_E_NOGPU;
  }
  m->n_sm = prop.multiProcessorCount;
  const ScanSwitches sw = scan_switches_from_env();
  m->use_tc_gemm = sw.tc_gemm;
  m->use_step_scan = sw.step;
  m->use_tma_gemm = sw.tma_gemm;
  m->use_persistent_scan = sw.persistent;
  if (const char* e = getenv("SBR_SCAN_FENCE")) m->scan_fence_mode = atoi(e);
  m->use_splitk_scan = sw.splitk;
  m->use_scan_multicast = sw.multicast;
  m->no_side_stream = getenv("SBR_NO_SIDE_STREAM") != nullptr;
  m->no_early_cost = getenv("SBR_NO_EARLY_COST") != nullptr;
  m->disable_tc = getenv("SBR_DISABLE_TC") != nullptr;
  m->disable_tc_bwd = sw.disable_tc_bwd;
  {
    // the critical path (scans) outranks the side stream: when both have CTAs pending, the 8-CTA clusters of a scan
    // must not queue behind the output-layer weight-gradient GEMM
    int lo = 0, hi = 0;
    CU_TRY(m, cudaDeviceGetStreamPriorityRange(&lo, &hi));
    const bool prio = !getenv("SBR_NO_STREAM_PRIORITY");
    CU_TRY(m, cudaStreamCreateWithPriority(&m->stream, cudaStreamNonBlocking, prio ? hi : 0));
    CU_TRY(m, cudaStreamCreateWithPriority(&m->side, cudaStreamNonBlocking, prio ? lo : 0));
    CU_TRY(m, cudaStreamCreateWithPriority(&m->aux, cudaStreamNonBlocking, prio ? hi : 0));
  }
  CU_TRY(m, cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming));
  CU_TRY(m, cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming));
  CU_TRY(m, cudaEventCreateWithFlags(&m->ev_staged, cudaEventDisableTiming));
  CU_TRY(m, cudaEventCreateWithFlags(&m->ev_aux_fork, cudaEventDisableTiming));
  CU_TRY(m, cudaEventCreateWithFlags(&m->ev_aux_join, cudaEventDisableTiming));
  CU_TRY(m, cudaEventCreateWithFlags(&m->ev_cost, cudaEventDisableTiming));
  for (auto& e : m->ev) CU_TRY(m, cudaEventCreate(&e));
  build_layout(m);

  const size_t arena = (size_t)m->P_pad + 4;
  int rc;
  if ((rc = dev_alloc(m, &m->params, arena))) return rc;
  if (c.n_ranks > 1 && !getenv("SBR_NO_NCCL_REGISTER")) {
    // the all-reduced buffer comes from NCCL's allocator and is registered with the communicator below
    std::string why;
    if (load_nccl(&why) && g_nccl.MemAlloc && g_nccl.MemFree && g_nccl.CommRegister) {
      void* p = nullptr;
      if (g_nccl.MemAlloc(&p, arena * sizeof(float)) == ncclSuccess && p) {
        m->grads = static_cast<float*>(p);
        m->grads_from_nccl = true;
        CU_TRY(m, cudaMemset(m->grads, 0, arena * sizeof(float)));
      }
    }
  }
  if (!m->grads && (rc = dev_alloc(m, &m->grads, arena))) return rc;
  if ((rc = dev_alloc(m, &m->opt_a, arena))) return rc;
  const bool two = c.updater == SBR_UPD_ADAM || c.updater == SBR_UPD_ADADELTA;
  if ((rc = dev_alloc(m, &m->opt_b, two ? arena : 4))) return rc;

  const size_t TB = (size_t)m->T * m->B, B = m->B;
  int maxHGH = 0;
  for (size_t li = 0; li < m->layers.size(); ++li) {
    LayerDesc& L = m->layers[li];
    const size_t H = L.H, GH = (size_t)L.G * L.H;
    maxHGH = std::max<int>(maxHGH, (int)(H * GH));
    if ((rc = dev_alloc(m, &L.Xg, TB * GH))) return rc;
    if (L.G > 1 && (rc = dev_alloc(m, &L.act, TB * 4 * H))) return rc;
    if ((rc = dev_alloc(m, &L.hs, (TB + B) * H))) return rc;
    if (L.G == 4 && (rc = dev_alloc(m, &L.cs, (TB + B) * H))) return rc;
    if ((rc = dev_alloc(m, &L.dXg, TB * GH))) return rc;
    if (L.G == 3 && (rc = dev_alloc(m, &L.dac, TB * H))) return rc;
    if (L.level + 1 < m->L && (rc = dev_alloc(m, &L.dhs, TB * H))) return rc;
    // K-major pre-split copies for the tensor-core weight-gradient GEMM (only where the tcgen05 scans run)
    if (tc_scan_applies(L.G, L.H) && m->B % 16 == 0 && !m->disable_tc && !getenv("SBR_DISABLE_TC_WGRAD")) {
      const size_t rq_h = (TB + B) / 4, rq_a = TB / 4;
      const size_t mts = (H + 127) / 128, nts = (GH + 127) / 128;
      L.hT_tile = (int64_t)rq_h * 512; L.hT_part = (int64_t)mts * L.hT_tile;
      L.aT_tile = (int64_t)rq_a * 512; L.aT_part = (int64_t)nts * L.aT_tile;
      if ((rc = dev_alloc(m, &L.hT, (size_t)2 * L.hT_part))) return rc;
      if ((rc = dev_alloc(m, &L.aT, (size_t)2 * L.aT_part))) return rc;
    }
  }
  if ((rc = dev_alloc(m, &m->WhidT, (size_t)maxHGH))) return rc;
  {
    int maxH = 0;
    for (const LayerDesc& L : m->layers) if (step_scan_applies(m, L.G, L.H) && !tc_scan_applies(L.G, L.H)) maxH = std::max(maxH, L.H);
    if (maxH > 0) {
      if ((rc = dev_alloc(m, &m->step_carry, B * maxH))) return rc;
      if ((rc = dev_alloc(m, &m->step_dcs, B * maxH))) return rc;
      if ((rc = dev_alloc(m, &m->step_dpe, 3 * B * maxH))) return rc;
      if ((rc = dev_alloc(m, &m->scan_sync, B / 32 + 8))) return rc;
    }
  }
  if (m->E > 0) {
    if ((rc = dev_alloc(m, &m->emb_out, TB * m->K * m->E))) return rc;
    if ((rc = dev_alloc(m, &m->demb, TB * m->K * m->E))) return rc;
  }
  if ((rc = dev_alloc(m, &m->h_last, B * m->H_last))) return rc;
  if ((rc = dev_alloc(m, &m->dh_last, B * m->H_last))) return rc;
  if ((rc = dev_alloc(m, &m->wg_list, 2 + TB / 32))) return rc;
  if (m->nd == 2) {
    size_t maxH = 0;
    for (const LayerDesc& L : m->layers) maxH = std::max<size_t>(maxH, L.H);
    if ((rc = dev_alloc(m, &m->X_rev, TB * m->K))) return rc;
    if ((rc = dev_alloc(m, &m->h_last_dir, 2 * B * maxH))) return rc;
    if ((rc = dev_alloc(m, &m->dh_last_dir, 2 * B * maxH))) return rc;
    if (m->L > 1) {
      if ((rc = dev_alloc(m, &m->cat_al, TB * 2 * maxH))) return rc;
      if ((rc = dev_alloc(m, &m->cat_rv, TB * 2 * maxH))) return rc;
      if ((rc = dev_alloc(m, &m->dcat_al, TB * 2 * maxH))) return rc;
      if ((rc = dev_alloc(m, &m->dcat_rv, TB * 2 * maxH))) return rc;
    }
    if (m->E > 0) {
      if ((rc = dev_alloc(m, &m->emb_out_rv, TB * m->K * m->E))) return rc;
      if ((rc = dev_alloc(m, &m->demb_rv, TB * m->K * m->E))) return rc;
    }
  }
  const bool sampled = (c.loss >= SBR_LOSS_BPR && c.loss <= SBR_LOSS_BLACKOUT) || m->n_clusters > 0;
  const bool margin = c.loss >= SBR_LOSS_HINGE;
  const size_t n_cells = (size_t)m->global_batch + std::max(1, c.n_samples);
  // rows padded to a multiple of 4 floats: 16-byte row pitch, so the score matrix can be a TMA operand of the gradient GEMMs
  if ((rc = dev_alloc(m, &m->logits, B * (size_t)round_up(std::max<size_t>(m->N, n_cells), 4)))) return rc;
  if ((rc = dev_alloc(m, &m->row_loss, B))) return rc;
  if (sampled) {
    if ((rc = dev_alloc(m, &m->cells, n_cells))) return rc;
    if ((rc = dev_alloc(m, &m->Wc, n_cells * m->H_last))) return rc;
    if ((rc = dev_alloc(m, &m->dWc, n_cells * m->H_last))) return rc;
    if ((rc = dev_alloc(m, &m->bc, 2 * n_cells))) return rc;
  }
  if (m->n_clusters > 0) {
    const size_t C = m->n_clusters, ncc = (size_t)m->global_batch + m->n_csamples, H = m->H_last;
    if ((rc = dev_alloc(m, &m->ccells, ncc))) return rc;
    if ((rc = dev_alloc(m, &m->cq, B * C))) return rc;
    if ((rc = dev_alloc(m, &m->cnoise, B * C))) return rc;
    if ((rc = dev_alloc(m, &m->cP, B * C))) return rc;
    if ((rc = dev_alloc(m, &m->cdP, B * C))) return rc;
    if ((rc = dev_alloc(m, &m->cdq, B * C))) return rc;
    if ((rc = dev_alloc(m, &m->cM, ncc * C))) return rc;
    if ((rc = dev_alloc(m, &m->cdM, ncc * C))) return rc;
    if ((rc = dev_alloc(m, &m->cS, B * (size_t)round_up(ncc, 4)))) return rc;
    if ((rc = dev_alloc(m, &m->crow_loss, B))) return rc;
    if ((rc = dev_alloc(m, &m->csel, B))) return rc;
    if ((rc = dev_alloc(m, &m->cnused, B))) return rc;
    if ((rc = dev_alloc(m, &m->cperm, B))) return rc;
    if ((rc = dev_alloc(m, &m->ch_sorted, B * H))) return rc;
    if ((rc = dev_alloc(m, &m->clse, m->N))) return rc;
    if ((rc = dev_alloc(m, &m->cl_off, C + 1))) return rc;
    if ((rc = dev_alloc(m, &m->cl_fb, m->N))) return rc;
    if ((rc = dev_alloc(m, &m->cl_cnt, (size_t)cdiv(m->N, 256) * C))) return rc;
  }
  if (margin) {
    // the dense [B, n_items] target / weight matrices of the reference exist only for callers of the dense entry point
    // (sbr_train_step_margin_dense allocates them on first use); the ragged entry point never materialises them
    if ((rc = dev_alloc(m, &m->tgt_off, B + 1))) return rc;
    if ((rc = dev_alloc(m, &m->w_neg, B))) return rc;
    if ((rc = dev_alloc(m, &m->def_tgt, m->N))) return rc;
  }
  if ((rc = dev_alloc(m, &m->excl_off, B + 1))) return rc;
  if ((rc = dev_alloc(m, &m->topk_ids, B * 64))) return rc;
  m->slots.resize(std::max(1, c.n_slots));
  for (BatchSlot& s : m->slots) {
    if ((rc = dev_alloc(m, &s.X, TB * m->K))) return rc;
    if ((rc = dev_alloc(m, &s.len, B))) return rc;
    if ((rc = dev_alloc(m, &s.Y, std::max<size_t>(B, m->global_batch)))) return rc;
    if ((rc = dev_alloc(m, &s.pop, B))) return rc;
  }
  CU_TRY(m, cudaMallocHost((void**)&m->h_len, (B + 1) * sizeof(int32_t)));
  CU_TRY(m, cudaMallocHost((void**)&m->h_cost, 4 * sizeof(float)));
  m->h_stage_bytes = TB * m->K * sizeof(int32_t);
  CU_TRY(m, cudaMallocHost(&m->h_stage, m->h_stage_bytes));
  CU_TRY(m, cudaEventCreate(&m->timer[0]));
  CU_TRY(m, cudaEventCreate(&m->timer[1]));

  if (c.n_ranks > 1) {
    std::string why;
    if (!load_nccl(&why)) {
      sbr_set_error(m, SBR_E_NCCL, "%s", why.c_str());
      return SBR_E_NCCL;
    }
    ncclUniqueId id;
    memcpy(&id, c.nccl_id, SBR_NCCL_ID_BYTES);
    ncclComm_t comm;
    ncclResult_t r = g_nccl.CommInitRank(&comm, c.n_ranks, id, c.rank);
    if (r != ncclSuccess) {
      sbr_set_error(m, SBR_E_NCCL, "ncclCommInitRank(rank %d/%d): %s", c.rank, c.n_ranks,
                    g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
      return SBR_E_NCCL;
    }
    m->nccl_comm = comm;
    if (m->grads_from_nccl) {
      void* handle = nullptr;
      if (g_nccl.CommRegister(comm, m->grads, ((size_t)m->P_pad + 4) * sizeof(float), &handle) == ncclSuccess) m->nccl_reg_handle = handle;
    }
  }
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  CU_TRY(m, cudaDeviceSynchronize());
  return 0;
}

static int create_model(const sbr_config* cfg, const sbr_cluster_config* ccfg, sbr_model** out);

extern "C" int sbr_create(const sbr_config* cfg, sbr_model** out) { return create_model(cfg, nullptr, out); }

extern "C" int sbr_create_cluster(const sbr_config* cfg, const sbr_cluster_config* ccfg, sbr_model** out) {
  if (!cfg || !ccfg || !out) { sbr_set_error(nullptr, SBR_E_ARG, "null argument"); return SBR_E_ARG; }
  *out = nullptr;
  if (ccfg->struct_size != (int32_t)sizeof(sbr_cluster_config)) {
    sbr_set_error(nullptr, SBR_E_ARG, "sbr_cluster_config.struct_size %d != %zu (ABI mismatch)", ccfg->struct_size, sizeof(sbr_cluster_config));
    return SBR_E_ARG;
  }
  auto bad = [&](const char* what) { sbr_set_error(nullptr, SBR_E_ARG, "unsupported cluster configuration: %s", what); return SBR_E_ARG; };
  if (ccfg->n_clusters < 1) return bad("n_clusters must be >= 1");
  if (ccfg->cluster_type < SBR_CLUSTER_SOFTMAX || ccfg->cluster_type > SBR_CLUSTER_SIGMOID) return bad("cluster_type");
  if (ccfg->loss < SBR_CLOSS_BLACKOUT || ccfg->loss > SBR_CLOSS_LIN) return bad("loss");
  if (ccfg->n_cluster_samples < 0) return bad("n_cluster_samples");
  if (cfg->n_samples < 1) return bad("n_samples must be >= 1");
  sbr_config c = *cfg;
  c.loss = SBR_LOSS_BLACKOUT;   // linear outputs, sampled-column buffers; the cluster loss is kept apart
  c.last_layer_tanh = 0;
  return create_model(&c, ccfg, out);
}

static int create_model(const sbr_config* cfg, const sbr_cluster_config* ccfg, sbr_model** out) {
  if (!cfg || !out) { sbr_set_error(nullptr, SBR_E_ARG, "null argument"); return SBR_E_ARG; }
  *out = nullptr;
  if (cfg->struct_size != (int32_t)sizeof(sbr_config)) {
    sbr_set_error(nullptr, SBR_E_ARG, "sbr_config.struct_size %d != %zu (ABI mismatch)", cfg->struct_size, sizeof(sbr_config));
    return SBR_E_ARG;
  }
  auto bad = [&](const char* what) { sbr_set_error(nullptr, SBR_E_ARG, "unsupported configuration: %s", what); return SBR_E_ARG; };
  if (cfg->cell < 0 || cfg->cell > SBR_CELL_VANILLA) return bad("cell");
  if (cfg->n_layers < 1 || cfg->n_layers > SBR_MAX_LAYERS) return bad("n_layers");
  if (cfg->bidirectional != 0 && cfg->bidirectional != 1) return bad("bidirectional must be 0 or 1");
  for (int i = 0; i < cfg->n_layers; ++i)
    if (cfg->layers[i] < 1 || cfg->layers[i] > 512) return bad("layer size must be in [1, 512]");
  if (cfg->n_items < 1 || cfg->n_extra_ids < 0 || cfg->ids_per_step < 1 || cfg->embedding < 0) return bad("sizes");
  if (cfg->max_length < 1 || cfg->batch_size < 1) return bad("max_length / batch_size");
  if (cfg->loss < 0 || cfg->loss > SBR_LOSS_LOGSIG) return bad("loss");
  if (cfg->updater < 0 || cfg->updater > SBR_UPD_NESTEROV) return bad("updater");
  if (cfg->n_ranks < 1 || cfg->rank < 0 || cfg->rank >= cfg->n_ranks) return bad("rank / n_ranks");
  if (cfg->math_mode != SBR_MATH_FP32) return bad("math_mode (only SBR_MATH_FP32 is implemented)");
  if (sbr_device_count() <= 0) {
    sbr_set_error(nullptr, SBR_E_NOGPU, "no CUDA device visible: libsbr_b200 has no CPU fallback");
    return SBR_E_NOGPU;
  }
  if (cfg->device < 0 || cfg->device >= sbr_device_count()) return bad("device ordinal");

  sbr_model* m = new sbr_model();
  m->cfg = *cfg;
  m->dev = cfg->device;
  m->B = cfg->batch_size; m->T = cfg->max_length; m->K = cfg->ids_per_step; m->N = cfg->n_items;
  m->n_in = cfg->n_items + cfg->n_extra_ids; m->E = cfg->embedding; m->L = cfg->n_layers;
  m->nd = cfg->bidirectional ? 2 : 1;
  m->global_batch = cfg->global_batch > 0 ? cfg->global_batch : cfg->batch_size * cfg->n_ranks;
  if (ccfg) {
    static const int kcode[] = {SBR_LOSS_BLACKOUT, SBR_LK_SCCE, SBR_LOSS_BPR, SBR_LOSS_TOP1, SBR_LK_BPRELU, SBR_LK_LIN};
    m->n_clusters = ccfg->n_clusters;
    m->cluster_type = ccfg->cluster_type;
    m->cluster_loss = kcode[ccfg->loss];
    m->n_csamples = ccfg->n_cluster_samples > 0 ? ccfg->n_cluster_samples : cfg->n_samples;
  }
  const int rc = create_impl(m);
  if (rc != 0) {
    g_create_error = m->err;
    sbr_destroy(m);
    return rc;
  }
  *out = m;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// parameters
// ------------------------------------------------------------------------------------------------
extern "C" int sbr_param_count(const sbr_model* m) { return m ? (int)m->views.size() : SBR_E_ARG; }
extern "C" int64_t sbr_total_params(const sbr_model* m) { return m ? m->P : SBR_E_ARG; }

extern "C" int sbr_param_info(const sbr_model* m, int idx, char* name, int name_cap, int* ndim, int64_t shape[4]) {
  if (!m || idx < 0 || idx >= (int)m->views.size()) return SBR_E_ARG;
  const ParamView& v = m->views[idx];
  if (name && name_cap > 0) {
    strncpy(name, v.name.c_str(), name_cap - 1);
    name[name_cap - 1] = 0;
  }
  if (ndim) *ndim = v.ndim;
  if (shape) { shape[0] = v.shape[0]; shape[1] = v.ndim > 1 ? v.shape[1] : 1; shape[2] = shape[3] = 1; }
  return 0;
}

static int copy_view(sbr_model* m, float* arena, int idx, float* host, bool to_host) {
  CHECK_STICKY(m);
  if (idx < 0 || idx >= (int)m->views.size() || !host) { sbr_set_error(m, SBR_E_ARG, "bad parameter index %d", idx); return SBR_E_ARG; }
  CU_TRY(m, cudaSetDevice(m->dev));
  const ParamView& v = m->views[idx];
  float* dev = arena + v.off;
  if (!v.transposed) {
    if (to_host)
      CU_TRY(m, cudaMemcpy2DAsync(host, v.cols * sizeof(float), dev, v.ld * sizeof(float), v.cols * sizeof(float), v.rows, cudaMemcpyDeviceToHost, m->stream));
    else
      CU_TRY(m, cudaMemcpy2DAsync(dev, v.ld * sizeof(float), host, v.cols * sizeof(float), v.cols * sizeof(float), v.rows, cudaMemcpyHostToDevice, m->stream));
    CU_TRY(m, cudaStreamSynchronize(m->stream));
    return 0;
  }
  // the arena keeps [cols, rows] (item-major output embeddings); the checkpoint wants [rows, cols]
  std::vector<float> tmp((size_t)v.rows * v.cols);
  if (to_host) {
    CU_TRY(m, cudaMemcpyAsync(tmp.data(), dev, tmp.size() * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
    CU_TRY(m, cudaStreamSynchronize(m->stream));
    for (int64_t r = 0; r < v.rows; ++r)
      for (int64_t c = 0; c < v.cols; ++c) host[r * v.cols + c] = tmp[c * v.rows + r];
  } else {
    for (int64_t r = 0; r < v.rows; ++r)
      for (int64_t c = 0; c < v.cols; ++c) tmp[c * v.rows + r] = host[r * v.cols + c];
    CU_TRY(m, cudaMemcpyAsync(dev, tmp.data(), tmp.size() * sizeof(float), cudaMemcpyHostToDevice, m->stream));
    CU_TRY(m, cudaStreamSynchronize(m->stream));
  }
  return 0;
}

extern "C" int sbr_get_param(sbr_model* m, int idx, float* host) { return copy_view(m, m ? m->params : nullptr, idx, host, true); }
extern "C" int sbr_set_param(sbr_model* m, int idx, const float* host) { return copy_view(m, m ? m->params : nullptr, idx, const_cast<float*>(host), false); }
extern "C" int sbr_get_grad(sbr_model* m, int idx, float* host) { return copy_view(m, m ? m->grads : nullptr, idx, host, true); }

extern "C" int sbr_reset_optimizer(sbr_model* m) {
  CHECK_STICKY(m);
  CU_TRY(m, cudaSetDevice(m->dev));
  const size_t arena = (size_t)m->P_pad + 4;
  CU_TRY(m, cudaMemsetAsync(m->opt_a, 0, arena * sizeof(float), m->stream));
  const bool two = m->cfg.updater == SBR_UPD_ADAM || m->cfg.updater == SBR_UPD_ADADELTA;
  if (two) CU_TRY(m, cudaMemsetAsync(m->opt_b, 0, arena * sizeof(float), m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  m->opt_t = 0;
  return 0;
}

extern "C" int sbr_set_skip_update(sbr_model* m, int flag) {
  if (!m) return SBR_E_ARG;
  // gradients of inspection steps stay in the arena (the optimizer kernel is what re-zeroes it): the next real step
  // must not accumulate on top of them
  if (m->skip_update && !flag) m->grads_dirty = true;
  m->skip_update = flag != 0;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// batch staging
// ------------------------------------------------------------------------------------------------
// mask [B,T] float -> lengths; rejects anything that is not a left-aligned run of ones
static int mask_to_len(sbr_model* m, const float* mask, const int32_t* X, int B, int* t_max) {
  // on the per-step host path: the scans below are written as branch-free reductions so that the compiler vectorises
  // them; the slow, index-reporting loops only run once something is wrong
  int mx = 0;
  const int T = m->T, K = m->K;
  const uint32_t n_in = (uint32_t)m->n_in;
  for (int b = 0; b < B; ++b) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(mask + (size_t)b * T);
    int L = 0;
    while (L < T && (r[L] & 0x7fffffffu) != 0u) ++L;      // != 0.f  (-0.f counts as zero)
    uint32_t tail = 0;
    for (int t = L; t < T; ++t) tail |= r[t] & 0x7fffffffu;
    if (tail) {
      sbr_set_error(m, SBR_E_MASK, "mask row %d is not a left-aligned run of ones (hole at %d)", b, L);
      return SBR_E_MASK;
    }
    m->h_len[b] = L;
    mx = std::max(mx, L);
    if (X) {
      const int32_t* x = X + (size_t)b * T * K;
      const int n = L * K;
      uint32_t bad = 0;
      for (int i = 0; i < n; ++i) bad |= (uint32_t)((uint32_t)x[i] >= n_in);   // negative ids wrap to huge values
      if (bad)
        for (int i = 0; i < n; ++i)
          if (x[i] < 0 || (uint32_t)x[i] >= n_in) {
            sbr_set_error(m, SBR_E_RANGE, "X[%d,%d,%d] = %d outside [0,%d)", b, i / K, i % K, x[i], m->n_in);
            return SBR_E_RANGE;
          }
    }
  }
  *t_max = mx;
  return 0;
}

static int stage_common(sbr_model* m, BatchSlot& s, const int32_t* X, const float* mask, int B) {
  if (m->staging_in_flight) {   // the previous batch must have left the pinned staging buffers (normally long ago)
    CU_TRY(m, cudaEventSynchronize(m->ev_staged));
    m->staging_in_flight = false;
  }
  if (B < 1 || B > m->B) { sbr_set_error(m, SBR_E_ARG, "B=%d outside [1,%d]", B, m->B); return SBR_E_ARG; }
  if (!X || !mask) { sbr_set_error(m, SBR_E_ARG, "null X/mask"); return SBR_E_ARG; }
  int t_max = 0;
  int rc = mask_to_len(m, mask, X, B, &t_max);
  if (rc) return rc;
  s.B = B;
  s.t_max = t_max;
  s.hlen.assign(m->h_len, m->h_len + B);
  // pageable caller buffer -> pinned staging -> device (one DMA, no driver-side bounce)
  const size_t xbytes = (size_t)B * m->T * m->K * sizeof(int32_t);
  memcpy(m->h_stage, X, xbytes);
  CU_TRY(m, cudaMemcpyAsync(s.X, m->h_stage, xbytes, cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(s.len, m->h_len, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  // the pinned staging buffers are reused by the next call: it must not start before these copies have left them
  CU_TRY(m, cudaEventRecord(m->ev_staged, m->stream));
  m->staging_in_flight = true;
  return 0;
}

static int stage_cce_impl(sbr_model* m, int slot, const int32_t* X, const float* mask, const int32_t* Y,
                          const float* pop, int B, bool sync) {
  CHECK_STICKY(m);
  if (slot < 0 || slot >= (int)m->slots.size() || !Y || !pop) { sbr_set_error(m, SBR_E_ARG, "bad slot or null Y/pop"); return SBR_E_ARG; }
  CU_TRY(m, cudaSetDevice(m->dev));
  BatchSlot& s = m->slots[slot];
  int rc = stage_common(m, s, X, mask, B);
  if (rc) return rc;
  for (int b = 0; b < B; ++b)
    if (Y[b] < 0 || Y[b] >= m->N) { sbr_set_error(m, SBR_E_RANGE, "Y[%d] = %d outside [0,%d)", b, Y[b], m->N); return SBR_E_RANGE; }
  s.n_all = B; s.row_offset = 0;
  CU_TRY(m, cudaMemcpyAsync(s.Y, Y, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(s.pop, pop, (size_t)B * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  if (sync) {   // Y / pop are caller buffers: they must be consumed before the call returns
    CU_TRY(m, cudaStreamSynchronize(m->stream));
    m->staging_in_flight = false;
  }
  return 0;
}

static int begin_step(sbr_model* m);
static int step_cce(sbr_model* m, const BatchSlot& s, float* cost);

extern "C" int sbr_dataset_upload(sbr_model* m, int n_seqs, const int32_t* offsets, const int32_t* ids) {
  CHECK_STICKY(m);
  if (n_seqs < 1 || !offsets || !ids || offsets[0] != 0) { sbr_set_error(m, SBR_E_ARG, "dataset_upload: bad arguments"); return SBR_E_ARG; }
  for (int i = 0; i < n_seqs; ++i)
    if (offsets[i + 1] < offsets[i]) { sbr_set_error(m, SBR_E_ARG, "dataset_upload: offsets must be non-decreasing"); return SBR_E_ARG; }
  const int64_t total = offsets[n_seqs];
  for (int64_t i = 0; i < total * m->K; ++i)
    if (ids[i] < 0 || ids[i] >= m->n_in) { sbr_set_error(m, SBR_E_RANGE, "dataset id %d outside [0,%d)", ids[i], m->n_in); return SBR_E_RANGE; }
  CU_TRY(m, cudaSetDevice(m->dev));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  if (m->ds_off) cudaFree(m->ds_off);
  if (m->ds_ids) cudaFree(m->ds_ids);
  m->ds_off = m->ds_ids = nullptr;
  int rc;
  if ((rc = dev_alloc(m, &m->ds_off, (size_t)n_seqs + 1, false))) return rc;
  if ((rc = dev_alloc(m, &m->ds_ids, (size_t)std::max<int64_t>(1, total * m->K), false))) return rc;
  if (!m->ds_rows && (rc = dev_alloc(m, &m->ds_rows, (size_t)3 * m->B))) return rc;
  CU_TRY(m, cudaMemcpyAsync(m->ds_off, offsets, ((size_t)n_seqs + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  if (total > 0) CU_TRY(m, cudaMemcpyAsync(m->ds_ids, ids, (size_t)total * m->K * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  m->ds_n = n_seqs;
  m->ds_hoff.assign(offsets, offsets + n_seqs + 1);
  return 0;
}

extern "C" int sbr_train_step_cce_rows(sbr_model* m, const int32_t* seq, const int32_t* start, const int32_t* len,
                                       const int32_t* Y, const float* pop, int B, float* cost) {
  CHECK_STICKY(m);
  if (m->cfg.loss != SBR_LOSS_CCE) { sbr_set_error(m, SBR_E_ARG, "model was not created with the CCE loss"); return SBR_E_ARG; }
  if (m->ds_n == 0) { sbr_set_error(m, SBR_E_ARG, "no dataset uploaded (sbr_dataset_upload)"); return SBR_E_ARG; }
  if (!seq || !start || !len || !Y || !pop || B < 1 || B > m->B) { sbr_set_error(m, SBR_E_ARG, "train_step_cce_rows: bad arguments"); return SBR_E_ARG; }
  int rc;
  if ((rc = begin_step(m))) return rc;
  stage_mark(m, 0);
  if (m->staging_in_flight) {
    CU_TRY(m, cudaEventSynchronize(m->ev_staged));
    m->staging_in_flight = false;
  }
  BatchSlot& s = m->slots[0];
  int32_t* h = static_cast<int32_t*>(m->h_stage);       // pinned: [3, B] triples (B*T*K*4 bytes available)
  int t_max = 0;
  for (int b = 0; b < B; ++b) {
    const int sq = seq[b], st = start[b], l = len[b];
    if (sq < 0 || sq >= m->ds_n || st < 0 || l < 0 || l > m->T || st + l > m->ds_hoff[sq + 1] - m->ds_hoff[sq]) {
      sbr_set_error(m, SBR_E_RANGE, "row %d: (sequence %d, start %d, length %d) outside the uploaded dataset / max_length %d", b, sq, st, l, m->T);
      return SBR_E_RANGE;
    }
    if (Y[b] < 0 || Y[b] >= m->N) { sbr_set_error(m, SBR_E_RANGE, "Y[%d] = %d outside [0,%d)", b, Y[b], m->N); return SBR_E_RANGE; }
    h[b] = sq; h[B + b] = st; h[2 * B + b] = l;
    m->h_len[b] = l;
    t_max = std::max(t_max, l);
  }
  s.B = B; s.t_max = t_max; s.n_all = B; s.row_offset = 0;
  s.hlen.assign(m->h_len, m->h_len + B);
  CU_TRY(m, cudaMemcpyAsync(m->ds_rows, h, (size_t)3 * B * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(s.Y, Y, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(s.pop, pop, (size_t)B * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaEventRecord(m->ev_staged, m->stream));
  m->staging_in_flight = true;
  const int64_t n = (int64_t)B * m->T * m->K;
  assemble_rows_kernel<<<cdiv(n, 256), 256, 0, m->stream>>>(m->ds_off, m->ds_ids, m->ds_rows, s.X, s.len, B, m->T, m->K);
  KERNEL_CHECK(m);
  float local_cost;
  return step_cce(m, s, cost ? cost : &local_cost);
}

extern "C" int sbr_stage_cce(sbr_model* m, int slot, const int32_t* X, const float* mask, const int32_t* Y,
                             const float* pop, int B) {
  return stage_cce_impl(m, slot, X, mask, Y, pop, B, true);
}

// ------------------------------------------------------------------------------------------------
// forward / backward building blocks
// ------------------------------------------------------------------------------------------------
static int bias_rows(sbr_model* m, float* out, const float* bias, int64_t rows, int cols) {
  if (rows == 0) return 0;
  fill_rows_kernel<<<cdiv(rows * cols, 256), 256, 0, m->stream>>>(out, bias, rows, cols);
  KERNEL_CHECK(m);
  return 0;
}

// ids -> final hidden state of the top level (m->h_last; [forward | backward] for a bidirectional stack)
static int forward_stack(sbr_model* m, const BatchSlot& s) {
  m->cur_hlen = (int)s.hlen.size() == s.B ? s.hlen.data() : nullptr;
  const int B = s.B, T = m->T, K = m->K, t_max = s.t_max, nd = m->nd;
  const int64_t rows = (int64_t)t_max * B;
  int rc;
  stage_mark(m, 1);
  if (nd == 2 && (rc = launch_reverse_ids(m, s.X, s.len, m->X_rev, B, T, K))) return rc;
  for (int li = 0; li < m->L; ++li) {
    for (int dir = 0; dir < nd; ++dir) {
      LayerDesc& L = m->layers[li * nd + dir];
      const int GH = L.G * L.H;
      const int32_t* X = dir ? m->X_rev : s.X;       // the backwards layer sees every row reversed
      if (li == 0 && m->E == 0) {
        if ((rc = launch_gather_rows(m, X, s.len, m->params + L.W_in, m->params + L.b, L.Xg, B, T, K, GH, t_max, m->n_in))) return rc;
      } else {
        const float* in;
        int I;
        if (li == 0) {
          float* eo = dir ? m->emb_out_rv : m->emb_out;
          if ((rc = launch_embed_gather(m, X, s.len, m->params + m->emb_W, eo, B, T, K, m->E, t_max))) return rc;
          in = eo; I = K * m->E;
        } else if (nd == 1) {
          in = m->layers[li - 1].hs + (int64_t)B * m->layers[li - 1].H;   // skip the init row block
          I = m->layers[li - 1].H;
        } else {
          in = dir ? m->cat_rv : m->cat_al;
          I = 2 * m->layers[(li - 1) * nd].H;
        }
        if ((rc = launch_gemm_bias(m, false, (int)rows, GH, I, in, I, m->params + L.W_in, GH, L.Xg, GH, m->params + L.b))) return rc;
      }
      if (li == 0 && dir == nd - 1) stage_mark(m, 2);
      float* h_last = nullptr;
      if (li == m->L - 1) h_last = nd == 1 ? m->h_last : m->h_last_dir + (size_t)dir * B * L.H;
      if ((rc = launch_rnn_forward(m, L, s.len, B, t_max, h_last))) return rc;
    }
    if (nd == 2) {
      const LayerDesc& Lf = m->layers[li * 2];
      const LayerDesc& Lb = m->layers[li * 2 + 1];
      const int H = Lf.H;
      if (li < m->L - 1) {
        // outputs of this depth for the next one, in both coordinate systems
        if ((rc = launch_bi_concat(m, Lf.hs + (int64_t)B * H, Lb.hs + (int64_t)B * H, s.len, m->cat_al, m->cat_rv, B, t_max, H))) return rc;
      } else {
        // final state = [forward state after the last item | backward state after the first item]
        CU_TRY(m, cudaMemcpy2DAsync(m->h_last, (size_t)2 * H * sizeof(float), m->h_last_dir, (size_t)H * sizeof(float),
                                    (size_t)H * sizeof(float), B, cudaMemcpyDeviceToDevice, m->stream));
        CU_TRY(m, cudaMemcpy2DAsync(m->h_last + H, (size_t)2 * H * sizeof(float), m->h_last_dir + (size_t)B * H, (size_t)H * sizeof(float),
                                    (size_t)H * sizeof(float), B, cudaMemcpyDeviceToDevice, m->stream));
      }
    }
  }
  stage_mark(m, 3);
  return 0;
}

static int side_fork(sbr_model* m);
static int side_return(sbr_model* m);
static int side_join(sbr_model* m);
static int launch_deferred_output_grads(sbr_model* m);

// BPTT through the stack given m->dh_last; fills the gradient arena of every stack parameter
static int backward_stack(sbr_model* m, const BatchSlot& s) {
  m->cur_hlen = (int)s.hlen.size() == s.B ? s.hlen.data() : nullptr;
  const int B = s.B, T = m->T, K = m->K, t_max = s.t_max, nd = m->nd;
  const int rows = t_max * B;
  int rc;
  if (nd == 2) {
    const int H = m->layers.back().H;     // split [forward | backward] of the gradient wrt the final state
    CU_TRY(m, cudaMemcpy2DAsync(m->dh_last_dir, (size_t)H * sizeof(float), m->dh_last, (size_t)2 * H * sizeof(float),
                                (size_t)H * sizeof(float), B, cudaMemcpyDeviceToDevice, m->stream));
    CU_TRY(m, cudaMemcpy2DAsync(m->dh_last_dir + (size_t)B * H, (size_t)H * sizeof(float), m->dh_last + H, (size_t)2 * H * sizeof(float),
                                (size_t)H * sizeof(float), B, cudaMemcpyDeviceToDevice, m->stream));
  }
  if ((rc = launch_wgrad_stage_list(m, s.len, B, rows))) return rc;
  for (int li = m->L - 1; li >= 0; --li) {
    for (int dir = 0; dir < nd; ++dir) {
      LayerDesc& L = m->layers[li * nd + dir];
      const int H = L.H, GH = L.G * L.H;
      const float* dh_last = nullptr;
      if (li == m->L - 1) dh_last = nd == 1 ? m->dh_last : m->dh_last_dir + (size_t)dir * B * H;
      if ((rc = launch_rnn_backward(m, L, s.len, B, t_max, dh_last))) return rc;
      // the scan is in the launch queue first, so its clusters get their SMs before the side-stream GEMM's CTAs do
      if (li == m->L - 1 && dir == 0 && (rc = launch_deferred_output_grads(m))) return rc;
      if (li == 0 && dir == nd - 1) stage_mark(m, 5);
      const bool gather_layer = (li == 0 && m->E == 0);
      const int32_t* X = dir ? m->X_rev : s.X;
      if (gather_layer) {
        // dW_in scatter on the side stream, concurrent with the weight-gradient GEMM below
        if ((rc = side_fork(m))) return rc;
        rc = launch_scatter_add_rows(m, X, s.len, L.dXg, m->grads + L.W_in, B, T, K, GH, t_max);
        side_return(m);
        m->side_pending = true;
        if (rc) return rc;
      }
      // dW_hid = sum_t h_{t-1}^T da_t  : one tall-K GEMM outside the scan -- on tcgen05 from the K-major copies the
      // tc scans wrote, else the generic GEMM (tcgen05 3xTF32 as well)
      const bool tc_wgrad = L.hT && L.aT && B % 16 == 0 && rows % 8 == 0 && rows > 0 && !m->disable_tc_bwd;
      if (tc_wgrad) {
        if ((rc = launch_wgrad_tc(m, L, rows, m->grads + L.W_hid, GH))) return rc;
      } else if (L.G == 3) {
        if ((rc = launch_gemm(m, true, false, H, 2 * H, rows, L.hs, H, L.dXg, GH, m->grads + L.W_hid, GH, 1.f, 1.f))) return rc;
        if ((rc = launch_gemm(m, true, false, H, H, rows, L.hs, H, L.dac, H, m->grads + L.W_hid + 2 * H, GH, 1.f, 1.f))) return rc;
      } else {
        if ((rc = launch_gemm(m, true, false, H, GH, rows, L.hs, H, L.dXg, GH, m->grads + L.W_hid, GH, 1.f, 1.f))) return rc;
      }
      // db = sum dXg: the tcgen05 BPTT kernels accumulate it themselves; the fallbacks need the column sum
      if (!m->bwd_did_bias)
        if ((rc = launch_colsum(m, L.dXg, rows, GH, GH, m->grads + L.b))) return rc;
      if (li == 0 && dir == nd - 1) stage_mark(m, 6);
      if (!gather_layer) {
        const float* in;
        float* din;
        int I;
        if (li == 0) {
          in = dir ? m->emb_out_rv : m->emb_out; din = dir ? m->demb_rv : m->demb; I = K * m->E;
        } else if (nd == 1) {
          in = m->layers[li - 1].hs + (int64_t)B * m->layers[li - 1].H; din = m->layers[li - 1].dhs; I = m->layers[li - 1].H;
        } else {
          in = dir ? m->cat_rv : m->cat_al; din = dir ? m->dcat_rv : m->dcat_al; I = 2 * m->layers[(li - 1) * nd].H;
        }
        if ((rc = launch_gemm(m, true, false, I, GH, rows, in, I, L.dXg, GH, m->grads + L.W_in, GH, 1.f, 1.f))) return rc;
        if ((rc = launch_gemm(m, false, true, rows, I, GH, L.dXg, GH, m->params + L.W_in, GH, din, I, 1.f, 0.f))) return rc;
        if (li == 0)
          if ((rc = launch_embed_scatter(m, X, s.len, din, m->grads + m->emb_W, B, T, K, m->E, t_max))) return rc;
      }
    }
    if (nd == 2 && li > 0) {
      // gradients wrt the outputs of the depth below: un-concatenate, bring both contributions into each layer's own
      // coordinate system, add.  The depth below needs ITS concatenated outputs again for its input-weight gradients.
      LayerDesc& Pf = m->layers[(li - 1) * 2];
      LayerDesc& Pb = m->layers[(li - 1) * 2 + 1];
      if ((rc = launch_bi_split(m, m->dcat_al, m->dcat_rv, s.len, Pf.dhs, Pb.dhs, B, t_max, Pf.H))) return rc;
      if (li - 1 > 0) {
        const LayerDesc& Qf = m->layers[(li - 2) * 2];
        const LayerDesc& Qb = m->layers[(li - 2) * 2 + 1];
        if ((rc = launch_bi_concat(m, Qf.hs + (int64_t)B * Qf.H, Qb.hs + (int64_t)B * Qb.H, s.len, m->cat_al, m->cat_rv, B, t_max, Qf.H))) return rc;
      }
    }
  }
  return 0;
}

// Fork / join of the side stream: work that is off the critical path (the output-layer weight gradients
// while the BPTT scan runs on 64 of the 148 SMs; the scatter while the weight-gradient GEMM runs) is
// launched on m->side between side_fork() and side_join(); the two streams write disjoint gradient blocks.
static int side_fork(sbr_model* m) {
  if (m->no_side_stream) return 0;   // diagnostics: everything on one stream
  CU_TRY(m, cudaEventRecord(m->ev_fork, m->stream));
  CU_TRY(m, cudaStreamWaitEvent(m->side, m->ev_fork, 0));
  std::swap(m->stream, m->side);     // launchers use m->stream
  m->on_side = true;
  return 0;
}
static int side_return(sbr_model* m) {   // back to the main stream; the side work keeps running
  if (m->no_side_stream) return 0;
  std::swap(m->stream, m->side);
  m->on_side = false;
  return 0;
}
static int side_join(sbr_model* m) {
  CU_TRY(m, cudaEventRecord(m->ev_join, m->side));
  CU_TRY(m, cudaStreamWaitEvent(m->stream, m->ev_join, 0));
  return 0;
}

// gradient of a full-catalog score matrix d[B,N] (already in m->logits): dW_out^T, db, dh_last
static int output_backward_full(sbr_model* m, int B) {
  const int N = m->N, H = m->H_last;
  int rc;
  // critical path: dh_last feeds the BPTT scan
  if ((rc = launch_gemm(m, false, false, B, H, N, m->logits, (int)round_up(N, 4), m->params + m->out_WT, H, m->dh_last, H, 1.f, 0.f))) return rc;
  // off the critical path: dW_out^T and db_out go to the side stream (joined before the all-reduce).  The fork point
  // is here (they only need the logit gradients and h_last), but the launches are issued AFTER the BPTT scan has
  // been launched on the main stream (launch_deferred_output_grads): a GEMM that reaches the SMs first would keep
  // some of the scan's 8-CTA clusters waiting for free SMs.
  if (!m->no_side_stream) CU_TRY(m, cudaEventRecord(m->ev_fork, m->stream));
  m->deferred_out_B = B;
  return 0;
}

static int launch_deferred_output_grads(sbr_model* m) {
  const int B = m->deferred_out_B;
  if (B <= 0) return 0;
  m->deferred_out_B = 0;
  const int N = m->N, H = m->H_last;
  const bool side = !m->no_side_stream;
  if (side) {
    CU_TRY(m, cudaStreamWaitEvent(m->side, m->ev_fork, 0));
    std::swap(m->stream, m->side);
    m->on_side = true;
  }
  int rc = launch_gemm(m, true, false, N, H, B, m->logits, (int)round_up(N, 4), m->h_last, H, m->grads + m->out_WT, H, 1.f, 1.f);
  if (!rc) rc = launch_colsum(m, m->logits, B, N, (int)round_up(N, 4), m->grads + m->out_b);
  if (side) {
    std::swap(m->stream, m->side);
    m->on_side = false;
    m->side_pending = true;
  }
  return rc;
}

static int begin_step(sbr_model* m) {
  CU_TRY(m, cudaSetDevice(m->dev));
  if (m->skip_update || m->grads_dirty) {  // gradients of the previous (inspection) step are still in the arena
    CU_TRY(m, cudaMemsetAsync(m->grads, 0, ((size_t)m->P_pad + 4) * sizeof(float), m->stream));
    m->grads_dirty = false;
  } else
    CU_TRY(m, cudaMemsetAsync(m->grads + m->cost_slot, 0, 4 * sizeof(float), m->stream));
  return 0;
}

static int finish_step(sbr_model* m, float* cost) {
  int rc;
  if (m->side_pending) {
    if ((rc = side_join(m))) return rc;
    m->side_pending = false;
  }
  stage_mark(m, 7);
  if (m->nccl_comm) {
    // the cost slot rides along (the cluster model's second cost in the slot after it)
    ncclResult_t r = g_nccl.AllReduce(m->grads, m->grads, (size_t)m->P_pad + (m->n_clusters > 0 ? 2 : 1), ncclFloat, ncclSum,
                                      (ncclComm_t)m->nccl_comm, m->stream);
    if (r != ncclSuccess) {
      sbr_set_error(m, SBR_E_NCCL, "ncclAllReduce: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
      return SBR_E_NCCL;
    }
  }
  stage_mark(m, 8);
  if (cost && !m->cost_early)
    CU_TRY(m, cudaMemcpyAsync(m->h_cost, m->grads + m->cost_slot, (m->n_clusters > 0 ? 2 : 1) * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
  if (!m->skip_update)
    if ((rc = launch_optimizer(m))) return rc;
  stage_mark(m, 9);
  if (m->cost_early && cost) {
    // the cost left the device right after the loss kernels: return as soon as it has landed.  The backward pass
    // and the update keep running; everything the caller can do next (another step, get/set_param, scores) is
    // ordered behind them on the same stream, and the host work of the next step overlaps them.
    m->cost_early = false;
    CU_TRY(m, cudaEventSynchronize(m->ev_cost));
    *cost = m->h_cost[0];
    return 0;
  }
  m->cost_early = false;
  if (cost || m->profiling) {
    CU_TRY(m, cudaStreamSynchronize(m->stream));
    m->staging_in_flight = false;
    if (cost) *cost = m->h_cost[0];
    if (m->profiling)
      for (int i = 0; i < SBR_N_STAGES; ++i) cudaEventElapsedTime(&m->stage_ms[i], m->ev[i], m->ev[i + 1]);
  }
  return 0;
}

static int step_cce(sbr_model* m, const BatchSlot& s, float* cost) {
  int rc;
  const float inv_gb = 1.f / (float)(m->cfg.global_batch > 0 ? m->cfg.global_batch : s.B * m->cfg.n_ranks);
  if ((rc = forward_stack(m, s))) return rc;
  const int B = s.B, N = m->N, H = m->H_last;
  if ((rc = launch_gemm(m, false, true, B, N, H, m->h_last, H, m->params + m->out_WT, H, m->logits, (int)round_up(N, 4), 1.f, 0.f))) return rc;
  if ((rc = launch_cce(m, m->logits, (int)round_up(N, 4), m->params + m->out_b, s.Y, s.pop, B, N, inv_gb, m->row_loss))) return rc;
  if ((rc = launch_reduce_cost(m, m->row_loss, B, m->grads + m->cost_slot))) return rc;
  if (m->cfg.regularization != 0.f)
    if ((rc = launch_bias_reg(m, m->params + m->out_b, m->grads + m->out_b, N, m->cfg.regularization / (float)m->cfg.n_ranks,
                              m->grads + m->cost_slot))) return rc;
  // single rank: the cost is final here (no all-reduce): start its way to the host now, before the backward pass
  if (cost && !m->nccl_comm && !m->profiling && !m->no_early_cost) {
    CU_TRY(m, cudaMemcpyAsync(m->h_cost, m->grads + m->cost_slot, sizeof(float), cudaMemcpyDeviceToHost, m->stream));
    CU_TRY(m, cudaEventRecord(m->ev_cost, m->stream));
    m->cost_early = true;
  }
  if ((rc = output_backward_full(m, B))) return rc;
  stage_mark(m, 4);
  if ((rc = backward_stack(m, s))) return rc;
  return finish_step(m, cost);
}

extern "C" int sbr_train_step_staged(sbr_model* m, int slot, float* cost) {
  CHECK_STICKY(m);
  if (slot < 0 || slot >= (int)m->slots.size()) { sbr_set_error(m, SBR_E_ARG, "bad slot"); return SBR_E_ARG; }
  if (m->cfg.loss != SBR_LOSS_CCE) { sbr_set_error(m, SBR_E_ARG, "staged steps are implemented for the CCE loss"); return SBR_E_ARG; }
  if (m->slots[slot].B == 0) { sbr_set_error(m, SBR_E_ARG, "slot %d is empty", slot); return SBR_E_ARG; }
  int rc;
  if ((rc = begin_step(m))) return rc;
  stage_mark(m, 0);
  return step_cce(m, m->slots[slot], cost);
}

extern "C" int sbr_train_step_cce(sbr_model* m, const int32_t* X, const float* mask, const int32_t* Y,
                                  const float* pop, int B, float* cost) {
  CHECK_STICKY(m);
  if (m->cfg.loss != SBR_LOSS_CCE) { sbr_set_error(m, SBR_E_ARG, "model was not created with the CCE loss"); return SBR_E_ARG; }
  int rc;
  if ((rc = begin_step(m))) return rc;
  stage_mark(m, 0);
  // X goes through the pinned staging buffer, Y / pop are small pageable copies that the driver stages at call
  // time: the caller's buffers are free when this call returns even though the device may still be working
  if ((rc = stage_cce_impl(m, 0, X, mask, Y, pop, B, false))) return rc;
  float local_cost;
  return step_cce(m, m->slots[0], cost ? cost : &local_cost);
}

extern "C" int sbr_synchronize(sbr_model* m, float* last_cost) {
  CHECK_STICKY(m);
  CU_TRY(m, cudaSetDevice(m->dev));
  if (last_cost) CU_TRY(m, cudaMemcpyAsync(m->h_cost, m->grads + m->cost_slot, sizeof(float), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  if (last_cost) *last_cost = m->h_cost[0];
  return 0;
}

static int sampled_output(sbr_model* m, int loss, bool tanh_out, const float* pop, int B, int n_all, int row_offset, int S,
                          float inv_gb);

extern "C" int sbr_train_step_sampled(sbr_model* m, const int32_t* X, const float* mask, const int32_t* Y_all,
                                      int n_all, int row_offset, const int32_t* samples, int S, const float* pop,
                                      int B, float* cost) {
  CHECK_STICKY(m);
  const int loss = m->cfg.loss;
  if (loss < SBR_LOSS_BPR || loss > SBR_LOSS_BLACKOUT || m->n_clusters > 0) { sbr_set_error(m, SBR_E_ARG, "model was not created with a sampling loss"); return SBR_E_ARG; }
  if (!Y_all || !samples || !pop || S < 1 || S > std::max(1, m->cfg.n_samples) || n_all < B || n_all > m->global_batch ||
      row_offset < 0 || row_offset + B > n_all) {
    sbr_set_error(m, SBR_E_ARG, "bad sampled-step arguments (S=%d n_all=%d row_offset=%d B=%d)", S, n_all, row_offset, B);
    return SBR_E_ARG;
  }
  int rc;
  if ((rc = begin_step(m))) return rc;
  stage_mark(m, 0);
  BatchSlot& s = m->slots[0];
  if ((rc = stage_common(m, s, X, mask, B))) return rc;
  const int nc = n_all + S;
  for (int i = 0; i < nc; ++i) {
    const int id = i < n_all ? Y_all[i] : samples[i - n_all];
    if (id < 0 || id >= m->N) { sbr_set_error(m, SBR_E_RANGE, "target/sample id %d outside [0,%d)", id, m->N); return SBR_E_RANGE; }
  }
  CU_TRY(m, cudaMemcpyAsync(m->cells, Y_all, (size_t)n_all * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(m->cells + n_all, samples, (size_t)S * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(s.pop, pop, (size_t)B * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  const float inv_gb = 1.f / (float)(m->cfg.global_batch > 0 ? m->cfg.global_batch : s.B * m->cfg.n_ranks);
  if ((rc = forward_stack(m, s))) return rc;
  if ((rc = sampled_output(m, loss, m->cfg.last_layer_tanh != 0, s.pop, B, n_all, row_offset, S, inv_gb))) return rc;
  stage_mark(m, 4);
  if ((rc = backward_stack(m, s))) return rc;
  return finish_step(m, cost);
}

// BlackoutLayer of the sampled models on the gathered columns m->cells = [Y_all; samples]: scores, loss (into the
// cost slot), the gradients of the gathered output rows / bias and m->dh_last
static int sampled_output(sbr_model* m, int loss, bool tanh_out, const float* pop, int B, int n_all, int row_offset, int S,
                          float inv_gb) {
  int rc;
  const int nc = n_all + S;
  const int H = m->H_last;
  const int ldc = (int)round_up(nc, 4);      // padded row pitch of the [B, n_all + S] score matrix
  float* bcg = m->bc + nc;   // gradient of the gathered bias entries
  // BlackoutLayer: scores of the gathered columns only (sparse_lstm.py:41-54)
  if ((rc = launch_gather_table_rows(m, m->params + m->out_WT, m->params + m->out_b, m->cells, nc, H, m->Wc, m->bc))) return rc;
  if ((rc = launch_gemm(m, false, true, B, nc, H, m->h_last, H, m->Wc, H, m->logits, ldc, 1.f, 0.f))) return rc;
  if ((rc = launch_sampling_loss(m, loss, tanh_out, m->logits, ldc, m->bc, pop, B, n_all, row_offset, S, inv_gb, m->row_loss))) return rc;
  if ((rc = launch_reduce_cost(m, m->row_loss, B, m->grads + m->cost_slot))) return rc;
  if ((rc = launch_gemm(m, true, false, nc, H, B, m->logits, ldc, m->h_last, H, m->dWc, H, 1.f, 0.f))) return rc;
  CU_TRY(m, cudaMemsetAsync(bcg, 0, (size_t)nc * sizeof(float), m->stream));
  if ((rc = launch_colsum(m, m->logits, B, nc, ldc, bcg))) return rc;
  if ((rc = launch_scatter_table_rows(m, m->dWc, bcg, m->cells, nc, H, m->grads + m->out_WT, m->grads + m->out_b))) return rc;
  return launch_gemm(m, false, false, B, H, nc, m->logits, ldc, m->Wc, H, m->dh_last, H, 1.f, 0.f);
}

struct MarginRagged { bool on = false; bool has_default = false; int exclude_seen = 0; int max_special = 0; };

static int step_margin(sbr_model* m, const BatchSlot& s, float* cost, const MarginRagged& rg = MarginRagged()) {
  int rc;
  const float inv_gb = 1.f / (float)(m->cfg.global_batch > 0 ? m->cfg.global_batch : s.B * m->cfg.n_ranks);
  if ((rc = forward_stack(m, s))) return rc;
  const int B = s.B, N = m->N, H = m->H_last;
  const int ldl = (int)round_up(N, 4);
  if ((rc = launch_gemm(m, false, true, B, N, H, m->h_last, H, m->params + m->out_WT, H, m->logits, ldl, 1.f, 0.f))) return rc;
  if (rg.on) {
    if ((rc = launch_margin_loss_ragged(m, m->cfg.loss, m->logits, ldl, m->params + m->out_b, m->tgt_off, m->tgt_ids, s.X, s.len, m->w_neg,
                                        rg.has_default ? m->def_tgt : nullptr, rg.exclude_seen, B, m->T, m->K, N, rg.max_special, inv_gb,
                                        m->row_loss))) return rc;
  } else if ((rc = launch_margin_loss(m, m->cfg.loss, m->logits, ldl, m->params + m->out_b, m->mY, m->mW, B, N, inv_gb, m->row_loss))) return rc;
  if ((rc = launch_reduce_cost(m, m->row_loss, B, m->grads + m->cost_slot))) return rc;
  if ((rc = output_backward_full(m, B))) return rc;
  stage_mark(m, 4);
  if ((rc = backward_stack(m, s))) return rc;
  return finish_step(m, cost);
}

extern "C" int sbr_train_step_margin_dense(sbr_model* m, const int32_t* X, const float* mask, const float* Ymat,
                                           const float* weight, int B, float* cost) {
  CHECK_STICKY(m);
  if (m->cfg.loss < SBR_LOSS_HINGE) { sbr_set_error(m, SBR_E_ARG, "model was not created with a margin loss"); return SBR_E_ARG; }
  if (!Ymat || !weight) { sbr_set_error(m, SBR_E_ARG, "null Ymat/weight"); return SBR_E_ARG; }
  int rc;
  if ((rc = begin_step(m))) return rc;
  stage_mark(m, 0);
  BatchSlot& s = m->slots[0];
  if ((rc = stage_common(m, s, X, mask, B))) return rc;
  if (!m->mY) {
    if ((rc = dev_alloc(m, &m->mY, (size_t)m->B * m->N, false))) return rc;
    if ((rc = dev_alloc(m, &m->mW, (size_t)m->B * m->N, false))) return rc;
  }
  CU_TRY(m, cudaMemcpyAsync(m->mY, Ymat, (size_t)B * m->N * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(m->mW, weight, (size_t)B * m->N * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  return step_margin(m, s, cost);
}

extern "C" int sbr_train_step_margin(sbr_model* m, const int32_t* X, const float* mask, const int32_t* target_offsets,
                                     const int32_t* target_ids, const float* w_neg, const float* default_target,
                                     int exclude_seen, int B, float* cost) {
  CHECK_STICKY(m);
  if (m->cfg.loss < SBR_LOSS_HINGE) { sbr_set_error(m, SBR_E_ARG, "model was not created with a margin loss"); return SBR_E_ARG; }
  if (!target_offsets || !target_ids || !w_neg) { sbr_set_error(m, SBR_E_ARG, "null ragged target arguments"); return SBR_E_ARG; }
  int rc;
  if ((rc = begin_step(m))) return rc;
  stage_mark(m, 0);
  BatchSlot& s = m->slots[0];
  if ((rc = stage_common(m, s, X, mask, B))) return rc;
  const int nt = target_offsets[B];
  if (target_offsets[0] != 0 || nt < 0) { sbr_set_error(m, SBR_E_ARG, "target_offsets must start at 0"); return SBR_E_ARG; }
  for (int b = 0; b < B; ++b)
    if (target_offsets[b + 1] < target_offsets[b]) { sbr_set_error(m, SBR_E_ARG, "target_offsets must be non-decreasing"); return SBR_E_ARG; }
  if (nt > m->tgt_cap) {
    if (m->tgt_ids) cudaFree(m->tgt_ids);
    m->tgt_ids = nullptr;
    m->tgt_cap = std::max(nt, 2 * m->tgt_cap);
    if ((rc = dev_alloc(m, &m->tgt_ids, (size_t)m->tgt_cap, false))) return rc;
  }
  CU_TRY(m, cudaMemcpyAsync(m->tgt_off, target_offsets, (size_t)(B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  if (nt > 0) CU_TRY(m, cudaMemcpyAsync(m->tgt_ids, target_ids, (size_t)nt * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(m->w_neg, w_neg, (size_t)B * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  if (default_target) CU_TRY(m, cudaMemcpyAsync(m->def_tgt, default_target, (size_t)m->N * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  MarginRagged rg;
  rg.on = true; rg.has_default = default_target != nullptr; rg.exclude_seen = exclude_seen;
  for (int b = 0; b < B; ++b)
    rg.max_special = std::max(rg.max_special, target_offsets[b + 1] - target_offsets[b] + (exclude_seen ? m->h_len[b] : 0));
  return step_margin(m, s, cost, rg);
}

// ------------------------------------------------------------------------------------------------
// predict / test
// ------------------------------------------------------------------------------------------------
static int scores_device(sbr_model* m, const int32_t* X, const float* mask, int B, int softmax) {
  int rc;
  CU_TRY(m, cudaSetDevice(m->dev));
  BatchSlot& s = m->slots[0];
  if ((rc = stage_common(m, s, X, mask, B))) return rc;
  const bool prof = m->profiling;
  m->profiling = false;
  rc = forward_stack(m, s);
  m->profiling = prof;
  if (rc) return rc;
  const int N = m->N, H = m->H_last;
  const int ldl = (int)round_up(N, 4);
  if ((rc = launch_gemm(m, false, true, B, N, H, m->h_last, H, m->params + m->out_WT, H, m->logits, ldl, 1.f, 0.f))) return rc;
  if (softmax) return launch_softmax_rows(m, m->logits, ldl, m->params + m->out_b, B, N);
  return launch_add_bias_rows(m, m->logits, ldl, m->params + m->out_b, B, N);
}

extern "C" int sbr_scores(sbr_model* m, const int32_t* X, const float* mask, int B, int softmax, float* scores) {
  CHECK_STICKY(m);
  if (!scores) { sbr_set_error(m, SBR_E_ARG, "null scores"); return SBR_E_ARG; }
  const int sm = (m->cfg.loss == SBR_LOSS_CCE) || softmax;
  int rc = scores_device(m, X, mask, B, sm);
  if (rc) return rc;
  CU_TRY(m, cudaMemcpy2DAsync(scores, (size_t)m->N * sizeof(float), m->logits, (size_t)round_up(m->N, 4) * sizeof(float),
                              (size_t)m->N * sizeof(float), B, cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  return 0;
}

// ragged exclusion lists -> m->excl_off / m->excl_ids (*d_off stays NULL when there are none)
static int upload_exclusions(sbr_model* m, int B, const int32_t* excl_offsets, const int32_t* excl_ids, const int32_t** d_off) {
  int rc;
  *d_off = nullptr;
  if (!excl_offsets || !excl_ids) return 0;
  const int ne = excl_offsets[B];
  if (ne > m->excl_cap) {
    if (m->excl_ids) cudaFree(m->excl_ids);
    m->excl_ids = nullptr;
    m->excl_cap = std::max(ne, 2 * m->excl_cap);
    if ((rc = dev_alloc(m, &m->excl_ids, (size_t)m->excl_cap, false))) return rc;
  }
  CU_TRY(m, cudaMemcpyAsync(m->excl_off, excl_offsets, (size_t)(B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  if (ne > 0) CU_TRY(m, cudaMemcpyAsync(m->excl_ids, excl_ids, (size_t)ne * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  *d_off = m->excl_off;
  return 0;
}

extern "C" int sbr_topk(sbr_model* m, const int32_t* X, const float* mask, int B, const int32_t* excl_offsets,
                        const int32_t* excl_ids, int k, int mode, int32_t* ids_out) {
  CHECK_STICKY(m);
  if (!ids_out || k < 1 || k > 64 || k > m->N) { sbr_set_error(m, SBR_E_ARG, "k must be in [1, min(64, n_items)]"); return SBR_E_ARG; }
  const int sm = (m->cfg.loss == SBR_LOSS_CCE) || (mode & 1);
  int rc = scores_device(m, X, mask, B, sm);
  if (rc) return rc;
  const int32_t* d_off = nullptr;
  if ((rc = upload_exclusions(m, B, excl_offsets, excl_ids, &d_off))) return rc;
  if ((rc = launch_topk(m, m->logits, (int)round_up(m->N, 4), B, m->N, d_off, m->excl_ids, k, (mode >> 1) & 1, m->topk_ids))) return rc;
  CU_TRY(m, cudaMemcpyAsync(ids_out, m->topk_ids, (size_t)B * k * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// RNNCluster (rnn_cluster.py)
// ------------------------------------------------------------------------------------------------
// The cluster branch of one step (rnn_cluster.py:232-251), after the recommendation branch.  It reads h_last but sends
// no gradient back to it: the cluster cost only reaches Wc and R (rnn_cluster.py:268-270).
static int cluster_branch(sbr_model* m, int B, int n_all, int row_offset, int Sc, bool noise, float scale, float inv_gb) {
  int rc;
  const int C = m->n_clusters, H = m->H_last, nc = n_all + Sc, lds = (int)round_up(nc, 4), type = m->cluster_type;
  const float* R = m->params + m->cl_R;
  if ((rc = launch_gemm(m, false, false, B, C, H, m->h_last, H, m->params + m->cl_W, C, m->cq, C, 1.f, 0.f))) return rc;
  if ((rc = launch_cluster_select(m, m->cq, noise ? m->cnoise : nullptr, B, C, scale, m->cP))) return rc;
  if ((rc = launch_cluster_members(m, R, m->ccells, nc, C, type, scale, m->cM))) return rc;
  if ((rc = launch_gemm(m, false, true, B, nc, C, m->cP, C, m->cM, C, m->cS, lds, 1.f, 0.f))) return rc;
  if ((rc = launch_sampling_loss(m, m->cluster_loss, false, m->cS, lds, nullptr, nullptr, B, n_all, row_offset, Sc, inv_gb, m->crow_loss))) return rc;
  if ((rc = launch_reduce_cost(m, m->crow_loss, B, m->grads + m->cost_slot + 1))) return rc;
  // dP = dS M, dM = dS^T P
  if ((rc = launch_gemm(m, false, false, B, C, nc, m->cS, lds, m->cM, C, m->cdP, C, 1.f, 0.f))) return rc;
  if ((rc = launch_gemm(m, true, false, nc, C, B, m->cS, lds, m->cP, C, m->cdM, C, 1.f, 0.f))) return rc;
  if ((rc = launch_cluster_dq(m, m->cP, m->cdP, B, C, scale, m->cdq))) return rc;
  if ((rc = launch_gemm(m, true, false, H, C, B, m->h_last, H, m->cdq, C, m->grads + m->cl_W, C, 1.f, 1.f))) return rc;
  return launch_cluster_dR(m, R, m->ccells, nc, C, type, scale, m->cdM, m->grads + m->cl_R);
}

extern "C" int sbr_train_step_cluster(sbr_model* m, const int32_t* X, const float* mask, const int32_t* Y_all, int n_all,
                                      int row_offset, const int32_t* samples, int S, const int32_t* cluster_samples, int Sc,
                                      const float* noise, float scale, int B, float* cost, float* cluster_cost) {
  CHECK_STICKY(m);
  if (m->n_clusters <= 0) { sbr_set_error(m, SBR_E_ARG, "model was not created with sbr_create_cluster"); return SBR_E_ARG; }
  if (!cluster_samples) Sc = S;
  if (!Y_all || !samples || S < 1 || S > m->cfg.n_samples || Sc < 1 || Sc > m->n_csamples || n_all < B || n_all > m->global_batch ||
      row_offset < 0 || row_offset + B > n_all || !(scale == scale)) {
    sbr_set_error(m, SBR_E_ARG, "bad cluster-step arguments (S=%d Sc=%d n_all=%d row_offset=%d B=%d)", S, Sc, n_all, row_offset, B);
    return SBR_E_ARG;
  }
  const int32_t* cs = cluster_samples ? cluster_samples : samples;
  int rc;
  if ((rc = begin_step(m))) return rc;
  stage_mark(m, 0);
  BatchSlot& s = m->slots[0];
  if ((rc = stage_common(m, s, X, mask, B))) return rc;
  for (int i = 0; i < n_all + std::max(S, Sc); ++i) {
    const int a = i < n_all ? Y_all[i] : (i - n_all < S ? samples[i - n_all] : 0);
    const int b = i < n_all ? 0 : (i - n_all < Sc ? cs[i - n_all] : 0);
    if (a < 0 || a >= m->N || b < 0 || b >= m->N) { sbr_set_error(m, SBR_E_RANGE, "target/sample id outside [0,%d)", m->N); return SBR_E_RANGE; }
  }
  CU_TRY(m, cudaMemcpyAsync(m->cells, Y_all, (size_t)n_all * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(m->cells + n_all, samples, (size_t)S * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(m->ccells, Y_all, (size_t)n_all * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(m->ccells + n_all, cs, (size_t)Sc * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  if (noise) CU_TRY(m, cudaMemcpyAsync(m->cnoise, noise, (size_t)B * m->n_clusters * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  const float inv_gb = 1.f / (float)(m->cfg.global_batch > 0 ? m->cfg.global_batch : s.B * m->cfg.n_ranks);
  if ((rc = forward_stack(m, s))) return rc;
  // recommendation branch: the sampled model's BlackoutLayer with unit weights and no tanh (rnn_cluster.py:222-228)
  if ((rc = sampled_output(m, m->cluster_loss, false, nullptr, B, n_all, row_offset, S, inv_gb))) return rc;
  if ((rc = cluster_branch(m, B, n_all, row_offset, Sc, noise != nullptr, scale, inv_gb))) return rc;
  stage_mark(m, 4);
  if ((rc = backward_stack(m, s))) return rc;
  float local_cost;
  if ((rc = finish_step(m, cost ? cost : &local_cost))) return rc;
  if (cluster_cost) *cluster_cost = m->h_cost[1];
  return 0;
}

extern "C" int sbr_cluster_test_topk(sbr_model* m, const int32_t* X, const float* mask, int B, const int32_t* excl_offsets,
                                     const int32_t* excl_ids, int k, int32_t* ids_full, int32_t* ids_cluster,
                                     int32_t* selected, float* n_used) {
  CHECK_STICKY(m);
  if (m->n_clusters <= 0) { sbr_set_error(m, SBR_E_ARG, "model was not created with sbr_create_cluster"); return SBR_E_ARG; }
  if (!ids_full || !ids_cluster || !selected || !n_used || k < 1 || k > 64 || k > m->N) {
    sbr_set_error(m, SBR_E_ARG, "cluster_test_topk: bad arguments (k must be in [1, min(64, n_items)])");
    return SBR_E_ARG;
  }
  int rc = scores_device(m, X, mask, B, /*softmax=*/1);
  if (rc) return rc;
  const int N = m->N, C = m->n_clusters, H = m->H_last, ld = (int)round_up(N, 4);
  if (!m->logits2 && (rc = dev_alloc(m, &m->logits2, (size_t)m->B * ld, false))) return rc;
  if ((rc = launch_gemm(m, false, false, B, C, H, m->h_last, H, m->params + m->cl_W, C, m->cq, C, 1.f, 0.f))) return rc;
  if ((rc = launch_cluster_hard(m, m->logits, ld, m->cq, m->params + m->cl_R, B, N, C, m->cluster_type, m->logits2, m->csel, m->cnused))) return rc;
  const int32_t* d_off = nullptr;
  if ((rc = upload_exclusions(m, B, excl_offsets, excl_ids, &d_off))) return rc;
  if ((rc = launch_topk(m, m->logits, ld, B, N, d_off, m->excl_ids, k, 0, m->topk_ids))) return rc;
  CU_TRY(m, cudaMemcpyAsync(ids_full, m->topk_ids, (size_t)B * k * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  if ((rc = launch_topk(m, m->logits2, ld, B, N, d_off, m->excl_ids, k, 0, m->topk_ids))) return rc;
  CU_TRY(m, cudaMemcpyAsync(ids_cluster, m->topk_ids, (size_t)B * k * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaMemcpyAsync(selected, m->csel, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaMemcpyAsync(n_used, m->cnused, (size_t)B * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  return 0;
}

extern "C" int sbr_cluster_build(sbr_model* m, int32_t* sizes) {
  CHECK_STICKY(m);
  if (m->n_clusters <= 0) { sbr_set_error(m, SBR_E_ARG, "model was not created with sbr_create_cluster"); return SBR_E_ARG; }
  CU_TRY(m, cudaSetDevice(m->dev));
  const int N = m->N, C = m->n_clusters;
  int rc;
  if ((rc = launch_cluster_csr(m, m->params + m->cl_R, N, C))) return rc;
  std::vector<int32_t> off(C + 1);
  CU_TRY(m, cudaMemcpyAsync(off.data(), m->cl_off, (C + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  const int64_t total = off[C];
  int max_size = 0;
  for (int j = 0; j < C; ++j) max_size = std::max(max_size, off[j + 1] - off[j]);
  if (total > m->cl_cap_items || !m->cl_items) {
    if (m->cl_items) cudaFree(m->cl_items);
    m->cl_items = nullptr;
    m->cl_cap_items = std::max<int64_t>(total, 1);
    if ((rc = dev_alloc(m, &m->cl_items, (size_t)m->cl_cap_items, false))) return rc;
  }
  if (max_size > m->cl_cap_rows || !m->cl_Wg) {
    if (m->cl_Wg) cudaFree(m->cl_Wg);
    m->cl_Wg = nullptr;
    m->cl_cap_rows = std::max(max_size, 1);
    if ((rc = dev_alloc(m, &m->cl_Wg, (size_t)m->cl_cap_rows * m->H_last, false))) return rc;
  }
  if ((rc = launch_cluster_fill(m, m->params + m->cl_R, N, C))) return rc;
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  m->cl_hoff = off;
  if (sizes)
    for (int j = 0; j < C; ++j) sizes[j] = off[j + 1] - off[j];
  return 0;
}

extern "C" int sbr_cluster_topk(sbr_model* m, const int32_t* X, const float* mask, int B, const int32_t* excl_offsets,
                                const int32_t* excl_ids, int k, int32_t* ids_out, int32_t* n_out, int32_t* selected_out,
                                int use_clusters) {
  CHECK_STICKY(m);
  if (m->n_clusters <= 0) { sbr_set_error(m, SBR_E_ARG, "model was not created with sbr_create_cluster"); return SBR_E_ARG; }
  if (!ids_out || !n_out || k < 1 || k > 64 || k > m->N) { sbr_set_error(m, SBR_E_ARG, "cluster_topk: k must be in [1, min(64, n_items)]"); return SBR_E_ARG; }
  const int N = m->N, C = m->n_clusters, H = m->H_last;
  int rc;
  if (!use_clusters) {   // --ignore_clusters: the whole catalog, raw scores, -inf exclusion (rnn_cluster.py:314-321)
    if ((rc = sbr_topk(m, X, mask, B, excl_offsets, excl_ids, k, 2, ids_out))) return rc;
    for (int b = 0; b < B; ++b) n_out[b] = N;
    if (selected_out)
      for (int b = 0; b < B; ++b) selected_out[b] = -1;
    return 0;
  }
  if (m->cl_hoff.empty()) { sbr_set_error(m, SBR_E_ARG, "cluster_topk: call sbr_cluster_build first"); return SBR_E_ARG; }
  BatchSlot& s = m->slots[0];
  CU_TRY(m, cudaSetDevice(m->dev));
  if ((rc = stage_common(m, s, X, mask, B))) return rc;
  const bool prof = m->profiling;
  m->profiling = false;
  rc = forward_stack(m, s);
  m->profiling = prof;
  if (rc) return rc;
  if ((rc = launch_gemm(m, false, false, B, C, H, m->h_last, H, m->params + m->cl_W, C, m->cq, C, 1.f, 0.f))) return rc;
  if ((rc = launch_cluster_argmax(m, m->cq, B, C, m->csel))) return rc;
  std::vector<int32_t> sel(B), perm(B);
  CU_TRY(m, cudaMemcpyAsync(sel.data(), m->csel, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  // rows grouped by selected cluster: each cluster's item rows are gathered once and scored by one GEMM
  for (int b = 0; b < B; ++b) perm[b] = b;
  std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return sel[a] < sel[b]; });
  const std::vector<int32_t>& off = m->cl_hoff;
  int ld = 4;
  for (int b = 0; b < B; ++b) ld = std::max<int>(ld, (int)round_up(off[sel[b] + 1] - off[sel[b]], 4));
  CU_TRY(m, cudaMemcpyAsync(m->cperm, perm.data(), (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  if ((rc = launch_gather_table_rows(m, m->h_last, nullptr, m->cperm, B, H, m->ch_sorted, nullptr))) return rc;
  for (int r0 = 0; r0 < B;) {
    const int c = sel[perm[r0]];
    int r1 = r0;
    while (r1 < B && sel[perm[r1]] == c) ++r1;
    const int nc = off[c + 1] - off[c];
    if (nc > 0) {
      if ((rc = launch_gather_table_rows(m, m->params + m->out_WT, nullptr, m->cl_items + off[c], nc, H, m->cl_Wg, nullptr))) return rc;
      if ((rc = launch_gemm(m, false, true, r1 - r0, nc, H, m->ch_sorted + (size_t)r0 * H, H, m->cl_Wg, H, m->logits + (size_t)r0 * ld, ld,
                            1.f, 0.f))) return rc;
    }
    r0 = r1;
  }
  const int32_t* d_off = nullptr;
  if ((rc = upload_exclusions(m, B, excl_offsets, excl_ids, &d_off))) return rc;
  if ((rc = launch_cluster_row_topk(m, m->logits, ld, B, m->cperm, m->csel, m->params + m->out_b, d_off, m->excl_ids, k, m->topk_ids))) return rc;
  CU_TRY(m, cudaMemcpyAsync(ids_out, m->topk_ids, (size_t)B * k * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  for (int b = 0; b < B; ++b) {
    n_out[b] = off[sel[b] + 1] - off[sel[b]];
    if (selected_out) selected_out[b] = sel[b];
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// measurement
// ------------------------------------------------------------------------------------------------
extern "C" const char* sbr_stage_name(int i) { return (i >= 0 && i < SBR_N_STAGES) ? kStageNames[i] : ""; }

extern "C" int sbr_set_profiling(sbr_model* m, int on) {
  if (!m) return SBR_E_ARG;
  m->profiling = on != 0;
  return 0;
}

extern "C" int sbr_stage_times(sbr_model* m, float ms[SBR_N_STAGES]) {
  if (!m || !ms) return SBR_E_ARG;
  for (int i = 0; i < SBR_N_STAGES; ++i) ms[i] = m->stage_ms[i];
  return 0;
}

extern "C" int64_t sbr_kernel_launches(const sbr_model* m) { return m ? m->launches : SBR_E_ARG; }
extern "C" int64_t sbr_scan_launches(const sbr_model* m) { return m ? m->scan_launches : SBR_E_ARG; }

extern "C" int sbr_debug_gemm(sbr_model* m, int engine, int ta, int tb, int M, int N, int K, const float* A, int lda,
                              const float* B, int ldb, float* C, int ldc, float alpha, float beta, const float* bias,
                              int reps, float* ms) {
  CHECK_STICKY(m);
  if (!A || !B || !C || M < 1 || N < 1 || K < 1 || reps < 1) { sbr_set_error(m, SBR_E_ARG, "debug_gemm: bad arguments"); return SBR_E_ARG; }
  CU_TRY(m, cudaSetDevice(m->dev));
  const size_t na = (size_t)(ta ? K : M) * lda, nb = (size_t)(tb ? N : K) * ldb, nc = (size_t)M * ldc;
  float *dA = nullptr, *dB = nullptr, *dC = nullptr, *dbias = nullptr;
  int rc = 0;
  if ((rc = dev_alloc(m, &dA, na, false)) || (rc = dev_alloc(m, &dB, nb, false)) || (rc = dev_alloc(m, &dC, nc, false))) return rc;
  if (bias && (rc = dev_alloc(m, &dbias, (size_t)N, false))) return rc;
  CU_TRY(m, cudaMemcpyAsync(dA, A, na * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaMemcpyAsync(dB, B, nb * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  if (bias) CU_TRY(m, cudaMemcpyAsync(dbias, bias, (size_t)N * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  const bool saved = m->use_tc_gemm;
  m->use_tc_gemm = engine != 0;
  CU_TRY(m, cudaMemcpyAsync(dC, C, nc * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  CU_TRY(m, cudaEventRecord(m->timer[0], m->stream));
  for (int r = 0; r < reps && rc == 0; ++r) {
    if (beta != 0.f && r > 0) CU_TRY(m, cudaMemcpyAsync(dC, C, nc * sizeof(float), cudaMemcpyHostToDevice, m->stream));
    if (bias) {
      if (engine != 0) { rc = launch_gemm_tc(m, ta != 0, tb != 0, M, N, K, dA, lda, dB, ldb, dC, ldc, alpha, beta, dbias); if (rc == 1) { sbr_set_error(m, SBR_E_ARG, "debug_gemm: tensor-core kernel does not apply"); rc = SBR_E_ARG; } }
      else rc = launch_gemm_bias(m, tb != 0, M, N, K, dA, lda, dB, ldb, dC, ldc, dbias);
    } else if (engine != 0) {
      rc = launch_gemm_tc(m, ta != 0, tb != 0, M, N, K, dA, lda, dB, ldb, dC, ldc, alpha, beta, nullptr);
      if (rc == 1) { sbr_set_error(m, SBR_E_ARG, "debug_gemm: tensor-core kernel does not apply"); rc = SBR_E_ARG; }
    } else {
      rc = launch_gemm(m, ta != 0, tb != 0, M, N, K, dA, lda, dB, ldb, dC, ldc, alpha, beta);
    }
  }
  m->use_tc_gemm = saved;
  if (rc == 0) {
    CU_TRY(m, cudaEventRecord(m->timer[1], m->stream));
    CU_TRY(m, cudaMemcpyAsync(C, dC, nc * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
    CU_TRY(m, cudaStreamSynchronize(m->stream));
    if (ms) CU_TRY(m, cudaEventElapsedTime(ms, m->timer[0], m->timer[1]));
  }
  cudaFree(dA); cudaFree(dB); cudaFree(dC); if (dbias) cudaFree(dbias);
  return rc;
}

extern "C" int sbr_timer_start(sbr_model* m) {
  CHECK_STICKY(m);
  CU_TRY(m, cudaSetDevice(m->dev));
  CU_TRY(m, cudaStreamSynchronize(m->stream));
  CU_TRY(m, cudaEventRecord(m->timer[0], m->stream));
  return 0;
}

extern "C" int sbr_timer_stop(sbr_model* m, float* ms) {
  CHECK_STICKY(m);
  if (!ms) return SBR_E_ARG;
  CU_TRY(m, cudaSetDevice(m->dev));
  CU_TRY(m, cudaEventRecord(m->timer[1], m->stream));
  CU_TRY(m, cudaEventSynchronize(m->timer[1]));
  CU_TRY(m, cudaEventElapsedTime(ms, m->timer[0], m->timer[1]));
  return 0;
}
