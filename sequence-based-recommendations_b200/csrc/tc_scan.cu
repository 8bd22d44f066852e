// tc_scan.cu -- persistent tensor-core scans for hidden sizes beyond the cluster-resident kernels of rnn_tc.cu
// (H > 224, H % 16 == 0): the whole recurrence of a layer (sparse_lstm.py:377-425,474-481 LSTM; :764-805,843-850 GRU;
// :1120-1152,1190-1197 vanilla) -- or its BPTT (theano.grad of the same, rnn_base.py:183) -- in ONE cooperative
// launch.  Per time step every CTA runs the tc_gemm.cu pipeline (TMA fp32 tiles -> 3xTF32 split -> tcgen05.mma with
// the A operand in TMEM) on its tile and the fused cell / gate-gradient math in the epilogue; the CTAs that share a
// batch tile hand each other the step's result through global memory and a per-tile release/acquire counter (no
// grid-wide barrier: batch tiles run their own number of steps and leave when their longest row is done).
//
//   forward   CTA = 128 batch rows x (G gates of 8 hidden units).  A = h_{t-1} tile [128 x H] streamed by TMA from
//             the state trajectory; B = the CTA's 8-unit slice of W_hid, split once in step 0 and kept resident in
//             shared memory; cell state and previous hidden state live in registers (thread = batch row).
//   backward  CTA = 128 hidden units k x 32 batch rows.  A = W_hid rows [128 x G*H] streamed by TMA every step (runs
//             ahead of the recurrence: it does not depend on it); B = da_{t+1} rows of the tile's 32 batch rows;
//             D[k][b] = sum_c W_hid[k][c] da_{t+1}[b][c].  The carried dh / d(cell state) of every (b, k) live in shared
//             memory, the bias / peephole gradient sums in registers (thread = k); the step "t = -1" yields the
//             gradients of the learned initial states.
#include <cooperative_groups.h>

#include "common.cuh"
#include "tc_common.cuh"

using namespace tcx;

namespace {

constexpr int SC_KC = 32;          // k per chunk (4 MMA k-steps)
constexpr int SC_ST = 7;           // converted-operand stages (TMEM slots of A, 64 columns each: 64 + 7*64 = 512 columns; shared-memory
                                   // slots of B in the backward).  Deep on purpose: a slot is only free again once the MMAs that read it
                                   // have COMPLETED (tcgen05.commit), ~1.5k cycles after the converter filled it
constexpr int SC_BN = 32;          // MMA N: forward 4 gates x 8 units, backward 32 batch rows
constexpr int SC_U = 8;
constexpr int SC_NT = 352;         // warps 0-3 A converters + epilogue, 4-7 B converters, 8 MMA, 9 A producer, 10 B producer
constexpr int SC_LOOK_MAX = 8;     // raw A ring depth (16 KB per stage)
constexpr int SC_LOOKB = 4;        // raw B ring depth (4 KB per stage)
constexpr int SC_MAX_CHUNKS = 16;  // forward: resident B covers K = H <= 512

struct ScanArgs {
  CUtensorMap tmA, tmB, tmB2;
  int B, H, G, t_max, n_chunks, look;
  const int32_t* len;
  const float* peep;
  unsigned int* sync;            // one counter per batch tile, zeroed before the launch
  // forward
  const float* Xg; float* hs; float* cs; float* act;
  // backward
  const float* act_r; const float* cs_r; const float* hs_r; const float* dhs; const float* dh_last;
  float* dXg; float* dac;
  float* g_h_init; float* g_c_init; float* g_peep; float* g_b;
  float clip;
  int relu;            // vanilla cell: rectifier instead of tanh (dense-input layers)
  int b_split;                   // GRU: k >= 2H of da comes from dac (tmB2)
  long long* dbg;                // optional clock64 phase sums of CTA (0,0,0) (SBR_SCAN_TIMELINE)
  int acq_spin;                  // experiments (SBR_SCAN_ACQ_SPIN): acquire loads in the counter spin / cluster-acquire barrier waits, as before
  int fence_mode;                // publication fences (SBR_SCAN_FENCE, experiments): see publish_step()
  int tile0;                     // first batch tile of this launch (large batches run as several launches over tile slices)
};

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Spin on a step counter: relaxed polls, ONE acquire fence once the value is there (an acquire load per poll drags an
// L1 invalidation -- CCTL.IVALL -- behind every iteration of the spin)
__device__ __forceinline__ void wait_counter_gpu(const unsigned int* p, unsigned int need) {
  unsigned int v;
  do { asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); } while (v < need);
  asm volatile("fence.acq_rel.gpu;" ::: "memory");
}
__device__ __forceinline__ void red_release_gpu(unsigned int* p, unsigned int v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// The 128 epilogue threads have stored this step's results to global memory; make them visible to the TMA loads of the
// other CTAs of the tile and count the CTA in.  mode 0: every thread fences (gpu scope + async proxy) before the
// barrier; 1: every thread only orders against the async proxy; 2: one thread fences after the barrier (the CTA barrier
// makes the other threads' stores cumulative with its release); 3 (default): only the gpu-scope release of the counter
// update -- the consumer pairs it with ld.acquire.gpu + fence.proxy.async before its TMA loads.
__device__ __forceinline__ void publish_step(int mode, int tid, uint64_t* tmem_empty, unsigned int* ctr) {
  if (mode == 0) { __threadfence(); fence_proxy_async_all(); }
  else if (mode == 1) fence_proxy_async_all();
  tc_fence_before();
  epi_bar();
  if (tid == 0) {
    mbar_arrive(tmem_empty);
    if (mode == 2) { __threadfence(); fence_proxy_async_all(); }
    red_release_gpu(ctr, 1u);      // mode 3: the release itself (gpu scope) after the CTA barrier is the only fence
  }
}

__device__ __forceinline__ uint32_t map_to_rank(uint32_t cta_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes, uint32_t mbar_cluster_addr) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(dst_cluster_addr), "r"(src_cta_addr), "r"(bytes), "r"(mbar_cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
               "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
               "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ void tma_load_2d_multicast(void* smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar, uint16_t mask) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
               :: "r"(smem_u32(smem_dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" :: "r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void fence_acq_rel_cluster() { asm volatile("fence.acq_rel.cluster;" ::: "memory"); }

struct ScanBars {
  uint64_t rawA_full[SC_LOOK_MAX], rawA_empty[SC_LOOK_MAX];
  uint64_t rawB_full[SC_LOOKB], rawB_empty[SC_LOOKB];
  uint64_t full[SC_ST], empty[SC_ST];           // converted operands of a stage ready / consumed by the MMAs
  uint64_t fullB[SC_MAX_CHUNKS];                 // forward: resident B chunk converted (once)
  uint64_t done, tmem_empty;
};

__device__ __forceinline__ void init_bars(ScanBars& b, int full_count) {
  for (int i = 0; i < SC_LOOK_MAX; ++i) { mbar_init(&b.rawA_full[i], 1); mbar_init(&b.rawA_empty[i], 4); }
  for (int i = 0; i < SC_LOOKB; ++i) { mbar_init(&b.rawB_full[i], 1); mbar_init(&b.rawB_empty[i], 4); }
  for (int i = 0; i < SC_ST; ++i) { mbar_init(&b.full[i], full_count); mbar_init(&b.empty[i], 1); }
  for (int i = 0; i < SC_MAX_CHUNKS; ++i) mbar_init(&b.fullB[i], 4);
  mbar_init(&b.done, 1);
  mbar_init(&b.tmem_empty, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// A converter: raw fp32 tile [128 rows][32 k] (TMA 128B swizzle) -> hi | lo in the stage's TMEM slot.  gc = running chunk index.
__device__ __forceinline__ void convert_a_chunk(ScanBars& bars, const uint8_t* rawA0, int look, uint32_t tA, uint32_t lane_off,
                                                int tid, int lane, int gc) {
  const int rs = gc % look;
  mbar_wait(&bars.rawA_full[rs], (gc / look) & 1);
  float cur[SC_KC];
  const float* src = reinterpret_cast<const float*>(rawA0 + (size_t)rs * (128 * SC_KC * 4));
#pragma unroll
  for (int q = 0; q < SC_KC / 4; ++q) {
    const float4 x = *reinterpret_cast<const float4*>(src + tid * 32 + ((q ^ (tid & 7)) << 2));
    cur[4 * q] = x.x; cur[4 * q + 1] = x.y; cur[4 * q + 2] = x.z; cur[4 * q + 3] = x.w;
  }
  __syncwarp();
  if (lane == 0) mbar_arrive(&bars.rawA_empty[rs]);
  const int s = gc % SC_ST;
  if (gc >= SC_ST) {
    mbar_wait(&bars.empty[s], ((gc / SC_ST) - 1) & 1);
    tc_fence_after();
  }
  const uint32_t dst = tA + (uint32_t)s * 64u + lane_off;
#pragma unroll
  for (int q = 0; q < SC_KC / 8; ++q) {
    uint32_t hi[8], lo[8];
    split8(cur + 8 * q, hi, lo);
    tmem_st8(dst + 8 * q, hi);
    tmem_st8(dst + SC_KC + 8 * q, lo);
  }
  tmem_wait_st();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(&bars.full[s]);
}

__device__ __forceinline__ void issue_chunk_mmas(uint32_t tD1, uint32_t tD2, uint32_t ta, uint32_t sb, uint32_t idesc, uint32_t& acc) {
  constexpr uint32_t lbo = SC_BN * 16u, part = SC_BN * SC_KC * 4u;
  // descriptors built once per chunk; a k-step advances the start-address field (16-byte units) by two core matrices
  uint64_t bhi = make_desc(sb, lbo, 128), blo = make_desc(sb + part, lbo, 128);
  constexpr uint64_t adv = (2u * lbo) >> 4;
#pragma unroll
  for (int ks = 0; ks < SC_KC / 8; ++ks) {
    mma_ts(tD1, ta + 8 * ks, bhi, idesc, acc);
    mma_ts(tD2, ta + 8 * ks, blo, idesc, acc);
    mma_ts(tD2, ta + SC_KC + 8 * ks, bhi, idesc, 1);
    acc = 1;
    bhi += adv; blo += adv;
  }
}

// split one 16-byte (n, 4k) element group into the canonical K-major tile [k/4][32][4], hi then lo
__device__ __forceinline__ void store_b_split(uint8_t* st, int n, int kq, float4 x) {
  float4 h, l;
  h.x = tf32_hi(x.x); h.y = tf32_hi(x.y); h.z = tf32_hi(x.z); h.w = tf32_hi(x.w);
  l.x = x.x - h.x; l.y = x.y - h.y; l.z = x.z - h.z; l.w = x.w - h.w;
  const uint32_t off = (uint32_t)kq * (SC_BN * 16u) + (uint32_t)n * 16u;
  *reinterpret_cast<float4*>(st + off) = h;
  *reinterpret_cast<float4*>(st + SC_BN * SC_KC * 4 + off) = l;
}

// ================================================================================================ forward
template <int G>
__global__ void __launch_bounds__(SC_NT, 1) tc_scan_fwd_kernel(const __grid_constant__ ScanArgs a) {
  extern __shared__ __align__(1024) uint8_t sc_smem[];
  __shared__ ScanBars bars;
  __shared__ __align__(8) uint64_t slot_free[SC_LOOK_MAX];     // every CTA of the cluster has consumed the raw A slot
  __shared__ uint32_t tmem_base_s;
  __shared__ int t_end_s;
  // The CTAs of a cluster are consecutive unit slices of the SAME batch tile: they all need the same h_{t-1} tile, so
  // each one fetches 128/CS of its rows per chunk and multicasts them into every CTA of the cluster (the tile leaves
  // L2 once per cluster instead of once per CTA).
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int CS = (int)cluster.num_blocks(), crank = (int)cluster.block_rank();
  uint8_t* const base = sc_smem + ((1024u - (smem_u32(sc_smem) & 1023u)) & 1023u);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int u0 = blockIdx.x * SC_U, m0 = (blockIdx.y + a.tile0) * 128;
  const int B = a.B, H = a.H, GH = G * H, NC = a.n_chunks, LOOK = a.look;
  constexpr uint32_t stageB = SC_BN * SC_KC * 8u;              // converted B chunk: hi + lo
  uint8_t* convB = base;                                        // [NC] resident converted W_hid slice
  uint8_t* rawA0 = convB + (size_t)NC * stageB;                 // [LOOK][128][32] fp32
  uint8_t* rawB0 = rawA0 + (size_t)LOOK * (128 * SC_KC * 4);    // [SC_LOOKB][G][32 k][8 units] fp32

  if (tid == 0) {
    t_end_s = 0;
    init_bars(bars, 4);
    for (int i = 0; i < SC_LOOK_MAX; ++i) mbar_init(&slot_free[i], CS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (tid < 128) {
    const int b = m0 + tid;
    const int l = b < B ? min(__ldg(a.len + b), a.t_max) : 0;
    atomicMax(&t_end_s, l);
  }
  __syncthreads();
  if (CS > 1) cluster.sync();       // every CTA's barriers exist before any multicast / remote arrive
  const int t_end = t_end_s;
  const uint32_t tmem = tmem_base_s;
  const uint32_t tD1 = tmem, tD2 = tmem + SC_BN, tA = tmem + 64;
  const int group_ctas = gridDim.x;
  unsigned int* ctr = a.sync + blockIdx.y;

  if (warp < 4) {
    // ------------------------------------------------------------ A converter + epilogue (thread = batch row)
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    const int b = m0 + tid;
    const int my_len = b < B ? min(__ldg(a.len + b), a.t_max) : 0;
    float hreg[8], creg[8], wci[8], wcf[8], wco[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      hreg[j] = __ldg(a.hs + u0 + j);          // block 0 row 0 == learned init (broadcast by the launcher)
      creg[j] = 0.f; wci[j] = wcf[j] = wco[j] = 0.f;
      if (G == 4) {
        creg[j] = __ldg(a.cs + u0 + j);
        wci[j] = __ldg(a.peep + u0 + j); wcf[j] = __ldg(a.peep + H + u0 + j); wco[j] = __ldg(a.peep + 2 * H + u0 + j);
      }
    }
    int gc = 0;
    const bool tl = a.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0;
    long long ph[6] = {0, 0, 0, 0, 0, 0}, tl0 = tl ? clock64() : 0;
#define SC_ACC(i) do { if (tl) { const long long n_ = clock64(); ph[i] += n_ - tl0; tl0 = n_; } } while (0)
    for (int t = 0; t < t_end; ++t) {
      for (int c = 0; c < NC; ++c, ++gc) {
        if (c == 1) SC_ACC(0);      // first chunk: includes the wait for the other CTAs and the first TMA tile
        convert_a_chunk(bars, rawA0, LOOK, tA, lane_off, tid, lane, gc);
      }
      SC_ACC(1);
      // this step's input pre-activations, requested before the accumulators are complete
      const bool active = t < my_len;
      float xg[G][8];
      if (active) {
#pragma unroll
        for (int g = 0; g < G; ++g) ld8(a.Xg + ((long long)t * B + b) * GH + g * H + u0, xg[g]);
      }
      mbar_wait(&bars.done, t & 1);
      tc_fence_after();
      SC_ACC(2);
      float pre[32];
      {
        float d0[16], d1[16], w0[16], w1[16];
        tmem_ld16(tD1 + lane_off, d0); tmem_ld16(tD1 + lane_off + 16, d1);
        tmem_ld16(tD2 + lane_off, w0); tmem_ld16(tD2 + lane_off + 16, w1);
#pragma unroll
        for (int i = 0; i < 16; ++i) { pre[i] = d0[i] + w0[i]; pre[16 + i] = d1[i] + w1[i]; }
      }
      float sv[4][8];
      if (active) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if constexpr (G == 4) {
            const float c_prev = creg[j];
            const float ig = sigmoid_fast(xg[0][j] + pre[j] + c_prev * wci[j]);
            const float fg = sigmoid_fast(xg[1][j] + pre[8 + j] + c_prev * wcf[j]);
            const float gg = tanh_fast(xg[2][j] + pre[16 + j]);
            const float c_new = fg * c_prev + ig * gg;
            const float og = sigmoid_fast(xg[3][j] + pre[24 + j] + c_new * wco[j]);
            hreg[j] = og * tanh_fast(c_new);
            creg[j] = c_new;
            sv[0][j] = ig; sv[1][j] = fg; sv[2][j] = gg; sv[3][j] = og;
          } else if constexpr (G == 3) {
            const float r = sigmoid_fast(pre[j] + xg[0][j]);
            const float uu = sigmoid_fast(pre[8 + j] + xg[1][j]);
            const float ac = pre[16 + j];
            const float cand = tanh_fast(xg[2][j] + r * ac);
            hreg[j] = (1.f - uu) * hreg[j] + uu * cand;
            sv[0][j] = r; sv[1][j] = uu; sv[2][j] = cand; sv[3][j] = ac;
          } else {
            const float z = xg[0][j] + pre[j];
            hreg[j] = a.relu ? fmaxf(z, 0.f) : tanh_fast(z);
          }
        }
        st8(a.hs + ((long long)(t + 1) * B + b) * H + u0, hreg);
      }
      SC_ACC(3);
      // publish: the state block t+1 of this CTA's units is in global memory; the accumulators may be overwritten
      publish_step(a.fence_mode, tid, &bars.tmem_empty, ctr);
      // what only the backward pass reads (cell state, gate activations) is stored after the release: it does not
      // have to drain before the other CTAs may start the next step
      if (active) {
        if (G == 4) st8(a.cs + ((long long)(t + 1) * B + b) * H + u0, creg);
        if (G > 1) {
#pragma unroll
          for (int g = 0; g < 4; ++g) st8(a.act + ((long long)t * B + b) * 4 * H + g * H + u0, sv[g]);
        }
      }
      SC_ACC(4);
    }
    if (tl) { for (int i = 0; i < 6; ++i) a.dbg[i] = ph[i]; a.dbg[6] = t_end; }
  } else if (warp < 8) {
    // ------------------------------------------------------------ B converter: W_hid slice, once
    const int bt = tid - 128;
    if (t_end > 0) {
      for (int c = 0; c < NC; ++c) {
        const int rs = c % SC_LOOKB;
        mbar_wait(&bars.rawB_full[rs], (c / SC_LOOKB) & 1);
        const float* src = reinterpret_cast<const float*>(rawB0 + (size_t)rs * (4 * SC_KC * SC_U * 4));
        float4 cur[2];
#pragma unroll
        for (int it = 0; it < 2; ++it) {
          const int idx = it * 128 + bt, kq = idx / SC_BN, n = idx - kq * SC_BN;
          const int g = n / SC_U, j = n - g * SC_U;
          const float* q = src + g * (SC_KC * SC_U) + (4 * kq) * SC_U + j;
          cur[it] = g < G ? make_float4(q[0], q[SC_U], q[2 * SC_U], q[3 * SC_U]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.rawB_empty[rs]);
#pragma unroll
        for (int it = 0; it < 2; ++it) {
          const int idx = it * 128 + bt, kq = idx / SC_BN, n = idx - kq * SC_BN;
          store_b_split(convB + (size_t)c * stageB, n, kq, cur[it]);
        }
        proxy_fence_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.fullB[c]);
      }
    }
  } else if (warp == 8) {
    // ------------------------------------------------------------ MMA issuer
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32(128, SC_BN);
      int gc = 0;
      for (int t = 0; t < t_end; ++t) {
        if (t > 0) { mbar_wait(&bars.tmem_empty, (t - 1) & 1); tc_fence_after(); }
        uint32_t acc = 0;
        for (int c = 0; c < NC; ++c, ++gc) {
          const int s = gc % SC_ST;
          mbar_wait(&bars.full[s], (gc / SC_ST) & 1);
          if (t == 0) mbar_wait(&bars.fullB[c], 0);
          tc_fence_after();
          issue_chunk_mmas(tD1, tD2, tA + (uint32_t)s * 64u, smem_u32(convB + (size_t)c * stageB), idesc, acc);
          umma_commit(&bars.empty[s]);
        }
        umma_commit(&bars.done);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------ A producer: h_{t-1} tile of every step
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmA) : "memory");
      int gc = 0;
      for (int t = 0; t < t_end; ++t) {
        const long long w0 = a.dbg ? clock64() : 0;
        if (t > 0) {
          const unsigned int need = (unsigned int)t * (unsigned int)group_ctas;
          if (a.acq_spin) { while (ld_acquire_gpu(ctr) < need) { } } else wait_counter_gpu(ctr, need);
          fence_proxy_async_all();
        }
        if (a.dbg && blockIdx.x == 0 && blockIdx.y == 0) a.dbg[8] += clock64() - w0;
        for (int c = 0; c < NC; ++c, ++gc) {
          const int rs = gc % LOOK;
          if (gc >= LOOK) {
            mbar_wait(&bars.rawA_empty[rs], ((gc / LOOK) - 1) & 1);        // this CTA's converters are done with the slot
            if (CS > 1) {
              // tell every CTA of the cluster, then wait until all of them have told me: only then may anybody multicast into it
              fence_acq_rel_cluster();
              for (int q = 0; q < CS; ++q) mbar_arrive_remote_relaxed(map_to_rank(smem_u32(&slot_free[rs]), q));
              mbar_wait_cluster(&slot_free[rs], ((gc / LOOK) - 1) & 1);
            }
          }
          mbar_arrive_expect_tx(&bars.rawA_full[rs], 128 * SC_KC * 4);
          if (CS > 1) {
            const int rows = 128 / CS;
            tma_load_2d_multicast(rawA0 + (size_t)rs * (128 * SC_KC * 4) + (size_t)crank * rows * (SC_KC * 4), &a.tmA, c * SC_KC,
                                  t * B + m0 + crank * rows, &bars.rawA_full[rs], (uint16_t)((1u << CS) - 1u));
          } else {
            tma_load_2d(rawA0 + (size_t)rs * (128 * SC_KC * 4), &a.tmA, c * SC_KC, t * B + m0, &bars.rawA_full[rs]);
          }
        }
      }
    }
  } else if (warp == 10) {
    // ------------------------------------------------------------ B producer: the 8-unit slice of W_hid, gate by gate
    if (lane == 0 && t_end > 0) {
      asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmB) : "memory");
      for (int c = 0; c < NC; ++c) {
        const int rs = c % SC_LOOKB;
        if (c >= SC_LOOKB) mbar_wait(&bars.rawB_empty[rs], ((c / SC_LOOKB) - 1) & 1);
        mbar_arrive_expect_tx(&bars.rawB_full[rs], (uint32_t)G * SC_KC * SC_U * 4u);
        uint8_t* dst = rawB0 + (size_t)rs * (4 * SC_KC * SC_U * 4);
        for (int g = 0; g < G; ++g) tma_load_2d(dst + g * (SC_KC * SC_U * 4), &a.tmB, g * H + u0, c * SC_KC, &bars.rawB_full[rs]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CS > 1) cluster.sync();       // nobody leaves while a peer may still multicast into / arrive on this CTA
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512));
}

// ================================================================================================ backward
template <int G>
__global__ void __launch_bounds__(SC_NT, 1) tc_scan_bwd_kernel(const __grid_constant__ ScanArgs a) {
  extern __shared__ __align__(1024) uint8_t sc_smem[];
  __shared__ ScanBars bars;
  __shared__ uint32_t tmem_base_s;
  __shared__ int t_end_s;
  uint8_t* const base = sc_smem + ((1024u - (smem_u32(sc_smem) & 1023u)) & 1023u);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n0 = (blockIdx.x + a.tile0) * SC_BN, m0 = blockIdx.y * 128;
  const int B = a.B, H = a.H, GH = G * H, NC = a.n_chunks, LOOK = a.look;
  constexpr uint32_t stageB = SC_BN * SC_KC * 8u;
  uint8_t* convB = base;                                                // [SC_ST] converted da chunks
  float* carry_s = reinterpret_cast<float*>(convB + SC_ST * stageB);    // [32 b][128 k] dh carried to the previous step
  float* dcs_s = carry_s + SC_BN * 128;                                 // [32 b][128 k] d(cell state)
  uint8_t* rawA0 = reinterpret_cast<uint8_t*>(dcs_s + SC_BN * 128);     // [LOOK][128][32]
  uint8_t* rawB0 = rawA0 + (size_t)LOOK * (128 * SC_KC * 4);            // [SC_LOOKB][32][32]

  if (tid == 0) { t_end_s = 0; init_bars(bars, 8); }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (tid < SC_BN) {
    const int b = n0 + tid;
    atomicMax(&t_end_s, b < B ? min(__ldg(a.len + b), a.t_max) : 0);
  }
  __syncthreads();
  const int t_end = t_end_s;
  // masked tail [t_end, t_max): exactly zero gradients wrt the input pre-activations
  for (int t = t_end; t < a.t_max; ++t)
    for (int i = tid; i < SC_BN * 128; i += SC_NT) {
      const int b = n0 + (i >> 7), k = m0 + (i & 127);
      if (b < B && k < H) {
        const long long row = (long long)t * B + b;
        for (int g = 0; g < G; ++g) a.dXg[row * GH + g * H + k] = 0.f;
        if (G == 3) a.dac[row * H + k] = 0.f;
      }
    }
  const uint32_t tmem = tmem_base_s;
  const uint32_t tD1 = tmem, tD2 = tmem + SC_BN, tA = tmem + 64;
  const int group_ctas = gridDim.y;
  unsigned int* ctr = a.sync + blockIdx.x;
  const int n_steps = t_end + 1;            // s = 0 .. t_end  <->  t = t_end-1 .. -1 ; the product exists for s >= 1

  if (warp < 4) {
    // ------------------------------------------------------------ A converter + epilogue (thread = hidden unit k)
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    const int k = m0 + tid;
    const bool k_ok = k < H;
    float wci = 0.f, wcf = 0.f, wco = 0.f;
    if (G == 4 && k_ok) { wci = __ldg(a.peep + k); wcf = __ldg(a.peep + H + k); wco = __ldg(a.peep + 2 * H + k); }
    for (int j = 0; j < SC_BN; ++j) {
      const int b = n0 + j;
      carry_s[j * 128 + tid] = (a.dh_last && k_ok && b < B) ? __ldg(a.dh_last + (long long)b * H + k) : 0.f;
      dcs_s[j * 128 + tid] = 0.f;
    }
    float dpe0 = 0.f, dpe1 = 0.f, dpe2 = 0.f, dbs[4] = {0.f, 0.f, 0.f, 0.f};
    int gc = 0;
    for (int s = 0; s < n_steps; ++s) {
      const int t = t_end - 1 - s;
      if (s > 0) {
        for (int c = 0; c < NC; ++c, ++gc) convert_a_chunk(bars, rawA0, LOOK, tA, lane_off, tid, lane, gc);
        mbar_wait(&bars.done, (s - 1) & 1);
        tc_fence_after();
      }
      float sum_h = 0.f, sum_c = 0.f;
      for (int c0 = 0; c0 < SC_BN; c0 += 16) {
        float P[16];
        if (s > 0) {
          float w[16];
          tmem_ld16(tD1 + lane_off + c0, P);
          tmem_ld16(tD2 + lane_off + c0, w);
#pragma unroll
          for (int i = 0; i < 16; ++i) P[i] += w[i];
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) P[i] = 0.f;
        }
        if (!k_ok) continue;
        if (t < 0) {
          // step "t = -1": dh flowing into the learned initial state, summed over the rows
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            if (n0 + c0 + j < B) { sum_h += carry_s[(c0 + j) * 128 + tid] + P[j]; sum_c += dcs_s[(c0 + j) * 128 + tid]; }
          }
          continue;
        }
        // four batch rows at a time: all their saved tensors are requested before the first one is used
#pragma unroll
        for (int j0 = 0; j0 < 16; j0 += 4) {
          float sv[4][7];
          bool act_[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int b = n0 + c0 + j0 + q;
            act_[q] = b < B && t < min(__ldg(a.len + b), a.t_max);
            if (act_[q]) {
              const long long row = (long long)t * B + b;
              if (G > 1) {
                const float* ap = a.act_r + row * 4 * H + k;
                sv[q][0] = __ldg(ap); sv[q][1] = __ldg(ap + H); sv[q][2] = __ldg(ap + 2 * H); sv[q][3] = __ldg(ap + 3 * H);
              }
              if (G == 4) { sv[q][4] = __ldg(a.cs_r + row * H + k); sv[q][5] = __ldg(a.cs_r + (row + B) * H + k); }
              if (G == 3) sv[q][4] = __ldg(a.hs_r + row * H + k);
              if (G == 1) sv[q][0] = __ldg(a.hs_r + (row + B) * H + k);
              sv[q][6] = a.dhs ? __ldg(a.dhs + row * H + k) : 0.f;
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int j = c0 + j0 + q, b = n0 + j;
            if (b >= B) continue;
            const float dh = carry_s[j * 128 + tid] + P[j0 + q];
            float dx[4] = {0.f, 0.f, 0.f, 0.f}, dacv = 0.f, carry_new = dh;
            if (act_[q]) {
              const float d = dh + sv[q][6];
              if constexpr (G == 4) {
                const float ig = sv[q][0], fg = sv[q][1], gg = sv[q][2], og = sv[q][3], c_prev = sv[q][4], c_new = sv[q][5];
                const float tc = tanh_fast(c_new);
                const float do_pre = d * (tc * og * (1.f - og));
                const float dct = dcs_s[j * 128 + tid] + d * (og * (1.f - tc * tc)) + do_pre * wco;
                const float di_pre = dct * (gg * ig * (1.f - ig));
                const float df_pre = dct * (c_prev * fg * (1.f - fg));
                const float dg_pre = dct * (ig * (1.f - gg * gg));
                dpe0 += di_pre * c_prev; dpe1 += df_pre * c_prev; dpe2 += do_pre * c_new;
                dcs_s[j * 128 + tid] = dct * fg + di_pre * wci + df_pre * wcf;
                dx[0] = clip_sym(di_pre, a.clip); dx[1] = clip_sym(df_pre, a.clip);
                dx[2] = clip_sym(dg_pre, a.clip); dx[3] = clip_sym(do_pre, a.clip);
                carry_new = 0.f;
              } else if constexpr (G == 3) {
                const float r = sv[q][0], uu = sv[q][1], cand = sv[q][2], ac = sv[q][3], h_prev = sv[q][4];
                const float du_pre = d * ((cand - h_prev) * uu * (1.f - uu));
                const float dq = clip_sym(d * (uu * (1.f - cand * cand)), a.clip);
                const float dr_pre = dq * (ac * r * (1.f - r));
                dx[0] = clip_sym(dr_pre, a.clip); dx[1] = clip_sym(du_pre, a.clip); dx[2] = dq;
                dacv = clip_sym(dq * r, a.clip);
                carry_new = d * (1.f - uu);
              } else {
                const float h_new = sv[q][0];
                dx[0] = clip_sym(d * (a.relu ? (h_new > 0.f ? 1.f : 0.f) : 1.f - h_new * h_new), a.clip);
                carry_new = 0.f;
              }
            }
            carry_s[j * 128 + tid] = carry_new;
            const long long row = (long long)t * B + b;
#pragma unroll
            for (int g = 0; g < G; ++g) { a.dXg[row * GH + g * H + k] = dx[g]; dbs[g] += dx[g]; }
            if (G == 3) a.dac[row * H + k] = dacv;
          }
        }
      }
      if (t < 0 && k_ok) {
        atomicAdd(a.g_h_init + k, sum_h);
        if (G == 4) {
          atomicAdd(a.g_c_init + k, sum_c);
          atomicAdd(a.g_peep + k, dpe0); atomicAdd(a.g_peep + H + k, dpe1); atomicAdd(a.g_peep + 2 * H + k, dpe2);
        }
#pragma unroll
        for (int g = 0; g < G; ++g) atomicAdd(a.g_b + g * H + k, dbs[g]);
      }
      publish_step(a.fence_mode, tid, &bars.tmem_empty, ctr);
    }
  } else if (warp < 8) {
    // ------------------------------------------------------------ B converter: da_{t+1} rows of the tile
    const int bt = tid - 128;
    int gc = 0;
    for (int s = 1; s < n_steps; ++s) {
      for (int c = 0; c < NC; ++c, ++gc) {
        const int rs = gc % SC_LOOKB;
        mbar_wait(&bars.rawB_full[rs], (gc / SC_LOOKB) & 1);
        const float* src = reinterpret_cast<const float*>(rawB0 + (size_t)rs * (SC_BN * SC_KC * 4));
        float4 cur[2];
        int nn[2], kk[2];
#pragma unroll
        for (int it = 0; it < 2; ++it) {
          const int idx = it * 128 + bt;
          nn[it] = ((idx >> 6) << 3) + (idx & 7); kk[it] = (idx >> 3) & 7;
          cur[it] = *reinterpret_cast<const float4*>(src + nn[it] * 32 + ((kk[it] ^ (nn[it] & 7)) << 2));
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.rawB_empty[rs]);
        const int st = gc % SC_ST;
        if (gc >= SC_ST) mbar_wait(&bars.empty[st], ((gc / SC_ST) - 1) & 1);
#pragma unroll
        for (int it = 0; it < 2; ++it) store_b_split(convB + (size_t)st * stageB, nn[it], kk[it], cur[it]);
        proxy_fence_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.full[st]);
      }
    }
  } else if (warp == 8) {
    // ------------------------------------------------------------ MMA issuer
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32(128, SC_BN);
      int gc = 0;
      for (int s = 1; s < n_steps; ++s) {
        mbar_wait(&bars.tmem_empty, (s - 1) & 1);          // the epilogue of step s-1 has drained the accumulators
        tc_fence_after();
        uint32_t acc = 0;
        for (int c = 0; c < NC; ++c, ++gc) {
          const int st = gc % SC_ST;
          mbar_wait(&bars.full[st], (gc / SC_ST) & 1);
          tc_fence_after();
          issue_chunk_mmas(tD1, tD2, tA + (uint32_t)st * 64u, smem_u32(convB + (size_t)st * stageB), idesc, acc);
          umma_commit(&bars.empty[st]);
        }
        umma_commit(&bars.done);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------ A producer: W_hid rows, independent of the recurrence
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmA) : "memory");
      int gc = 0;
      for (int s = 1; s < n_steps; ++s)
        for (int c = 0; c < NC; ++c, ++gc) {
          const int rs = gc % LOOK;
          if (gc >= LOOK) mbar_wait(&bars.rawA_empty[rs], ((gc / LOOK) - 1) & 1);
          mbar_arrive_expect_tx(&bars.rawA_full[rs], 128 * SC_KC * 4);
          tma_load_2d(rawA0 + (size_t)rs * (128 * SC_KC * 4), &a.tmA, c * SC_KC, m0, &bars.rawA_full[rs]);
        }
    }
  } else if (warp == 10) {
    // ------------------------------------------------------------ B producer: waits for the step that wrote da_{t+1}
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmB) : "memory");
      int gc = 0;
      for (int s = 1; s < n_steps; ++s) {
        const int t = t_end - 1 - s;
        const unsigned int need = (unsigned int)s * (unsigned int)group_ctas;
        if (a.acq_spin) { while (ld_acquire_gpu(ctr) < need) { } } else wait_counter_gpu(ctr, need);
        fence_proxy_async_all();
        for (int c = 0; c < NC; ++c, ++gc) {
          const int rs = gc % SC_LOOKB;
          if (gc >= SC_LOOKB) mbar_wait(&bars.rawB_empty[rs], ((gc / SC_LOOKB) - 1) & 1);
          mbar_arrive_expect_tx(&bars.rawB_full[rs], SC_BN * SC_KC * 4);
          const int k0 = c * SC_KC;
          uint8_t* dst = rawB0 + (size_t)rs * (SC_BN * SC_KC * 4);
          if (G == 3 && k0 >= a.b_split) tma_load_2d(dst, &a.tmB2, k0 - a.b_split, (t + 1) * B + n0, &bars.rawB_full[rs]);
          else tma_load_2d(dst, &a.tmB, k0, (t + 1) * B + n0, &bars.rawB_full[rs]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512));
}

// ================================================================================================ backward, split-K cluster
// The BPTT product contracts over the G*H gate columns -- 4x the forward's K with 1/4 of its output -- so one CTA per
// (128 hidden units x 32 batch rows) tile would serialise 32-64 k chunks per step.  Here a cluster of KS CTAs shares
// the tile: CTA r contracts over its slice of the gate columns (its own chunks of W_hid rows and of da_{t+1}), drains
// its partial D[k][b] to shared memory and bulk-copies the 32/KS batch columns owned by each peer into the peer's
// receive buffer (cp.async.bulk shared::cta -> shared::cluster, completion on the peer's mbarrier: the exchange idiom
// of rnn_tc.cu).  Every CTA then sums KS partials for ITS 32/KS batch rows and runs the gate-gradient epilogue for them.
constexpr int SC_KS = 4;                     // cluster size along K
constexpr int SC_OWN = SC_BN / SC_KS;        // batch rows owned by a CTA in the epilogue

template <int G>
__global__ void __launch_bounds__(SC_NT, 1) tc_scan_bwd2_kernel(const __grid_constant__ ScanArgs a) {
  extern __shared__ __align__(1024) uint8_t sc_smem[];
  __shared__ ScanBars bars;
  __shared__ __align__(8) uint64_t recv_full[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ int t_end_s;
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();          // K slice and owned batch rows
  uint8_t* const base = sc_smem + ((1024u - (smem_u32(sc_smem) & 1023u)) & 1023u);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n0 = (blockIdx.x + a.tile0) * SC_BN, m0 = blockIdx.y * 128;
  const int B = a.B, H = a.H, GH = G * H, LOOK = a.look;
  const int per = (a.n_chunks + SC_KS - 1) / SC_KS;
  const int c_lo = min(a.n_chunks, rank * per), c_hi = min(a.n_chunks, c_lo + per);
  const int NC = c_hi - c_lo;                          // this CTA's chunks of the contraction (may be 0)
  constexpr uint32_t stageB = SC_BN * SC_KC * 8u;
  uint8_t* convB = base;                                                          // [SC_ST] converted da chunks (24 KB)
  float* part_s = reinterpret_cast<float*>(convB + SC_ST * stageB);               // [32 b][128 k] own partial D (16 KB)
  float* recv_s = part_s + SC_BN * 128;                                           // [2][KS][OWN][128] partials of my rows from every rank
  float* carry_s = recv_s + 2 * SC_KS * SC_OWN * 128;                             // [OWN][128]
  float* dcs_s = carry_s + SC_OWN * 128;                                          // [OWN][128]
  uint8_t* rawA0 = reinterpret_cast<uint8_t*>(dcs_s + SC_OWN * 128);              // [LOOK][128][32]
  uint8_t* rawB0 = rawA0 + (size_t)LOOK * (128 * SC_KC * 4);                      // [SC_LOOKB][32][32]

  if (tid == 0) {
    t_end_s = 0;
    init_bars(bars, 8);
    mbar_init(&recv_full[0], 1); mbar_init(&recv_full[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (tid < SC_BN) {
    const int b = n0 + tid;
    atomicMax(&t_end_s, b < B ? min(__ldg(a.len + b), a.t_max) : 0);
  }
  __syncthreads();
  const int t_end = t_end_s;
  const int jb = rank * SC_OWN;                        // first owned batch column of the tile
  // masked tail [t_end, t_max) of the owned rows: exactly zero gradients wrt the input pre-activations
  for (int t = t_end; t < a.t_max; ++t)
    for (int i = tid; i < SC_OWN * 128; i += SC_NT) {
      const int b = n0 + jb + (i >> 7), k = m0 + (i & 127);
      if (b < B && k < H) {
        const long long row = (long long)t * B + b;
        for (int g = 0; g < G; ++g) a.dXg[row * GH + g * H + k] = 0.f;
        if (G == 3) a.dac[row * H + k] = 0.f;
      }
    }
  const uint32_t tmem = tmem_base_s;
  const uint32_t tD1 = tmem, tD2 = tmem + SC_BN, tA = tmem + 64;
  const int group_ctas = gridDim.y * SC_KS;
  unsigned int* ctr = a.sync + blockIdx.x;
  const int n_steps = t_end + 1;
  constexpr uint32_t slice_bytes = SC_OWN * 128 * 4;   // one rank's partial of my rows
  if (tid == 0) {
    mbar_arrive_expect_tx(&recv_full[0], (SC_KS - 1) * slice_bytes);
    mbar_arrive_expect_tx(&recv_full[1], (SC_KS - 1) * slice_bytes);
  }
  cluster.sync();        // barriers of every CTA initialised and armed before any remote traffic

  if (warp < 4) {
    // ------------------------------------------------------------ A converter + exchange + epilogue (thread = hidden unit k)
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    const int k = m0 + tid;
    const bool k_ok = k < H;
    float wci = 0.f, wcf = 0.f, wco = 0.f;
    if (G == 4 && k_ok) { wci = __ldg(a.peep + k); wcf = __ldg(a.peep + H + k); wco = __ldg(a.peep + 2 * H + k); }
    for (int j = 0; j < SC_OWN; ++j) {
      const int b = n0 + jb + j;
      carry_s[j * 128 + tid] = (a.dh_last && k_ok && b < B) ? __ldg(a.dh_last + (long long)b * H + k) : 0.f;
      dcs_s[j * 128 + tid] = 0.f;
    }
    float dpe0 = 0.f, dpe1 = 0.f, dpe2 = 0.f, dbs[4] = {0.f, 0.f, 0.f, 0.f};
    int gc = 0, n_done = 0;
    const bool tl = a.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && tid == 0;
    long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tl0 = tl ? clock64() : 0;
    for (int s = 0; s < n_steps; ++s) {
      const int t = t_end - 1 - s;
      float P[SC_OWN];
#pragma unroll
      for (int j = 0; j < SC_OWN; ++j) P[j] = 0.f;
      // saved tensors of step t for the owned rows: they do not depend on this step's product, so they are requested
      // before the contraction and have landed by the time the partial sums arrive
      float sv[SC_OWN][7];
      bool act_[SC_OWN];
#pragma unroll
      for (int q = 0; q < SC_OWN; ++q) {
        const int b = n0 + jb + q;
        act_[q] = k_ok && t >= 0 && b < B && t < min(__ldg(a.len + b), a.t_max);
        if (act_[q]) {
          const long long row = (long long)t * B + b;
          if (G > 1) {
            const float* ap = a.act_r + row * 4 * H + k;
            sv[q][0] = __ldg(ap); sv[q][1] = __ldg(ap + H); sv[q][2] = __ldg(ap + 2 * H); sv[q][3] = __ldg(ap + 3 * H);
          }
          if (G == 4) { sv[q][4] = __ldg(a.cs_r + row * H + k); sv[q][5] = __ldg(a.cs_r + (row + B) * H + k); }
          if (G == 3) sv[q][4] = __ldg(a.hs_r + row * H + k);
          if (G == 1) sv[q][0] = __ldg(a.hs_r + (row + B) * H + k);
          sv[q][6] = a.dhs ? __ldg(a.dhs + row * H + k) : 0.f;
        }
      }
      if (s > 0) {
        const int buf = (s - 1) & 1;
        for (int c = 0; c < NC; ++c, ++gc) convert_a_chunk(bars, rawA0, LOOK, tA, lane_off, tid, lane, gc);
        SC_ACC(0);
        // partial D of this CTA's K slice -> shared memory [b][k]
        if (NC > 0) {
          mbar_wait(&bars.done, n_done & 1);
          tc_fence_after();
          SC_ACC(1);
          for (int c0 = 0; c0 < SC_BN; c0 += 16) {
            float d[16], w[16];
            tmem_ld16(tD1 + lane_off + c0, d);
            tmem_ld16(tD2 + lane_off + c0, w);
#pragma unroll
            for (int i = 0; i < 16; ++i) part_s[(c0 + i) * 128 + tid] = d[i] + w[i];
          }
        } else {
          for (int j = 0; j < SC_BN; ++j) part_s[j * 128 + tid] = 0.f;
        }
        proxy_fence_smem();
        tc_fence_before();
        epi_bar();
        if (tid == 0) {
          if (NC > 0) { mbar_arrive(&bars.tmem_empty); }
          // rows owned by rank q: columns q*OWN .. of my partial -> q's receive slot [buf][my rank]
          for (int q = 0; q < SC_KS; ++q) {
            if (q == rank) continue;
            const uint32_t src = smem_u32(part_s + q * SC_OWN * 128);
            const uint32_t dst = map_to_rank(smem_u32(recv_s + ((buf * SC_KS + rank) * SC_OWN) * 128), q);
            bulk_copy_to_peer(dst, src, slice_bytes, map_to_rank(smem_u32(&recv_full[buf]), q));
          }
        }
        if (NC > 0) ++n_done;
        SC_ACC(2);
        // the other ranks' partials of my rows
        if (a.acq_spin) mbar_wait_cluster(&recv_full[buf], ((s - 1) >> 1) & 1); else mbar_wait(&recv_full[buf], ((s - 1) >> 1) & 1);   // bulk-copy complete_tx: no cluster acquire needed
        SC_ACC(3);
        if (tid == 0) mbar_arrive_expect_tx(&recv_full[buf], (SC_KS - 1) * slice_bytes);     // next use of this buffer (two steps later)
#pragma unroll
        for (int j = 0; j < SC_OWN; ++j) {
          float v = part_s[(jb + j) * 128 + tid];
#pragma unroll
          for (int q = 0; q < SC_KS; ++q)
            if (q != rank) v += recv_s[((buf * SC_KS + q) * SC_OWN + j) * 128 + tid];
          P[j] = v;
        }
      }
      if (k_ok) {
        if (t < 0) {
          float sum_h = 0.f, sum_c = 0.f;
#pragma unroll
          for (int j = 0; j < SC_OWN; ++j)
            if (n0 + jb + j < B) { sum_h += carry_s[j * 128 + tid] + P[j]; sum_c += dcs_s[j * 128 + tid]; }
          atomicAdd(a.g_h_init + k, sum_h);
          if (G == 4) {
            atomicAdd(a.g_c_init + k, sum_c);
            atomicAdd(a.g_peep + k, dpe0); atomicAdd(a.g_peep + H + k, dpe1); atomicAdd(a.g_peep + 2 * H + k, dpe2);
          }
#pragma unroll
          for (int g = 0; g < G; ++g) atomicAdd(a.g_b + g * H + k, dbs[g]);
        } else {
          {
#pragma unroll
            for (int q = 0; q < SC_OWN; ++q) {
              const int j = q, b = n0 + jb + j;
              if (b >= B) continue;
              const float dh = carry_s[j * 128 + tid] + P[j];
              float dx[4] = {0.f, 0.f, 0.f, 0.f}, dacv = 0.f, carry_new = dh;
              if (act_[q]) {
                const float d = dh + sv[q][6];
                if constexpr (G == 4) {
                  const float ig = sv[q][0], fg = sv[q][1], gg = sv[q][2], og = sv[q][3], c_prev = sv[q][4], c_new = sv[q][5];
                  const float tc = tanh_fast(c_new);
                  const float do_pre = d * (tc * og * (1.f - og));
                  const float dct = dcs_s[j * 128 + tid] + d * (og * (1.f - tc * tc)) + do_pre * wco;
                  const float di_pre = dct * (gg * ig * (1.f - ig));
                  const float df_pre = dct * (c_prev * fg * (1.f - fg));
                  const float dg_pre = dct * (ig * (1.f - gg * gg));
                  dpe0 += di_pre * c_prev; dpe1 += df_pre * c_prev; dpe2 += do_pre * c_new;
                  dcs_s[j * 128 + tid] = dct * fg + di_pre * wci + df_pre * wcf;
                  dx[0] = clip_sym(di_pre, a.clip); dx[1] = clip_sym(df_pre, a.clip);
                  dx[2] = clip_sym(dg_pre, a.clip); dx[3] = clip_sym(do_pre, a.clip);
                  carry_new = 0.f;
                } else if constexpr (G == 3) {
                  const float r = sv[q][0], uu = sv[q][1], cand = sv[q][2], ac = sv[q][3], h_prev = sv[q][4];
                  const float du_pre = d * ((cand - h_prev) * uu * (1.f - uu));
                  const float dq = clip_sym(d * (uu * (1.f - cand * cand)), a.clip);
                  const float dr_pre = dq * (ac * r * (1.f - r));
                  dx[0] = clip_sym(dr_pre, a.clip); dx[1] = clip_sym(du_pre, a.clip); dx[2] = dq;
                  dacv = clip_sym(dq * r, a.clip);
                  carry_new = d * (1.f - uu);
                } else {
                  const float h_new = sv[q][0];
                  dx[0] = clip_sym(d * (a.relu ? (h_new > 0.f ? 1.f : 0.f) : 1.f - h_new * h_new), a.clip);
                  carry_new = 0.f;
                }
              }
              carry_s[j * 128 + tid] = carry_new;
              const long long row = (long long)t * B + b;
#pragma unroll
              for (int g = 0; g < G; ++g) { a.dXg[row * GH + g * H + k] = dx[g]; dbs[g] += dx[g]; }
              if (G == 3) a.dac[row * H + k] = dacv;
            }
          }
        }
      }
      SC_ACC(4);
      // publish the step (the accumulators were released right after the drain)
      if (a.fence_mode == 0) { __threadfence(); fence_proxy_async_all(); }
      else if (a.fence_mode == 1) fence_proxy_async_all();
      epi_bar();
      if (tid == 0) {
        if (a.fence_mode == 2) { __threadfence(); fence_proxy_async_all(); }
        red_release_gpu(ctr, 1u);
      }
      SC_ACC(5);
    }
    if (tl) { for (int i = 0; i < 8; ++i) a.dbg[16 + i] = ph[i]; a.dbg[24] = n_steps; }
  } else if (warp < 8) {
    // ------------------------------------------------------------ B converter: da_{t+1} rows, this CTA's K slice
    const int bt = tid - 128;
    int gc = 0;
    for (int s = 1; s < n_steps; ++s) {
      for (int c = 0; c < NC; ++c, ++gc) {
        const int rs = gc % SC_LOOKB;
        mbar_wait(&bars.rawB_full[rs], (gc / SC_LOOKB) & 1);
        const float* src = reinterpret_cast<const float*>(rawB0 + (size_t)rs * (SC_BN * SC_KC * 4));
        float4 cur[2];
        int nn[2], kk[2];
#pragma unroll
        for (int it = 0; it < 2; ++it) {
          const int idx = it * 128 + bt;
          nn[it] = ((idx >> 6) << 3) + (idx & 7); kk[it] = (idx >> 3) & 7;
          cur[it] = *reinterpret_cast<const float4*>(src + nn[it] * 32 + ((kk[it] ^ (nn[it] & 7)) << 2));
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.rawB_empty[rs]);
        const int st = gc % SC_ST;
        if (gc >= SC_ST) mbar_wait(&bars.empty[st], ((gc / SC_ST) - 1) & 1);
#pragma unroll
        for (int it = 0; it < 2; ++it) store_b_split(convB + (size_t)st * stageB, nn[it], kk[it], cur[it]);
        proxy_fence_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.full[st]);
      }
    }
  } else if (warp == 8) {
    // ------------------------------------------------------------ MMA issuer
    if (NC > 0 && elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32(128, SC_BN);
      int gc = 0;
      for (int s = 1; s < n_steps; ++s) {
        if (s > 1) { mbar_wait(&bars.tmem_empty, (s - 2) & 1); tc_fence_after(); }     // the previous drain is over
        uint32_t acc = 0;
        for (int c = 0; c < NC; ++c, ++gc) {
          const int st = gc % SC_ST;
          mbar_wait(&bars.full[st], (gc / SC_ST) & 1);
          tc_fence_after();
          issue_chunk_mmas(tD1, tD2, tA + (uint32_t)st * 64u, smem_u32(convB + (size_t)st * stageB), idesc, acc);
          umma_commit(&bars.empty[st]);
        }
        umma_commit(&bars.done);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------ A producer: W_hid rows, this CTA's gate columns
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmA) : "memory");
      int gc = 0;
      for (int s = 1; s < n_steps; ++s)
        for (int c = 0; c < NC; ++c, ++gc) {
          const int rs = gc % LOOK;
          if (gc >= LOOK) mbar_wait(&bars.rawA_empty[rs], ((gc / LOOK) - 1) & 1);
          mbar_arrive_expect_tx(&bars.rawA_full[rs], 128 * SC_KC * 4);
          tma_load_2d(rawA0 + (size_t)rs * (128 * SC_KC * 4), &a.tmA, (c_lo + c) * SC_KC, m0, &bars.rawA_full[rs]);
        }
    }
  } else if (warp == 10) {
    // ------------------------------------------------------------ B producer: waits for the step that wrote da_{t+1}
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmB) : "memory");
      int gc = 0;
      for (int s = 1; s < n_steps; ++s) {
        const int t = t_end - 1 - s;
        const long long w0 = a.dbg ? clock64() : 0;
        if (NC > 0) {
          const unsigned int need = (unsigned int)s * (unsigned int)group_ctas;
          if (a.acq_spin) { while (ld_acquire_gpu(ctr) < need) { } } else wait_counter_gpu(ctr, need);
          fence_proxy_async_all();
        }
        if (a.dbg && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) a.dbg[26] += clock64() - w0;
        for (int c = 0; c < NC; ++c, ++gc) {
          const int rs = gc % SC_LOOKB;
          if (gc >= SC_LOOKB) mbar_wait(&bars.rawB_empty[rs], ((gc / SC_LOOKB) - 1) & 1);
          mbar_arrive_expect_tx(&bars.rawB_full[rs], SC_BN * SC_KC * 4);
          const int k0 = (c_lo + c) * SC_KC;
          uint8_t* dst = rawB0 + (size_t)rs * (SC_BN * SC_KC * 4);
          if (G == 3 && k0 >= a.b_split) tma_load_2d(dst, &a.tmB2, k0 - a.b_split, (t + 1) * B + n0, &bars.rawB_full[rs]);
          else tma_load_2d(dst, &a.tmB, k0, (t + 1) * B + n0, &bars.rawB_full[rs]);
        }
      }
    }
  }
  tc_fence_before();
  cluster.sync();        // nobody leaves while a peer may still copy into this CTA's shared memory
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512));
}

__global__ void bcast_rows2_kernel(float* __restrict__ out, const float* __restrict__ v, int64_t rows, int cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) out[i] = v[i % cols];
}
__global__ void gather_last_state2_kernel(const float* __restrict__ hs, const int32_t* __restrict__ len, float* __restrict__ out,
                                          int B, int H, int t_max) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * H) return;
  const int b = (int)(i / H), k = (int)(i - (long long)b * H);
  out[i] = hs[((long long)min(len[b], t_max) * B + b) * H + k];
}

constexpr size_t SC_SMEM_MAX = 232448 - 2048;

long long* g_scan_dbg = nullptr;
long long* scan_dbg_buffer(sbr_model* m) {
  static const bool want = getenv("SBR_SCAN_TIMELINE") != nullptr;
  if (!want) return nullptr;
  if (!g_scan_dbg) cudaMalloc(&g_scan_dbg, 64 * sizeof(long long));
  cudaMemsetAsync(g_scan_dbg, 0, 64 * sizeof(long long), m->stream);
  return g_scan_dbg;
}
void scan_dbg_print(sbr_model* m, const char* what) {
  if (!g_scan_dbg) return;
  long long h[64];
  cudaStreamSynchronize(m->stream);
  cudaMemcpy(h, g_scan_dbg, sizeof(h), cudaMemcpyDeviceToHost);
  const double nf = (double)(h[6] > 0 ? h[6] : 1), nb = (double)(h[24] > 0 ? h[24] : 1);
  if (h[6] > 0)
    fprintf(stderr, "[scan fwd %s, cycles/step over %lld steps] first_chunk(sync+tma) %.0f conv_rest %.0f wait_done %.0f ldtm+math+stores %.0f publish %.0f | producer spin %.0f\n",
            what, h[6], h[0] / nf, h[1] / nf, h[2] / nf, h[3] / nf, h[4] / nf, h[8] / nf);
  if (h[24] > 0)
    fprintf(stderr, "[scan bwd %s, cycles/step over %lld steps] conv(sync+tma+conv) %.0f wait_done %.0f drain+send %.0f wait_recv %.0f epilogue %.0f publish %.0f | B producer spin %.0f\n",
            what, h[24], h[16] / nb, h[17] / nb, h[18] / nb, h[19] / nb, h[20] / nb, h[21] / nb, h[26] / nb);
}

template <typename Kern>
int launch_coop(sbr_model* m, Kern kern, dim3 grid, size_t smem, const ScanArgs& a) {
  static std::vector<std::pair<int, const void*>> attr_done;     // (device, kernel): opt-in shared memory is per device
  bool have = false;
  for (auto& kv : attr_done) have |= kv.first == m->dev && kv.second == (const void*)kern;
  if (!have) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SC_SMEM_MAX);
    if (e != cudaSuccess) { sbr_set_error(m, SBR_E_CUDA, "tc_scan attr: %s", cudaGetErrorString(e)); return SBR_E_CUDA; }
    attr_done.push_back({m->dev, (const void*)kern});
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = dim3(SC_NT, 1, 1); cfg.dynamicSmemBytes = smem; cfg.stream = m->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;     // all CTAs co-resident: they wait for each other through global counters
  attr[0].val.cooperative = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
  if (e != cudaSuccess) { sbr_set_error(m, SBR_E_CUDA, "persistent scan launch (%u x %u CTAs) failed: %s", grid.x, grid.y, cudaGetErrorString(e)); return SBR_E_CUDA; }
  m->launches++;
  m->scan_launches++;
  return 0;
}

template <typename Kern>
int launch_cluster_coop(sbr_model* m, Kern kern, dim3 grid, dim3 cl, size_t smem, const ScanArgs& a) {
  static std::vector<std::pair<int, const void*>> attr_done;
  bool have = false;
  for (auto& kv : attr_done) have |= kv.first == m->dev && kv.second == (const void*)kern;
  if (!have) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SC_SMEM_MAX);
    if (e != cudaSuccess) { sbr_set_error(m, SBR_E_CUDA, "tc_scan attr: %s", cudaGetErrorString(e)); return SBR_E_CUDA; }
    attr_done.push_back({m->dev, (const void*)kern});
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = dim3(SC_NT, 1, 1); cfg.dynamicSmemBytes = smem; cfg.stream = m->stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cl.x; attr[0].val.clusterDim.y = cl.y; attr[0].val.clusterDim.z = cl.z;
  attr[1].id = cudaLaunchAttributeCooperative;
  attr[1].val.cooperative = 1;
  // SBR_SCAN_NO_COOP: plain cluster launch (Nsight Compute cannot replay a cooperative cluster launch; the grid is sized
  // to be co-resident on an otherwise idle GPU)
  static const bool no_coop = getenv("SBR_SCAN_NO_COOP") != nullptr;
  cfg.attrs = attr; cfg.numAttrs = no_coop ? 1 : 2;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
  if (e != cudaSuccess && !no_coop) {
    // cooperative + cluster not accepted together: the grid is sized to be co-resident, launch it as a plain cluster grid
    cudaGetLastError();
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, kern, a);
  }
  if (e != cudaSuccess) { sbr_set_error(m, SBR_E_CUDA, "split-K scan launch (%u x %u x %u CTAs) failed: %s", grid.x, grid.y, grid.z, cudaGetErrorString(e)); return SBR_E_CUDA; }
  m->launches++;
  m->scan_launches++;
  return 0;
}

template <typename Kern>
int max_clusters(Kern kern, dim3 cl, size_t smem) {
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SC_SMEM_MAX);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(cl.x * 64, cl.y, cl.z); cfg.blockDim = dim3(SC_NT, 1, 1); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cl.x; attr[0].val.clusterDim.y = cl.y; attr[0].val.clusterDim.z = cl.z;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

}  // namespace

// 1 when the persistent kernels take this layer: tensor maps possible (always for arena / workspace arrays with H % 16
// == 0), the resident forward W_hid slice fits, and the per-launch grid can be made co-resident by slicing the batch
int persistent_scan_applies(const ScanSwitches& s, int H) {
  return (s.tc_gemm && s.step && s.persistent && s.tma_gemm && H % 16 == 0 && H >= 32 && H <= 512) ? 1 : 0;
}
int persistent_scan_applies(const sbr_model* m, int G, int H) {
  (void)G;
  return persistent_scan_applies(scan_switches(m), H);
}

// shared memory of the split-K backward CTA (independent of the layer: the ring depth fills what is left)
static size_t splitk_smem(int* look) {
  const size_t fixed2 = (size_t)SC_ST * SC_BN * SC_KC * 8 + (size_t)SC_BN * 128 * 4 + (size_t)2 * SC_KS * SC_OWN * 128 * 4 +
                        (size_t)2 * SC_OWN * 128 * 4 + (size_t)SC_LOOKB * SC_BN * SC_KC * 4 + 1024;
  *look = (int)std::min<size_t>(SC_LOOK_MAX, (SC_SMEM_MAX - fixed2) / (128 * SC_KC * 4));
  return fixed2 + (size_t)*look * 128 * SC_KC * 4;
}
int persistent_splitk_slots() {
  static int slots = -1;
  if (slots < 0) {
    int look = 0;
    const size_t smem2 = splitk_smem(&look);
    slots = max_clusters(tc_scan_bwd2_kernel<4>, dim3(1, 1, SC_KS), smem2);
  }
  return slots;
}
// forward: one CTA per 8 hidden units and 128-row tile, one CTA per SM
PersistentSlicing persistent_fwd_slicing(int n_sm, int H, int B) {
  const int unit_ctas = cdiv(H, SC_U);
  return PersistentSlicing{128, cdiv(B, 128), std::max(1, n_sm / unit_ctas), SC_U, false};
}
// backward: per 32-row tile, one 128-unit CTA (or split-K cluster of SC_KS CTAs) per 128 hidden units; split-K when at
// least one tile's clusters are co-resident
PersistentSlicing persistent_bwd_slicing(int n_sm, int H, int B, bool use_splitk, int splitk_slots) {
  const int m_ctas = cdiv(H, 128);
  PersistentSlicing s{SC_BN, cdiv(B, SC_BN), 0, 128, false};
  if (use_splitk && splitk_slots / m_ctas >= 1) {
    s.splitk = true;
    s.tiles_per_launch = splitk_slots / m_ctas;
  } else {
    s.tiles_per_launch = std::max(1, n_sm / m_ctas);
  }
  return s;
}

int launch_rnn_forward_persistent(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last) {
  const int H = L.H, G = L.G, GH = G * H;
  bcast_rows2_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, m->stream>>>(L.hs, m->params + L.h_init, (int64_t)B, H);
  KERNEL_CHECK(m);
  if (G == 4) {
    bcast_rows2_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, m->stream>>>(L.cs, m->params + L.c_init, (int64_t)B, H);
    KERNEL_CHECK(m);
  }
  ScanArgs a{};
  a.fence_mode = m->scan_fence_mode;
  a.acq_spin = getenv("SBR_SCAN_ACQ_SPIN") ? 1 : 0;
  a.dbg = scan_dbg_buffer(m);
  a.B = B; a.H = H; a.G = G; a.t_max = t_max; a.n_chunks = cdiv(H, SC_KC);
  a.relu = L.relu;
  a.len = len; a.peep = m->params + L.peep; a.Xg = L.Xg; a.hs = L.hs; a.cs = L.cs; a.act = L.act;
  const int unit_ctas = cdiv(H, SC_U), n_tiles = cdiv(B, 128);
  if (unit_ctas > m->n_sm) return 1;
  // cluster of CS consecutive unit slices shares the h tile through TMA multicast
  int CS = 1;
  if (m->use_scan_multicast)
    for (int c = 4; c >= 2; c >>= 1) if (unit_ctas % c == 0) { CS = c; break; }
  if (!get_tmap(&a.tmA, L.hs, H, (uint64_t)(m->T + 1) * m->B, H, SC_KC, 128 / CS, true) ||
      !get_tmap(&a.tmB, m->params + L.W_hid, GH, H, GH, SC_U, SC_KC, false))
    return 1;
  const size_t fixed = (size_t)a.n_chunks * SC_BN * SC_KC * 8 + (size_t)SC_LOOKB * 4 * SC_KC * SC_U * 4 + 1024;
  a.look = (int)std::min<size_t>(SC_LOOK_MAX, (SC_SMEM_MAX - fixed) / (128 * SC_KC * 4));
  if (a.look < 2) return 1;
  const size_t smem = fixed + (size_t)a.look * 128 * SC_KC * 4;
  // batch tiles per launch: all CTAs of a launch must be co-resident (one per SM); rows are independent, so a larger
  // batch runs as several launches over slices of its tiles
  int tiles_per_launch = persistent_fwd_slicing(m->n_sm, H, B).tiles_per_launch;
  if (CS > 1) {
    static int slots[5] = {-1, -1, -1, -1, -1};
    if (slots[CS] < 0) slots[CS] = max_clusters(tc_scan_fwd_kernel<4>, dim3(CS, 1, 1), smem);
    tiles_per_launch = slots[CS] / (unit_ctas / CS);
    if (tiles_per_launch < 1) { CS = 1; tiles_per_launch = std::max(1, m->n_sm / unit_ctas); get_tmap(&a.tmA, L.hs, H, (uint64_t)(m->T + 1) * m->B, H, SC_KC, 128, true); }
  }
  CU_TRY(m, cudaMemsetAsync(m->scan_sync, 0, (size_t)std::max(n_tiles, cdiv(B, SC_BN)) * sizeof(unsigned int), m->stream));
  for (int t0 = 0; t0 < n_tiles; t0 += tiles_per_launch) {
    const int nt = std::min(tiles_per_launch, n_tiles - t0);
    ScanArgs v = a;
    v.sync = m->scan_sync + t0;
    v.tile0 = t0;
    int rc;
    const dim3 grid(unit_ctas, nt, 1), cl(CS, 1, 1);
    if (G == 4) rc = launch_cluster_coop(m, tc_scan_fwd_kernel<4>, grid, cl, smem, v);
    else if (G == 3) rc = launch_cluster_coop(m, tc_scan_fwd_kernel<3>, grid, cl, smem, v);
    else rc = launch_cluster_coop(m, tc_scan_fwd_kernel<1>, grid, cl, smem, v);
    if (rc) return rc;
  }
  if (h_last) {
    gather_last_state2_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, m->stream>>>(L.hs, len, h_last, B, H, t_max);
    KERNEL_CHECK(m);
  }
  scan_dbg_print(m, "");
  return 0;
}

int launch_rnn_backward_persistent(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, const float* dh_last) {
  const int H = L.H, G = L.G, GH = G * H;
  ScanArgs a{};
  a.fence_mode = m->scan_fence_mode;
  a.acq_spin = getenv("SBR_SCAN_ACQ_SPIN") ? 1 : 0;
  a.dbg = scan_dbg_buffer(m);
  a.B = B; a.H = H; a.G = G; a.t_max = t_max; a.n_chunks = cdiv(GH, SC_KC);
  a.relu = L.relu;
  a.len = len; a.peep = m->params + L.peep;
  a.act_r = L.act; a.cs_r = L.cs; a.hs_r = L.hs; a.dhs = dh_last ? nullptr : L.dhs; a.dh_last = dh_last;
  a.dXg = L.dXg; a.dac = L.dac; a.clip = m->cfg.grad_clip; a.b_split = 2 * H;
  a.g_h_init = m->grads + L.h_init; a.g_c_init = m->grads + L.c_init; a.g_peep = m->grads + L.peep; a.g_b = m->grads + L.b;
  if (!get_tmap(&a.tmA, m->params + L.W_hid, GH, H, GH, SC_KC, 128, true) ||
      !get_tmap(&a.tmB, L.dXg, GH, (uint64_t)m->T * m->B, GH, SC_KC, SC_BN, true))
    return 1;
  if (G == 3 && !get_tmap(&a.tmB2, L.dac, H, (uint64_t)m->T * m->B, H, SC_KC, SC_BN, true)) return 1;
  const int m_ctas0 = cdiv(H, 128), n_tiles0 = cdiv(B, SC_BN);
  const PersistentSlicing sl = persistent_bwd_slicing(m->n_sm, H, B, m->use_splitk_scan,
                                                      m->use_splitk_scan ? persistent_splitk_slots() : 0);
  if (sl.splitk) {
    // split-K clusters: KS CTAs per (hidden tile, batch tile)
    ScanArgs v = a;
    const size_t smem2 = splitk_smem(&v.look);
    const int tiles_per = sl.tiles_per_launch;      // batch tiles whose clusters are all co-resident
    {
      CU_TRY(m, cudaMemsetAsync(m->scan_sync, 0, (size_t)std::max(n_tiles0, cdiv(B, 128)) * sizeof(unsigned int), m->stream));
      for (int t0 = 0; t0 < n_tiles0; t0 += tiles_per) {
        const int nt = std::min(tiles_per, n_tiles0 - t0);
        v.sync = m->scan_sync + t0;
        v.tile0 = t0;
        int rc;
        if (G == 4) rc = launch_cluster_coop(m, tc_scan_bwd2_kernel<4>, dim3(nt, m_ctas0, SC_KS), dim3(1, 1, SC_KS), smem2, v);
        else if (G == 3) rc = launch_cluster_coop(m, tc_scan_bwd2_kernel<3>, dim3(nt, m_ctas0, SC_KS), dim3(1, 1, SC_KS), smem2, v);
        else rc = launch_cluster_coop(m, tc_scan_bwd2_kernel<1>, dim3(nt, m_ctas0, SC_KS), dim3(1, 1, SC_KS), smem2, v);
        if (rc) return rc;
      }
      scan_dbg_print(m, "split-K");
      return 0;
    }
  }
  const size_t fixed = (size_t)SC_ST * SC_BN * SC_KC * 8 + (size_t)2 * SC_BN * 128 * 4 + (size_t)SC_LOOKB * SC_BN * SC_KC * 4 + 1024;
  a.look = (int)std::min<size_t>(SC_LOOK_MAX, (SC_SMEM_MAX - fixed) / (128 * SC_KC * 4));
  const size_t smem = fixed + (size_t)a.look * 128 * SC_KC * 4;
  const int m_ctas = cdiv(H, 128), n_tiles = cdiv(B, SC_BN);
  const int tiles_per_launch = sl.tiles_per_launch;
  CU_TRY(m, cudaMemsetAsync(m->scan_sync, 0, (size_t)std::max(n_tiles, cdiv(B, 128)) * sizeof(unsigned int), m->stream));
  for (int t0 = 0; t0 < n_tiles; t0 += tiles_per_launch) {
    const int nt = std::min(tiles_per_launch, n_tiles - t0);
    ScanArgs v = a;
    v.sync = m->scan_sync + t0;
    v.tile0 = t0;
    int rc;
    if (G == 4) rc = launch_coop(m, tc_scan_bwd_kernel<4>, dim3(nt, m_ctas, 1), smem, v);
    else if (G == 3) rc = launch_coop(m, tc_scan_bwd_kernel<3>, dim3(nt, m_ctas, 1), smem, v);
    else rc = launch_coop(m, tc_scan_bwd_kernel<1>, dim3(nt, m_ctas, 1), smem, v);
    if (rc) return rc;
  }
  return 0;
}
