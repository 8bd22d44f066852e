// rnn_tc.cu -- stage 2 on the 5th-generation tensor cores: the recurrent scan (and its BPTT) with the
// per-step gate GEMM on tcgen05.mma, fp32-accurate through the 3xTF32 split.
//
// Same reference semantics as rnn_cluster.cu (sparse_lstm.py:377-425, :764-805, :1120-1152) and the
// same ownership: a cluster of C CTAs owns a tile of BT = 8 or 16 batch rows for all T steps; CTA r owns the
// hidden units [r*Hs, (r+1)*Hs) of every gate.  What changes is how a step is computed:
//
//   * the CTA's slice of W_hid is the **A operand, resident in TMEM** for the whole scan
//     (tcgen05.st once): row m = 4*j + g (unit j, gate g) of a 128-row tile, K along the columns,
//     stored twice -- hi = fp32 rounded to the 19 bits kind::tf32 reads, lo = w - hi;
//   * h_{t-1} (forward) / da_t (backward) is the **B operand in shared memory** [k/4][hi|lo][BT rows][4]
//     (K-major, no swizzle: 8x16B core matrices), already split hi/lo by its producer;
//   * D[128 x 16] = A_hi*B_hi, A_hi*B_lo, A_lo*B_hi in separate fp32 TMEM accumulators, one accumulation chain per
//     issuing warp (elect.sync); tcgen05.commit -> mbarrier -> tcgen05.ld (thread = gate row) -> shared memory;
//   * the fused gate math runs on one (row, unit) [8-row tiles] or (row, 2 units) [16-row tiles] per thread; the
//     new h_t slice is written pre-split into the local copy of the next B operand and sent to every peer CTA
//     with ONE bulk copy (cp.async.bulk shared::cta -> shared::cluster) that completes on the peer's mbarrier:
//     no cluster-wide barrier in the loop, no receiver-side work;
//   * the per-step inputs from global memory (Xg forward; saved gates / cell states / upstream gradient backward)
//     are streamed by the TMA engine (cp.async.bulk.tensor.2d, 4-stage ring, 3 steps ahead) so that the
//     fence.proxy.async every thread executes before the MMA never has an outstanding global load to drain.
//
// The backward keeps W_hid^T-style tiles in TMEM (rows = hidden index k, columns = own gate columns):
// dh_{t-1}[b][k] partial = sum over OWN gate columns of da[b][gj] W_hid[k][gj] (split-K), reduce-
// scattered to the owners with bulk copies.  It also writes the K-major hi/lo copies of da (and the forward those of
// h) that wgrad_tc.cu contracts, and accumulates the bias gradient.
//
// Host side: schedule_tiles() orders the tiles longest-first and chooses the tile height from the host copy of the
// lengths (15 eight-CTA clusters are co-resident on a B200; a batch of 128 rows is 16 eight-row tiles).
//
// Applicability: H % 4 == 0, H <= 224 (hi+lo copies of the K extent must fit in 512 TMEM columns),
// otherwise launch_rnn_* falls back to the FFMA cluster kernels.
#include <cooperative_groups.h>
#include <cuda.h>
#include <string.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int TC_N = 16;     // MMA N (minimum for M = 128); the cluster tile holds BT = 16 or 8 live batch rows
constexpr int GSM_LD = 132;  // padded row of the gate staging buffer

struct TcArgs {
  const float* Xg; const float* W_hid; const float* W_hidT; const float* peep; const float* h_init; const float* c_init;
  const int32_t* len;
  float* hs; float* cs; float* act; float* h_last;
  const float* dh_last; const float* dhs; float* dXg; float* dac; float* g_peep; float* g_h_init; float* g_c_init;
  float clip;
  int relu;            // vanilla cell: rectifier instead of tanh (dense-input layers)
  int B, H, Hs, Kp, t_max;
  long long* dbg;   // optional phase timeline of CTA 0 / thread 0 (8 stamps per step)
  float* hT; float* aT;                 // K-major pre-split copies for the tensor-core wgrad GEMM (may be null)
  float* g_b;                           // bias gradient slot (backward accumulates sum dXg itself when set)
  long long hT_part, hT_tile, aT_part, aT_tile;
  int ld_p;                             // backward: steps of saved activations in flight (TMA staging ring)
  // 2-D tiled tensor maps over the saved tensors, box = [BT rows x Hs units]: the backward kernel streams its
  // slice of a step with one TMA load per array (async proxy: nothing for the thread fences to wait on)
  CUtensorMap tm_act, tm_cs, tm_hs, tm_dhs;
  CUtensorMap tm_xg;                    // forward: input pre-activations Xg [rows x G*H]
  int xflags;                           // SBR_TC_EXPERIMENT bit mask (timing experiments only: results are wrong)
  int use_order;                        // cluster c works on tile order[c] (longest tiles first) instead of tile c
  unsigned char order[64];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// top 19 bits of v, rounded to nearest: exactly what kind::tf32 reads; lo = v - hi is exact in fp32
__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u); }
// gate nonlinearities on the SFU: ex2.approx + rcp.approx (relative error ~1e-7 in the working range)
__device__ __forceinline__ float sigmoidf_(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanhf_(float x) { return 1.f - __fdividef(2.f, __expf(2.f * x) + 1.f); }
__device__ __forceinline__ float clipf_(float x, float c) { return c > 0.f ? fminf(fmaxf(x, -c), c) : x; }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version 1 (sm_100); layout SWIZZLE_NONE
  return d;
}
// kind::tf32, fp32 accumulate, K-major A and B
__device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
               :: "r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait_cta(uint64_t* bar, uint32_t parity) {
  asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
               "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
               "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// wait with cluster-scope acquire: pairs with the remote arrive.release.cluster of the producers
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
               "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
               "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(uint32_t cta_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(cta_addr), "r"(rank));
  return r;
}
// bulk asynchronous copy of a contiguous block of THIS CTA's shared memory into a peer CTA's shared memory
// (TMA engine, no per-thread stores); the peer's mbarrier receives complete_tx(bytes) when it has landed
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes,
                                                  uint32_t mbar_cluster_addr) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(dst_cluster_addr), "r"(src_cta_addr), "r"(bytes), "r"(mbar_cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// one elected lane of a converged warp (same idiom as cute::elect_one_sync): lets the compiler keep the
// tcgen05.mma operands in uniform registers without per-instruction election loops
__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred = 0, laneid = 0;
  asm volatile("{\n.reg .b32 %%rx;\n.reg .pred %%px;\n     elect.sync %%rx|%%px, %2;\n@%%px mov.s32 %1, 1;\n     mov.s32 %0, %%rx;\n}\n"
               : "+r"(laneid), "+r"(pred) : "r"(0xFFFFFFFF));
  return pred;
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t addr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(addr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st8(uint32_t addr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "r"(addr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
#define TC_FENCE_BEFORE() asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory")
#define TC_FENCE_AFTER() asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory")
#define PROXY_FENCE_SMEM() asm volatile("fence.proxy.async.shared::cta;" ::: "memory")

__device__ __forceinline__ void tmem_ld8(uint32_t addr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(addr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
template <int N> __device__ __forceinline__ void tmem_ldn(uint32_t addr, float (&v)[N]) {
  if constexpr (N == 16) tmem_ld16(addr, v); else tmem_ld8(addr, v);
}
// NU consecutive floats (NU = 1 or 2) as one access
template <int N> __device__ __forceinline__ void ldn(const float* p, float (&d)[N]) {
  if constexpr (N == 2) { const float2 v = *reinterpret_cast<const float2*>(p); d[0] = v.x; d[1] = v.y; } else d[0] = *p;
}
template <int N> __device__ __forceinline__ void ldgn(const float* p, float (&d)[N]) {
  if constexpr (N == 2) { const float2 v = __ldg(reinterpret_cast<const float2*>(p)); d[0] = v.x; d[1] = v.y; } else d[0] = __ldg(p);
}
template <int N> __device__ __forceinline__ void stn(float* p, const float (&d)[N]) {
  if constexpr (N == 2) *reinterpret_cast<float2*>(p) = make_float2(d[0], d[1]); else *p = d[0];
}

// 3xTF32: D1[128x16] = A_hi*B_hi ; D2[128x16] = A_hi*B_lo + A_lo*B_hi over KS k-chunks of 8.  The
// accumulator add of the tensor core truncates, so the large term and the 2^-11-times-smaller
// correction terms are kept in separate TMEM accumulators (D2 = D1 + 16 columns) and summed in fp32
// by the epilogue: the chain into the large accumulator is KS adds instead of 3*KS.
// one accumulation chain: D[128x16] (=|+=) sum_ks A(ks) * B(ks); each chain is issued by its own warp so that
// the (issue-bound) tensor-core work of a step is spread over several instruction streams
__device__ __forceinline__ void issue_chain(uint32_t tD, uint32_t tA, uint32_t b_addr, uint32_t lbo_bytes, int KS,
                                            uint32_t idesc, uint32_t acc_first) {
  uint64_t d = make_desc(b_addr, lbo_bytes, 128);
  const uint64_t adv = (uint64_t)(2 * lbo_bytes) >> 4;
  mma_ts(tD, tA, d, idesc, acc_first);
#pragma unroll 4
  for (int ks = 1; ks < KS; ++ks) {
    d += adv;
    tA += 8;
    mma_ts(tD, tA, d, idesc, 1);
  }
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
constexpr int FWD_NT = 256;  // forward: 8 warps (warp w reaches TMEM lane quadrant w % 4)

// BT = live batch rows of the cluster tile.  The MMA is always N = 16; with BT = 8 the B operand keeps only 8 rows
// per core-matrix column and the descriptor's second 8-row group aliases the neighbouring block (its accumulator
// columns are never read), so the exchange moves half the bytes, every thread owns ONE unit of the gate math, and a
// batch of 128 rows spreads over 16 clusters = 128 SMs instead of 64.
template <int G, int BT>
__global__ void __launch_bounds__(FWD_NT, 1) rnn_fwd_tc_kernel(const __grid_constant__ TcArgs a) {
  constexpr int TC_BT = BT;
  constexpr int TPR = FWD_NT / BT;     // threads per batch row
  constexpr int NU = 32 / TPR;         // hidden units per thread (Hs <= 32)
  constexpr int KCB = BT * 8;          // floats per 4-wide k block of the B operand: hi[BT][4] | lo[BT][4]
  constexpr int QB = BT / 4;           // row quads per tile
  cg::cluster_group cluster = cg::this_cluster();
  const int C = cluster.num_blocks();
  const int rank = cluster.block_rank();
  const int tile = a.use_order ? (int)a.order[blockIdx.x / C] : (int)(blockIdx.x / C);
  const int b0 = tile * TC_BT;
  const int H = a.H, Hs = a.Hs, Kp = a.Kp, GH = G * H, B = a.B;
  const int KS = Kp / 8;
  const int j0 = rank * Hs;
  const int nj = max(0, min(Hs, H - j0));
  const int tid = threadIdx.x, warp = tid >> 5;
  const int quad = warp & 3;
  const uint32_t lane_off = (uint32_t)(quad * 32) << 16;

  extern __shared__ __align__(128) float smem[];
  // h exchange buffers = the MMA B operand itself: hbuf[2][Kp/4][hi|lo][16][4]; every CTA keeps the FULL h_{t-1}
  // (hi and lo = h - hi), its own Hs-unit slice written locally, the rest bulk-copied in by the owners
  float* hbuf = smem;
  const int HB = Kp * TC_BT * 2;                 // floats per buffer (Kp/4 blocks of 128 floats)
  float* gsm = hbuf + 2 * HB;                    // [16][GSM_LD] gate pre-activations, row b, column m = 4j+g
  // input pre-activations Xg of the CTA's slice, streamed by the TMA engine 3 steps ahead: ring [4][G][BT][Hs]
  // (ordinary prefetch loads would be drained by the fence.proxy.async before the h exchange, see the backward)
  float* xs = gsm + TC_BT * GSM_LD;
  const int XAS = TC_BT * Hs, XSB = G * XAS;
  __shared__ __align__(8) uint64_t x_full[4];
  __shared__ __align__(8) uint64_t raw_full[2];
  __shared__ __align__(8) uint64_t mma_done;
  __shared__ uint32_t tmem_base_s;
  __shared__ int lens_s[TC_BT];
  __shared__ int t_end_s;

#ifdef SBR_TC_TIMELINE_BUILD   // in-kernel clock64 timeline: compiled in only for profiling builds (build.py --timeline)
#define TC_KSTAMP(i) do { if (a.dbg && blockIdx.x == 0 && tid == 0) a.dbg[512 + (i)] = clock64(); } while (0)
#else
#define TC_KSTAMP(i) do { } while (0)
#endif
  TC_KSTAMP(0);
  if (tid < TC_BT) lens_s[tid] = (b0 + tid < B) ? min(a.len[b0 + tid], a.t_max) : 0;
  if (tid == 0) {
    mbar_init(&raw_full[0], 1);
    mbar_init(&raw_full[1], 1);
    mbar_init(&mma_done, 3);
    for (int i = 0; i < 4; ++i) mbar_init(&x_full[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // h_{-1} = learned init, broadcast over the rows: straight into the split B operand
  for (int i = tid; i < Kp * TC_BT; i += FWD_NT) {
    const int kc = i / (TC_BT * 4), rem = i - kc * (TC_BT * 4);
    const int k = kc * 4 + (rem & 3);
    const float v = k < H ? a.h_init[k] : 0.f;
    const float hi = tf32_hi(v);
    hbuf[kc * KCB + rem] = hi;
    hbuf[kc * KCB + BT * 4 + rem] = v - hi;
    hbuf[HB + kc * KCB + rem] = 0.f;
    hbuf[HB + kc * KCB + BT * 4 + rem] = 0.f;
  }
  TC_FENCE_BEFORE();
  __syncthreads();
  TC_FENCE_AFTER();
  if (tid == 0) {
    int mx = 0;
    for (int b = 0; b < TC_BT; ++b) mx = max(mx, lens_s[b]);
    t_end_s = mx;
  }
  const uint32_t tmem = tmem_base_s;
  const uint32_t tD = tmem;                 // three 16-column accumulators: hi*hi, hi*lo, lo*hi
  const uint32_t tAhi = tmem + 64;          // Kp columns
  const uint32_t tAlo = tmem + 64 + Kp;     // Kp columns (64 + 2*Kp <= 512)

  // ---- A operand: row m = 4*j + g  <->  W_hid[:, g*H + j0 + j]; K along the TMEM columns.
  //      A thread reads ITS row (a warp request touches 32 rows = 32 sectors: the prologue is bound by sector
  //      requests, 13 000 cycles when every row was read twice), so each word is loaded once: warps 0-3 stage the
  //      first half of K, warps 4-7 the second (same lane quadrants), hi and lo copies from the same registers;
  //      8 independent 16-byte loads in flight per thread.
  {
    const int m = quad * 32 + (tid & 31);
    const int j = m >> 2, g = m & 3;
    const bool live = (g < G) && (j < nj);
    const float* src = a.W_hidT + (int64_t)(g * H + j0 + j) * H;   // k contiguous
    const int kmid = min(Kp, ((Kp / 2 + 31) / 32) * 32);
    const int kb0 = warp >= 4 ? kmid : 0, kb1 = warp >= 4 ? Kp : kmid;
    for (int kb = kb0; kb < kb1; kb += 32) {
      float4 v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int k = kb + 4 * q;
        v[q] = make_float4(0.f, 0.f, 0.f, 0.f);                   // H % 4 == 0: 16-byte loads, guarded per quad
        if (live && k < H) v[q] = __ldg(reinterpret_cast<const float4*>(src + k));
      }
#pragma unroll
      for (int q = 0; q < 8; q += 2) {
        if (kb + 4 * q >= Kp) break;
        const float vv[8] = {v[q].x, v[q].y, v[q].z, v[q].w, v[q + 1].x, v[q + 1].y, v[q + 1].z, v[q + 1].w};
        uint32_t rh[8], rl[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float h = tf32_hi(vv[i]);
          rh[i] = __float_as_uint(h);
          rl[i] = __float_as_uint(vv[i] - h);
        }
        tmem_st8(tAhi + lane_off + kb + 4 * q, rh);
        tmem_st8(tAlo + lane_off + kb + 4 * q, rl);
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }

  TC_KSTAMP(1);
  // ---- gate-math ownership: row eb, units ju .. ju+NU-1 of the slice
  // 16-row tiles: a warp = 2 rows x 16 unit pairs (global accesses of a row are contiguous).  8-row tiles: a warp =
  // all 8 rows x 4 consecutive units, so that its writes into the B operand ([unit/4][row][4]) cover 32 consecutive
  // words instead of hitting one bank group 8 times.
  const int eb = (BT == 8) ? (tid & 7) : tid / TPR;
  const int ju = (BT == 8) ? (warp * 4 + ((tid & 31) >> 3)) : NU * (tid % TPR);
  const bool own = ju < nj;                       // nj is a multiple of 4 (H % 4 == 0, Hs % 4 == 0)
  const bool row_ok = b0 + eb < B;
  float cst[NU], wci[NU], wcf[NU], wco[NU];
#pragma unroll
  for (int u = 0; u < NU; ++u) {
    cst[u] = wci[u] = wcf[u] = wco[u] = 0.f;
    if (G == 4 && own) {
      wci[u] = a.peep[j0 + ju + u];
      wcf[u] = a.peep[H + j0 + ju + u];
      wco[u] = a.peep[2 * H + j0 + ju + u];
      cst[u] = a.c_init[j0 + ju + u];
    }
  }
  if (own && row_ok) {
#pragma unroll
    for (int u = 0; u < NU; ++u) {
      a.hs[(int64_t)(b0 + eb) * H + j0 + ju + u] = a.h_init[j0 + ju + u];
      if (G == 4) a.cs[(int64_t)(b0 + eb) * H + j0 + ju + u] = a.c_init[j0 + ju + u];
    }
  }
  float xc[G][NU];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int u = 0; u < NU; ++u) xc[g][u] = 0.f;
  auto x_issue = [&](int t) {        // executed by ONE thread: G boxes [BT rows x Hs units] of step t
    float* dst = xs + (t & 3) * XSB;
    mbar_arrive_expect_tx(&x_full[t & 3], (uint32_t)(XSB * 4));
#pragma unroll
    for (int g = 0; g < G; ++g)
      asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                   :: "r"(smem_u32(dst + g * XAS)), "l"(&a.tm_xg), "r"(smem_u32(&x_full[t & 3])), "r"(g * H + j0), "r"(t * B + b0)
                   : "memory");
  };
  auto x_fetch = [&](int t, float (&x)[G][NU]) {
    mbar_wait_cta(&x_full[t & 3], (t >> 2) & 1);
    if (own && t < lens_s[eb]) {
      const float* src = xs + (t & 3) * XSB + eb * Hs + ju;
#pragma unroll
      for (int g = 0; g < G; ++g) ldn<NU>(src + g * XAS, x[g]);
    }
  };
  PROXY_FENCE_SMEM();       // hbuf was written through the generic proxy
  TC_FENCE_BEFORE();
  __syncthreads();
  TC_FENCE_AFTER();
  const int t_end = t_end_s;
  if (tid == FWD_NT - 32 && !(a.xflags & 16)) {     // lane 0 of warp 7 (never issues MMAs)
    asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tm_xg) : "memory");
    for (int t = 0; t < 3 && t < t_end; ++t) x_issue(t);
  }
  // K-major copy of the own slice of a state block (hi and lo) for the weight-gradient GEMM: one 16-byte chunk =
  // (part, unit, 4 consecutive rows); `blk` = index of the hs block (0 = learned init, t+1 = state after step t)
  auto dump_hT = [&](const float* buf, int blk) {
    if (!a.hT) return;
    for (int c = tid; c < 2 * nj * QB; c += FWD_NT) {
      const int part = c / (nj * QB), rem = c - part * (nj * QB), j = rem / QB, q = rem - j * QB;
      const int k = j0 + j;
      const float* src = buf + (k >> 2) * KCB + part * (BT * 4) + (4 * q) * 4 + (k & 3);
      const float4 v = make_float4(src[0], src[4], src[8], src[12]);
      const long long rq = ((long long)blk * B + b0) / 4 + q;
      *reinterpret_cast<float4*>(a.hT + part * a.hT_part + (k >> 7) * a.hT_tile + (rq * 128 + (k & 127)) * 4) = v;
    }
  };
  dump_hT(hbuf, 0);
  // one phase of raw_full[x] = the h_t slices (hi + lo, BT rows) of all the OTHER owners have landed
  const uint32_t tx_bytes = (uint32_t)((H - nj) * BT * 8);
  if (tid == 0) {
    mbar_arrive_expect_tx(&raw_full[0], tx_bytes);
    mbar_arrive_expect_tx(&raw_full[1], tx_bytes);
  }
  cluster.sync();           // barriers initialised and armed everywhere before remote traffic

  const uint32_t idesc = make_idesc_tf32(128, TC_N);
  const uint32_t hbuf_addr = smem_u32(hbuf);
  const uint32_t bar_addr[2] = {smem_u32(&raw_full[0]), smem_u32(&raw_full[1])};
  const int hoff = ((j0 + ju) >> 2) * KCB + eb * 4 + (ju & 3);   // float offset of this thread's units in a buffer

  TC_KSTAMP(2);
#ifdef SBR_TC_TIMELINE_BUILD
  if (a.dbg && blockIdx.x == 0 && tid == 0) a.dbg[512 + 5] = t_end;
  long long ph[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, last_stamp = 0;
#define TC_STAMP(i) do { if (a.dbg && blockIdx.x == 0 && tid == 0) { const long long now_ = clock64(); if ((i) > 0) ph[i] += now_ - last_stamp; last_stamp = now_; } } while (0)
#else
#define TC_STAMP(i) do { } while (0)
#endif
  for (int t = 0; t < t_end; ++t) {
    const int cur = t & 1, nxt = cur ^ 1;
    TC_STAMP(0);
    const float* hprev = hbuf + cur * HB;
    if (t > 0) {
      // the slices of h_{t-1} owned by the other CTAs have landed (bulk copies, async proxy) next to our own
      const int use = (t - (cur == 0 ? 2 : 1)) >> 1;
      mbar_wait_cluster(&raw_full[cur], use & 1);
      TC_STAMP(1);
      if (tid == 0) mbar_arrive_expect_tx(&raw_full[cur], tx_bytes);   // arm the next use of this buffer
      TC_FENCE_AFTER();
    }
    TC_STAMP(2);
    if (warp >= 4 && warp < 7) {
      // warp 4: D1 = A_hi B_hi, warp 5: D2 = A_hi B_lo, warp 6: D3 = A_lo B_hi  (3xTF32 split, one chain per warp)
      if (elect_one_sync()) {
        const int c = warp - 4;
        const uint32_t bbase = hbuf_addr + cur * HB * 4 + (c == 1 ? BT * 16 : 0);
        issue_chain(tD + c * TC_N, c == 2 ? tAlo : tAhi, bbase, KCB * 4, KS, idesc, 0);
        umma_commit(&mma_done);
      }
      __syncwarp();
    }
    TC_STAMP(3);
    // stage (t + 3) % 4 was last read in the gate math of step t-1, before the barrier that ended it: refill it;
    // then this step's input pre-activations (landed steps ago) while the tensor core works
    if (!(a.xflags & 16)) {
      if (tid == FWD_NT - 32 && t + 3 < t_end) x_issue(t + 3);
      x_fetch(t, xc);
    }
    mbar_wait_cta(&mma_done, t & 1);
    TC_STAMP(4);
    TC_FENCE_AFTER();
    if (warp < 4) {
      float v[BT], w[BT], x[BT];
      tmem_ldn<BT>(tD + lane_off, v);
      tmem_ldn<BT>(tD + TC_N + lane_off, w);
      tmem_ldn<BT>(tD + 2 * TC_N + lane_off, x);
#pragma unroll
      for (int b = 0; b < BT; ++b) gsm[b * GSM_LD + tid] = v[b] + (w[b] + x[b]);
    }
    TC_FENCE_BEFORE();
    __syncthreads();
    TC_STAMP(5);

    float hn[NU];
#pragma unroll
    for (int u = 0; u < NU; ++u) hn[u] = 0.f;
    float sv[NU][4];
    bool active = false;
    if (own) {
      active = t < lens_s[eb];
      float hph[NU], hpl[NU], hp[NU];
      ldn<NU>(hprev + hoff, hph);
      ldn<NU>(hprev + hoff + BT * 4, hpl);
#pragma unroll
      for (int u = 0; u < NU; ++u) hp[u] = hph[u] + hpl[u];
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        const float4 p4 = *reinterpret_cast<const float4*>(gsm + eb * GSM_LD + 4 * (ju + u));
        const float pre[4] = {p4.x, p4.y, p4.z, p4.w};
        float xg[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int g = 0; g < G; ++g) xg[g] = xc[g][u];
        hn[u] = hp[u];
        sv[u][0] = sv[u][1] = sv[u][2] = sv[u][3] = 0.f;
        if (active) {
          if constexpr (G == 4) {
            const float c_prev = cst[u];
            const float ig = sigmoidf_(xg[0] + pre[0] + c_prev * wci[u]);
            const float fg = sigmoidf_(xg[1] + pre[1] + c_prev * wcf[u]);
            const float gg = tanhf_(xg[2] + pre[2]);
            const float c_new = fg * c_prev + ig * gg;
            const float og = sigmoidf_(xg[3] + pre[3] + c_new * wco[u]);
            hn[u] = og * tanhf_(c_new);
            cst[u] = c_new;
            sv[u][0] = ig; sv[u][1] = fg; sv[u][2] = gg; sv[u][3] = og;
          } else if constexpr (G == 3) {
            const float r = sigmoidf_(pre[0] + xg[0]);
            const float uu = sigmoidf_(pre[1] + xg[1]);
            const float ac = pre[2];
            const float cand = tanhf_(xg[2] + r * ac);
            hn[u] = (1.f - uu) * hp[u] + uu * cand;
            sv[u][0] = r; sv[u][1] = uu; sv[u][2] = cand; sv[u][3] = ac;
          } else {
            const float z = xg[0] + pre[0];
            hn[u] = a.relu ? fmaxf(z, 0.f) : tanhf_(z);
          }
        }
      }
      // h_t pair of this thread, pre-split, into the LOCAL copy of the next buffer
      float hh[NU], hl[NU];
#pragma unroll
      for (int u = 0; u < NU; ++u) { hh[u] = tf32_hi(hn[u]); hl[u] = hn[u] - hh[u]; }
      stn<NU>(hbuf + nxt * HB + hoff, hh);
      stn<NU>(hbuf + nxt * HB + hoff + BT * 4, hl);
    }
    TC_STAMP(6);
    // own slice complete in shared memory -> one bulk copy per peer CTA (hi and lo blocks are contiguous);
    // lane 0 of warp w serves peer w: the C-1 copies are issued concurrently by different warps.  (Measured:
    // the exchange is bound by the ~20 B/clk DSMEM egress of the SM; per-thread st.async of the same bytes and
    // fp32-only st.async + receiver-side split were both slower, see DESIGN.md.)
    PROXY_FENCE_SMEM();
    TC_STAMP(8);
    __syncthreads();
    TC_STAMP(9);
    if ((tid & 31) == 0 && nj > 0) {
      const uint32_t src = hbuf_addr + (uint32_t)(nxt * HB + (j0 >> 2) * KCB) * 4u;
      const uint32_t bytes = (uint32_t)(nj >> 2) * (uint32_t)(KCB * 4);
      for (int rr = warp; rr < C; rr += FWD_NT / 32)
        if (rr != rank) bulk_copy_to_peer(map_to_rank(src, rr), src, bytes, map_to_rank(bar_addr[nxt], rr));
    }
    TC_STAMP(10);
    // saved trajectories for the backward pass: issued last so that nothing on the critical path waits on them
    if (own && row_ok && !(a.xflags & 32)) {
      const int64_t row1 = (int64_t)(t + 1) * B + b0 + eb;
      stn<NU>(a.hs + row1 * H + j0 + ju, hn);
      if (G == 4) stn<NU>(a.cs + row1 * H + j0 + ju, cst);
      if (active && G > 1) {
        float* ap = a.act + ((int64_t)t * B + b0 + eb) * 4 * H + j0 + ju;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float o[NU];
#pragma unroll
          for (int u = 0; u < NU; ++u) o[u] = sv[u][g];
          stn<NU>(ap + g * H, o);
        }
      }
    }
    if (!(a.xflags & 64)) dump_hT(hbuf + nxt * HB, t + 1);
    TC_STAMP(7);
  }

  TC_KSTAMP(3);
#ifdef SBR_TC_TIMELINE_BUILD
  if (a.dbg && blockIdx.x == 0 && tid == 0) for (int i = 0; i < 12; ++i) a.dbg[i] = ph[i];
#endif
  // final state: wait for the last exchange (only the own slice is written out)
  if (t_end > 0) {
    const int fin = t_end & 1;
    const int use = (t_end - (fin == 0 ? 2 : 1)) >> 1;
    mbar_wait_cluster(&raw_full[fin], use & 1);
  }
  if (a.h_last && own && row_ok) {
    const int fin = t_end & 1;
    float hh[NU], hl[NU];
    ldn<NU>(hbuf + fin * HB + hoff, hh);
    ldn<NU>(hbuf + fin * HB + hoff + BT * 4, hl);
#pragma unroll
    for (int u = 0; u < NU; ++u) hh[u] += hl[u];
    stn<NU>(a.h_last + (int64_t)(b0 + eb) * H + j0 + ju, hh);
  }
  TC_FENCE_BEFORE();
  cluster.sync();   // nobody exits while peers may still write to / arrive on this CTA's shared memory
  TC_KSTAMP(4);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512));
}

// ------------------------------------------------------------------------------------------------
// backward (BPTT)
// ------------------------------------------------------------------------------------------------
// TMEM map (MT = number of 128-row tiles of the hidden index k, Kb = 4*Hs own gate columns):
//   D1_mt at 32*mt, D2_mt at 32*mt+16; A_mt_hi at 32*MT + mt*2*Kb, A_mt_lo right after it.
// The saved activations of a step (gates, cell states, gradient from the layer above) come from global memory.  When
// the compute threads fetched them with ordinary loads, the fence.proxy.async every thread executes before the MMA
// and before the bulk copies (a MEMBAR that drains the thread's outstanding loads) put the full L2/HBM latency of
// that prefetch on the per-step critical path (0.33 -> 0.22 ms for the whole scan without the loads).  They are now
// streamed by the TMA engine: one elected thread issues one 2-D tiled load per array ([BT rows x Hs units] box) three
// steps ahead into a 4-stage shared-memory ring, completion lands on an mbarrier, and the compute threads read the
// stage with plain LDS.
constexpr int bwd_threads(int) { return FWD_NT; }

template <int G, int MT, int BT>
__global__ void __launch_bounds__(bwd_threads(BT), 1) rnn_bwd_tc_kernel(const __grid_constant__ TcArgs a) {
  constexpr int TC_BT = BT;
  constexpr int TPR = FWD_NT / BT;
  constexpr int NU = 32 / TPR;
  constexpr int QB = BT / 4;

  cg::cluster_group cluster = cg::this_cluster();
  const int C = cluster.num_blocks();
  const int rank = cluster.block_rank();
  const int tile = a.use_order ? (int)a.order[blockIdx.x / C] : (int)(blockIdx.x / C);
  const int b0 = tile * TC_BT;
  const int H = a.H, Hs = a.Hs, GH = G * H, B = a.B;
  const int Kb = 4 * Hs;                 // contraction length: own gate columns, kk = 4*j + g
  const int KS = Kb / 8;
  const int HP = MT * 128;               // padded hidden extent of the partial dh
  const int j0 = rank * Hs;
  const int nj = max(0, min(Hs, H - j0));
  const int tid = threadIdx.x, warp = tid >> 5;
  const int quad = warp & 3;
  const uint32_t lane_off = (uint32_t)(quad * 32) << 16;

  extern __shared__ __align__(128) float smem[];
  float* Bhi = smem;                            // [Kb/4][16][4]  da (hi)
  float* Blo = Bhi + Kb * TC_BT;                // da (lo)
  float* part = Blo + Kb * TC_BT;               // [2][C][16][Hs] partial dh received from the peers (bulk copies)
  float* sbuf = part + 2 * C * TC_BT * Hs;      // [2][C][16][Hs] partial dh of this CTA, grouped by owner (send buffer)
  const int PB = C * TC_BT * Hs;                // floats per part / send buffer
  float* stag = sbuf + 2 * PB;                  // [4][7][BT][Hs] saved tensors of a step, filled by the loader warps
  const int SGB = 7 * TC_BT * Hs;
  __shared__ __align__(8) uint64_t sv_full[4];
  __shared__ __align__(8) uint64_t part_full[2];
  __shared__ __align__(8) uint64_t mma_done;
  __shared__ uint32_t tmem_base_s;
  __shared__ int lens_s[TC_BT];
  __shared__ int t_end_s;

  if (tid < TC_BT) lens_s[tid] = (b0 + tid < B) ? min(a.len[b0 + tid], a.t_max) : 0;
  if (tid == 0) {
    mbar_init(&part_full[0], 1);
    mbar_init(&part_full[1], 1);
    mbar_init(&mma_done, MT + 1);
    for (int i = 0; i < 4; ++i) mbar_init(&sv_full[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  {
    for (int i = tid; i < 2 * Kb * TC_BT; i += FWD_NT) Bhi[i] = 0.f;            // Bhi and Blo are contiguous
    for (int i = tid; i < 4 * C * TC_BT * Hs; i += FWD_NT) part[i] = 0.f;          // part and sbuf are contiguous
  }
  TC_FENCE_BEFORE();
  __syncthreads();
  TC_FENCE_AFTER();
  if (tid == 0) {
    int mx = 0;
    for (int b = 0; b < TC_BT; ++b) mx = max(mx, lens_s[b]);
    t_end_s = mx;
  }
  const uint32_t tmem = tmem_base_s;

  // ---- A operand tiles: row = hidden index k, column kk = 4*j + g  <->  W_hid[k][g*H + j0 + j]
  //      every word is loaded once: warps 0-3 stage the first half of the columns, warps 4-7 the second, hi and lo
  //      copies from the same registers (the prologue is bound by sector requests: a warp request = 32 rows)
  {
    const int cmid = min(Kb, ((Kb / 2 + 31) / 32) * 32);
    const int cb0 = warp >= 4 ? cmid : 0, cb1 = warp >= 4 ? Kb : cmid;
    for (int mt = 0; mt < MT; ++mt) {
      const int k = mt * 128 + quad * 32 + (tid & 31);
      const float* src = a.W_hid + (int64_t)k * GH + j0;
      const uint32_t dst = tmem + 32 * MT + mt * 2 * Kb + lane_off;
      for (int cb = cb0; cb < cb1; cb += 32) {                    // two passes of 4 units x 4 gates: 8 loads in flight
       float4 vgs[2][4];
#pragma unroll
       for (int h2 = 0; h2 < 2; ++h2)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int jb = (cb + 16 * h2) >> 2;
          vgs[h2][g] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (k < H && g < G && jb < nj) vgs[h2][g] = __ldg(reinterpret_cast<const float4*>(src + g * H + jb));   // nj % 4 == 0
        }
#pragma unroll
       for (int h2 = 0; h2 < 2; ++h2) {
        const int c0 = cb + 16 * h2;
        if (c0 >= Kb) break;
        float4 vg[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) vg[g] = vgs[h2][g];
        uint32_t r0[8], r1[8], l0[8], l1[8];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float u4[4] = {vg[g].x, vg[g].y, vg[g].z, vg[g].w};
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const float h = tf32_hi(u4[jj]);
            const uint32_t hb = __float_as_uint(h), lb = __float_as_uint(u4[jj] - h);
            if (jj < 2) { r0[4 * jj + g] = hb; l0[4 * jj + g] = lb; } else { r1[4 * (jj - 2) + g] = hb; l1[4 * (jj - 2) + g] = lb; }
          }
        }
        tmem_st8(dst + c0, r0);
        tmem_st8(dst + Kb + c0, l0);
        if (c0 + 8 < Kb) { tmem_st8(dst + c0 + 8, r1); tmem_st8(dst + Kb + c0 + 8, l1); }
       }
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }

  // thread <-> (row, unit) as in the forward kernel: with 8-row tiles a warp's 16-byte stores of da into the B
  // operand ([unit][row][4 gates]) are 512 contiguous bytes (conflict-free) instead of 32 hits on one bank group
  const int eb = (BT == 8) ? (tid & 7) : tid / TPR;
  const int ju = (BT == 8) ? (warp * 4 + ((tid & 31) >> 3)) : NU * (tid % TPR);
  const bool own = ju < nj;
  const bool row_ok = b0 + eb < B;
  float carry[NU], dcs[NU], dpe[NU][3], wci[NU], wcf[NU], wco[NU];
  float dbias[NU][4];                                                   // sum over steps of dXg (bias gradient)
#pragma unroll
  for (int u = 0; u < NU; ++u) {
    dbias[u][0] = dbias[u][1] = dbias[u][2] = dbias[u][3] = 0.f;
    carry[u] = (a.dh_last && own && row_ok) ? a.dh_last[(int64_t)(b0 + eb) * H + j0 + ju + u] : 0.f;
    dcs[u] = 0.f;
    dpe[u][0] = dpe[u][1] = dpe[u][2] = 0.f;
    wci[u] = wcf[u] = wco[u] = 0.f;
    if (G == 4 && own) {
      wci[u] = a.peep[j0 + ju + u];
      wcf[u] = a.peep[H + j0 + ju + u];
      wco[u] = a.peep[2 * H + j0 + ju + u];
    }
  }
  TC_FENCE_BEFORE();
  __syncthreads();
  TC_FENCE_AFTER();
  const int t_end = t_end_s;

  // K-major copy of da (hi | lo) for the weight-gradient GEMM.  Thread <-> (part, row quad q, unit j): it reads the
  // 4 rows x 4 gates block of that unit with four 16-byte shared loads and writes one 16-byte chunk per gate
  // (= 4 consecutive rows of one gate column); consecutive lanes hold consecutive units = consecutive chunks.
  int dmp_src = -1;
  long long dmp_dst[4] = {0, 0, 0, 0};
  if (a.aT && tid < 2 * QB * nj) {
    const int part = tid / (QB * nj), rem = tid - part * (QB * nj), q = rem / nj, j = rem - q * nj;
    dmp_src = part * (Kb * TC_BT) + j * (TC_BT * 4) + (4 * q) * 4;     // Blo follows Bhi
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int col = g * H + j0 + j;
      dmp_dst[g] = part * a.aT_part + (long long)(col >> 7) * a.aT_tile + ((long long)q * 128 + (col & 127)) * 4;
    }
  }
  auto dump_aT = [&](int t, bool zero) {
    if (dmp_src < 0) return;
    float4 v[4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
      v[r] = zero ? make_float4(0.f, 0.f, 0.f, 0.f) : *reinterpret_cast<const float4*>(Bhi + dmp_src + r * 4);
    const long long tb = (((long long)t * B + b0) / 4) * 512;
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const float4 o = g == 0 ? make_float4(v[0].x, v[1].x, v[2].x, v[3].x)
                     : g == 1 ? make_float4(v[0].y, v[1].y, v[2].y, v[3].y)
                     : g == 2 ? make_float4(v[0].z, v[1].z, v[2].z, v[3].z)
                              : make_float4(v[0].w, v[1].w, v[2].w, v[3].w);
      *reinterpret_cast<float4*>(a.aT + dmp_dst[g] + tb) = o;
    }
  };
  // masked tail [t_end, t_max): exactly zero gradients
  for (int t = t_end; t < a.t_max; ++t) dump_aT(t, true);
  for (int t = t_end; t < a.t_max; ++t) {
    if (own && row_ok) {
      const int64_t row = (int64_t)t * B + b0 + eb;
#pragma unroll
      float z[NU];
#pragma unroll
      for (int u = 0; u < NU; ++u) z[u] = 0.f;
#pragma unroll
      for (int g = 0; g < G; ++g) stn<NU>(a.dXg + row * GH + g * H + j0 + ju, z);
      if (G == 3) stn<NU>(a.dac + row * H + j0 + ju, z);
    }
  }

  // saved tensors of a step for this thread's units: [slot][unit]
  //  LSTM: i f g o c_prev c_new | GRU: r u cand a_c h_prev | Vanilla: h_new ; last slot: dhs from above
  constexpr int NSAVE = (G == 4) ? 6 : (G == 3 ? 5 : 1);
  const int NA = NSAVE + (a.dhs ? 1 : 0);          // arrays staged per step
  float sv[NSAVE + 1][NU];
#pragma unroll
  for (int s = 0; s <= NSAVE; ++s)
#pragma unroll
    for (int u = 0; u < NU; ++u) sv[s][u] = 0.f;

  // ---- TMA staging ring: LD_D stages, LD_P steps ahead (the activations come back from HBM with ~2 us latency
  //      under load, i.e. more than one step)
  constexpr int LD_D = 4;
  const int LD_P = a.ld_p;                          // 1 .. 3
  const int AS = TC_BT * Hs;                        // floats per array per stage (multiple of 32: 128-byte aligned)
  auto tma2d = [](float* dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
  };
  auto sv_issue = [&](int t) {       // executed by ONE thread
    if (t < 0 || (a.xflags & 128)) return;
    float* sg = stag + (t & (LD_D - 1)) * SGB;
    uint64_t* bar = &sv_full[t & (LD_D - 1)];
    mbar_arrive_expect_tx(bar, (uint32_t)(NA * AS * 4));
    const int r = t * B + b0;
    if constexpr (G == 4) {
#pragma unroll
      for (int g = 0; g < 4; ++g) tma2d(sg + g * AS, &a.tm_act, g * H + j0, r, bar);
      tma2d(sg + 4 * AS, &a.tm_cs, j0, r, bar);
      tma2d(sg + 5 * AS, &a.tm_cs, j0, r + B, bar);
    } else if constexpr (G == 3) {
#pragma unroll
      for (int g = 0; g < 4; ++g) tma2d(sg + g * AS, &a.tm_act, g * H + j0, r, bar);
      tma2d(sg + 4 * AS, &a.tm_hs, j0, r, bar);
    } else {
      tma2d(sg, &a.tm_hs, j0, r + B, bar);
    }
    if (a.dhs) tma2d(sg + NSAVE * AS, &a.tm_dhs, j0, r, bar);
  };
  // compute threads: this step's saved tensors out of the staging buffer (rows past their length are never used)
  auto fetch_saved = [&](int t) {
    if (!(a.xflags & 128)) mbar_wait_cta(&sv_full[t & (LD_D - 1)], ((t_end - 1 - t) >> 2) & 1);
    if (own && t < lens_s[eb]) {
      const float* sg = stag + (t & (LD_D - 1)) * SGB + eb * Hs + ju;
#pragma unroll
      for (int s2 = 0; s2 < NSAVE + 1; ++s2)
        if (s2 < NA) ldn<NU>(sg + s2 * TC_BT * Hs, sv[s2]);
    }
  };
  if (tid == FWD_NT - 32) {     // lane 0 of warp 7 (the one compute warp that never issues MMAs)
    asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tm_act) : "memory");
    for (int i = 1; i <= LD_P; ++i) sv_issue(t_end - i);
  }

  // one phase of part_full[x] = the partial dh blocks of my units have landed from the C-1 other CTAs
  const uint32_t tx_bytes = (a.xflags & 8) ? (uint32_t)((C - 1) * 16) : (uint32_t)((C - 1) * TC_BT * Hs * 4);
  if (tid == 0) {
    mbar_arrive_expect_tx(&part_full[0], tx_bytes);
    mbar_arrive_expect_tx(&part_full[1], tx_bytes);
  }
  cluster.sync();

  const uint32_t idesc = make_idesc_tf32(128, TC_N);
  const uint32_t part_addr = smem_u32(part);
  const uint32_t sbuf_addr = smem_u32(sbuf);
  const uint32_t bar_addr[2] = {smem_u32(&part_full[0]), smem_u32(&part_full[1])};
  int n_wait[2] = {0, 0};      // completed phases of each part_full barrier

#ifdef SBR_TC_TIMELINE_BUILD
  long long bph[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, blast = 0;
#define TC_BSTAMP(i) do { if (a.dbg && blockIdx.x == 0 && tid == 0) { const long long now_ = clock64(); if ((i) > 0) bph[i] += now_ - blast; blast = now_; } } while (0)
  const long long bstart = a.dbg ? clock64() : 0;
#else
#define TC_BSTAMP(i) do { } while (0)
#endif
  // TMEM lane of this thread = hidden index k of tile warp/4; its owner CTA and slot there (loop-invariant)
  const int k_mine = (warp >> 2) * 128 + quad * 32 + (tid & 31);
  const int sb_off = (k_mine < H && (warp >> 2) < MT) ? ((k_mine / Hs) * TC_BT) * Hs + (k_mine % Hs) : -1;
  for (int t = t_end - 1; t >= 0; --t) {
    const int par = t & 1, rpar = par ^ 1;
    TC_BSTAMP(0);
    if (!(a.xflags & 4)) fetch_saved(t);

    // ---- everything of the gate gradients that does not depend on dh_t is computed BEFORE waiting for the
    //      partial sums of step t+1 (the exchange is in flight meanwhile): after the wait only a short chain of
    //      multiplies by these coefficients remains on the critical path
    const bool active = own && t < lens_s[eb];
    float kc[NU][5];
#pragma unroll
    for (int u = 0; u < NU; ++u) {
      kc[u][0] = kc[u][1] = kc[u][2] = kc[u][3] = kc[u][4] = 0.f;
      if (active) {
        if constexpr (G == 4) {
          const float ig = sv[0][u], fg = sv[1][u], gg = sv[2][u], og = sv[3][u], c_prev = sv[4][u];
          const float tc = tanhf_(sv[5][u]);
          kc[u][0] = tc * og * (1.f - og);          // do_pre = d * kc0
          kc[u][1] = og * (1.f - tc * tc);          // dct    = dcs + d * kc1 + do_pre * wco
          kc[u][2] = gg * ig * (1.f - ig);          // di_pre = dct * kc2
          kc[u][3] = c_prev * fg * (1.f - fg);      // df_pre = dct * kc3
          kc[u][4] = ig * (1.f - gg * gg);          // dg_pre = dct * kc4
        } else if constexpr (G == 3) {
          const float r = sv[0][u], uu = sv[1][u], cand = sv[2][u], ac = sv[3][u], h_prev = sv[4][u];
          kc[u][0] = (cand - h_prev) * uu * (1.f - uu);   // du_pre = d * kc0
          kc[u][1] = uu * (1.f - cand * cand);            // dq     = clip(d * kc1)
          kc[u][2] = ac * r * (1.f - r);                  // dr_pre = dq * kc2
          kc[u][3] = 1.f - uu;                            // carry  = d * kc3
        } else {
          kc[u][0] = a.relu ? (sv[0][u] > 0.f ? 1.f : 0.f) : 1.f - sv[0][u] * sv[0][u];   // dq = clip(d * kc0)
        }
      }
    }

    // ---- phase A: dh_t = carry + partials of step t+1 (+ gradient from the layer above); gate gradients
    if (t < t_end - 1) {
      mbar_wait_cluster(&part_full[rpar], n_wait[rpar] & 1);
      n_wait[rpar]++;
      if (tid == 0) mbar_arrive_expect_tx(&part_full[rpar], tx_bytes);
    }
    TC_BSTAMP(1);
    float dx_out[NU][4], dac_out[NU];
    if (own) {
      float dh[NU];
#pragma unroll
      for (int u = 0; u < NU; ++u) dh[u] = carry[u];
      if (t < t_end - 1) {
        // own contribution straight from the send buffer of step t+1, the others from the received blocks;
        // all loads first (independent), then the adds
        float p[8][NU];
#pragma unroll
        for (int src = 0; src < 8; ++src) {
#pragma unroll
          for (int u = 0; u < NU; ++u) p[src][u] = 0.f;
          if (src < C) {
            const float* base = (src == rank) ? sbuf + rpar * PB : part + rpar * PB;
            ldn<NU>(base + (src * TC_BT + eb) * Hs + ju, p[src]);
          }
        }
#pragma unroll
        for (int u = 0; u < NU; ++u)
          dh[u] += ((p[0][u] + p[1][u]) + (p[2][u] + p[3][u])) + ((p[4][u] + p[5][u]) + (p[6][u] + p[7][u]));
      }
      float da[NU][4], dx[NU][4];   // [unit][gate]
#pragma unroll
      for (int u = 0; u < NU; ++u) {
#pragma unroll
        for (int g = 0; g < 4; ++g) da[u][g] = dx[u][g] = 0.f;
        float carry_new = dh[u];
        if (active) {
          const float d = dh[u] + sv[NSAVE][u];
          if constexpr (G == 4) {
            const float fg = sv[1][u], c_prev = sv[4][u], c_new = sv[5][u];
            const float do_pre = d * kc[u][0];
            const float dct = dcs[u] + d * kc[u][1] + do_pre * wco[u];
            const float di_pre = dct * kc[u][2];
            const float df_pre = dct * kc[u][3];
            const float dg_pre = dct * kc[u][4];
            dpe[u][0] += di_pre * c_prev;
            dpe[u][1] += df_pre * c_prev;
            dpe[u][2] += do_pre * c_new;
            dcs[u] = dct * fg + di_pre * wci[u] + df_pre * wcf[u];
            da[u][0] = clipf_(di_pre, a.clip);
            da[u][1] = clipf_(df_pre, a.clip);
            da[u][2] = clipf_(dg_pre, a.clip);
            da[u][3] = clipf_(do_pre, a.clip);
#pragma unroll
            for (int g = 0; g < 4; ++g) dx[u][g] = da[u][g];
            carry_new = 0.f;
          } else if constexpr (G == 3) {
            const float r = sv[0][u];
            const float du_pre = d * kc[u][0];
            const float dq = clipf_(d * kc[u][1], a.clip);
            const float dr_pre = dq * kc[u][2];
            da[u][0] = clipf_(dr_pre, a.clip);
            da[u][1] = clipf_(du_pre, a.clip);
            da[u][2] = clipf_(dq * r, a.clip);
            dx[u][0] = da[u][0];
            dx[u][1] = da[u][1];
            dx[u][2] = dq;
            carry_new = d * kc[u][3];
          } else {
            const float dq = clipf_(d * kc[u][0], a.clip);
            da[u][0] = dq;
            dx[u][0] = dq;
            carry_new = 0.f;
          }
        }
        carry[u] = carry_new;
        // B operand element (row eb, kk = 4*(ju+u) + g): one 16-byte store per unit, hi and lo
        float4 h4, l4;
        h4.x = tf32_hi(da[u][0]); h4.y = tf32_hi(da[u][1]); h4.z = tf32_hi(da[u][2]); h4.w = tf32_hi(da[u][3]);
        l4.x = da[u][0] - h4.x; l4.y = da[u][1] - h4.y; l4.z = da[u][2] - h4.z; l4.w = da[u][3] - h4.w;
        *reinterpret_cast<float4*>(Bhi + (ju + u) * (TC_BT * 4) + eb * 4) = h4;
        *reinterpret_cast<float4*>(Blo + (ju + u) * (TC_BT * 4) + eb * 4) = l4;
      }
#pragma unroll
      for (int u = 0; u < NU; ++u)
#pragma unroll
        for (int g = 0; g < 4; ++g) { dx_out[u][g] = dx[u][g]; dac_out[u] = da[u][2]; dbias[u][g] += dx[u][g]; }
    }
    TC_BSTAMP(2);
    PROXY_FENCE_SMEM();
    TC_BSTAMP(3);
    TC_FENCE_BEFORE();
    __syncthreads();
    TC_FENCE_AFTER();
    TC_BSTAMP(4);
    // stage (t - LD_P) % LD_D last held step t+1, which every thread read before the barrier above: refill it
    if (tid == FWD_NT - 32) sv_issue(t - LD_P);

    // ---- phase B: partial dh_{t-1}[b][k] = sum_kk da[b][kk] * W_hid[k][kk], all k (MT tiles of 128 rows)
    if (warp >= 4 && warp <= 4 + MT) {
      // warp 4: the main chains D1_mt = A_hi B_hi of every hidden tile; warp 5+mt: the correction chain
      // D2_mt = A_hi B_lo + A_lo B_hi of tile mt  (MT + 1 instruction streams, MT + 1 commits)
      if (elect_one_sync()) {
        const uint32_t bhi = smem_u32(Bhi), blo = smem_u32(Blo);
        if (warp == 4) {
          for (int mt = 0; mt < MT; ++mt) issue_chain(tmem + 32 * mt, tmem + 32 * MT + mt * 2 * Kb, bhi, TC_BT * 16, KS, idesc, 0);
        } else {
          const int mt = warp - 5;
          const uint32_t tAhi = tmem + 32 * MT + mt * 2 * Kb;
          issue_chain(tmem + 32 * mt + 16, tAhi, blo, TC_BT * 16, KS, idesc, 0);
          issue_chain(tmem + 32 * mt + 16, tAhi + Kb, bhi, TC_BT * 16, KS, idesc, 1);
        }
        umma_commit(&mma_done);
      }
      __syncwarp();
    }
    // K-major copy of this step's da for the weight-gradient GEMM and the gradient wrt the input pre-activations:
    // streamed out while the tensor core works (right after this step's proxy fence, a full step before the next
    // one, so no fence ever waits on these stores)
    if (!(a.xflags & 1)) dump_aT(t, false);
    if (own && row_ok && !(a.xflags & 2)) {
      const int64_t row = (int64_t)t * B + b0 + eb;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float o[NU];
#pragma unroll
        for (int u = 0; u < NU; ++u) o[u] = dx_out[u][g];
        stn<NU>(a.dXg + row * GH + g * H + j0 + ju, o);
      }
      if (G == 3) stn<NU>(a.dac + row * H + j0 + ju, dac_out);
    }
    TC_BSTAMP(5);
    mbar_wait_cta(&mma_done, (t_end - 1 - t) & 1);
    TC_FENCE_AFTER();
    TC_BSTAMP(6);
    {
      // hidden tile mt is drained by warps 4*mt .. 4*mt+3 (MT == 2), or by warps 0-3 alone (MT == 1)
      float* sb = sbuf + par * PB;
      const int mt = warp >> 2;
      if (mt < MT) {
        float v[BT], w[BT];
        tmem_ldn<BT>(tmem + 32 * mt + lane_off, v);
        tmem_ldn<BT>(tmem + 32 * mt + 16 + lane_off, w);
        if (sb_off >= 0) {
#pragma unroll
          for (int b = 0; b < BT; ++b) sb[sb_off + b * Hs] = v[b] + w[b];
        }
      }
    }
    // ---- phase C: reduce-scatter: one bulk copy of the [BT x Hs] block per peer, into slot [par][my rank]
    TC_BSTAMP(7);
    PROXY_FENCE_SMEM();
    TC_BSTAMP(8);
    TC_FENCE_BEFORE();
    __syncthreads();
    TC_BSTAMP(9);
    if ((tid & 31) == 0) {
      const uint32_t bytes = (a.xflags & 8) ? 16u : (uint32_t)(TC_BT * Hs * 4);
      for (int rr = warp; rr < C; rr += FWD_NT / 32) {
        if (rr == rank) continue;
        const uint32_t src = sbuf_addr + (uint32_t)(par * PB + rr * TC_BT * Hs) * 4u;
        const uint32_t dst = part_addr + (uint32_t)(par * PB + rank * TC_BT * Hs) * 4u;
        bulk_copy_to_peer(map_to_rank(dst, rr), src, bytes, map_to_rank(bar_addr[par], rr));
      }
    }
    TC_BSTAMP(10);
  }
#ifdef SBR_TC_TIMELINE_BUILD
  if (a.dbg && blockIdx.x == 0 && tid == 0) {
    for (int i = 0; i < 12; ++i) a.dbg[64 + i] = bph[i];
    a.dbg[76] = clock64() - bstart;
    a.dbg[77] = t_end;
  }
#endif

  // ---- gradients of the learned initial states and of the peepholes
  if (t_end > 0) {
    mbar_wait_cluster(&part_full[0], n_wait[0] & 1);   // step t = 0 wrote buffer 0
  }
  if (own && row_ok) {
#pragma unroll
    for (int u = 0; u < NU; ++u) {
      float dh = carry[u];
      if (t_end > 0)
        for (int src = 0; src < C; ++src) dh += ((src == rank) ? sbuf : part)[(src * TC_BT + eb) * Hs + ju + u];   // buffer 0
      atomicAdd(a.g_h_init + j0 + ju + u, dh);
      if (a.g_b) {
#pragma unroll
        for (int g = 0; g < G; ++g) atomicAdd(a.g_b + g * H + j0 + ju + u, dbias[u][g]);
      }
      if (G == 4) {
        atomicAdd(a.g_c_init + j0 + ju + u, dcs[u]);
        atomicAdd(a.g_peep + j0 + ju + u, dpe[u][0]);
        atomicAdd(a.g_peep + H + j0 + ju + u, dpe[u][1]);
        atomicAdd(a.g_peep + 2 * H + j0 + ju + u, dpe[u][2]);
      }
    }
  }
  TC_FENCE_BEFORE();
  cluster.sync();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512));
}

// ------------------------------------------------------------------------------------------------
// launch plumbing
// ------------------------------------------------------------------------------------------------
struct TcPlan { int C, Hs, Kp, MT; size_t smem, smem_bwd; bool ok, bwd_ok; };

TcPlan tc_plan(int G, int H) {
  TcPlan p{};
  p.ok = false;
  if (getenv("SBR_DISABLE_TC")) return p;
  if (H % 4 != 0 || H < 8) return p;
  p.Kp = (int)round_up(H, 8);
  if (64 + 2 * p.Kp > 512) return p;
  for (int C = 8; C >= 1; C >>= 1) {
    const int Hs = (int)round_up(cdiv(H, C), 4);
    if (Hs > 32) break;
    if (Hs * (C - 1) < H) { p.C = C; p.Hs = Hs; p.ok = true; break; }
  }
  if (!p.ok) return p;
  constexpr int TC_BT = 16;   // sized for the larger tile; the 8-row tile needs half
  size_t f = (size_t)4 * p.Kp * TC_BT + (size_t)TC_BT * GSM_LD + (size_t)4 * 4 * TC_BT * p.Hs;
  p.smem = std::max<size_t>(f * sizeof(float), 120 * 1024);   // > half an SM: one CTA (one TMEM allocation) per SM
  // backward: MT tiles of 128 hidden rows, Kb = 4*Hs own gate columns, hi+lo: 32*MT + 2*MT*Kb TMEM columns
  p.MT = cdiv(H, 128);
  p.bwd_ok = (32 * p.MT + 2 * p.MT * 4 * p.Hs) <= 512;
  p.smem_bwd = 0;   // depends on the tile height: tc_bwd_smem()
  return p;
}

// Rows per cluster tile.  8-row tiles halve the per-step exchange and gate math but need twice the clusters: use
// them when all the clusters of the batch are co-resident (B = 128 -> 16 clusters x 8 CTAs = 128 of the 148 SMs).
// SBR_TC_BT=8|16 forces a choice (tests run both).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// row-major fp32 matrix [rows x cols] -> 2-D tiled map with a [box_rows x box_cols] box, no swizzle, OOB reads = 0
bool make_map2d(CUtensorMap* tm, const float* base, uint64_t rows, uint64_t cols, uint32_t box_cols, uint32_t box_rows) {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  if (!fn || !base) return false;
  // the maps only depend on the allocation and the box: encode once (cuTensorMapEncodeTiled costs ~10 us of host time)
  // (device pointers are unique across the devices of a process under UVA, so the base address identifies the device)
  struct Key { const float* base; uint64_t rows, cols; uint32_t bc, br; CUtensorMap tm; };
  static std::vector<Key> cache;
  for (const Key& k : cache)
    if (k.base == base && k.rows == rows && k.cols == cols && k.bc == box_cols && k.br == box_rows) { *tm = k.tm; return true; }
  const cuuint64_t gdim[2] = {cols, rows};
  const cuuint64_t gstride[1] = {cols * sizeof(float)};
  const cuuint32_t box[2] = {box_cols, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  if (fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  if (cache.size() > 256) cache.clear();   // allocations of destroyed handles
  cache.push_back(Key{base, rows, cols, box_cols, box_rows, *tm});
  return true;
}

// backward: B operand (da hi|lo), partial-dh receive + send buffers, 4-deep staging ring of the saved tensors;
// at least 120 KB so that a second scan CTA (one TMEM allocation each) never lands on the same SM, and small enough
// that a side-stream GEMM CTA still fits next to it
size_t tc_bwd_smem(const TcPlan& p, int BT) {
  const size_t f = (size_t)2 * 4 * p.Hs * BT + (size_t)4 * p.C * BT * p.Hs + (size_t)4 * 7 * BT * p.Hs;
  return std::max<size_t>(f * sizeof(float), 120 * 1024);
}

template <typename Kern>
int max_active_clusters(Kern kern, const TcPlan& p, size_t smem) {
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(p.C * 64, 1, 1);
  cfg.blockDim = dim3(FWD_NT, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
int resident_clusters(const TcPlan& p) {
  // co-resident clusters depend on the device, the cluster size and the shared-memory request: one entry per triple
  struct Entry { int dev, C; size_t smem; int n; };
  static std::vector<Entry> cache;
  int dev = 0;
  cudaGetDevice(&dev);
  for (const Entry& e : cache)
    if (e.dev == dev && e.C == p.C && e.smem == p.smem) return e.n;
  const int n = max_active_clusters(rnn_fwd_tc_kernel<4, 8>, p, p.smem);
  cache.push_back(Entry{dev, p.C, p.smem, n});
  if (getenv("SBR_TC_VERBOSE")) fprintf(stderr, "[tc] device %d: clusters of %d CTAs co-resident: %d\n", dev, p.C, n);
  return n;
}
// Tile schedule of one scan launch.  The hardware hands clusters to free SM groups in blockIdx order, i.e. list
// scheduling on `slots` machines (15 eight-CTA clusters fit on a B200: seven GPCs take two, one takes one).  With
// the host copy of the lengths the launcher (a) sorts the tiles longest first, so that when there are more tiles
// than slots the short ones queue behind clusters that finish early, and (b) takes 8-row tiles only when their
// makespan (x the measured per-step cost ratio of an 8-row vs a 16-row tile) beats the 16-row tiling.
// extra16 >= 0: MIXED tiling -- the 16-row group `extra16` (rows 16g .. 16g+15, the shortest one) runs as one 16-row
// tile on a second stream while the remaining rows run as 8-row tiles: B = 128 is then 14 + 1 = 15 clusters, all
// co-resident, instead of 16 eight-row tiles of which one has to queue.
struct TileSched { int BT; int n_tiles; int use_order; unsigned char order[64]; int extra16; };
int makespan(const int* t_end, int n, int slots) {   // t_end sorted descending
  std::vector<int> busy(std::max(1, slots), 0);
  for (int i = 0; i < n; ++i) {
    auto it = std::min_element(busy.begin(), busy.end());
    *it += t_end[i];
  }
  return *std::max_element(busy.begin(), busy.end());
}
// pure host planner (no CUDA calls): exported for the CPU tests as sbr_plan_scan_tiles
TileSched plan_tiles(const int32_t* hl, int B, int t_max, int slots, float ratio8) {
  TileSched sc{};
  sc.extra16 = -1;
  auto tiles_of = [&](int BT, int* t_end, unsigned char* order) {
    const int n = cdiv(B, BT);
    std::vector<std::pair<int, int>> v(n);
    for (int i = 0; i < n; ++i) {
      int mx = 0;
      for (int b = i * BT; b < std::min(B, (i + 1) * BT); ++b) mx = std::max(mx, std::min(hl[b], t_max));
      v[i] = {-mx, i};
    }
    std::sort(v.begin(), v.end());
    for (int i = 0; i < n; ++i) { t_end[i] = -v[i].first; order[i] = (unsigned char)v[i].second; }
    return n;
  };
  int forced = 0;
  if (const char* e = getenv("SBR_TC_BT")) { const int v = atoi(e); if (v == 8 || v == 16) forced = v; }
  if (!hl || cdiv(B, 8) > 64) {           // no host lengths (or too many tiles to reorder): static rule
    sc.BT = forced ? forced : ((B % 8 == 0 && B / 8 <= slots) ? 8 : 16);
    sc.n_tiles = cdiv(B, sc.BT);
    return sc;
  }
  int t8[64], t16[64];
  unsigned char o8[64], o16[64];
  const int n8 = tiles_of(8, t8, o8), n16 = tiles_of(16, t16, o16);
  int BT = forced;
  if (!BT) {
    const float c8 = ratio8 * (float)makespan(t8, n8, slots), c16 = (float)makespan(t16, n16, slots);
    BT = (B % 8 == 0 && c8 < c16) ? 8 : 16;
    // one tile too many for the co-resident slots: fold the two shortest adjacent 8-row tiles into one 16-row tile
    const bool force_mixed = getenv("SBR_TC_FORCE_MIXED") != nullptr;     // tests
    if (B % 16 == 0 && ((n8 == slots + 1 && !getenv("SBR_TC_NO_MIXED")) || (force_mixed && n8 >= 4))) {
      const int g = o16[n16 - 1];                       // shortest 16-row group (t16 / o16 are sorted descending)
      int rest = 0;
      for (int i = 0; i < n8; ++i) if ((o8[i] >> 1) != g) rest = std::max(rest, t8[i]);
      const float cmix = std::max(ratio8 * (float)rest, (float)t16[n16 - 1]);
      if (cmix < std::min(c8, c16) || force_mixed) {
        sc.BT = 8;
        sc.use_order = 1;
        sc.extra16 = g;
        int n = 0;
        for (int i = 0; i < n8; ++i) if ((o8[i] >> 1) != g) sc.order[n++] = o8[i];
        sc.n_tiles = n;
        return sc;
      }
    }
  }
  sc.BT = BT;
  sc.n_tiles = BT == 8 ? n8 : n16;
  sc.use_order = 1;
  memcpy(sc.order, BT == 8 ? o8 : o16, 64);
  return sc;
}
TileSched schedule_tiles(const sbr_model* m, const TcPlan& p, int B, int t_max, float ratio8) {
  return plan_tiles(m->cur_hlen, B, t_max, resident_clusters(p), ratio8);
}
constexpr float TC_RATIO8_FWD = 0.71f;   // fwd: 2914 vs 4114 cycles per step (8 vs 16 rows)
constexpr float TC_RATIO8_BWD = 0.75f;   // bwd: 4118 vs 5477 cycles per step (8 vs 16 rows)

template <typename Kern>
int launch_tc(sbr_model* m, Kern kern, const TcPlan& p, int n_tiles, const TcArgs& args, int threads, cudaStream_t stream) {
  cudaError_t e = cudaSuccess;
  // raise the opt-in shared-memory limit once per kernel, not on every launch (Kern is the same function-pointer
  // TYPE for every instantiation, so the cache is keyed by the pointer value)
  // (the attribute is per device: the cache is keyed by (device, kernel pointer))
  struct SmemKey { int dev; const void* kern; size_t bytes; };
  static std::vector<SmemKey> smem_set;
  size_t* have = nullptr;
  for (auto& kv : smem_set) if (kv.dev == m->dev && kv.kern == (const void*)kern) have = &kv.bytes;
  if (!have) { smem_set.push_back(SmemKey{m->dev, (const void*)kern, 0}); have = &smem_set.back().bytes; }
  if (p.smem > *have) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
    if (e != cudaSuccess) { sbr_set_error(m, SBR_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return SBR_E_CUDA; }
    *have = p.smem;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(p.C * n_tiles, 1, 1);
  cfg.blockDim = dim3(threads, 1, 1);
  cfg.dynamicSmemBytes = p.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, kern, args);
  if (e != cudaSuccess) { sbr_set_error(m, SBR_E_CUDA, "tcgen05 scan launch (C=%d) failed: %s", p.C, cudaGetErrorString(e)); return SBR_E_CUDA; }
  m->launches++;
  m->scan_launches++;
  return 0;
}

}  // namespace

// returns 1 when the tensor-core path does not apply (caller falls back), 0 on success, <0 on error
int launch_rnn_forward_tc(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last) {
  const TcPlan p = tc_plan(L.G, L.H);
  if (!p.ok) return 1;
  int rc = launch_transpose(m, m->params + L.W_hid, L.H, L.G * L.H, L.G * L.H, m->WhidT);
  if (rc) return rc;
  TcArgs a{};
  a.Xg = L.Xg; a.W_hid = m->params + L.W_hid; a.W_hidT = m->WhidT;
  a.peep = m->params + L.peep; a.h_init = m->params + L.h_init; a.c_init = m->params + L.c_init;
  a.len = len; a.hs = L.hs; a.cs = L.cs; a.act = L.act; a.h_last = h_last;
  a.clip = m->cfg.grad_clip; a.relu = L.relu; a.B = B; a.H = L.H; a.Hs = p.Hs; a.Kp = p.Kp; a.t_max = t_max;
  if (const char* e = getenv("SBR_TC_EXPERIMENT")) a.xflags = atoi(e);
  const TileSched sc = schedule_tiles(m, p, B, t_max, TC_RATIO8_FWD);
  const int BT = sc.BT;
  static long long* dbg = nullptr;
  if (getenv("SBR_TC_TIMELINE")) {
    if (!dbg) { cudaMalloc(&dbg, 80 * 8 * sizeof(long long)); cudaMemset(dbg, 0, 80 * 8 * sizeof(long long)); }
    a.dbg = dbg;
  }
  // one launch = one tile height: tensor map with the matching box, tile order, stream
  auto launch_one = [&](int bt, int n_tiles, const unsigned char* order, int use_order, cudaStream_t stream) -> int {
    TcArgs v = a;
    v.use_order = use_order;
    if (order) memcpy(v.order, order, sizeof(v.order));
    if (L.hT && B % bt == 0) { v.hT = L.hT; v.hT_part = L.hT_part; v.hT_tile = L.hT_tile; }
    if (!make_map2d(&v.tm_xg, L.Xg, (uint64_t)m->T * m->B, (uint64_t)L.G * L.H, p.Hs, bt)) {
      sbr_set_error(m, SBR_E_CUDA, "cuTensorMapEncodeTiled failed (Xg, H=%d Hs=%d BT=%d)", L.H, p.Hs, bt);
      return SBR_E_CUDA;
    }
#define SBR_FWD_CASE(G_, BT_) if (L.G == G_ && bt == BT_) return launch_tc(m, rnn_fwd_tc_kernel<G_, BT_>, p, n_tiles, v, FWD_NT, stream);
    SBR_FWD_CASE(4, 16) SBR_FWD_CASE(4, 8) SBR_FWD_CASE(3, 16) SBR_FWD_CASE(3, 8) SBR_FWD_CASE(1, 16) SBR_FWD_CASE(1, 8)
#undef SBR_FWD_CASE
    return 1;
  };
  if (sc.extra16 >= 0) {
    // mixed tiling: the shortest 16-row group as ONE 16-row tile on the aux stream, concurrent with the 8-row tiles
    unsigned char one[64] = {(unsigned char)sc.extra16};
    CU_TRY(m, cudaEventRecord(m->ev_aux_fork, m->stream));
    CU_TRY(m, cudaStreamWaitEvent(m->aux, m->ev_aux_fork, 0));
    if ((rc = launch_one(16, 1, one, 1, m->aux))) return rc;
    CU_TRY(m, cudaEventRecord(m->ev_aux_join, m->aux));
  }
  rc = launch_one(BT, sc.n_tiles, sc.order, sc.use_order, m->stream);
  if (sc.extra16 >= 0 && rc == 0) CU_TRY(m, cudaStreamWaitEvent(m->stream, m->ev_aux_join, 0));
  if (rc == 0 && a.dbg && L.G == 4) {
    static int calls = 0;
    if (++calls == 8) {
      long long h[80 * 8];
      cudaStreamSynchronize(m->stream);
      cudaMemcpy(h, dbg, sizeof(h), cudaMemcpyDeviceToHost);
      double acc[12] = {0};
      int n = (int)(h[517] > 0 ? h[517] : 1);
      for (int i = 1; i < 12; ++i) acc[i] = (double)h[i];
      fprintf(stderr, "[tc fwd BT=%d tail] proxy_fence %.0f barrier %.0f bulk_issue %.0f stores+loop %.0f\n", BT, acc[8] / n, acc[9] / n, acc[10] / n, acc[7] / n);
      fprintf(stderr, "[tc fwd kernel, cycles] t_end %lld | entry->A_init_done %lld | ->loop_start %lld | loop %lld (%.0f/step) | ->exit %lld\n", h[517],
              h[513] - h[512], h[514] - h[513], h[515] - h[514], (double)(h[515] - h[514]) / (double)(h[517] > 0 ? h[517] : 1), h[516] - h[515]);
      fprintf(stderr, "[tc fwd timeline, cycles/step] wait_peers %.0f arm %.0f mma_issue %.0f mma_wait %.0f ldtm+bar %.0f gate %.0f\n",
              acc[1] / n, acc[2] / n, acc[3] / n, acc[4] / n, acc[5] / n, acc[6] / n);
    }
  }
  return rc;
}

int launch_rnn_backward_tc(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, const float* dh_last) {
  TcPlan p = tc_plan(L.G, L.H);
  if (!p.ok || !p.bwd_ok) return 1;
  TcArgs a{};
  a.W_hid = m->params + L.W_hid; a.peep = m->params + L.peep; a.len = len; a.hs = L.hs; a.cs = L.cs; a.act = L.act;
  a.dh_last = dh_last; a.dhs = dh_last ? nullptr : L.dhs; a.dXg = L.dXg; a.dac = L.dac;
  a.g_peep = m->grads + L.peep; a.g_h_init = m->grads + L.h_init; a.g_c_init = m->grads + L.c_init;
  a.clip = m->cfg.grad_clip; a.relu = L.relu; a.B = B; a.H = L.H; a.Hs = p.Hs; a.Kp = p.Kp; a.t_max = t_max;
  const TileSched sc = schedule_tiles(m, p, B, t_max, TC_RATIO8_BWD);
  const int BT = sc.BT;
  a.g_b = m->grads + L.b;
  a.ld_p = 3;
  if (const char* e = getenv("SBR_TC_LDP")) a.ld_p = std::max(1, std::min(3, atoi(e)));
  if (const char* e = getenv("SBR_TC_EXPERIMENT")) a.xflags = atoi(e);
  if (getenv("SBR_TC_TIMELINE")) {
    static long long* bdbg = nullptr;
    static int calls = 0;
    if (!bdbg) { cudaMalloc(&bdbg, 80 * 8 * sizeof(long long)); cudaMemset(bdbg, 0, 80 * 8 * sizeof(long long)); }
    a.dbg = bdbg;
    if (++calls == 9) {
      long long h[80];
      cudaStreamSynchronize(m->stream);
      cudaMemcpy(h, bdbg + 64, 16 * sizeof(long long), cudaMemcpyDeviceToHost);
      const double n = (double)(h[13] > 0 ? h[13] : 1);
      fprintf(stderr, "[tc bwd BT=%d, cycles/step] total %.0f (t_end %lld) | issue_prefetch %.0f wait_parts+arm %.0f gate_grad %.0f fence %.0f barrier %.0f "
              "dump+stores %.0f mma_wait %.0f ldtm+sbuf %.0f fence %.0f barrier %.0f bulk+copy %.0f\n", BT, h[12] / n, h[13],
              0.0, h[1] / n, h[2] / n, h[3] / n, h[4] / n, h[5] / n, h[6] / n, h[7] / n, h[8] / n, h[9] / n, h[10] / n);
    }
  }
  auto launch_one = [&](int bt, int n_tiles, const unsigned char* order, int use_order, cudaStream_t stream) -> int {
    TcArgs v = a;
    TcPlan q = p;
    q.smem = tc_bwd_smem(p, bt);
    v.use_order = use_order;
    if (order) memcpy(v.order, order, sizeof(v.order));
    if (L.aT && B % bt == 0) { v.aT = L.aT; v.aT_part = L.aT_part; v.aT_tile = L.aT_tile; }
    // tensor maps over the whole allocations ([T*Bmax (+Bmax)] rows): box = [bt x Hs]
    const uint64_t TB = (uint64_t)m->T * m->B;
    bool ok = true;
    if (L.G > 1) ok = ok && make_map2d(&v.tm_act, L.act, TB, 4 * (uint64_t)L.H, p.Hs, bt);
    if (L.G == 4) ok = ok && make_map2d(&v.tm_cs, L.cs, TB + m->B, L.H, p.Hs, bt);
    ok = ok && make_map2d(&v.tm_hs, L.hs, TB + m->B, L.H, p.Hs, bt);
    if (v.dhs) ok = ok && make_map2d(&v.tm_dhs, L.dhs, TB, L.H, p.Hs, bt);
    if (!ok) { sbr_set_error(m, SBR_E_CUDA, "cuTensorMapEncodeTiled failed (H=%d Hs=%d BT=%d)", L.H, p.Hs, bt); return SBR_E_CUDA; }
#define SBR_BWD_CASE(G_, MT_) \
    if (L.G == G_ && p.MT == MT_ && bt == 16) return launch_tc(m, rnn_bwd_tc_kernel<G_, MT_, 16>, q, n_tiles, v, bwd_threads(16), stream); \
    if (L.G == G_ && p.MT == MT_ && bt == 8) return launch_tc(m, rnn_bwd_tc_kernel<G_, MT_, 8>, q, n_tiles, v, bwd_threads(8), stream);
    SBR_BWD_CASE(4, 1) SBR_BWD_CASE(4, 2) SBR_BWD_CASE(3, 1) SBR_BWD_CASE(3, 2) SBR_BWD_CASE(1, 1) SBR_BWD_CASE(1, 2)
#undef SBR_BWD_CASE
    return 1;
  };
  int rc = 0;
  if (sc.extra16 >= 0) {
    unsigned char one[64] = {(unsigned char)sc.extra16};
    CU_TRY(m, cudaEventRecord(m->ev_aux_fork, m->stream));
    CU_TRY(m, cudaStreamWaitEvent(m->aux, m->ev_aux_fork, 0));
    if ((rc = launch_one(16, 1, one, 1, m->aux))) return rc;
    CU_TRY(m, cudaEventRecord(m->ev_aux_join, m->aux));
  }
  rc = launch_one(BT, sc.n_tiles, sc.order, sc.use_order, m->stream);
  if (sc.extra16 >= 0 && rc == 0) CU_TRY(m, cudaStreamWaitEvent(m->stream, m->ev_aux_join, 0));
  return rc;
}

// Host-only view of the scan launch plan for a batch with the given lengths on `slots` co-resident cluster slots
// (diagnostics / CPU tests; touches no device).  tile_rows = 8 or 16 for the main launch; order[0..n_tiles) = its
// tiles in launch order (units of tile_rows rows); extra16 = the 16-row group of the second launch, or -1.
extern "C" SBR_API int sbr_plan_scan_tiles(const int32_t* lens, int B, int t_max, int slots, float ratio8,
                                           int* tile_rows, int* n_tiles, int* extra16, unsigned char* order64) {
  if (B < 1 || slots < 1 || !tile_rows || !n_tiles || !extra16 || !order64) return SBR_E_ARG;
  const TileSched sc = plan_tiles(lens, B, t_max, slots, ratio8);
  *tile_rows = sc.BT; *n_tiles = sc.n_tiles; *extra16 = sc.extra16;
  if (sc.use_order) memcpy(order64, sc.order, 64);
  else for (int i = 0; i < 64; ++i) order64[i] = (unsigned char)i;
  return 0;
}

int tc_scan_applies(int G, int H) {
  const TcPlan p = tc_plan(G, H);
  return (p.ok && p.bwd_ok) ? 1 : 0;
}

TcShape tc_scan_shape(int G, int H) {
  const TcPlan p = tc_plan(G, H);
  return TcShape{p.ok, p.ok && p.bwd_ok, p.C, p.Hs, p.MT};
}
int tc_scan_slots(int G, int H) {
  const TcPlan p = tc_plan(G, H);
  return p.ok ? resident_clusters(p) : 0;
}
// tile height of the main launch and number of launches (the mixed tiling adds the 16-row launch on the aux stream)
void tc_scan_schedule(const int32_t* hl, int B, int t_max, int slots, bool backward, int* tile_rows, int* n_launches) {
  const TileSched sc = plan_tiles(hl, B, t_max, slots, backward ? TC_RATIO8_BWD : TC_RATIO8_FWD);
  *tile_rows = sc.BT;
  *n_launches = 1 + (sc.extra16 >= 0 ? 1 : 0);
}
