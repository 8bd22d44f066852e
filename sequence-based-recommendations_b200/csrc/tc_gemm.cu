// tc_gemm.cu -- the fp32-accurate tensor-core GEMM of the path (tcgen05, 3xTF32) and the recurrent steps built on it.
//
// One kernel, templated on its epilogue, computes D[128 x BN] = A[128 x K] * B[BN x K]^T per CTA with fp32 operands
// read straight from their row-major homes (no pre-split or pre-transposed copies in HBM):
//
//   * A operand: warps 0-3, thread = tile row.  A thread reads its row's 32 k-values of a stage from global memory
//     (16-byte loads when k is the contiguous index, coalesced 4-byte loads when the row index is), splits them
//     hi = tf32(x), lo = x - hi in registers and writes them into the stage's TMEM slot with tcgen05.st
//     (hi | lo, 64 columns per stage): the MMA reads A from TMEM (TS form), so A never touches shared memory;
//   * B operand: warps 4-7 read the [BN x 32] slice, split it the same way and store it as the canonical no-swizzle
//     K-major core-matrix tile ([k/4][BN][4] floats, hi then lo) in a 3-stage shared-memory ring;
//     both loaders keep 3 chunks in flight through thread-private cp.async cells (no registers held across the
//     global-memory latency, no barrier: a thread only ever reads back what it copied itself);
//   * warp 8 (one elected lane) issues per 8-wide k-step  D1 += A_hi B_hi,  D2 += A_hi B_lo,  D2 += A_lo B_hi
//     (two fp32 TMEM accumulators: the tensor core's accumulate truncates, the 2^-11-smaller correction terms stay
//     apart and are added by the epilogue) and releases the stage with tcgen05.commit;
//   * warps 0-3 drain TMEM (thread = tile row) into the epilogue.
//
// Epilogues:
//   EPI_STORE      C = alpha * D (+ bias[n]) (+ C), split-K through fp32 reductions: every GEMM-shaped stage that is
//                  not a recurrent step -- layer>=1 / embedding input GEMMs and their two gradients
//                  (recurrent_layers.py:47-50,94-104), the output projection and its gradients (rnn_one_hot.py:65,
//                  rnn_margin.py:103, sparse_lstm.py:41-54), the BPTT weight gradients.
//   EPI_*_FWD      one time step of the recurrent scan for hidden sizes the cluster-resident kernels of rnn_tc.cu do
//                  not hold (H > 224): rows = batch rows, columns = the G gates of 8 hidden units; fused LSTM / GRU /
//                  vanilla cell (sparse_lstm.py:377-425, :764-805, :1120-1152) incl. peepholes and the length mask.
//   EPI_*_BWD      one BPTT step: rows = hidden units k, columns = batch rows, D = da_{t+1} W_hid^T; fused gate
//                  gradients with grad_clip at the reference's sites (sparse_lstm.py:386-388,768-772,789-791).
//   EPI_INIT_GRAD  the step "t = -1": gradients of the learned initial states and the peepholes.
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"

using namespace tcx;

namespace {

constexpr int TG_KC = 32;        // k per pipeline stage = 4 MMA k-steps
#ifndef SBR_TG_STAGES
#define SBR_TG_STAGES 3
#endif
constexpr int TG_STAGES = SBR_TG_STAGES;      // converted-operand ring: TMEM slots of A (64 columns each) + shared-memory tiles of B
constexpr int TG_LOOK_MAX = 8;    // raw fp32 ring: up to this many 32-wide k chunks in flight (args.look, sized by the shared-memory budget)
constexpr int TG_NT = 544;       // warps 0-3: A converters + epilogue, 4-7: B converters, 8: MMA issuer, 9-12: A loaders, 13-16: B loaders
constexpr int TG_A0 = 256;       // first TMEM column of the A ring (D1 | D2 occupy 2*BN <= 256 columns)
constexpr int STEP_U = 8;        // hidden units per CTA of a forward step (BN = 32 = 4 gates x 8 units)
constexpr int STEP_BN = 32;

enum { EPI_STORE = 0, EPI_LSTM_FWD, EPI_GRU_FWD, EPI_VAN_FWD, EPI_LSTM_BWD, EPI_GRU_BWD, EPI_VAN_BWD, EPI_INIT_GRAD };

struct StepArgs {
  int t, B, H, G;
  const int32_t* len;
  const float* peep;                 // LSTM [3,H]
  // forward (pointers already offset to step t)
  const float* Xg_t; const float* hs_t; const float* cs_t;
  float* hs_n; float* cs_n; float* act_t;
  // backward
  const float* act_r; const float* cs_r; const float* cs_rn; const float* hs_r; const float* dhs_t;
  float* dXg_t; float* dac_t;
  float* carry; float* dcs; float* dpe;     // [B,H] scratch (dpe: [3][B,H])
  float* g_h_init; float* g_c_init; float* g_peep;
  float clip;
  int relu;            // vanilla cell: rectifier instead of tanh (dense-input layers)
};

struct TgArgs {
  const float* A; long long lda; int a_mode;      // 0: A[m*lda + k]   1: A[k*lda + m]
  const float* B; long long ldb; int b_mode;      // 0: B[n*ldb + k]   1: B[k*ldb + n]   2: gate columns of B[k*ldb + .]
  const float* B2; long long ldb2; int b_split;   // b_mode 0: k >= b_split comes from B2[n*ldb2 + k - b_split]
  int M, N, K, BN, k_per_split;
  int a_vec, b_vec;
  float* C; long long ldc; float alpha; int accumulate; const float* bias; int c_vec;
  long long* dbg;                                 // optional clock64 timeline of CTA (0,0,0) (SBR_TG_TIMELINE)
  // raw-ring loaders: TMA tiled loads where the operand allows a tensor map (16-byte aligned base, ld % 4 == 0)
  CUtensorMap tmA, tmB, tmB2;
  int tma_a, tma_b;
  int a_off, b_off, b2_off;                       // row offsets of the tile origin inside the mapped arrays (recurrent steps)
  int look;                                       // raw ring depth
  StepArgs st;
};

template <int EPI>
__global__ void __launch_bounds__(TG_NT, 1) tc_gemm_kernel(const __grid_constant__ TgArgs a) {
  extern __shared__ __align__(1024) uint8_t tg_smem[];   // B ring: [stage][hi | lo][KC/4][BN][4] floats
  __shared__ __align__(8) uint64_t full[TG_STAGES];
  __shared__ __align__(8) uint64_t empty[TG_STAGES];
  __shared__ __align__(8) uint64_t done;
  __shared__ __align__(8) uint64_t rawA_full[TG_LOOK_MAX], rawA_empty[TG_LOOK_MAX], rawB_full[TG_LOOK_MAX], rawB_empty[TG_LOOK_MAX];
  __shared__ uint32_t tmem_base_s;

  uint8_t* const tg_base = tg_smem + ((1024u - (smem_u32(tg_smem) & 1023u)) & 1023u);   // TMA swizzle atoms are 1 KB
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int BN = a.BN;
  const int m0 = blockIdx.y * 128, n0 = blockIdx.x * BN;
  const int k_begin = blockIdx.z * a.k_per_split;
  int k_end = min(a.K, k_begin + a.k_per_split);
  constexpr bool FWD = EPI == EPI_LSTM_FWD || EPI == EPI_GRU_FWD || EPI == EPI_VAN_FWD;
  constexpr bool BWD = EPI == EPI_LSTM_BWD || EPI == EPI_GRU_BWD || EPI == EPI_VAN_BWD;

  // ---- recurrent steps: CTA-uniform decisions from the lengths, before anything is allocated
  if constexpr (FWD) {
    // rows = batch rows: nothing to do when no row of the tile is still inside its sequence
    const int b = m0 + tid;
    const int act = (tid < 128 && b < a.st.B && a.st.t < a.st.len[b]) ? 1 : 0;
    if (!__syncthreads_or(act)) return;
  }
  if constexpr (BWD) {
    // columns = batch rows n0 .. n0+BN-1.  No row active at step t: dXg of the tile is exactly zero, nothing else
    // changes (the carried gradient passes through).  No row active at t+1: da_{t+1} = 0, the product is skipped.
    const int b = n0 + tid;
    const bool in = tid < BN && b < a.st.B;
    const int l = in ? a.st.len[b] : 0;
    const int any_t = __syncthreads_or(in && a.st.t < l);
    const int any_t1 = __syncthreads_or(in && a.st.t + 1 < l);
    if (!any_t) {
      const int GH = a.st.G * a.st.H;
      for (int i = tid; i < BN * 128; i += TG_NT) {
        const int bb = n0 + i / 128, k = m0 + (i & 127);
        if (bb < a.st.B && k < a.st.H) {
          for (int g = 0; g < a.st.G; ++g) a.st.dXg_t[(long long)bb * GH + g * a.st.H + k] = 0.f;
          if (EPI == EPI_GRU_BWD) a.st.dac_t[(long long)bb * a.st.H + k] = 0.f;
        }
      }
      return;
    }
    if (!any_t1) k_end = k_begin;
  }
  const int n_chunks = k_end > k_begin ? (k_end - k_begin + TG_KC - 1) / TG_KC : 0;
  const bool tl = a.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
  const long long t_start = tl ? clock64() : 0;
#define TG_T0() long long t0_ = tl ? clock64() : 0
#define TG_ACC(var) do { if (tl) { const long long n_ = clock64(); var += n_ - t0_; t0_ = n_; } } while (0)

  if (tid == 0) {
    for (int s = 0; s < TG_STAGES; ++s) { mbar_init(&full[s], 8); mbar_init(&empty[s], 1); }
    mbar_init(&done, 1);
    for (int i = 0; i < TG_LOOK_MAX; ++i) {
      // TMA: one arrive.expect_tx by the producer + the bytes; cp.async: one completion arrive per loader thread
      mbar_init(&rawA_full[i], a.tma_a ? 1 : 128); mbar_init(&rawB_full[i], a.tma_b ? 1 : 128);
      mbar_init(&rawA_empty[i], 4); mbar_init(&rawB_empty[i], 4);        // one arrive per converter warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t tD1 = tmem, tD2 = tmem + BN, tA = tmem + TG_A0;
  const uint32_t stage_bytes = (uint32_t)BN * TG_KC * 8u;       // hi + lo
  const uint32_t part_bytes = (uint32_t)BN * TG_KC * 4u;

  // Warp roles.  The threads that wait on global memory (loaders) are NOT the ones that publish operands to the
  // tensor core: fence.proxy.async / tcgen05.wait::st drain the executing thread's outstanding global accesses, so a
  // thread that both prefetches and publishes pays the full memory latency per stage.  Loaders fill a raw fp32 ring
  // (TMA tiled loads issued by one thread when the operand's base / leading dimension allow a tensor map, else
  // cp.async from 128 threads) and signal an mbarrier; converters only touch shared memory / TMEM.
  //
  // Raw tile layouts (the same whichever loader filled them):
  //   A mode 0  [128 rows][32 k], 128-byte rows with the TMA 128B swizzle: 16-byte chunk q of row r sits at q ^ (r & 7)
  //   A mode 1  [32 k][128 rows]
  //   B mode 0  [BN rows][32 k], swizzled like A mode 0;  B mode 1  [32 k][BN];  B mode 2  [gate][32 k][8 units]
  const int LOOK = a.look;
  const uint32_t rawA_bytes = 128u * TG_KC * 4u, rawB_bytes = (uint32_t)BN * TG_KC * 4u;
  uint8_t* rawA0 = tg_base + (size_t)TG_STAGES * stage_bytes;
  uint8_t* rawB0 = rawA0 + (size_t)LOOK * rawA_bytes;
  const int bn_shift = 31 - __clz(BN);
  auto b_coords = [&](int idx, int& n, int& kq) {
    if (a.b_mode == 0) { n = ((idx >> 6) << 3) + (idx & 7); kq = (idx >> 3) & 7; }
    else { kq = idx >> bn_shift; n = idx & (BN - 1); }       // BN is a power of two (an integer division here cost more than the conversion)
  };

  if (warp < 4) {
    // =================================================================================== A converter (thread = row)
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    long long w_raw = 0, w_empty = 0, w_work = 0;
    TG_T0();
    for (int c = 0; c < n_chunks; ++c) {
      const int rs = c % LOOK;
      mbar_wait(&rawA_full[rs], (c / LOOK) & 1);
      TG_ACC(w_raw);
      float cur[TG_KC];
      const float* src = reinterpret_cast<const float*>(rawA0 + (size_t)rs * rawA_bytes);
      if (a.a_mode == 0) {
#pragma unroll
        for (int q = 0; q < TG_KC / 4; ++q) {
          const float4 x = *reinterpret_cast<const float4*>(src + tid * 32 + ((q ^ (tid & 7)) << 2));
          cur[4 * q] = x.x; cur[4 * q + 1] = x.y; cur[4 * q + 2] = x.z; cur[4 * q + 3] = x.w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < TG_KC; ++i) cur[i] = src[i * 128 + tid];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&rawA_empty[rs]);       // the raw cells are in registers
      const int s = c % TG_STAGES;
      if (c >= TG_STAGES) {
        mbar_wait(&empty[s], ((c / TG_STAGES) - 1) & 1);
        tc_fence_after();
      }
      TG_ACC(w_empty);
      const uint32_t dst = tA + (uint32_t)s * 64u + lane_off;
#pragma unroll
      for (int q = 0; q < TG_KC / 8; ++q) {
        uint32_t hi[8], lo[8];
        split8(cur + 8 * q, hi, lo);
        tmem_st8(dst + 8 * q, hi);
        tmem_st8(dst + TG_KC + 8 * q, lo);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
      TG_ACC(w_work);
    }
    if (tl && tid == 0) { a.dbg[0] = w_raw; a.dbg[1] = w_empty; a.dbg[2] = w_work; a.dbg[3] = clock64() - t_start; }
  } else if (warp < 8) {
    // =================================================================================== B converter
    const int bt = tid - 128;
    const int per = BN / 16;                       // 16-byte chunks (n, 4 k) per thread per stage
    long long w_raw = 0, w_empty = 0, w_work = 0;
    TG_T0();
    for (int c = 0; c < n_chunks; ++c) {
      const int rs = c % LOOK;
      mbar_wait(&rawB_full[rs], (c / LOOK) & 1);
      TG_ACC(w_raw);
      const float* src = reinterpret_cast<const float*>(rawB0 + (size_t)rs * rawB_bytes);
      float4 cur[8];
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        if (it >= per) break;
        int n, kq;
        b_coords(it * 128 + bt, n, kq);
        if (a.b_mode == 0) {
          cur[it] = *reinterpret_cast<const float4*>(src + n * 32 + ((kq ^ (n & 7)) << 2));
        } else if (a.b_mode == 1) {
          const float* q = src + (4 * kq) * BN + n;
          cur[it] = make_float4(q[0], q[BN], q[2 * BN], q[3 * BN]);
        } else {
          const int g = n / STEP_U, j = n - g * STEP_U;
          const float* q = src + g * (TG_KC * STEP_U) + (4 * kq) * STEP_U + j;
          cur[it] = g < a.st.G ? make_float4(q[0], q[STEP_U], q[2 * STEP_U], q[3 * STEP_U]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&rawB_empty[rs]);
      const int s = c % TG_STAGES;
      if (c >= TG_STAGES) mbar_wait(&empty[s], ((c / TG_STAGES) - 1) & 1);
      TG_ACC(w_empty);
      uint8_t* st = tg_base + (size_t)s * stage_bytes;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        if (it >= per) break;
        int n, kq;
        b_coords(it * 128 + bt, n, kq);
        const float4 x = cur[it];
        float4 h, l;
        h.x = tf32_hi(x.x); h.y = tf32_hi(x.y); h.z = tf32_hi(x.z); h.w = tf32_hi(x.w);
        l.x = x.x - h.x; l.y = x.y - h.y; l.z = x.z - h.z; l.w = x.w - h.w;
        const uint32_t off = (uint32_t)kq * (uint32_t)BN * 16u + (uint32_t)n * 16u;
        *reinterpret_cast<float4*>(st + off) = h;
        *reinterpret_cast<float4*>(st + part_bytes + off) = l;
      }
      proxy_fence_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
      TG_ACC(w_work);
    }
    if (tl && tid == 128) { a.dbg[8] = w_raw; a.dbg[9] = w_empty; a.dbg[10] = w_work; a.dbg[11] = clock64() - t_start; }
  } else if (warp == 8) {
    // =================================================================================== MMA issuer
    if (elect_one_sync()) {
      const uint32_t idesc = make_idesc_tf32(128, BN);
      const uint32_t lbo = (uint32_t)BN * 16u;
      uint32_t acc = 0;
      long long w_full = 0, w_issue = 0;
      TG_T0();
      for (int c = 0; c < n_chunks; ++c) {
        const int s = c % TG_STAGES;
        mbar_wait(&full[s], (c / TG_STAGES) & 1);
        tc_fence_after();
        TG_ACC(w_full);
        const uint32_t sb = smem_u32(tg_base + (size_t)s * stage_bytes);
        const uint32_t ta = tA + (uint32_t)s * 64u;
        uint64_t bhi = make_desc(sb, lbo, 128), blo = make_desc(sb + part_bytes, lbo, 128);
        const uint64_t adv = (uint64_t)((2u * lbo) >> 4);      // two core matrices along K, in the descriptor's 16-byte units
#pragma unroll
        for (int ks = 0; ks < TG_KC / 8; ++ks) {
          mma_ts(tD1, ta + 8 * ks, bhi, idesc, acc);
          mma_ts(tD2, ta + 8 * ks, blo, idesc, acc);
          mma_ts(tD2, ta + TG_KC + 8 * ks, bhi, idesc, 1);
          acc = 1;
          bhi += adv; blo += adv;
        }
        umma_commit(&empty[s]);        // the stage (TMEM slot + shared-memory slot) is free once these MMAs have read it
        TG_ACC(w_issue);
      }
      if (n_chunks > 0) umma_commit(&done);
      if (tl) { a.dbg[16] = w_full; a.dbg[17] = w_issue; a.dbg[18] = clock64() - t_start; a.dbg[19] = n_chunks; }
    }
    __syncwarp();
    } else if (warp < 13) {
    // =================================================================================== A loader
    const int r = tid - 9 * 32;
    long long w_wait = 0, w_work = 0;
    TG_T0();
    if (a.tma_a) {
      // ---- TMA producer: ONE thread issues the tiled loads of the A operand
      if (r == 0) {
        asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmA) : "memory");
        for (int c = 0; c < n_chunks; ++c) {
          const int rs = c % LOOK;
          if (c >= LOOK) mbar_wait(&rawA_empty[rs], ((c / LOOK) - 1) & 1);
          TG_ACC(w_wait);
          const int k0 = k_begin + c * TG_KC;
          mbar_arrive_expect_tx(&rawA_full[rs], rawA_bytes);
          if (a.a_mode == 0) tma_load_2d(rawA0 + (size_t)rs * rawA_bytes, &a.tmA, k0, a.a_off + m0, &rawA_full[rs]);
          else tma_load_2d(rawA0 + (size_t)rs * rawA_bytes, &a.tmA, a.a_off + m0, k0, &rawA_full[rs]);
          TG_ACC(w_work);
        }
      }
    }
    if (!a.tma_a) {
      // ---- cp.async fallback (unaligned base / leading dimension): thread r copies row r's cells
      const int row = m0 + r;
      const bool row_ok = row < a.M;
      const bool vec = a.a_mode == 0 && a.a_vec;
      for (int c = 0; c < n_chunks; ++c) {
        const int rs = c % LOOK;
        if (c >= LOOK) mbar_wait(&rawA_empty[rs], ((c / LOOK) - 1) & 1);
        TG_ACC(w_wait);
        const int k0 = k_begin + c * TG_KC;
        float* dst = reinterpret_cast<float*>(rawA0 + (size_t)rs * rawA_bytes);
        if (vec) {
          const float* src = a.A + (long long)(a.a_off + row) * a.lda + k0;
#pragma unroll
          for (int q = 0; q < TG_KC / 4; ++q) {
            const int left = row_ok ? (k_end - (k0 + 4 * q)) * 4 : 0;
            const int nb = left >= 16 ? 16 : (left > 0 ? left : 0);
            cp_async16(dst + r * 32 + ((q ^ (r & 7)) << 2), nb > 0 ? src + 4 * q : a.A, nb);
          }
        } else if (a.a_mode == 0) {
          const float* src = a.A + (long long)(a.a_off + row) * a.lda + k0;
#pragma unroll
          for (int i = 0; i < TG_KC; ++i) {
            const bool ok = row_ok && k0 + i < k_end;
            cp_async4(dst + r * 32 + (((i >> 2) ^ (r & 7)) << 2) + (i & 3), ok ? src + i : a.A, ok ? 4 : 0);
          }
        } else {
          const float* src = a.A + (long long)k0 * a.lda + a.a_off + row;
#pragma unroll
          for (int i = 0; i < TG_KC; ++i) {
            const bool ok = row_ok && k0 + i < k_end;
            cp_async4(dst + i * 128 + r, ok ? src + (long long)i * a.lda : a.A, ok ? 4 : 0);
          }
        }
        cp_async_arrive(&rawA_full[rs]);
        TG_ACC(w_work);
      }
    }
    if (tl && r == 0) { a.dbg[24] = w_wait; a.dbg[25] = w_work; a.dbg[26] = clock64() - t_start; }
  } else if (a.tma_b) {
    // =================================================================================== B loader: TMA producer (one thread)
    if (tid == 13 * 32) {
      long long w_wait = 0, w_work = 0;
      TG_T0();
      asm volatile("prefetch.tensormap [%0];" :: "l"(&a.tmB) : "memory");
      for (int c = 0; c < n_chunks; ++c) {
        const int rs = c % LOOK;
        if (c >= LOOK) mbar_wait(&rawB_empty[rs], ((c / LOOK) - 1) & 1);
        TG_ACC(w_wait);
        const int k0 = k_begin + c * TG_KC;
        uint8_t* dst = rawB0 + (size_t)rs * rawB_bytes;
        if (a.b_mode == 0) {
          mbar_arrive_expect_tx(&rawB_full[rs], rawB_bytes);
          if (a.B2 && k0 >= a.b_split) tma_load_2d(dst, &a.tmB2, k0 - a.b_split, a.b2_off + n0, &rawB_full[rs]);
          else tma_load_2d(dst, &a.tmB, k0, a.b_off + n0, &rawB_full[rs]);
        } else if (a.b_mode == 1) {
          mbar_arrive_expect_tx(&rawB_full[rs], rawB_bytes);
          tma_load_2d(dst, &a.tmB, a.b_off + n0, k0, &rawB_full[rs]);
        } else {
          mbar_arrive_expect_tx(&rawB_full[rs], (uint32_t)a.st.G * TG_KC * STEP_U * 4u);
          for (int g = 0; g < a.st.G; ++g)
            tma_load_2d(dst + g * (TG_KC * STEP_U * 4), &a.tmB, g * a.st.H + (int)blockIdx.x * STEP_U, k0, &rawB_full[rs]);
        }
        TG_ACC(w_work);
      }
      if (tl) { a.dbg[32] = w_wait; a.dbg[33] = w_work; a.dbg[34] = clock64() - t_start; }
    }
  } else {
    // =================================================================================== B loader (cp.async fallback)
    const int bt = tid - 13 * 32;
    const int per = BN / 16;
    long long w_wait = 0, w_work = 0;
    TG_T0();
    for (int c = 0; c < n_chunks; ++c) {
      const int rs = c % LOOK;
      if (c >= LOOK) mbar_wait(&rawB_empty[rs], ((c / LOOK) - 1) & 1);
      TG_ACC(w_wait);
      const int k0 = k_begin + c * TG_KC;
      float* dst = reinterpret_cast<float*>(rawB0 + (size_t)rs * rawB_bytes);
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        if (it >= per) break;
        int n, kq;
        b_coords(it * 128 + bt, n, kq);
        const int k = k0 + 4 * kq;
        if (a.b_mode == 0) {
          float* cell = dst + n * 32 + ((kq ^ (n & 7)) << 2);
          const bool ok = n0 + n < a.N && k < k_end;
          const float* src = a.B;
          if (ok) src = (a.B2 && k >= a.b_split) ? a.B2 + (long long)(a.b2_off + n0 + n) * a.ldb2 + (k - a.b_split)
                                                 : a.B + (long long)(a.b_off + n0 + n) * a.ldb + k;
          if (a.b_vec) {
            const int left = ok ? (k_end - k) * 4 : 0;
            cp_async16(cell, src, left >= 16 ? 16 : (left > 0 ? left : 0));
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) { const bool oe = ok && k + e < k_end; cp_async4(cell + e, oe ? src + e : a.B, oe ? 4 : 0); }
          }
        } else {
          long long col = -1;
          float* cell;
          if (a.b_mode == 1) {
            if (n0 + n < a.N) col = a.b_off + n0 + n;
            cell = dst + (4 * kq) * BN + n;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const bool oe = col >= 0 && k + e < k_end;
              cp_async4(cell + e * BN, oe ? a.B + (long long)(k + e) * a.ldb + col : a.B, oe ? 4 : 0);
            }
          } else {
            const int g = n / STEP_U, j = n - g * STEP_U, u = blockIdx.x * STEP_U + j;
            if (g < a.st.G && u < a.st.H) col = (long long)g * a.st.H + u;
            cell = dst + g * (TG_KC * STEP_U) + (4 * kq) * STEP_U + j;
            if (g < 4) {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const bool oe = col >= 0 && k + e < k_end;
                cp_async4(cell + e * STEP_U, oe ? a.B + (long long)(k + e) * a.ldb + col : a.B, oe ? 4 : 0);
              }
            }
          }
        }
      }
      cp_async_arrive(&rawB_full[rs]);
      TG_ACC(w_work);
    }
    if (tl && bt == 0) { a.dbg[32] = w_wait; a.dbg[33] = w_work; a.dbg[34] = clock64() - t_start; }
  }

  // ======================================================================================= epilogue (thread = row)
  if (warp < 4) {
    // bias of this thread's output columns, fetched before the accumulators are waited for (EPI_STORE: pass p, columns
    // n0 + 32 p + 4 (lane & 7) ..)
    float bias_pre[4][4];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int col = n0 + 32 * p + (lane & 7) * 4 + e;
        bias_pre[p][e] = (EPI == EPI_STORE && a.bias && blockIdx.z == 0 && 32 * p < BN && col < a.N) ? __ldg(a.bias + col) : 0.f;
      }
    if (n_chunks > 0) {
      mbar_wait(&done, 0);
      tc_fence_after();
    }
    if (tl && tid == 0) a.dbg[4] = clock64() - t_start;       // accumulators complete
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    const int row = m0 + tid;
    auto load_d = [&](int c0, float (&d)[16]) {     // D1 + D2 of 16 columns (warp-collective)
      if (n_chunks > 0) {
        float w[16];
        tmem_ld16(tD1 + lane_off + c0, d);
        tmem_ld16(tD2 + lane_off + c0, w);
#pragma unroll
        for (int i = 0; i < 16; ++i) d[i] += w[i];
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) d[i] = 0.f;
      }
    };

    if constexpr (EPI == EPI_STORE) {
      // TMEM holds the tile with one ROW per thread; written straight from there a warp store would touch 32 different
      // rows.  Each warp therefore transposes 32 rows x 32 columns through a shared-memory patch (the raw ring is idle by
      // now) and writes full 128-byte row segments: lane = (row within a group of 4, 16-byte column chunk).
      const bool atomic_out = gridDim.z > 1;
      constexpr int PITCH = 36;                                    // floats per patch row: 16-byte aligned, conflict-free
      float* patch = reinterpret_cast<float*>(rawA0) + warp * 32 * PITCH;
      const int r_in = lane >> 3, c4 = (lane & 7) * 4;             // read-back position: row r_in (+4 per pass), columns c4..c4+3
      for (int c0 = 0; c0 < BN; c0 += 32) {
        {
          float d[16];
          load_d(c0, d);
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(patch + lane * PITCH + i) = make_float4(d[i], d[i + 1], d[i + 2], d[i + 3]);
          if (c0 + 16 < BN) {
            load_d(c0 + 16, d);
#pragma unroll
            for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(patch + lane * PITCH + 16 + i) = make_float4(d[i], d[i + 1], d[i + 2], d[i + 3]);
          }
        }
        __syncwarp();
        const int col = n0 + c0 + c4;
        const bool col_in = col < a.N && c0 + c4 < BN;
        float bias4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) bias4[e] = bias_pre[0][e];
#pragma unroll
        for (int p = 1; p < 4; ++p)
          if (c0 == 32 * p) {
#pragma unroll
            for (int e = 0; e < 4; ++e) bias4[e] = bias_pre[p][e];
          }
#pragma unroll
        for (int rr = 0; rr < 32; rr += 4) {
          const int grow = m0 + warp * 32 + rr + r_in;
          if (grow >= a.M || !col_in) continue;
          const float4 v = *reinterpret_cast<const float4*>(patch + (rr + r_in) * PITCH + c4);
          float o[4] = {a.alpha * v.x + bias4[0], a.alpha * v.y + bias4[1], a.alpha * v.z + bias4[2], a.alpha * v.w + bias4[3]};
          float* dst = a.C + (long long)grow * a.ldc + col;
          const bool v4 = a.c_vec && col + 3 < a.N;
          if (atomic_out) {
            if (v4) asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" :: "l"(dst), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]) : "memory");
            else {
#pragma unroll
              for (int e = 0; e < 4; ++e) if (col + e < a.N) atomicAdd(dst + e, o[e]);
            }
          } else if (v4) {
            float4 r = make_float4(o[0], o[1], o[2], o[3]);
            if (a.accumulate) { const float4 p = *reinterpret_cast<const float4*>(dst); r.x += p.x; r.y += p.y; r.z += p.z; r.w += p.w; }
            *reinterpret_cast<float4*>(dst) = r;
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) if (col + e < a.N) dst[e] = a.accumulate ? dst[e] + o[e] : o[e];
          }
        }
        __syncwarp();
      }
    }

    if constexpr (FWD) {
      // row = batch row b, columns: gate g of unit u0 + j at g*8 + j
      constexpr int G = EPI == EPI_LSTM_FWD ? 4 : (EPI == EPI_GRU_FWD ? 3 : 1);
      const StepArgs& s = a.st;
      float pre[32];
      {
        float d0[16], d1[16];
        load_d(0, d0);
        load_d(16, d1);
#pragma unroll
        for (int i = 0; i < 16; ++i) { pre[i] = d0[i]; pre[16 + i] = d1[i]; }
      }
      const int b = row, u0 = blockIdx.x * STEP_U;
      if (b < s.B && s.t < __ldg(s.len + b)) {
        const int H = s.H, GH = G * H;
        float xg[4][8], hp[8], hn[8], cp[8], cn[8], sv[4][8];
#pragma unroll
        for (int g = 0; g < G; ++g) ld8(s.Xg_t + (long long)b * GH + g * H + u0, xg[g]);
        ld8(s.hs_t + (long long)b * H + u0, hp);
        if (G == 4) ld8(s.cs_t + (long long)b * H + u0, cp);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if constexpr (G == 4) {
            const float wci = __ldg(s.peep + u0 + j), wcf = __ldg(s.peep + H + u0 + j), wco = __ldg(s.peep + 2 * H + u0 + j);
            const float c_prev = cp[j];
            const float ig = sigmoid_fast(xg[0][j] + pre[j] + c_prev * wci);
            const float fg = sigmoid_fast(xg[1][j] + pre[8 + j] + c_prev * wcf);
            const float gg = tanh_fast(xg[2][j] + pre[16 + j]);
            const float c_new = fg * c_prev + ig * gg;
            const float og = sigmoid_fast(xg[3][j] + pre[24 + j] + c_new * wco);
            hn[j] = og * tanh_fast(c_new);
            cn[j] = c_new;
            sv[0][j] = ig; sv[1][j] = fg; sv[2][j] = gg; sv[3][j] = og;
          } else if constexpr (G == 3) {
            const float r = sigmoid_fast(pre[j] + xg[0][j]);
            const float uu = sigmoid_fast(pre[8 + j] + xg[1][j]);
            const float ac = pre[16 + j];
            const float cand = tanh_fast(xg[2][j] + r * ac);
            hn[j] = (1.f - uu) * hp[j] + uu * cand;
            sv[0][j] = r; sv[1][j] = uu; sv[2][j] = cand; sv[3][j] = ac;
          } else {
            const float z = xg[0][j] + pre[j];
            hn[j] = s.relu ? fmaxf(z, 0.f) : tanh_fast(z);
          }
        }
        st8(s.hs_n + (long long)b * H + u0, hn);
        if (G == 4) st8(s.cs_n + (long long)b * H + u0, cn);
        if (G > 1) {
#pragma unroll
          for (int g = 0; g < 4; ++g) st8(s.act_t + (long long)b * 4 * H + g * H + u0, sv[g]);
        }
      }
    }

    if constexpr (BWD) {
      // row = hidden unit k, columns = batch rows n0 + j;  D[k][j] = sum_c W_hid[k][c] da_{t+1}[b][c]
      constexpr int G = EPI == EPI_LSTM_BWD ? 4 : (EPI == EPI_GRU_BWD ? 3 : 1);
      const StepArgs& s = a.st;
      const int k = row, H = s.H, GH = G * H;
      const bool k_ok = k < H;
      float wci = 0.f, wcf = 0.f, wco = 0.f;
      if (G == 4 && k_ok) { wci = __ldg(s.peep + k); wcf = __ldg(s.peep + H + k); wco = __ldg(s.peep + 2 * H + k); }
      for (int c0 = 0; c0 < BN; c0 += 16) {
        float P[16];
        load_d(c0, P);
        if (!k_ok) continue;
#pragma unroll 4
        for (int j = 0; j < 16; ++j) {
          const int b = n0 + c0 + j;
          if (b >= s.B) break;
          const long long idx = (long long)b * H + k;
          const float dh = s.carry[idx] + P[j];
          const bool active = s.t < __ldg(s.len + b);
          float dx[4] = {0.f, 0.f, 0.f, 0.f}, dacv = 0.f, carry_new = dh;
          if (active) {
            const float d = dh + (s.dhs_t ? __ldg(s.dhs_t + idx) : 0.f);
            const float* ap = s.act_r + (long long)b * 4 * H + k;
            if constexpr (G == 4) {
              const float ig = __ldg(ap), fg = __ldg(ap + H), gg = __ldg(ap + 2 * H), og = __ldg(ap + 3 * H);
              const float c_prev = __ldg(s.cs_r + idx), c_new = __ldg(s.cs_rn + idx);
              const float tc = tanh_fast(c_new);
              const float do_pre = d * (tc * og * (1.f - og));
              const float dct = s.dcs[idx] + d * (og * (1.f - tc * tc)) + do_pre * wco;
              const float di_pre = dct * (gg * ig * (1.f - ig));
              const float df_pre = dct * (c_prev * fg * (1.f - fg));
              const float dg_pre = dct * (ig * (1.f - gg * gg));
              const long long BH = (long long)s.B * H;
              s.dpe[idx] += di_pre * c_prev;
              s.dpe[BH + idx] += df_pre * c_prev;
              s.dpe[2 * BH + idx] += do_pre * c_new;
              s.dcs[idx] = dct * fg + di_pre * wci + df_pre * wcf;
              dx[0] = clip_sym(di_pre, s.clip); dx[1] = clip_sym(df_pre, s.clip);
              dx[2] = clip_sym(dg_pre, s.clip); dx[3] = clip_sym(do_pre, s.clip);
              carry_new = 0.f;
            } else if constexpr (G == 3) {
              const float r = __ldg(ap), uu = __ldg(ap + H), cand = __ldg(ap + 2 * H), ac = __ldg(ap + 3 * H);
              const float h_prev = __ldg(s.hs_r + idx);
              const float du_pre = d * ((cand - h_prev) * uu * (1.f - uu));
              const float dq = clip_sym(d * (uu * (1.f - cand * cand)), s.clip);
              const float dr_pre = dq * (ac * r * (1.f - r));
              dx[0] = clip_sym(dr_pre, s.clip);
              dx[1] = clip_sym(du_pre, s.clip);
              dx[2] = dq;
              dacv = clip_sym(dq * r, s.clip);
              carry_new = d * (1.f - uu);
            } else {
              const float h_new = __ldg(s.hs_r + idx);          // hs_r = state AFTER step t for the vanilla cell
              dx[0] = clip_sym(d * (s.relu ? (h_new > 0.f ? 1.f : 0.f) : 1.f - h_new * h_new), s.clip);
              carry_new = 0.f;
            }
          }
          s.carry[idx] = carry_new;
#pragma unroll
          for (int g = 0; g < G; ++g) s.dXg_t[(long long)b * GH + g * H + k] = dx[g];
          if (G == 3) s.dac_t[idx] = dacv;
        }
      }
    }

    if constexpr (EPI == EPI_INIT_GRAD) {
      const StepArgs& s = a.st;
      const int k = row, H = s.H;
      float sh = 0.f, sc = 0.f, sp0 = 0.f, sp1 = 0.f, sp2 = 0.f;
      const long long BH = (long long)s.B * H;
      for (int c0 = 0; c0 < BN; c0 += 16) {
        float P[16];
        load_d(c0, P);
        if (k >= H) continue;
        for (int j = 0; j < 16; ++j) {
          const int b = n0 + c0 + j;
          if (b >= s.B) break;
          const long long idx = (long long)b * H + k;
          sh += s.carry[idx] + P[j];
          if (s.G == 4) { sc += s.dcs[idx]; sp0 += s.dpe[idx]; sp1 += s.dpe[BH + idx]; sp2 += s.dpe[2 * BH + idx]; }
        }
      }
      if (k < H) {
        atomicAdd(s.g_h_init + k, sh);
        if (s.G == 4) {
          atomicAdd(s.g_c_init + k, sc);
          atomicAdd(s.g_peep + k, sp0);
          atomicAdd(s.g_peep + H + k, sp1);
          atomicAdd(s.g_peep + 2 * H + k, sp2);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tl && tid == 0) a.dbg[5] = clock64() - t_start;         // epilogue done
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512));
#undef TG_T0
#undef TG_ACC
}

// h_last[b] = state after the last valid step of row b = block len[b] of the trajectory (block 0 = learned init)
__global__ void gather_last_state_kernel(const float* __restrict__ hs, const int32_t* __restrict__ len, float* __restrict__ out,
                                         int B, int H, int t_max) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * H) return;
  const int b = (int)(i / H), k = (int)(i - (long long)b * H);
  const int l = min(len[b], t_max);
  out[i] = hs[((long long)l * B + b) * H + k];
}

__global__ void bcast_rows_kernel(float* __restrict__ out, const float* __restrict__ v, int64_t rows, int cols) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) out[i] = v[i % cols];
}

__global__ void zero2d_kernel(float* C, int M, int N, long long ldc) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)M * N) return;
  C[(i / N) * ldc + (i % N)] = 0.f;
}

constexpr size_t TG_SMEM_MAX = 232448 - 1024;      // 227 KB opt-in limit minus the static barriers

size_t tg_conv_bytes(int BN) { return (size_t)TG_STAGES * BN * TG_KC * 8; }
size_t tg_raw_stage_bytes(int BN) { return (size_t)128 * TG_KC * 4 + (size_t)BN * TG_KC * 4; }
int tg_look(int BN) {
  const size_t left = TG_SMEM_MAX - 1024 - tg_conv_bytes(BN);
  return (int)std::max<size_t>(2, std::min<size_t>(TG_LOOK_MAX, left / tg_raw_stage_bytes(BN)));
}

template <int EPI>
int launch_tg(sbr_model* m, const TgArgs& a, dim3 grid) {
  // converted B ring + raw fp32 ring (A tile 16 KB + B tile BN*128 B per stage) + 1 KB alignment slack
  const size_t smem = tg_conv_bytes(a.BN) + (size_t)a.look * tg_raw_stage_bytes(a.BN) + 1024;
  // opt-in shared-memory limit: per (kernel instantiation, device) -- the attribute is per device
  static std::vector<int> done_dev;
  if (std::find(done_dev.begin(), done_dev.end(), m->dev) == done_dev.end()) {
    cudaError_t e = cudaFuncSetAttribute(tc_gemm_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TG_SMEM_MAX);
    if (e != cudaSuccess) { sbr_set_error(m, SBR_E_CUDA, "tc_gemm attr: %s", cudaGetErrorString(e)); return SBR_E_CUDA; }
    done_dev.push_back(m->dev);
  }
  tc_gemm_kernel<EPI><<<grid, TG_NT, smem, m->stream>>>(a);
  KERNEL_CHECK(m);
  return 0;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

// C[M,N] = alpha * op(A) * op(B) (+ bias[n]) (+ C);  ta: A stored [K, lda] ; tb: B stored [N, ldb] (same meaning as
// launch_gemm).  Returns 1 when the tensor-core kernel does not apply (caller falls back to the FFMA kernels).
int launch_gemm_tc(sbr_model* m, bool ta, bool tb, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                   float* C, int ldc, float alpha, float beta, const float* bias) {
  if (M <= 0 || N <= 0) return 0;
  if (!m->use_tc_gemm || K <= 0) return 1;
  if (beta != 0.f && beta != 1.f) return 1;
  TgArgs a{};
  a.A = A; a.lda = lda; a.a_mode = ta ? 1 : 0;
  a.B = B; a.ldb = ldb; a.b_mode = tb ? 0 : 1;
  a.M = M; a.N = N; a.K = K;
  a.BN = N <= 16 ? 16 : (N <= 32 ? 32 : (N <= 64 ? 64 : 128));
  // small outputs (the C2 score matrix is 29 tiles of 128 columns on 148 SMs): 64-column tiles halve the B conversion and
  // the epilogue of every CTA and double the CTAs
  // (not for side-stream work: it runs beside a cluster scan that needs whole GPCs free, fewer and fatter CTAs interfere less)
  if (a.BN == 128 && K <= 512 && !m->on_side && cdiv(M, 128) * cdiv(N, 128) * 2 <= m->n_sm) a.BN = 64;   // short K only: with a long K the A tile would be converted twice as often
  a.a_vec = (!ta && lda % 4 == 0 && aligned16(A)) ? 1 : 0;
  a.b_vec = (tb && ldb % 4 == 0 && aligned16(B)) ? 1 : 0;
  a.C = C; a.ldc = ldc; a.alpha = alpha; a.accumulate = beta == 1.f ? 1 : 0; a.bias = bias;
  a.c_vec = (ldc % 4 == 0 && aligned16(C)) ? 1 : 0;
  a.look = tg_look(a.BN);
  if (m->use_tma_gemm) {
    a.tma_a = ta ? get_tmap(&a.tmA, A, M, K, lda, 128, TG_KC, false) : get_tmap(&a.tmA, A, K, M, lda, TG_KC, 128, true);
    a.tma_b = tb ? get_tmap(&a.tmB, B, K, N, ldb, TG_KC, a.BN, true) : get_tmap(&a.tmB, B, N, K, ldb, a.BN, TG_KC, false);
  }
  const int tiles = cdiv(M, 128) * cdiv(N, a.BN);
  int splits = 1;
  if (tiles < m->n_sm) splits = std::max(1, std::min(m->n_sm / tiles, K / 128));   // tall-K, small output: fill the SMs
  int kps = (int)round_up(cdiv(K, splits), TG_KC);
  splits = cdiv(K, kps);
  a.k_per_split = kps;
  if (splits > 1 && beta == 0.f) {
    if (ldc == N) {
      CU_TRY(m, cudaMemsetAsync(C, 0, (size_t)M * N * sizeof(float), m->stream));
    } else {
      zero2d_kernel<<<cdiv((int64_t)M * N, 256), 256, 0, m->stream>>>(C, M, N, ldc);
      KERNEL_CHECK(m);
    }
  }
  static long long* dbg = nullptr;
  static const bool want_tl = getenv("SBR_TG_TIMELINE") != nullptr;
  if (want_tl) {
    if (!dbg) { cudaMalloc(&dbg, 64 * sizeof(long long)); }
    cudaMemsetAsync(dbg, 0, 64 * sizeof(long long), m->stream);
    a.dbg = dbg;
  }
  const int rc = launch_tg<EPI_STORE>(m, a, dim3(cdiv(N, a.BN), cdiv(M, 128), splits));
  if (want_tl && rc == 0) {
    long long h[64];
    cudaStreamSynchronize(m->stream);
    cudaMemcpy(h, dbg, sizeof(h), cudaMemcpyDeviceToHost);
    fprintf(stderr, "[tg timeline M=%d N=%d K=%d BN=%d splits=%d chunks=%lld] Aconv: wait_raw %lld wait_empty %lld work %lld total %lld | Bconv: wait_raw %lld wait_empty %lld work %lld total %lld | "
            "MMA: wait_full %lld issue %lld total %lld | Aload: wait %lld work %lld total %lld | Bload: wait %lld work %lld total %lld | acc_done %lld epi_done %lld\n",
            M, N, K, a.BN, splits, h[19], h[0], h[1], h[2], h[3], h[8], h[9], h[10], h[11], h[16], h[17], h[18], h[24], h[25], h[26], h[32], h[33], h[34], h[4], h[5]);
  }
  return rc;
}

// 1 when the per-step tensor-core scan handles this layer (hidden sizes beyond the cluster-resident kernels)
int step_scan_applies(const ScanSwitches& s, int H) {
  // H % 16: the GRU backward switches its B source (dXg | dac) at k = 2H, which must be a 32-wide chunk boundary
  return (s.tc_gemm && s.step && H % 16 == 0 && H >= 32) ? 1 : 0;
}
int step_scan_applies(const sbr_model* m, int G, int H) {
  (void)G;
  return step_scan_applies(scan_switches(m), H);
}

int launch_rnn_forward_steps(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last) {
  const int H = L.H, G = L.G, GH = G * H;
  // block 0 of the trajectories = the learned initial state, broadcast over the rows
  bcast_rows_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, m->stream>>>(L.hs, m->params + L.h_init, (int64_t)B, H);
  KERNEL_CHECK(m);
  if (G == 4) {
    bcast_rows_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, m->stream>>>(L.cs, m->params + L.c_init, (int64_t)B, H);
    KERNEL_CHECK(m);
  }
  TgArgs a{};
  a.lda = H; a.a_mode = 0; a.a_vec = 1;
  a.B = m->params + L.W_hid; a.ldb = GH; a.b_mode = 2;
  a.M = B; a.N = STEP_BN; a.K = H; a.BN = STEP_BN; a.k_per_split = (int)round_up(H, TG_KC);
  a.look = tg_look(a.BN);
  a.A = L.hs;
  if (m->use_tma_gemm) {
    a.tma_a = get_tmap(&a.tmA, L.hs, H, (uint64_t)(m->T + 1) * m->B, H, TG_KC, 128, true);
    a.tma_b = get_tmap(&a.tmB, m->params + L.W_hid, GH, H, GH, STEP_U, TG_KC, false);
  }
  a.st.B = B; a.st.H = H; a.st.G = G; a.st.len = len; a.st.peep = m->params + L.peep; a.st.relu = L.relu;
  const dim3 grid(cdiv(H, STEP_U), cdiv(B, 128), 1);
  for (int t = 0; t < t_max; ++t) {
    a.a_off = t * B;       // rows t*B .. of the state trajectory
    a.st.t = t;
    a.st.Xg_t = L.Xg + (int64_t)t * B * GH;
    a.st.hs_t = L.hs + (int64_t)t * B * H;
    a.st.hs_n = L.hs + (int64_t)(t + 1) * B * H;
    a.st.cs_t = L.cs ? L.cs + (int64_t)t * B * H : nullptr;
    a.st.cs_n = L.cs ? L.cs + (int64_t)(t + 1) * B * H : nullptr;
    a.st.act_t = L.act ? L.act + (int64_t)t * B * 4 * H : nullptr;
    int rc;
    if (G == 4) rc = launch_tg<EPI_LSTM_FWD>(m, a, grid);
    else if (G == 3) rc = launch_tg<EPI_GRU_FWD>(m, a, grid);
    else rc = launch_tg<EPI_VAN_FWD>(m, a, grid);
    if (rc) return rc;
    m->scan_launches++;
  }
  if (h_last) {
    gather_last_state_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, m->stream>>>(L.hs, len, h_last, B, H, t_max);
    KERNEL_CHECK(m);
  }
  return 0;
}

int launch_rnn_backward_steps(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, const float* dh_last) {
  const int H = L.H, G = L.G, GH = G * H;
  const size_t BH = (size_t)B * H;
  // carried state of the scan: dh flowing to the previous step, d(cell state), peephole gradient partial sums
  if (dh_last) CU_TRY(m, cudaMemcpyAsync(m->step_carry, dh_last, BH * sizeof(float), cudaMemcpyDeviceToDevice, m->stream));
  else CU_TRY(m, cudaMemsetAsync(m->step_carry, 0, BH * sizeof(float), m->stream));
  if (G == 4) {
    CU_TRY(m, cudaMemsetAsync(m->step_dcs, 0, BH * sizeof(float), m->stream));
    CU_TRY(m, cudaMemsetAsync(m->step_dpe, 0, 3 * BH * sizeof(float), m->stream));
  }
  TgArgs a{};
  a.A = m->params + L.W_hid; a.lda = GH; a.a_mode = 0; a.a_vec = 1;
  a.b_mode = 0; a.b_vec = 1;
  a.M = H; a.N = B; a.K = GH; a.BN = STEP_BN; a.k_per_split = (int)round_up(GH, TG_KC);
  a.look = tg_look(a.BN);
  a.B = L.dXg; a.ldb = GH;
  if (G == 3) { a.B2 = L.dac; a.ldb2 = H; a.b_split = 2 * H; }
  if (m->use_tma_gemm) {
    a.tma_a = get_tmap(&a.tmA, m->params + L.W_hid, GH, H, GH, TG_KC, 128, true);
    a.tma_b = get_tmap(&a.tmB, L.dXg, GH, (uint64_t)m->T * m->B, GH, TG_KC, STEP_BN, true);
    if (G == 3) a.tma_b = a.tma_b && get_tmap(&a.tmB2, L.dac, H, (uint64_t)m->T * m->B, H, TG_KC, STEP_BN, true);
  }
  StepArgs& s = a.st;
  s.B = B; s.H = H; s.G = G; s.len = len; s.peep = m->params + L.peep; s.clip = m->cfg.grad_clip; s.relu = L.relu;
  s.carry = m->step_carry; s.dcs = m->step_dcs; s.dpe = m->step_dpe;
  s.g_h_init = m->grads + L.h_init; s.g_c_init = m->grads + L.c_init; s.g_peep = m->grads + L.peep;
  const dim3 grid(cdiv(B, STEP_BN), cdiv(H, 128), 1);
  for (int t = t_max - 1; t >= -1; --t) {
    // B operand = da_{t+1}: dXg rows of step t+1 (GRU: the candidate's hidden pre-activation gradient comes from dac)
    if (t + 1 < t_max) {
      a.b_off = a.b2_off = (t + 1) * B;
      a.K = GH;
    } else {
      a.b_off = a.b2_off = 0; a.K = 0;        // first step: nothing flows in from t+1
    }
    s.t = t;
    int rc;
    if (t >= 0) {
      const int64_t r = (int64_t)t * B;
      s.act_r = L.act ? L.act + r * 4 * H : nullptr;
      s.cs_r = L.cs ? L.cs + r * H : nullptr;
      s.cs_rn = L.cs ? L.cs + (r + B) * H : nullptr;
      s.hs_r = L.hs + (G == 1 ? r + B : r) * H;
      s.dhs_t = (!dh_last && L.dhs) ? L.dhs + r * H : nullptr;
      s.dXg_t = L.dXg + r * GH;
      s.dac_t = L.dac ? L.dac + r * H : nullptr;
      if (G == 4) rc = launch_tg<EPI_LSTM_BWD>(m, a, grid);
      else if (G == 3) rc = launch_tg<EPI_GRU_BWD>(m, a, grid);
      else rc = launch_tg<EPI_VAN_BWD>(m, a, grid);
    } else {
      rc = launch_tg<EPI_INIT_GRAD>(m, a, grid);
    }
    if (rc) return rc;
    m->scan_launches++;
  }
  return 0;
}
