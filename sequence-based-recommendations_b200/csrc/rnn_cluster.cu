// rnn_cluster.cu -- stage 2 of the hot path: the recurrent scan and its BPTT as persistent
// thread-block-cluster kernels.
//
// Reference semantics (neural_networks/sparse_lstm.py):
//   LSTM step   :377-415  gates = Xg_t + h W_hid ; peepholes ; c = f c + i g ; h = o tanh(c)
//   GRU step    :764-796  a = h W_hid ; r,u = sigma(a + x) ; cand = tanh(x_c + r a_c) ; h = (1-u) h + u cand
//   Vanilla     :1120-1143 h = tanh(x + h W_hid)
//   masking     :417-425, :798-805  masked rows keep their state
//   learned init:438-445, :817-819  h0/c0 rows broadcast over the batch
//   scan        :474-481, :843-850  T strictly sequential steps (theano.scan), full BPTT
//   grad_clip   :386-388, :768-772, :789-791  clamp of the incoming gradient to +-100
//
// B200 mapping.  Batch rows are independent, so the batch is cut into tiles of BT rows and each
// tile is owned by ONE thread-block cluster of C CTAs that runs all T steps without any grid-wide
// synchronisation.  CTA r of the cluster owns the hidden units [r*Hs, (r+1)*Hs) for ALL gates, keeps
// its slice of W_hid resident in shared memory for the whole scan (H x G*Hs floats), and keeps the
// tile's full previous state h_{t-1} [H x BT] in shared memory.  Per step a CTA computes its
// [BT x G*Hs] slice of the gate pre-activations, applies the fused gate math, and publishes its
// [BT x Hs] slice of h_t into the shared memory of every CTA of the cluster (DSMEM stores), double
// buffered, followed by one cluster barrier.  The backward kernel keeps the same ownership and the
// same weight slice: dh_{t-1} = dgates W_hid^T is computed split-K (each CTA contracts over ITS gate
// columns for all H outputs) and the partial sums are reduce-scattered to their owners through
// DSMEM.  Weight gradients are NOT accumulated inside the scan: the kernels stream dgates to HBM and
// dW_hid / dW_in / db are formed afterwards by one big GEMM / scatter (gemm.cu, gather_scatter.cu).
//
// Arithmetic: fp32 FFMA with fp32 accumulation (SBR_MATH_FP32).
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int NT = 256;  // threads per CTA (8 warps)

struct RnnArgs {
  // forward inputs
  const float* Xg;      // [T*B, G*H]
  const float* W_hid;   // [H, G*H]
  const float* W_hidT;  // [G*H, H] (backward)
  const float* peep;    // LSTM [3, H]
  const float* h_init;  // [H]
  const float* c_init;  // [H]
  const int32_t* len;   // [B]
  // saved / produced
  float* hs;            // [(T+1)*B, H]
  float* cs;            // [(T+1)*B, H]
  float* act;           // [T*B, 4H]
  float* h_last;        // [B, H] (forward output, may be null)
  // backward
  const float* dh_last; // [B, H] gradient of the final state (top layer) or null
  const float* dhs;     // [T*B, H] gradient from the layer above (lower layers) or null
  float* dXg;           // [T*B, G*H]
  float* dac;           // GRU [T*B, H]
  float* g_peep;        // gradient arena slots
  float* g_h_init;
  float* g_c_init;
  float clip;
  int relu;            // vanilla cell: rectifier instead of tanh (dense-input layers)
  int B, H, Hs, t_max;
};

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float clipf_(float x, float c) { return c > 0.f ? fminf(fmaxf(x, -c), c) : x; }

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <int G, int BT, int JU, bool WSMEM>
__global__ void __launch_bounds__(NT, 1) rnn_fwd_kernel(const RnnArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  const int C = cluster.num_blocks();
  const int rank = cluster.block_rank();
  const int tile = blockIdx.x / C;
  const int b0 = tile * BT;
  const int H = a.H, Hs = a.Hs, GH = G * H, B = a.B;
  const int j0 = rank * Hs;
  const int nj = max(0, min(Hs, H - j0));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NRG = BT / 8;
  constexpr int NKS = 8 / NRG;
  constexpr int JP = 32 * JU;
  constexpr int NP = BT * JP / NT;
  static_assert(NP >= 1 && NP <= 4, "pairs per thread");

  extern __shared__ __align__(16) float smem[];
  float* hbuf = smem;                        // [2][H][BT]
  float* cst = hbuf + 2 * H * BT;            // [BT][JP]
  float* red = cst + BT * JP;                // [NKS][BT][G][JP]
  float* Wf = red + NKS * BT * G * JP;       // [H][G*Hs]  (WSMEM only)
  __shared__ int lens_s[BT];
  __shared__ int t_end_s;

  if (tid < BT) lens_s[tid] = (b0 + tid < B) ? min(a.len[b0 + tid], a.t_max) : 0;
  __syncthreads();
  if (tid == 0) {
    int mx = 0;
    for (int b = 0; b < BT; ++b) mx = max(mx, lens_s[b]);
    t_end_s = mx;
  }
  if (WSMEM) {
    const int per_k = G * nj;
    for (int idx = tid; idx < H * per_k; idx += NT) {
      const int k = idx / per_k, rem = idx - k * per_k;
      const int g = rem / nj, j = rem - g * nj;
      Wf[k * (G * Hs) + g * Hs + j] = a.W_hid[(int64_t)k * GH + g * H + j0 + j];
    }
  }
  for (int idx = tid; idx < H * BT; idx += NT) hbuf[idx] = a.h_init[idx / BT];
  for (int idx = tid; idx < BT * JP; idx += NT) {
    const int j = idx % JP;
    cst[idx] = (G == 4 && j < nj) ? a.c_init[j0 + j] : 0.f;
  }
  // state 0 of the saved trajectories
  for (int idx = tid; idx < BT * nj; idx += NT) {
    const int b = idx / nj, j = idx - b * nj;
    if (b0 + b < B) {
      a.hs[(int64_t)(b0 + b) * H + j0 + j] = a.h_init[j0 + j];
      if (G == 4) a.cs[(int64_t)(b0 + b) * H + j0 + j] = a.c_init[j0 + j];
    }
  }
  __syncthreads();
  const int t_end = t_end_s;

  float wci[NP], wcf[NP], wco[NP];
  float xc[NP][G], xn[NP][G];
#pragma unroll
  for (int q = 0; q < NP; ++q) {
    const int p = tid + NT * q, j = p % JP;
    wci[q] = wcf[q] = wco[q] = 0.f;
    if (G == 4 && j < nj) {
      wci[q] = a.peep[j0 + j];
      wcf[q] = a.peep[H + j0 + j];
      wco[q] = a.peep[2 * H + j0 + j];
    }
#pragma unroll
    for (int g = 0; g < G; ++g) xc[q][g] = xn[q][g] = 0.f;
  }
  auto load_x = [&](int t, float (&x)[NP][G]) {
#pragma unroll
    for (int q = 0; q < NP; ++q) {
      const int p = tid + NT * q, b = p / JP, j = p % JP;
      if (j < nj && t < lens_s[b]) {
        const float* src = a.Xg + ((int64_t)t * B + b0 + b) * GH + j0 + j;
#pragma unroll
        for (int g = 0; g < G; ++g) x[q][g] = __ldg(src + g * H);
      }
    }
  };
  if (t_end > 0) load_x(0, xc);

  cluster.sync();  // every CTA's buffers are initialised before any remote store lands

  const int rg = warp % NRG, ks = warp / NRG;
  const int kc = (H + NKS - 1) / NKS;
  const int kb = ks * kc, ke = min(H, kb + kc);
  int jj[JU];
#pragma unroll
  for (int ju = 0; ju < JU; ++ju) jj[ju] = max(0, min(lane + 32 * ju, nj - 1));

  for (int t = 0; t < t_end; ++t) {
    const int cur = t & 1, nxt = cur ^ 1;
    if (t + 1 < t_end) load_x(t + 1, xn);

    // ---- partial gate pre-activations: acc[r][g][ju] = sum_{k in split} h[b][k] * W[k][g][j]
    float acc[8][G][JU];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int g = 0; g < G; ++g)
#pragma unroll
        for (int ju = 0; ju < JU; ++ju) acc[r][g][ju] = 0.f;
    if (nj > 0) {
      const float* hb = hbuf + cur * H * BT + rg * 8;
#pragma unroll 4
      for (int k = kb; k < ke; ++k) {
        const float4 h0 = *reinterpret_cast<const float4*>(hb + k * BT);
        const float4 h1 = *reinterpret_cast<const float4*>(hb + k * BT + 4);
        const float hv[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
        for (int ju = 0; ju < JU; ++ju) {
#pragma unroll
          for (int g = 0; g < G; ++g) {
            const float w = WSMEM ? Wf[k * (G * Hs) + g * Hs + jj[ju]]
                                  : __ldg(a.W_hid + (int64_t)k * GH + g * H + j0 + jj[ju]);
#pragma unroll
            for (int r = 0; r < 8; ++r) acc[r][g][ju] = fmaf(hv[r], w, acc[r][g][ju]);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int g = 0; g < G; ++g)
#pragma unroll
          for (int ju = 0; ju < JU; ++ju)
            red[((ks * BT + rg * 8 + r) * G + g) * JP + lane + 32 * ju] = acc[r][g][ju];
    }
    __syncthreads();

    // ---- fused gate math for the (b, j) pairs this thread owns
#pragma unroll
    for (int q = 0; q < NP; ++q) {
      const int p = tid + NT * q, b = p / JP, j = p % JP;
      if (j < nj) {
        float pre[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float s = 0.f;
#pragma unroll
          for (int s2 = 0; s2 < NKS; ++s2) s += red[((s2 * BT + b) * G + g) * JP + j];
          pre[g] = s;
        }
        const bool active = t < lens_s[b];
        const float h_prev = hbuf[cur * H * BT + (j0 + j) * BT + b];
        float h_new = h_prev;
        const int64_t row = (int64_t)t * B + b0 + b;
        if (active) {
          if constexpr (G == 4) {
            const float c_prev = cst[b * JP + j];
            const float ig = sigmoidf_(xc[q][0] + pre[0] + c_prev * wci[q]);
            const float fg = sigmoidf_(xc[q][1] + pre[1] + c_prev * wcf[q]);
            const float gg = tanhf(xc[q][2] + pre[2]);
            const float c_new = fg * c_prev + ig * gg;
            const float og = sigmoidf_(xc[q][G - 1] + pre[G - 1] + c_new * wco[q]);
            h_new = og * tanhf(c_new);
            cst[b * JP + j] = c_new;
            float* ap = a.act + row * 4 * H + j0 + j;
            ap[0] = ig; ap[H] = fg; ap[2 * H] = gg; ap[3 * H] = og;
          } else if constexpr (G == 3) {
            const float r = sigmoidf_(pre[0] + xc[q][0]);
            const float u = sigmoidf_(pre[1] + xc[q][1]);
            const float ac = pre[G - 1];
            const float cand = tanhf(xc[q][G - 1] + r * ac);
            h_new = (1.f - u) * h_prev + u * cand;
            float* ap = a.act + row * 4 * H + j0 + j;
            ap[0] = r; ap[H] = u; ap[2 * H] = cand; ap[3 * H] = ac;
          } else {
            const float z = xc[q][0] + pre[0];
            h_new = a.relu ? fmaxf(z, 0.f) : tanhf(z);
          }
        }
        // publish h_t[b, j0+j] to every CTA of the cluster (distributed shared memory)
        const int off = nxt * H * BT + (j0 + j) * BT + b;
        for (int rr = 0; rr < C; ++rr) cluster.map_shared_rank(hbuf, rr)[off] = h_new;
        if (b0 + b < B) {
          a.hs[((int64_t)(t + 1) * B + b0 + b) * H + j0 + j] = h_new;
          if (G == 4) a.cs[((int64_t)(t + 1) * B + b0 + b) * H + j0 + j] = cst[b * JP + j];
        }
      }
    }
#pragma unroll
    for (int q = 0; q < NP; ++q)
#pragma unroll
      for (int g = 0; g < G; ++g) xc[q][g] = xn[q][g];
    cluster.sync();
  }

  if (a.h_last) {
    const int fin = t_end & 1;
    for (int idx = tid; idx < BT * nj; idx += NT) {
      const int b = idx / nj, j = idx - b * nj;
      if (b0 + b < B) a.h_last[(int64_t)(b0 + b) * H + j0 + j] = hbuf[fin * H * BT + (j0 + j) * BT + b];
    }
  }
  cluster.sync();  // no CTA exits while a peer may still address its shared memory
}

// ------------------------------------------------------------------------------------------
// backward (BPTT)
// ------------------------------------------------------------------------------------------
template <int G, int BT, int JU, bool WSMEM>
__global__ void __launch_bounds__(NT, 1) rnn_bwd_kernel(const RnnArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  const int C = cluster.num_blocks();
  const int rank = cluster.block_rank();
  const int tile = blockIdx.x / C;
  const int b0 = tile * BT;
  const int H = a.H, Hs = a.Hs, GH = G * H, B = a.B;
  const int j0 = rank * Hs;
  const int nj = max(0, min(Hs, H - j0));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NRG = BT / 8;
  constexpr int JP = 32 * JU;
  constexpr int NP = BT * JP / NT;
  constexpr int NSAVE = (G == 4) ? 6 : (G == 3 ? 5 : 1);

  extern __shared__ __align__(16) float smem[];
  float* dg = smem;                           // [G*Hs][BT]   da of this CTA's gate columns
  float* part = dg + G * Hs * BT;             // [2][C][BT][Hs] partial dh received from the peers
  float* carry = part + 2 * C * BT * Hs;      // [BT][JP] elementwise part of dh_{t-1}
  float* dcs = carry + BT * JP;               // [BT][JP] dc (LSTM)
  float* Wb = dcs + BT * JP;                  // [G*Hs][H] (WSMEM only), k contiguous
  __shared__ int lens_s[BT];
  __shared__ int t_end_s;

  if (tid < BT) lens_s[tid] = (b0 + tid < B) ? min(a.len[b0 + tid], a.t_max) : 0;
  __syncthreads();
  if (tid == 0) {
    int mx = 0;
    for (int b = 0; b < BT; ++b) mx = max(mx, lens_s[b]);
    t_end_s = mx;
  }
  if (WSMEM) {
    for (int idx = tid; idx < G * nj * H; idx += NT) {
      const int gj = idx / H, k = idx - gj * H;
      const int g = gj / nj, j = gj - g * nj;
      Wb[(g * Hs + j) * H + k] = a.W_hidT[(int64_t)(g * H + j0 + j) * H + k];
    }
  }
  for (int idx = tid; idx < 2 * C * BT * Hs; idx += NT) part[idx] = 0.f;
  for (int idx = tid; idx < G * Hs * BT; idx += NT) dg[idx] = 0.f;
  for (int idx = tid; idx < BT * JP; idx += NT) {
    const int b = idx / JP, j = idx % JP;
    float v = 0.f;
    if (a.dh_last && j < nj && b0 + b < B) v = a.dh_last[(int64_t)(b0 + b) * H + j0 + j];
    carry[idx] = v;
    dcs[idx] = 0.f;
  }
  __syncthreads();
  const int t_end = t_end_s;

  // masked tail [t_end, t_max): gradients are exactly zero there
  for (int t = t_end; t < a.t_max; ++t) {
    for (int idx = tid; idx < BT * G * nj; idx += NT) {
      const int b = idx / (G * nj), rem = idx - b * (G * nj);
      const int g = rem / nj, j = rem - g * nj;
      if (b0 + b < B) {
        a.dXg[((int64_t)t * B + b0 + b) * GH + g * H + j0 + j] = 0.f;
        if (G == 3 && g == 0) a.dac[((int64_t)t * B + b0 + b) * H + j0 + j] = 0.f;
      }
    }
  }

  float wci[NP], wcf[NP], wco[NP], dpe[NP][3];
  float sv[NP][NSAVE + 1], svn[NP][NSAVE + 1];
#pragma unroll
  for (int q = 0; q < NP; ++q) {
    const int p = tid + NT * q, j = p % JP;
    wci[q] = wcf[q] = wco[q] = 0.f;
    dpe[q][0] = dpe[q][1] = dpe[q][2] = 0.f;
    if (G == 4 && j < nj) {
      wci[q] = a.peep[j0 + j];
      wcf[q] = a.peep[H + j0 + j];
      wco[q] = a.peep[2 * H + j0 + j];
    }
#pragma unroll
    for (int s = 0; s <= NSAVE; ++s) sv[q][s] = svn[q][s] = 0.f;
  }
  // saved tensors of step t for this thread's pairs:
  //  LSTM: i f g o c_prev c_new | GRU: r u cand a_c h_prev | Vanilla: h_new ; last slot: dhs from above
  auto load_saved = [&](int t, float (&s)[NP][NSAVE + 1]) {
#pragma unroll
    for (int q = 0; q < NP; ++q) {
      const int p = tid + NT * q, b = p / JP, j = p % JP;
      if (j < nj && t < lens_s[b]) {
        const int64_t row = (int64_t)t * B + b0 + b;
        if constexpr (G == 4) {
          const float* ap = a.act + row * 4 * H + j0 + j;
          s[q][0] = __ldg(ap); s[q][1] = __ldg(ap + H); s[q][2] = __ldg(ap + 2 * H); s[q][3] = __ldg(ap + 3 * H);
          s[q][4] = __ldg(a.cs + row * H + j0 + j);
          s[q][NSAVE - 1] = __ldg(a.cs + (row + B) * H + j0 + j);
        } else if constexpr (G == 3) {
          const float* ap = a.act + row * 4 * H + j0 + j;
          s[q][0] = __ldg(ap); s[q][1] = __ldg(ap + H); s[q][2] = __ldg(ap + 2 * H); s[q][3] = __ldg(ap + 3 * H);
          s[q][NSAVE - 1] = __ldg(a.hs + row * H + j0 + j);
        } else {
          s[q][0] = __ldg(a.hs + (row + B) * H + j0 + j);
        }
        s[q][NSAVE] = a.dhs ? __ldg(a.dhs + row * H + j0 + j) : 0.f;
      }
    }
  };
  if (t_end > 0) load_saved(t_end - 1, sv);

  cluster.sync();

  const int NKG = (H + 31) / 32;
  for (int t = t_end - 1; t >= 0; --t) {
    const int par = t & 1;        // partials produced at step t go to buffer `par`
    const int rpar = par ^ 1;     // ... and the ones produced at step t+1 are read from `rpar`
    if (t > 0) load_saved(t - 1, svn);

    // ---- phase A: elementwise gate gradients for the pairs this thread owns
#pragma unroll
    for (int q = 0; q < NP; ++q) {
      const int p = tid + NT * q, b = p / JP, j = p % JP;
      if (j < nj) {
        float dh = carry[b * JP + j];
        for (int src = 0; src < C; ++src) dh += part[((rpar * C + src) * BT + b) * Hs + j];
        const bool active = t < lens_s[b];
        const int64_t row = (int64_t)t * B + b0 + b;
        float da[G], dx[G];
#pragma unroll
        for (int g = 0; g < G; ++g) da[g] = dx[g] = 0.f;
        float carry_new = dh;
        if (active) {
          dh += sv[q][NSAVE];
          if constexpr (G == 4) {
            const float ig = sv[q][0], fg = sv[q][1], gg = sv[q][2], og = sv[q][3];
            const float c_prev = sv[q][4], c_new = sv[q][NSAVE - 1];
            const float tc = tanhf(c_new);
            const float do_pre = dh * tc * og * (1.f - og);
            const float dct = dcs[b * JP + j] + dh * og * (1.f - tc * tc) + do_pre * wco[q];
            const float di_pre = dct * gg * ig * (1.f - ig);
            const float df_pre = dct * c_prev * fg * (1.f - fg);
            const float dg_pre = dct * ig * (1.f - gg * gg);
            dpe[q][0] += di_pre * c_prev;
            dpe[q][1] += df_pre * c_prev;
            dpe[q][2] += do_pre * c_new;
            dcs[b * JP + j] = dct * fg + di_pre * wci[q] + df_pre * wcf[q];
            da[0] = clipf_(di_pre, a.clip);
            da[1] = clipf_(df_pre, a.clip);
            da[2] = clipf_(dg_pre, a.clip);
            da[G - 1] = clipf_(do_pre, a.clip);
#pragma unroll
            for (int g = 0; g < G; ++g) dx[g] = da[g];
            carry_new = 0.f;
          } else if constexpr (G == 3) {
            const float r = sv[q][0], u = sv[q][1], cand = sv[q][2], ac = sv[q][3], h_prev = sv[q][NSAVE - 1];
            const float du_pre = dh * (cand - h_prev) * u * (1.f - u);
            const float dq = clipf_(dh * u * (1.f - cand * cand), a.clip);
            const float dr_pre = dq * ac * r * (1.f - r);
            da[0] = clipf_(dr_pre, a.clip);
            da[1] = clipf_(du_pre, a.clip);
            da[G - 1] = clipf_(dq * r, a.clip);
            dx[0] = da[0];
            dx[1] = da[1];
            dx[G - 1] = dq;
            carry_new = dh * (1.f - u);
          } else {
            const float h_new = sv[q][0];
            const float dq = clipf_(dh * (a.relu ? (h_new > 0.f ? 1.f : 0.f) : 1.f - h_new * h_new), a.clip);
            da[0] = dq;
            dx[0] = dq;
            carry_new = 0.f;
          }
        }
        carry[b * JP + j] = carry_new;
#pragma unroll
        for (int g = 0; g < G; ++g) dg[(g * Hs + j) * BT + b] = da[g];
        if (b0 + b < B) {
          float* dxp = a.dXg + row * GH + j0 + j;
#pragma unroll
          for (int g = 0; g < G; ++g) dxp[g * H] = dx[g];
          if (G == 3) a.dac[row * H + j0 + j] = da[G - 1];
        }
      }
    }
    __syncthreads();

    // ---- phase B: partial dh_{t-1}[b][k] = sum_{(g,j) in my slice} da[b][g][j] * W_hid[k][g][j], all k
    if (nj > 0) {
      for (int item = warp; item < NKG * NRG; item += NT / 32) {
        const int kg = item / NRG, rg2 = item - kg * NRG;
        const int k = kg * 32 + lane;
        const int kk = min(k, H - 1);
        float acc[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) acc[r] = 0.f;
        for (int g = 0; g < G; ++g) {
#pragma unroll 4
          for (int j = 0; j < nj; ++j) {
            const int gj = g * Hs + j;
            const float w = WSMEM ? Wb[gj * H + kk] : __ldg(a.W_hidT + (int64_t)(g * H + j0 + j) * H + kk);
            const float4 d0 = *reinterpret_cast<const float4*>(dg + gj * BT + rg2 * 8);
            const float4 d1 = *reinterpret_cast<const float4*>(dg + gj * BT + rg2 * 8 + 4);
            acc[0] = fmaf(d0.x, w, acc[0]); acc[1] = fmaf(d0.y, w, acc[1]);
            acc[2] = fmaf(d0.z, w, acc[2]); acc[3] = fmaf(d0.w, w, acc[3]);
            acc[4] = fmaf(d1.x, w, acc[4]); acc[5] = fmaf(d1.y, w, acc[5]);
            acc[6] = fmaf(d1.z, w, acc[6]); acc[7] = fmaf(d1.w, w, acc[7]);
          }
        }
        if (k < H) {
          const int rr = k / Hs, jo = k - rr * Hs;
          float* dst = cluster.map_shared_rank(part, rr) + ((par * C + rank) * BT + rg2 * 8) * Hs + jo;
#pragma unroll
          for (int r = 0; r < 8; ++r) dst[r * Hs] = acc[r];
        }
      }
    }
#pragma unroll
    for (int q = 0; q < NP; ++q)
#pragma unroll
      for (int s = 0; s <= NSAVE; ++s) sv[q][s] = svn[q][s];
    cluster.sync();
  }

  // ---- gradients of the learned initial states and of the peepholes
  const int fpar = 0;  // step t = 0 wrote buffer 0
#pragma unroll
  for (int q = 0; q < NP; ++q) {
    const int p = tid + NT * q, b = p / JP, j = p % JP;
    if (j < nj && b0 + b < B) {
      float dh = carry[b * JP + j];
      if (t_end > 0)
        for (int src = 0; src < C; ++src) dh += part[((fpar * C + src) * BT + b) * Hs + j];
      atomicAdd(a.g_h_init + j0 + j, dh);
      if (G == 4) {
        atomicAdd(a.g_c_init + j0 + j, dcs[b * JP + j]);
        atomicAdd(a.g_peep + j0 + j, dpe[q][0]);
        atomicAdd(a.g_peep + H + j0 + j, dpe[q][1]);
        atomicAdd(a.g_peep + 2 * H + j0 + j, dpe[q][2]);
      }
    }
  }
  cluster.sync();
}

// ------------------------------------------------------------------------------------------
// launch plumbing
// ------------------------------------------------------------------------------------------
struct Plan {
  int C, Hs, BT, JU;
  bool wsmem;
  size_t smem;
};

size_t fwd_smem(int G, int BT, int JU, int H, int Hs, bool wsmem) {
  const int NRG = BT / 8, NKS = 8 / NRG, JP = 32 * JU;
  size_t f = (size_t)2 * H * BT + (size_t)BT * JP + (size_t)NKS * BT * G * JP;
  if (wsmem) f += (size_t)H * G * Hs;
  return f * sizeof(float);
}
size_t bwd_smem(int G, int BT, int JU, int H, int Hs, int C, bool wsmem) {
  const int JP = 32 * JU;
  size_t f = (size_t)G * Hs * BT + (size_t)2 * C * BT * Hs + (size_t)2 * BT * JP;
  if (wsmem) f += (size_t)G * Hs * H;
  return f * sizeof(float);
}

// cluster size, batch tile and weight residency for one layer
Plan make_plan(int n_sm, int G, int H, int B, bool backward) {
  const size_t limit = 227 * 1024 - 1024;  // static shared memory of the kernels is < 1 KB
  Plan best{};
  int C = 8;
  while (C > 1 && H / C < 16) C >>= 1;     // keep at least ~16 hidden units per CTA
  const int Hs = cdiv(H, C);
  const int JU = Hs <= 32 ? 1 : 2;
  if (Hs > 64) {                            // very wide layers: more CTAs per cluster is not portable;
    best.C = 0;                             // handled by the caller as an error for now
    return best;
  }
  const int bts[3] = {8, 16, 32};
  bool found = false;
  for (int pass = 0; pass < 2 && !found; ++pass) {
    const bool wsmem = pass == 0;
    // smallest tile whose grid still fits in one wave, else the largest tile that fits in smem
    int pick = -1;
    for (int i = 0; i < 3; ++i) {
      const int BT = bts[i];
      if (BT * JU > 32) continue;
      const size_t s = backward ? bwd_smem(G, BT, JU, H, Hs, C, wsmem) : fwd_smem(G, BT, JU, H, Hs, wsmem);
      if (s > limit) continue;
      pick = i;
      if (cdiv(B, BT) * C <= n_sm) break;
    }
    if (pick >= 0) {
      best.C = C; best.Hs = Hs; best.BT = bts[pick]; best.JU = JU; best.wsmem = wsmem;
      best.smem = backward ? bwd_smem(G, best.BT, JU, H, Hs, C, wsmem) : fwd_smem(G, best.BT, JU, H, Hs, wsmem);
      found = true;
    }
  }
  if (!found) best.C = 0;
  return best;
}

template <typename Kern>
int launch_cluster(sbr_model* m, Kern kern, const Plan& p, int n_tiles, const RnnArgs& args) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
  if (e != cudaSuccess) {
    sbr_set_error(m, SBR_E_CUDA, "cudaFuncSetAttribute(smem=%zu): %s", p.smem, cudaGetErrorString(e));
    return SBR_E_CUDA;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(p.C * n_tiles, 1, 1);
  cfg.blockDim = dim3(NT, 1, 1);
  cfg.dynamicSmemBytes = p.smem;
  cfg.stream = m->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, kern, args);
  if (e != cudaSuccess) {
    sbr_set_error(m, SBR_E_CUDA, "cluster launch (C=%d, BT=%d, smem=%zu) failed: %s", p.C, p.BT, p.smem,
                  cudaGetErrorString(e));
    return SBR_E_CUDA;
  }
  m->launches++;
  m->scan_launches++;
  return 0;
}

// The FFMA scan variants <G, BT, JU, WSMEM> per direction: exactly the ones make_plan returns for some layer (H <= 512)
// and batch.  JU = 1 layers (Hs <= 32) always hold their weight slice in shared memory, so no JU = 1 global-weight
// variant is compiled; tests/test_scan_dispatch.py checks these lists against the planner.
template <int G, bool BWD>
int dispatch(sbr_model* m, const Plan& p, int n_tiles, const RnnArgs& a) {
#define SBR_FFMA_FWD(G_, BT_, JU_, WS_)                                                      \
  if constexpr (!BWD && G == G_)                                                             \
    if (p.BT == BT_ && p.JU == JU_ && p.wsmem == WS_)                                        \
      return launch_cluster(m, rnn_fwd_kernel<G_, BT_, JU_, WS_>, p, n_tiles, a);
#define SBR_FFMA_BWD(G_, BT_, JU_, WS_)                                                      \
  if constexpr (BWD && G == G_)                                                              \
    if (p.BT == BT_ && p.JU == JU_ && p.wsmem == WS_)                                        \
      return launch_cluster(m, rnn_bwd_kernel<G_, BT_, JU_, WS_>, p, n_tiles, a);
  // LSTM: the 16-row JU = 2 forward tile never fits next to a resident weight slice
  SBR_FFMA_FWD(4, 8, 1, true) SBR_FFMA_FWD(4, 16, 1, true) SBR_FFMA_FWD(4, 32, 1, true)
  SBR_FFMA_FWD(4, 8, 2, true) SBR_FFMA_FWD(4, 8, 2, false) SBR_FFMA_FWD(4, 16, 2, false)
  SBR_FFMA_BWD(4, 8, 1, true) SBR_FFMA_BWD(4, 16, 1, true) SBR_FFMA_BWD(4, 32, 1, true)
  SBR_FFMA_BWD(4, 8, 2, true) SBR_FFMA_BWD(4, 16, 2, true) SBR_FFMA_BWD(4, 8, 2, false) SBR_FFMA_BWD(4, 16, 2, false)
  SBR_FFMA_FWD(3, 8, 1, true) SBR_FFMA_FWD(3, 16, 1, true) SBR_FFMA_FWD(3, 32, 1, true)
  SBR_FFMA_FWD(3, 8, 2, true) SBR_FFMA_FWD(3, 16, 2, true) SBR_FFMA_FWD(3, 8, 2, false) SBR_FFMA_FWD(3, 16, 2, false)
  SBR_FFMA_BWD(3, 8, 1, true) SBR_FFMA_BWD(3, 16, 1, true) SBR_FFMA_BWD(3, 32, 1, true)
  SBR_FFMA_BWD(3, 8, 2, true) SBR_FFMA_BWD(3, 16, 2, true) SBR_FFMA_BWD(3, 8, 2, false) SBR_FFMA_BWD(3, 16, 2, false)
  // Vanilla: the weight slice of H <= 512 always fits in shared memory
  SBR_FFMA_FWD(1, 8, 1, true) SBR_FFMA_FWD(1, 16, 1, true) SBR_FFMA_FWD(1, 32, 1, true)
  SBR_FFMA_FWD(1, 8, 2, true) SBR_FFMA_FWD(1, 16, 2, true)
  SBR_FFMA_BWD(1, 8, 1, true) SBR_FFMA_BWD(1, 16, 1, true) SBR_FFMA_BWD(1, 32, 1, true)
  SBR_FFMA_BWD(1, 8, 2, true) SBR_FFMA_BWD(1, 16, 2, true)
#undef SBR_FFMA_FWD
#undef SBR_FFMA_BWD
  sbr_set_error(m, SBR_E_ARG, "no recurrent kernel for G=%d BT=%d JU=%d wsmem=%d", G, p.BT, p.JU, (int)p.wsmem);
  return SBR_E_ARG;
}

}  // namespace

int launch_rnn_forward(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max, float* h_last) {
  {
    const int rc = launch_rnn_forward_tc(m, L, len, B, t_max, h_last);   // tcgen05 3xTF32 scan when it applies
    if (rc <= 0) return rc;
  }
  // larger hidden sizes: the persistent tensor-core scan (tc_scan.cu), else one tensor-core step kernel per time step
  if (persistent_scan_applies(m, L.G, L.H)) {
    const int rc = launch_rnn_forward_persistent(m, L, len, B, t_max, h_last);
    if (rc <= 0) return rc;
  }
  if (step_scan_applies(m, L.G, L.H)) return launch_rnn_forward_steps(m, L, len, B, t_max, h_last);
  const Plan p = make_plan(m->n_sm, L.G, L.H, B, false);
  if (p.C == 0) {
    sbr_set_error(m, SBR_E_ARG, "hidden size %d is not supported by the cluster scan (max 512)", L.H);
    return SBR_E_ARG;
  }
  RnnArgs a{};
  a.Xg = L.Xg; a.W_hid = m->params + L.W_hid; a.W_hidT = nullptr;
  a.peep = m->params + L.peep; a.h_init = m->params + L.h_init; a.c_init = m->params + L.c_init;
  a.len = len; a.hs = L.hs; a.cs = L.cs; a.act = L.act; a.h_last = h_last;
  a.clip = m->cfg.grad_clip; a.relu = L.relu; a.B = B; a.H = L.H; a.Hs = p.Hs; a.t_max = t_max;
  const int n_tiles = cdiv(B, p.BT);
  if (L.G == 4) return dispatch<4, false>(m, p, n_tiles, a);
  if (L.G == 3) return dispatch<3, false>(m, p, n_tiles, a);
  return dispatch<1, false>(m, p, n_tiles, a);
}

int launch_rnn_backward(sbr_model* m, const LayerDesc& L, const int32_t* len, int B, int t_max,
                        const float* dh_last) {
  m->bwd_did_bias = false;
  if (!m->disable_tc_bwd) {
    const int rc = launch_rnn_backward_tc(m, L, len, B, t_max, dh_last);   // tcgen05 3xTF32 BPTT when it applies
    if (rc <= 0) { m->bwd_did_bias = true; return rc; }
  }
  if (!tc_scan_applies(L.G, L.H)) {
    if (persistent_scan_applies(m, L.G, L.H)) {
      const int rc = launch_rnn_backward_persistent(m, L, len, B, t_max, dh_last);
      if (rc <= 0) { m->bwd_did_bias = true; return rc; }
    }
    if (step_scan_applies(m, L.G, L.H)) return launch_rnn_backward_steps(m, L, len, B, t_max, dh_last);
  }
  const Plan p = make_plan(m->n_sm, L.G, L.H, B, true);
  if (p.C == 0) {
    sbr_set_error(m, SBR_E_ARG, "hidden size %d is not supported by the cluster scan (max 512)", L.H);
    return SBR_E_ARG;
  }
  // k-contiguous copy of W_hid for the split-K contraction
  int rc = launch_transpose(m, m->params + L.W_hid, L.H, L.G * L.H, L.G * L.H, m->WhidT);
  if (rc) return rc;
  RnnArgs a{};
  a.W_hid = m->params + L.W_hid; a.W_hidT = m->WhidT;
  a.peep = m->params + L.peep; a.len = len; a.hs = L.hs; a.cs = L.cs; a.act = L.act;
  a.dh_last = dh_last; a.dhs = dh_last ? nullptr : L.dhs; a.dXg = L.dXg; a.dac = L.dac;
  a.g_peep = m->grads + L.peep; a.g_h_init = m->grads + L.h_init; a.g_c_init = m->grads + L.c_init;
  a.clip = m->cfg.grad_clip; a.relu = L.relu; a.B = B; a.H = L.H; a.Hs = p.Hs; a.t_max = t_max;
  const int n_tiles = cdiv(B, p.BT);
  if (L.G == 4) return dispatch<4, true>(m, p, n_tiles, a);
  if (L.G == 3) return dispatch<3, true>(m, p, n_tiles, a);
  return dispatch<1, true>(m, p, n_tiles, a);
}

// Which scan variant launch_rnn_forward / launch_rnn_backward run for one layer and batch: the same decisions in the
// same order (tc_plan + plan_tiles, the persistent slicing, step_scan_applies, make_plan).
extern "C" SBR_API int sbr_plan_layer_scan(const sbr_model* m, int cell, int H, int B, const int32_t* lens, int t_max,
                                           int backward, int n_sm, const int32_t* tc_slots, int splitk_slots,
                                           sbr_scan_plan* out) {
  const int G = cell == SBR_CELL_LSTM ? 4 : cell == SBR_CELL_GRU ? 3 : cell == SBR_CELL_VANILLA ? 1 : 0;
  if (!out || G == 0 || H < 1 || B < 1 || t_max < 1) return SBR_E_ARG;
  if (!m && (n_sm < 1 || !tc_slots)) return SBR_E_ARG;
  const ScanSwitches sw = m ? scan_switches(m) : scan_switches_from_env();
  if (sw.multicast) return SBR_E_ARG;     // the multicast forward sizes its launches from another occupancy query
  if (m) {
    n_sm = m->n_sm;
    if (cudaSetDevice(m->dev) != cudaSuccess) return SBR_E_CUDA;
  }
  *out = sbr_scan_plan{};
  out->G = G;
  const TcShape tc = tc_scan_shape(G, H);
  if (backward ? (tc.bwd_ok && !sw.disable_tc_bwd) : tc.ok) {
    const int slots = m ? tc_scan_slots(G, H) : tc_slots[tc.C == 8 ? 3 : tc.C == 4 ? 2 : tc.C == 2 ? 1 : 0];
    out->family = SBR_SCAN_TC_CLUSTER;
    out->C = tc.C; out->Hs = tc.Hs; out->MT = backward ? tc.MT : 0;
    tc_scan_schedule(lens, B, t_max, slots, backward != 0, &out->BT, &out->launches);
    return 0;
  }
  // the backward of a tcgen05-shaped layer under SBR_DISABLE_TC_BWD goes straight to the FFMA scan
  const bool others = !backward || !tc.bwd_ok;
  if (others && persistent_scan_applies(sw, H)) {
    const PersistentSlicing sl = backward ? persistent_bwd_slicing(n_sm, H, B, sw.splitk,
                                                                   sw.splitk ? (m ? persistent_splitk_slots() : splitk_slots) : 0)
                                          : persistent_fwd_slicing(n_sm, H, B);
    out->family = SBR_SCAN_PERSISTENT;
    out->BT = sl.tile_rows; out->splitk = sl.splitk ? 1 : 0;
    out->Hs = sl.owner; out->C = cdiv(H, sl.owner);
    out->tiles_per_launch = sl.tiles_per_launch;
    out->launches = cdiv(sl.n_tiles, sl.tiles_per_launch);
    return 0;
  }
  if (others && step_scan_applies(sw, H)) {
    out->family = SBR_SCAN_STEP;
    out->C = 1; out->Hs = H;
    out->launches = t_max + (backward ? 1 : 0);   // one per time step (the backward adds the initial-state step)
    return 0;
  }
  const Plan p = make_plan(n_sm, G, H, B, backward != 0);
  if (p.C == 0) return SBR_E_ARG;
  out->family = SBR_SCAN_FFMA;
  out->C = p.C; out->Hs = p.Hs; out->BT = p.BT; out->JU = p.JU; out->wsmem = p.wsmem ? 1 : 0;
  out->launches = 1;
  return 0;
}
