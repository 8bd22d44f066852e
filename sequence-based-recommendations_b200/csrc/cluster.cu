// cluster.cu -- the cluster branch of RNNCluster and its test paths (reference neural_networks/rnn_cluster.py).
//
//   training   q = h Wc (+ noise), P = softmax(s q)                          rnn_cluster.py:235-239
//              M = act(s R[cells_c])  softmax | softmax + sigmoid | sigmoid  :241-248
//              dq = s P (dP - <dP, P>) ; dR[cells_c] += s act'(dM)          (backward of the above; no gradient to h)
//   validation hard[:, c] = softmax(100 R)[:, c] | clip(softmax + sigmoid) | sigmoid(100 R)[:, c] ; c = argmax(h Wc)
//              score2 = score1 * hard[:, c], n_used = sum hard[:, c]         :275-282, :327-355
//   prepare    item CSR of the hard clusters, ascending ids per cluster      :461-487
//   top-k      raw scores of the selected cluster's items, -inf exclusion    :293-305
//
// C (clusters) is small next to everything else: one warp owns one row of length C.  The GEMM-shaped products
// (h Wc, P M^T, dS M, dS^T P, h^T dq, and the per-cluster scoring) run through launch_gemm in model.cu.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int WPB = 8;   // warps per block of the warp-per-row kernels

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float sigm(float x) { return 1.f / (1.f + expf(-x)); }

// first arg-max of x[0:C] over one warp (np.argmax / theano argmax: the lowest index among equal maxima)
__device__ __forceinline__ int warp_argmax(const float* x, int C) {
  const int lane = threadIdx.x & 31;
  float best = -CUDART_INF_F;
  int bi = 0x7fffffff;
  for (int c = lane; c < C; c += 32) {
    const float v = x[c];
    if (v > best || (v == best && c < bi)) { best = v; bi = c; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
  }
  return bi == 0x7fffffff ? 0 : bi;
}

// P[b, :] = softmax(s (q[b, :] + noise[b, :]))
__global__ void __launch_bounds__(WPB * 32) cluster_select_kernel(const float* __restrict__ q, const float* __restrict__ noise,
                                                                   int B, int C, float s, float* __restrict__ P) {
  const int b = blockIdx.x * WPB + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* qr = q + (int64_t)b * C;
  const float* nr = noise ? noise + (int64_t)b * C : nullptr;
  float mx = -CUDART_INF_F;
  for (int c = lane; c < C; c += 32) mx = fmaxf(mx, s * (qr[c] + (nr ? nr[c] : 0.f)));
  mx = wmax(mx);
  float sum = 0.f;
  for (int c = lane; c < C; c += 32) sum += expf(s * (qr[c] + (nr ? nr[c] : 0.f)) - mx);
  const float inv = 1.f / wsum(sum);
  for (int c = lane; c < C; c += 32) P[(int64_t)b * C + c] = expf(s * (qr[c] + (nr ? nr[c] : 0.f)) - mx) * inv;
}

// softmax over the C entries of one membership row, scaled by s: returns max and 1/sum for the lane loop
__device__ __forceinline__ void row_softmax_stats(const float* r, int C, float s, float& mx, float& inv) {
  const int lane = threadIdx.x & 31;
  float m = -CUDART_INF_F;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, s * r[c]);
  m = wmax(m);
  float sum = 0.f;
  for (int c = lane; c < C; c += 32) sum += expf(s * r[c] - m);
  mx = m;
  inv = 1.f / wsum(sum);
}

// M[j, :] = act(s R[cells[j], :])
__global__ void __launch_bounds__(WPB * 32) cluster_members_kernel(const float* __restrict__ R, const int32_t* __restrict__ cells,
                                                                    int n, int C, int type, float s, float* __restrict__ M) {
  const int j = blockIdx.x * WPB + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= n) return;
  const float* r = R + (int64_t)cells[j] * C;
  float mx = 0.f, inv = 0.f;
  if (type != SBR_CLUSTER_SIGMOID) row_softmax_stats(r, C, s, mx, inv);
  for (int c = lane; c < C; c += 32) {
    const float z = s * r[c];
    float v = 0.f;
    if (type != SBR_CLUSTER_SIGMOID) v += expf(z - mx) * inv;
    if (type != SBR_CLUSTER_SOFTMAX) v += sigm(z);
    M[(int64_t)j * C + c] = v;
  }
}

// dq[b, :] = s P (dP - <dP, P>)   (softmax of s q; the noise is an additive constant)
__global__ void __launch_bounds__(WPB * 32) cluster_dq_kernel(const float* __restrict__ P, const float* __restrict__ dP, int B, int C,
                                                               float s, float* __restrict__ dq) {
  const int b = blockIdx.x * WPB + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* p = P + (int64_t)b * C;
  const float* g = dP + (int64_t)b * C;
  float dot = 0.f;
  for (int c = lane; c < C; c += 32) dot += p[c] * g[c];
  dot = wsum(dot);
  for (int c = lane; c < C; c += 32) dq[(int64_t)b * C + c] = s * p[c] * (g[c] - dot);
}

// gR[cells[j], :] += d act(s R[cells[j], :]) / dR  . dM[j, :]   -- duplicate cells accumulate
__global__ void __launch_bounds__(WPB * 32) cluster_dR_kernel(const float* __restrict__ R, const int32_t* __restrict__ cells, int n,
                                                               int C, int type, float s, const float* __restrict__ dM,
                                                               float* __restrict__ gR) {
  const int j = blockIdx.x * WPB + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= n) return;
  const int id = cells[j];
  const float* r = R + (int64_t)id * C;
  const float* g = dM + (int64_t)j * C;
  float mx = 0.f, inv = 0.f, dot = 0.f;
  if (type != SBR_CLUSTER_SIGMOID) {
    row_softmax_stats(r, C, s, mx, inv);
    for (int c = lane; c < C; c += 32) dot += expf(s * r[c] - mx) * inv * g[c];
    dot = wsum(dot);
  }
  for (int c = lane; c < C; c += 32) {
    const float z = s * r[c];
    float d = 0.f;
    if (type != SBR_CLUSTER_SIGMOID) d += expf(z - mx) * inv * (g[c] - dot);
    if (type != SBR_CLUSTER_SOFTMAX) { const float sg = sigm(z); d += sg * (1.f - sg) * g[c]; }
    atomicAdd(gR + (int64_t)id * C + c, s * d);
  }
}

__global__ void __launch_bounds__(WPB * 32) cluster_argmax_kernel(const float* __restrict__ q, int B, int C, int32_t* __restrict__ sel) {
  const int b = blockIdx.x * WPB + (threadIdx.x >> 5);
  if (b >= B) return;
  const int c = warp_argmax(q + (int64_t)b * C, C);
  if ((threadIdx.x & 31) == 0) sel[b] = c;
}

// lse[n] = logsumexp_c(100 R[n, c])  (row-wise lasagne softmax of 100 R, rnn_cluster.py:277,280)
__global__ void __launch_bounds__(WPB * 32) cluster_lse100_kernel(const float* __restrict__ R, int N, int C, float* __restrict__ lse) {
  const int n = blockIdx.x * WPB + (threadIdx.x >> 5);
  if (n >= N) return;
  float mx, inv;
  row_softmax_stats(R + (int64_t)n * C, C, 100.f, mx, inv);
  if ((threadIdx.x & 31) == 0) lse[n] = mx - logf(inv);
}

// one block per row: c = argmax q[b, :]; scores2 = scores * hard[:, c]; n_used = sum_n hard[n, c]
__global__ void __launch_bounds__(256) cluster_hard_kernel(const float* __restrict__ scores, int ld, const float* __restrict__ q,
                                                           const float* __restrict__ R, const float* __restrict__ lse, int N, int C,
                                                           int type, float* __restrict__ scores2, int32_t* __restrict__ sel,
                                                           float* __restrict__ n_used) {
  __shared__ int sc;
  __shared__ float sh[8];
  const int b = blockIdx.x;
  if (threadIdx.x < 32) {
    const int c = warp_argmax(q + (int64_t)b * C, C);
    if (threadIdx.x == 0) { sc = c; sel[b] = c; }
  }
  __syncthreads();
  const int c = sc;
  const float* row = scores + (int64_t)b * ld;
  float* out = scores2 + (int64_t)b * ld;
  float used = 0.f;
  for (int n = threadIdx.x; n < N; n += 256) {
    const float z = 100.f * R[(int64_t)n * C + c];
    float h;
    if (type == SBR_CLUSTER_SOFTMAX) h = expf(z - lse[n]);
    else if (type == SBR_CLUSTER_MIX) h = fminf(fmaxf(expf(z - lse[n]) + sigm(z), 0.f), 1.f);
    else h = sigm(z);
    out[n] = row[n] * h;
    used += h;
  }
  used = wsum(used);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = used;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += sh[i];
    n_used[b] = t;
  }
}

// ---- item CSR of the hard clusters (prepare_tests) ----------------------------------------------------------------
constexpr int CHUNK = 256;   // items per block of the count / fill passes

// fb[n] = -1 when row n has a positive entry, else the first arg-max of the row (rnn_cluster.py:468-480)
__global__ void __launch_bounds__(WPB * 32) cluster_fallback_kernel(const float* __restrict__ R, int N, int C, int32_t* __restrict__ fb) {
  const int n = blockIdx.x * WPB + (threadIdx.x >> 5);
  if (n >= N) return;
  const float* r = R + (int64_t)n * C;
  bool pos = false;
  for (int c = threadIdx.x & 31; c < C; c += 32) pos |= r[c] > 0.f;
  pos = __any_sync(0xffffffffu, pos);
  const int am = warp_argmax(r, C);
  if ((threadIdx.x & 31) == 0) fb[n] = pos ? -1 : am;
}

__device__ __forceinline__ bool is_member(const float* R, const int32_t* fb, int n, int N, int C, int j) {
  if (n >= N) return false;
  return fb[n] < 0 ? R[(int64_t)n * C + j] > 0.f : fb[n] == j;
}

__global__ void __launch_bounds__(CHUNK) cluster_count_kernel(const float* __restrict__ R, const int32_t* __restrict__ fb, int N, int C,
                                                              int32_t* __restrict__ cnt) {
  const int n = blockIdx.x * CHUNK + threadIdx.x;
  for (int j = 0; j < C; ++j) {
    const int k = __syncthreads_count(is_member(R, fb, n, N, C, j));
    if (threadIdx.x == 0) cnt[(int64_t)blockIdx.x * C + j] = k;
  }
}

// per cluster: exclusive scan of the chunk counts (in place); off = exclusive scan of the cluster sizes
__global__ void cluster_scan_kernel(int32_t* __restrict__ cnt, int chunks, int C, int32_t* __restrict__ off) {
  for (int j = threadIdx.x; j < C; j += blockDim.x) {
    int acc = 0;
    for (int k = 0; k < chunks; ++k) {
      const int v = cnt[(int64_t)k * C + j];
      cnt[(int64_t)k * C + j] = acc;
      acc += v;
    }
    off[j + 1] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    off[0] = 0;
    for (int j = 0; j < C; ++j) off[j + 1] += off[j];
  }
}

// items of cluster j in ascending id: block-ordered chunks, rank inside the chunk by a ballot prefix count
__global__ void __launch_bounds__(CHUNK) cluster_fill_kernel(const float* __restrict__ R, const int32_t* __restrict__ fb, int N, int C,
                                                             const int32_t* __restrict__ cnt, const int32_t* __restrict__ off,
                                                             int32_t* __restrict__ items) {
  __shared__ int wc[CHUNK / 32];
  const int n = blockIdx.x * CHUNK + threadIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int j = 0; j < C; ++j) {
    const bool f = is_member(R, fb, n, N, C, j);
    const unsigned bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) wc[w] = __popc(bal);
    __syncthreads();
    int base = 0;
    for (int i = 0; i < w; ++i) base += wc[i];
    if (f) items[off[j] + cnt[(int64_t)blockIdx.x * C + j] + base + __popc(bal & ((1u << lane) - 1u))] = n;
    __syncthreads();
  }
}

// ---- cluster-restricted top-k -------------------------------------------------------------------------------------
// One block per row in cluster-grouped order (perm[r] = original row).  scores[r, :n_c] hold h W[:, items]; add the
// bias, set excluded ids to -inf (binary search in the ascending item list), then k rounds of arg-max; a picked entry
// becomes NaN so that -inf entries can still be picked once each.  Ties resolve to the lowest id.
__global__ void __launch_bounds__(256) cluster_row_topk_kernel(float* __restrict__ scores, int ld, const int32_t* __restrict__ perm,
                                                               const int32_t* __restrict__ sel, const int32_t* __restrict__ off,
                                                               const int32_t* __restrict__ items, const float* __restrict__ bias,
                                                               const int32_t* __restrict__ eoff, const int32_t* __restrict__ eids,
                                                               int k, int32_t* __restrict__ ids_out) {
  __shared__ float sv[8];
  __shared__ int si[8];
  const int r = blockIdx.x, b = perm[r], c = sel[b];
  const int lo = off[c], nc = off[c + 1] - lo;
  const int32_t* it = items + lo;
  float* row = scores + (int64_t)r * ld;
  for (int i = threadIdx.x; i < nc; i += 256) row[i] += bias[it[i]];
  __syncthreads();
  if (eoff) {
    for (int e = eoff[b] + threadIdx.x; e < eoff[b + 1]; e += 256) {
      const int id = eids[e];
      int a = 0, z = nc;   // first position with it[pos] >= id
      while (a < z) { const int mid = (a + z) >> 1; if (it[mid] < id) a = mid + 1; else z = mid; }
      if (a < nc && it[a] == id) row[a] = -CUDART_INF_F;
    }
    __syncthreads();
  }
  const int keff = min(k, nc);
  for (int q = 0; q < k; ++q) {
    if (q >= keff) {
      if (threadIdx.x == 0) ids_out[(int64_t)b * k + q] = -1;
      continue;
    }
    float best = -CUDART_INF_F;
    int bi = 0x7fffffff;
    for (int i = threadIdx.x; i < nc; i += 256) {
      const float v = row[i];
      if (v == v && (v > best || (v == best && i < bi))) { best = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 1; i < 8; ++i)
        if (sv[i] > best || (sv[i] == best && si[i] < bi)) { best = sv[i]; bi = si[i]; }
      ids_out[(int64_t)b * k + q] = it[bi];
      row[bi] = CUDART_NAN_F;
    }
    __syncthreads();
  }
}

inline int warp_rows_grid(int n) { return cdiv(n, WPB); }

}  // namespace

int launch_cluster_select(sbr_model* m, const float* q, const float* noise, int B, int C, float scale, float* P) {
  if (B == 0) return 0;
  cluster_select_kernel<<<warp_rows_grid(B), WPB * 32, 0, m->stream>>>(q, noise, B, C, scale, P);
  KERNEL_CHECK(m);
  return 0;
}

int launch_cluster_members(sbr_model* m, const float* R, const int32_t* cells, int n, int C, int type, float scale, float* M) {
  cluster_members_kernel<<<warp_rows_grid(n), WPB * 32, 0, m->stream>>>(R, cells, n, C, type, scale, M);
  KERNEL_CHECK(m);
  return 0;
}

int launch_cluster_dq(sbr_model* m, const float* P, const float* dP, int B, int C, float scale, float* dq) {
  if (B == 0) return 0;
  cluster_dq_kernel<<<warp_rows_grid(B), WPB * 32, 0, m->stream>>>(P, dP, B, C, scale, dq);
  KERNEL_CHECK(m);
  return 0;
}

int launch_cluster_dR(sbr_model* m, const float* R, const int32_t* cells, int n, int C, int type, float scale,
                      const float* dM, float* gR) {
  cluster_dR_kernel<<<warp_rows_grid(n), WPB * 32, 0, m->stream>>>(R, cells, n, C, type, scale, dM, gR);
  KERNEL_CHECK(m);
  return 0;
}

int launch_cluster_argmax(sbr_model* m, const float* q, int B, int C, int32_t* sel) {
  if (B == 0) return 0;
  cluster_argmax_kernel<<<warp_rows_grid(B), WPB * 32, 0, m->stream>>>(q, B, C, sel);
  KERNEL_CHECK(m);
  return 0;
}

int launch_cluster_hard(sbr_model* m, const float* scores, int ld, const float* q, const float* R, int B, int N, int C,
                        int type, float* scores2, int32_t* sel, float* n_used) {
  if (B == 0) return 0;
  if (type != SBR_CLUSTER_SIGMOID) {
    cluster_lse100_kernel<<<warp_rows_grid(N), WPB * 32, 0, m->stream>>>(R, N, C, m->clse);
    KERNEL_CHECK(m);
  }
  cluster_hard_kernel<<<B, 256, 0, m->stream>>>(scores, ld, q, R, m->clse, N, C, type, scores2, sel, n_used);
  KERNEL_CHECK(m);
  return 0;
}

int launch_cluster_csr(sbr_model* m, const float* R, int N, int C) {
  const int chunks = cdiv(N, CHUNK);
  cluster_fallback_kernel<<<warp_rows_grid(N), WPB * 32, 0, m->stream>>>(R, N, C, m->cl_fb);
  KERNEL_CHECK(m);
  cluster_count_kernel<<<chunks, CHUNK, 0, m->stream>>>(R, m->cl_fb, N, C, m->cl_cnt);
  KERNEL_CHECK(m);
  cluster_scan_kernel<<<1, 256, 0, m->stream>>>(m->cl_cnt, chunks, C, m->cl_off);
  KERNEL_CHECK(m);
  return 0;
}

// second half of the CSR build, once the caller knows the total (m->cl_items sized)
int launch_cluster_fill(sbr_model* m, const float* R, int N, int C) {
  cluster_fill_kernel<<<cdiv(N, CHUNK), CHUNK, 0, m->stream>>>(R, m->cl_fb, N, C, m->cl_cnt, m->cl_off, m->cl_items);
  KERNEL_CHECK(m);
  return 0;
}

int launch_cluster_row_topk(sbr_model* m, float* scores, int ld, int B, const int32_t* perm, const int32_t* sel,
                            const float* bias, const int32_t* excl_off, const int32_t* excl_ids, int k, int32_t* ids_out) {
  if (B == 0) return 0;
  cluster_row_topk_kernel<<<B, 256, 0, m->stream>>>(scores, ld, perm, sel, m->cl_off, m->cl_items, bias, excl_off, excl_ids, k,
                                                    ids_out);
  KERNEL_CHECK(m);
  return 0;
}
