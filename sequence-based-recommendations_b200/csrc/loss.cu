// loss.cu -- stage 3 epilogues: the row-wise losses that follow the catalog projection.
//
//   CCE      softmax + categorical_crossentropy / pop, mean            rnn_one_hot.py:65-71
//   bias reg L2 (reg>0) / L1 (reg<0) on the OUTPUT BIAS only           rnn_one_hot.py:73-77
//   sampling BPR / BPRI / TOP1 / Blackout on [B, n_all+S] scores       rnn_sampling.py:68-91,137
//   margin   hinge / logit / logsig with per-item targets and weights   rnn_margin.py:61-68,109
//   margin inputs rebuilt from ragged lists                             rnn_margin.py:121-149
//   test     exclude + sorted top-k                                     rnn_base.py:196-213,154-159
//
// Every loss kernel turns the score matrix into its own gradient IN PLACE (one read + one write of
// [B, C]) and emits one already-scaled loss term per row; rows are reduced by a single CTA in a
// fixed order so that the cost does not depend on scheduling.  One CTA per row, 256 threads,
// 128-bit accesses are not needed here: the row lives in L2 (it was just written by the GEMM).
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int LT = 256;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ float block_sum(float v, float* sh) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  for (int i = 0; i < (blockDim.x >> 5); ++i) r += sh[i];
  return r;
}
__device__ float block_max(float v, float* sh) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = -CUDART_INF_F;
  for (int i = 0; i < (blockDim.x >> 5); ++i) r = fmaxf(r, sh[i]);
  return r;
}
__device__ __forceinline__ float sigm(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float softplus(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }

// z = logits + bias ; lse ; loss ; dz = (softmax - onehot) * scale     (in place)
__global__ void __launch_bounds__(LT) cce_kernel(float* __restrict__ logits, int ld, const float* __restrict__ bias,
                                                  const int32_t* __restrict__ Y, const float* __restrict__ pop, int N,
                                                  float inv_gb, float* __restrict__ row_loss) {
  __shared__ float sh[LT / 32];
  const int b = blockIdx.x;
  float* row = logits + (int64_t)b * ld;
  float mx = -CUDART_INF_F;
  for (int n = threadIdx.x; n < N; n += LT) {
    const float z = row[n] + bias[n];
    row[n] = z;
    mx = fmaxf(mx, z);
  }
  mx = block_max(mx, sh);
  float s = 0.f;
  for (int n = threadIdx.x; n < N; n += LT) s += expf(row[n] - mx);
  s = block_sum(s, sh);
  const float lse = mx + logf(s);
  const int y = Y[b];
  const float scale = inv_gb / pop[b];
  if (threadIdx.x == 0) row_loss[b] = -(row[y] - lse) * scale;
  __syncthreads();
  for (int n = threadIdx.x; n < N; n += LT) {
    float p = expf(row[n] - lse);
    if (n == y) p -= 1.f;
    row[n] = p * scale;
  }
}

__global__ void __launch_bounds__(LT) softmax_rows_kernel(float* __restrict__ logits, int ld,
                                                           const float* __restrict__ bias, int N) {
  __shared__ float sh[LT / 32];
  float* row = logits + (int64_t)blockIdx.x * ld;
  float mx = -CUDART_INF_F;
  for (int n = threadIdx.x; n < N; n += LT) {
    const float z = row[n] + (bias ? bias[n] : 0.f);
    row[n] = z;
    mx = fmaxf(mx, z);
  }
  mx = block_max(mx, sh);
  float s = 0.f;
  for (int n = threadIdx.x; n < N; n += LT) {
    const float e = expf(row[n] - mx);
    row[n] = e;
    s += e;
  }
  s = block_sum(s, sh);
  const float inv = 1.f / s;
  for (int n = threadIdx.x; n < N; n += LT) row[n] *= inv;
}

__global__ void add_bias_rows_kernel(float* __restrict__ logits, int ld, const float* __restrict__ bias, int B, int N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * N) return;
  const int b = (int)(i / N), n = (int)(i % N);
  logits[(int64_t)b * ld + n] += bias[n];
}

// Sampling losses.  Columns [0, n_all) are the targets of the whole global batch, [n_all, n_all+S)
// the shared negative samples; the positive of local row b is column row_offset + b.  The cluster model
// (rnn_cluster.py:151-180) passes pop = NULL (unit weights), bias_cells = NULL for its cluster scores, and three more
// codes: SBR_LK_SCCE (-log softmax over the B+S columns, no negative term), SBR_LK_BPRELU (leaky_rectify(d + 0.5),
// leakiness 0.01, Theano slope 0.505 at 0) and SBR_LK_LIN (sum of the negatives minus the positive, not a mean).
__global__ void __launch_bounds__(LT) sampling_loss_kernel(int loss, int tanh_out, float* __restrict__ A, int ld,
                                                            const float* __restrict__ bias_cells,
                                                            const float* __restrict__ pop, int n_all, int row_offset,
                                                            int S, float inv_gb, float* __restrict__ row_loss) {
  __shared__ float sh[LT / 32];
  const int b = blockIdx.x;
  const int Ccols = n_all + S;
  float* row = A + (int64_t)b * ld;
  const int pc = row_offset + b;
  const float scale = pop ? inv_gb / pop[b] : inv_gb;
  if (loss == SBR_LOSS_BLACKOUT || loss == SBR_LK_SCCE) {
    const bool negs = loss == SBR_LOSS_BLACKOUT;
    float mx = -CUDART_INF_F;
    for (int n = threadIdx.x; n < Ccols; n += LT) {
      const float z = row[n] + (bias_cells ? bias_cells[n] : 0.f);
      row[n] = z;
      mx = fmaxf(mx, z);
    }
    mx = block_max(mx, sh);
    float s = 0.f;
    for (int n = threadIdx.x; n < Ccols; n += LT) s += expf(row[n] - mx);
    s = block_sum(s, sh);
    const float inv = 1.f / s;
    // loss = -log P_pos - sum_s log(1 - P_s) ;  g = dL/dP ;  dA_j = P_j (g_j - sum_k g_k P_k)
    float lpart = 0.f, gp = 0.f;
    for (int n = threadIdx.x; n < Ccols; n += LT) {
      const float p = expf(row[n] - mx) * inv;
      if (n == pc) { lpart += -logf(p); gp += -1.f; }           // g * p = -1
      if (negs && n >= n_all) { lpart += -logf(1.f - p); gp += p / (1.f - p); }
    }
    const float l = block_sum(lpart, sh);
    const float gdot = block_sum(gp, sh);
    if (threadIdx.x == 0) row_loss[b] = l * scale;
    __syncthreads();
    for (int n = threadIdx.x; n < Ccols; n += LT) {
      const float p = expf(row[n] - mx) * inv;
      float g = 0.f;
      if (n == pc) g += -1.f / p;
      if (negs && n >= n_all) g += 1.f / (1.f - p);
      row[n] = p * (g - gdot) * scale;
    }
    return;
  }
  // BPR / BPRI / TOP1 (and the cluster model's BPRelu / lin)
  float posv = row[pc] + (bias_cells ? bias_cells[pc] : 0.f);
  if (tanh_out) posv = tanhf(posv);
  __syncthreads();
  float lpart = 0.f, gsum = 0.f;
  const float invS = 1.f / (float)S;
  for (int n = threadIdx.x; n < Ccols; n += LT) {
    float out = 0.f;
    if (n >= n_all) {
      float v = row[n] + (bias_cells ? bias_cells[n] : 0.f);
      if (tanh_out) v = tanhf(v);
      const float d = v - posv;
      const float sd = sigm(d);
      float gd, gn = 0.f;
      if (loss == SBR_LOSS_BPR) { lpart += softplus(d) * invS; gd = sd * invS; }
      else if (loss == SBR_LOSS_BPRI) { lpart += (fminf(d, 0.f) - log1pf(expf(-fabsf(d)))) * invS; gd = (1.f - sd) * invS; }
      else if (loss == SBR_LK_BPRELU) {
        // Theano relu(x, a) = 0.5 (1 + a) x + 0.5 (1 - a) |x|: slope 1 / 0.505 / 0.01 for x > 0 / = 0 / < 0
        const float x = d + 0.5f;
        lpart += (x > 0.f ? x : 0.01f * x) * invS;
        gd = (x > 0.f ? 1.f : (x == 0.f ? 0.505f : 0.01f)) * invS;
      } else if (loss == SBR_LK_LIN) { lpart += v; gd = 0.f; gn = 1.f; }   // the positive is handled below
      else {
        const float sn = sigm(v * v);
        lpart += (sd + sn) * invS;
        gd = sd * (1.f - sd) * invS;
        gn = sn * (1.f - sn) * 2.f * v * invS;
      }
      gsum += gd;
      out = (gd + gn) * scale;
      if (tanh_out) out *= (1.f - v * v);
    }
    if (n != pc) row[n] = out;
  }
  const float l = block_sum(lpart, sh);
  const float gs = block_sum(gsum, sh);
  if (threadIdx.x == 0) {
    row_loss[b] = (loss == SBR_LK_LIN ? l - posv : l) * scale;
    float dp = (loss == SBR_LK_LIN ? -1.f : -gs) * scale;
    if (tanh_out) dp *= (1.f - posv * posv);
    row[pc] = dp;
  }
}

__global__ void __launch_bounds__(LT) margin_loss_kernel(int loss, float* __restrict__ pred, int ld,
                                                          const float* __restrict__ bias, const float* __restrict__ Y,
                                                          const float* __restrict__ W, int N, float inv_gb,
                                                          float* __restrict__ row_loss) {
  __shared__ float sh[LT / 32];
  const int b = blockIdx.x;
  float* row = pred + (int64_t)b * ld;
  const float* y = Y + (int64_t)b * N;
  const float* w = W + (int64_t)b * N;
  float lpart = 0.f;
  for (int n = threadIdx.x; n < N; n += LT) {
    const float p = row[n] + bias[n];
    const float wt = w[n], yt = y[n];
    float d;
    if (loss == SBR_LOSS_HINGE) {
      const float z = (p - yt) * wt;
      lpart += fmaxf(z, 0.f);
      d = (z > 0.f ? 1.f : (z == 0.f ? 0.5f : 0.f)) * wt;   // theano relu = 0.5 (x + |x|)
    } else if (loss == SBR_LOSS_LOGIT) {
      const float s = sigm(p - yt);
      lpart += s * wt;
      d = s * (1.f - s) * wt;
    } else {
      const float z = (yt - p) * wt;
      lpart += softplus(-z);            // -log sigmoid(z)
      d = (1.f - sigm(z)) * wt;
    }
    row[n] = d * inv_gb;
  }
  const float l = block_sum(lpart, sh);
  if (threadIdx.x == 0) row_loss[b] = l * inv_gb;
}

// one element of a margin loss (rnn_margin.py:61-68): contribution to the row loss and d loss / d pred
__device__ __forceinline__ void margin_elem(int loss, float p, float yt, float wt, float& l, float& d) {
  if (loss == SBR_LOSS_HINGE) {
    const float z = (p - yt) * wt;
    l = fmaxf(z, 0.f);
    d = (z > 0.f ? 1.f : (z == 0.f ? 0.5f : 0.f)) * wt;   // theano relu = 0.5 (x + |x|)
  } else if (loss == SBR_LOSS_LOGIT) {
    const float sg = sigm(p - yt);
    l = sg * wt;
    d = sg * (1.f - sg) * wt;
  } else {
    const float z = (yt - p) * wt;
    l = softplus(-z);            // -log sigmoid(z)
    d = (1.f - sigm(z)) * wt;
  }
}

// The same loss straight from the ragged description of a row (rnn_margin.py:121-149 builds dense [B, n_items] target
// and weight matrices on the host; they are never materialised here): weight = w_neg[b], target = default everywhere,
// except the row's targets (target 1, weight -1) and -- after them, so they win -- the items of its input window
// (target 0, weight 0).  The S = n_targets + len special entries keep their original prediction in shared memory
// while the dense pass overwrites the row with the default gradient; then every DISTINCT special id is corrected once
// by its last entry in the list (targets first, seen items second: the reference's override order).
__global__ void __launch_bounds__(LT) margin_loss_ragged_kernel(int loss, float* __restrict__ pred, int ld, const float* __restrict__ bias,
                                                                 const int32_t* __restrict__ toff, const int32_t* __restrict__ tids,
                                                                 const int32_t* __restrict__ X, const int32_t* __restrict__ len,
                                                                 const float* __restrict__ w_neg, const float* __restrict__ def_tgt,
                                                                 int exclude_seen, int T, int K, int N, float inv_gb,
                                                                 float* __restrict__ row_loss) {
  extern __shared__ __align__(16) unsigned char ms_smem[];
  __shared__ float sh[LT / 32];
  const int b = blockIdx.x;
  const int nt = toff[b + 1] - toff[b], ns = exclude_seen ? len[b] : 0, S = nt + ns;
  int32_t* sp_id = reinterpret_cast<int32_t*>(ms_smem);
  float* sp_p = reinterpret_cast<float*>(sp_id + S);
  float* row = pred + (int64_t)b * ld;
  const float w0 = w_neg[b];
  for (int i = threadIdx.x; i < S; i += LT) {
    const int id = i < nt ? tids[toff[b] + i] : X[((int64_t)b * T + (i - nt)) * K];
    sp_id[i] = id;
    sp_p[i] = (id >= 0 && id < N) ? row[id] + bias[id] : 0.f;
  }
  __syncthreads();
  float lpart = 0.f;
  for (int n = threadIdx.x; n < N; n += LT) {
    float l, d;
    margin_elem(loss, row[n] + bias[n], def_tgt ? def_tgt[n] : 0.f, w0, l, d);
    lpart += l;
    row[n] = d * inv_gb;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < S; i += LT) {
    const int id = sp_id[i];
    if (id < 0 || id >= N) continue;
    bool last = true;
    for (int j = i + 1; j < S && last; ++j) last = sp_id[j] != id;
    if (!last) continue;
    float l0, d0, l1, d1;
    margin_elem(loss, sp_p[i], def_tgt ? def_tgt[id] : 0.f, w0, l0, d0);
    if (i < nt) margin_elem(loss, sp_p[i], 1.f, -1.f, l1, d1);
    else margin_elem(loss, sp_p[i], 0.f, 0.f, l1, d1);
    lpart += l1 - l0;
    row[id] = d1 * inv_gb;
  }
  const float l = block_sum(lpart, sh);
  if (threadIdx.x == 0) row_loss[b] = l * inv_gb;
}

// weight[b,:] = w_neg[b] ; Y[b,:] = default ; then targets (Y=1, w=-1)
__global__ void margin_fill_kernel(float* __restrict__ Y, float* __restrict__ W, const int32_t* __restrict__ toff,
                                   const int32_t* __restrict__ tids, const float* __restrict__ w_neg,
                                   const float* __restrict__ def_tgt, int N) {
  const int b = blockIdx.x;
  const float w = w_neg[b];
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    Y[(int64_t)b * N + n] = def_tgt ? def_tgt[n] : 0.f;
    W[(int64_t)b * N + n] = w;
  }
  __syncthreads();
  for (int i = toff[b] + threadIdx.x; i < toff[b + 1]; i += blockDim.x) {
    const int id = tids[i];
    if (id >= 0 && id < N) {
      Y[(int64_t)b * N + id] = 1.f;
      W[(int64_t)b * N + id] = -1.f;
    }
  }
}

// seen items override the targets (rnn_margin.py:140-145)
__global__ void margin_seen_kernel(float* __restrict__ Y, float* __restrict__ W, const int32_t* __restrict__ X,
                                   const int32_t* __restrict__ len, int T, int K, int N) {
  const int b = blockIdx.x;
  const int L = len[b];
  for (int t = threadIdx.x; t < L; t += blockDim.x) {
    const int id = X[((int64_t)b * T + t) * K];
    if (id >= 0 && id < N) {
      Y[(int64_t)b * N + id] = 0.f;
      W[(int64_t)b * N + id] = 0.f;
    }
  }
}

__global__ void __launch_bounds__(LT) bias_reg_kernel(const float* __restrict__ b, float* __restrict__ db, int N,
                                                       float reg, float* __restrict__ cost_acc) {
  __shared__ float sh[LT / 32];
  float part = 0.f;
  for (int n = blockIdx.x * LT + threadIdx.x; n < N; n += gridDim.x * LT) {
    const float v = b[n];
    if (reg > 0.f) { part += reg * v * v; atomicAdd(db + n, 2.f * reg * v); }
    else { part += -reg * fabsf(v); atomicAdd(db + n, -reg * (v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f))); }
  }
  const float s = block_sum(part, sh);
  if (threadIdx.x == 0) atomicAdd(cost_acc, s);
}

__global__ void __launch_bounds__(LT) reduce_cost_kernel(const float* __restrict__ row_loss, int B,
                                                          float* __restrict__ cost_acc) {
  __shared__ float sh[LT / 32];
  float part = 0.f;
  for (int b = threadIdx.x; b < B; b += LT) part += row_loss[b];
  const float s = block_sum(part, sh);
  if (threadIdx.x == 0) atomicAdd(cost_acc, s);
}

__global__ void exclude_kernel(float* __restrict__ scores, int ld, const int32_t* __restrict__ off,
                               const int32_t* __restrict__ ids, int N, int neg_inf) {
  const int b = blockIdx.x;
  for (int i = off[b] + threadIdx.x; i < off[b + 1]; i += blockDim.x) {
    const int id = ids[i];
    if (id >= 0 && id < N) scores[(int64_t)b * ld + id] = neg_inf ? -CUDART_INF_F : 0.f * scores[(int64_t)b * ld + id];
  }
}

// k rounds of block-wide arg-max (k is ~10); ties resolve to the smallest id
__global__ void __launch_bounds__(LT) topk_kernel(float* __restrict__ scores, int ld, int N, int k,
                                                   int32_t* __restrict__ ids_out) {
  __shared__ float sv[LT / 32];
  __shared__ int si[LT / 32];
  const int b = blockIdx.x;
  float* row = scores + (int64_t)b * ld;
  for (int r = 0; r < k; ++r) {
    float best = -CUDART_INF_F;
    int bi = 0x7fffffff;
    for (int n = threadIdx.x; n < N; n += LT) {
      const float v = row[n];
      if (v > best || (v == best && n < bi)) { best = v; bi = n; }
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
      for (int i = 1; i < LT / 32; ++i)
        if (sv[i] > best || (sv[i] == best && si[i] < bi)) { best = sv[i]; bi = si[i]; }
      if (bi == 0x7fffffff) bi = 0;
      ids_out[b * k + r] = bi;
      row[bi] = -CUDART_INF_F;   // remove from the next rounds (NaN-free inputs assumed)
      si[0] = bi;
    }
    __syncthreads();
    // a picked -inf must not be picked again: mark with NaN-free sentinel by skipping equal ids
  }
}

}  // namespace

int launch_cce(sbr_model* m, float* logits, int ld, const float* bias, const int32_t* Y, const float* pop, int B,
               int N, float inv_gb, float* row_loss) {
  if (B == 0) return 0;
  cce_kernel<<<B, LT, 0, m->stream>>>(logits, ld, bias, Y, pop, N, inv_gb, row_loss);
  KERNEL_CHECK(m);
  return 0;
}

int launch_softmax_rows(sbr_model* m, float* logits, int ld, const float* bias, int B, int N) {
  if (B == 0) return 0;
  softmax_rows_kernel<<<B, LT, 0, m->stream>>>(logits, ld, bias, N);
  KERNEL_CHECK(m);
  return 0;
}

int launch_add_bias_rows(sbr_model* m, float* logits, int ld, const float* bias, int B, int N) {
  if (B == 0) return 0;
  add_bias_rows_kernel<<<cdiv((int64_t)B * N, 256), 256, 0, m->stream>>>(logits, ld, bias, B, N);
  KERNEL_CHECK(m);
  return 0;
}

int launch_sampling_loss(sbr_model* m, int loss, bool tanh_out, float* A, int ld, const float* bias_cells,
                         const float* pop, int B, int n_all, int row_offset, int S, float inv_gb, float* row_loss) {
  if (B == 0) return 0;
  sampling_loss_kernel<<<B, LT, 0, m->stream>>>(loss, tanh_out ? 1 : 0, A, ld, bias_cells, pop, n_all, row_offset, S,
                                                inv_gb, row_loss);
  KERNEL_CHECK(m);
  return 0;
}

int launch_margin_loss(sbr_model* m, int loss, float* pred, int ld, const float* bias, const float* Y,
                       const float* W, int B, int N, float inv_gb, float* row_loss) {
  if (B == 0) return 0;
  margin_loss_kernel<<<B, LT, 0, m->stream>>>(loss, pred, ld, bias, Y, W, N, inv_gb, row_loss);
  KERNEL_CHECK(m);
  return 0;
}

int launch_margin_loss_ragged(sbr_model* m, int loss, float* pred, int ld, const float* bias, const int32_t* toff,
                              const int32_t* tids, const int32_t* X, const int32_t* len, const float* w_neg,
                              const float* def_tgt, int exclude_seen, int B, int T, int K, int N, int max_special,
                              float inv_gb, float* row_loss) {
  if (B == 0) return 0;
  const size_t smem = (size_t)std::max(1, max_special) * 8;
  if (smem > 200 * 1024) { sbr_set_error(m, SBR_E_ARG, "margin step: %d targets + seen items in one row", max_special); return SBR_E_ARG; }
  static std::vector<int> attr_devs;
  if (smem > 48 * 1024 && std::find(attr_devs.begin(), attr_devs.end(), m->dev) == attr_devs.end()) {
    cudaFuncSetAttribute(margin_loss_ragged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_devs.push_back(m->dev);
  }
  margin_loss_ragged_kernel<<<B, LT, smem, m->stream>>>(loss, pred, ld, bias, toff, tids, X, len, w_neg, def_tgt, exclude_seen,
                                                        T, K, N, inv_gb, row_loss);
  KERNEL_CHECK(m);
  return 0;
}

int launch_margin_fill(sbr_model* m, float* Y, float* W, const int32_t* X, const int32_t* len, const int32_t* toff,
                       const int32_t* tids, const float* w_neg, const float* def_tgt, int exclude_seen, int B,
                       int T, int K, int N) {
  if (B == 0) return 0;
  margin_fill_kernel<<<B, 256, 0, m->stream>>>(Y, W, toff, tids, w_neg, def_tgt, N);
  KERNEL_CHECK(m);
  if (exclude_seen) {
    margin_seen_kernel<<<B, 128, 0, m->stream>>>(Y, W, X, len, T, K, N);
    KERNEL_CHECK(m);
  }
  return 0;
}

int launch_bias_reg(sbr_model* m, const float* b, float* db, int N, float reg, float* cost_acc) {
  if (reg == 0.f) return 0;
  bias_reg_kernel<<<std::min(cdiv(N, LT), m->n_sm), LT, 0, m->stream>>>(b, db, N, reg, cost_acc);
  KERNEL_CHECK(m);
  return 0;
}

int launch_reduce_cost(sbr_model* m, const float* row_loss, int B, float* cost_acc) {
  reduce_cost_kernel<<<1, LT, 0, m->stream>>>(row_loss, B, cost_acc);
  KERNEL_CHECK(m);
  return 0;
}

int launch_topk(sbr_model* m, float* scores, int ld, int B, int N, const int32_t* excl_off, const int32_t* excl_ids,
                int k, int neg_inf, int32_t* ids_out) {
  if (B == 0) return 0;
  if (excl_off) {
    exclude_kernel<<<B, 128, 0, m->stream>>>(scores, ld, excl_off, excl_ids, N, neg_inf);
    KERNEL_CHECK(m);
  }
  topk_kernel<<<B, LT, 0, m->stream>>>(scores, ld, N, k, ids_out);
  KERNEL_CHECK(m);
  return 0;
}
