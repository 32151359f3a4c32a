// Molecule-level head of the training step (SURVEY.md section 8f-2): what follows the aggregation in
// chemprop/models/model.py:126-161 -- BatchNorm1d over the b x d fingerprints, the FFN (chemprop/nn/ffn.py:38-61; its
// GEMMs run on dmpnn_linear_fwd / dmpnn_linear_x3) and the masked, weighted MSE criterion (chemprop/nn/metrics.py:78-123,
// 139-141).  b x d is tiny next to the E x h work of the encoder: these kernels exist so that the WHOLE step is
// libdmpnn launches with no host round trip (and therefore capturable in one CUDA graph), not for their own speed.
//
//   dmpnn_bn_train_fwd   batch statistics (biased variance, two-pass, fixed summation order) + normalisation + affine, one
//                        launch; updates running_mean / running_var (momentum, unbiased variance) like nn.BatchNorm1d
//   dmpnn_bn_bwd         dX, dgamma, dbeta from the saved x_hat / invstd
//   dmpnn_mse_loss       loss = sum(w_b * tw_t * mask * (p - y)^2) / sum(mask) and dLoss/dp, NaN targets masked, one launch
//   dmpnn_bce_loss       the same with binary cross entropy on logits (BinaryClassificationFFN + BCELoss)
//   dmpnn_ce_loss        the same with cross entropy over groups of C logits (MulticlassClassificationFFN + CrossEntropyLoss)
//   dmpnn_class_probs    eval output of the classifiers: sigmoid (C == 1) or per-group softmax; _bwd: its mirror
#include <cooperative_groups.h>

#include "common.cuh"

namespace dmpnn {
namespace head {

constexpr int kWarps = 8;          // block = 8 warps x 32 lanes; lane = column of the block's 32-column strip

// column strip [32 * blockIdx.x, +32); warps stride over the rows; fixed-order reductions (deterministic)
__global__ void __launch_bounds__(kWarps * 32)
k_bn_train_fwd(const float* __restrict__ X, int64_t ldx, int64_t B, int d, const float* __restrict__ gamma,
               const float* __restrict__ beta, float eps, float momentum, float* __restrict__ running_mean,
               float* __restrict__ running_var, float* __restrict__ Y, int64_t ldy, float* __restrict__ Xhat, int64_t ldh,
               float* __restrict__ save_mean, float* __restrict__ save_invstd) {
  __shared__ float red[kWarps][32];
  __shared__ float s_mean[32], s_inv[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * 32 + lane;
  const bool cv = c < d;
  // pass 1: mean
  float s = 0.f;
  for (int64_t r = warp; r < B; r += kWarps) s += cv ? X[r * ldx + c] : 0.f;
  red[warp][lane] = s;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) t += red[w][lane];
    s_mean[lane] = t / (float)B;
  }
  __syncthreads();
  const float mean = s_mean[lane];
  // pass 2: variance around the mean (the strip is L2-resident)
  float q = 0.f;
  for (int64_t r = warp; r < B; r += kWarps) {
    const float dlt = cv ? X[r * ldx + c] - mean : 0.f;
    q = fmaf(dlt, dlt, q);
  }
  __syncthreads();
  red[warp][lane] = q;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) t += red[w][lane];
    const float var = t / (float)B;                       // biased: what normalises the batch
    s_inv[lane] = rsqrtf(var + eps);
    if (cv) {
      save_mean[c] = mean;
      save_invstd[c] = s_inv[lane];
      if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
      if (running_var) running_var[c] = (1.f - momentum) * running_var[c] + momentum * (B > 1 ? t / (float)(B - 1) : var);
    }
  }
  __syncthreads();
  const float inv = s_inv[lane];
  const float g = (cv && gamma) ? gamma[c] : 1.f, bt = (cv && beta) ? beta[c] : 0.f;
  for (int64_t r = warp; r < B; r += kWarps) {
    if (!cv) continue;
    const float xh = (X[r * ldx + c] - mean) * inv;
    Xhat[r * ldh + c] = xh;
    Y[r * ldy + c] = fmaf(xh, g, bt);
  }
}

__global__ void __launch_bounds__(kWarps * 32)
k_bn_bwd(const float* __restrict__ dY, int64_t lddy, const float* __restrict__ Xhat, int64_t ldh, int64_t B, int d,
         const float* __restrict__ gamma, const float* __restrict__ invstd, float* __restrict__ dX, int64_t lddx,
         float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ float red1[kWarps][32], red2[kWarps][32];
  __shared__ float s_sdy[32], s_sdyx[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * 32 + lane;
  const bool cv = c < d;
  float a = 0.f, b = 0.f;
  for (int64_t r = warp; r < B; r += kWarps) {
    if (!cv) continue;
    const float g = dY[r * lddy + c];
    a += g;
    b = fmaf(g, Xhat[r * ldh + c], b);
  }
  red1[warp][lane] = a;
  red2[warp][lane] = b;
  __syncthreads();
  if (warp == 0) {
    float ta = 0.f, tb = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) { ta += red1[w][lane]; tb += red2[w][lane]; }
    s_sdy[lane] = ta;
    s_sdyx[lane] = tb;
    if (cv) {
      if (dbeta) dbeta[c] = ta;
      if (dgamma) dgamma[c] = tb;
    }
  }
  __syncthreads();
  if (!cv) return;
  const float sdy = s_sdy[lane], sdyx = s_sdyx[lane];
  const float k = (gamma ? gamma[c] : 1.f) * invstd[c] / (float)B;
  for (int64_t r = warp; r < B; r += kWarps)
    dX[r * lddx + c] = k * ((float)B * dY[r * lddy + c] - sdy - Xhat[r * ldh + c] * sdyx);
}

// Fixed-order sum of (l, n) over the block: lanes (shuffle tree), then the warp partials in warp order by thread 0.
// Every thread gets the totals.  Deterministic for a fixed blockDim; contains __syncthreads (call from all threads).
__device__ __forceinline__ float2 block_sum2(float l, float n) {
  __shared__ float s_l[32], s_n[32];
  __shared__ float s_tot[2];
  for (int o = 16; o > 0; o >>= 1) {
    l += __shfl_down_sync(0xffffffffu, l, o);
    n += __shfl_down_sync(0xffffffffu, n, o);
  }
  if ((threadIdx.x & 31) == 0) { s_l[threadIdx.x >> 5] = l; s_n[threadIdx.x >> 5] = n; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float tl = 0.f, tn = 0.f;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) { tl += s_l[k]; tn += s_n[k]; }
    s_tot[0] = tl;
    s_tot[1] = tn;
  }
  __syncthreads();
  return make_float2(s_tot[0], s_tot[1]);
}

// one block: loss[0] = sum_{b,t} w_b tw_t m_bt (p - y)^2 / sum m,  dP = 2 w tw m (p - y) / sum m   (m = isfinite(y))
__global__ void __launch_bounds__(1024)
k_mse_loss(const float* __restrict__ P, int64_t ldp, const float* __restrict__ Y, int64_t ldy, const float* __restrict__ w,
           const float* __restrict__ tw, int64_t B, int T, float* __restrict__ loss, float* __restrict__ dP, int64_t lddp) {
  const int64_t n = B * (int64_t)T;
  float l = 0.f, cnt = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t b = i / T;
    const int t = (int)(i - b * T);
    const float y = Y[b * ldy + t];
    if (isfinite(y)) {
      const float e = P[b * ldp + t] - y;
      l = fmaf((w ? w[b] : 1.f) * (tw ? tw[t] : 1.f) * e, e, l);
      cnt += 1.f;
    }
  }
  const float2 tot = block_sum2(l, cnt);
  if (threadIdx.x == 0) loss[0] = tot.y > 0.f ? tot.x / tot.y : 0.f;
  const float inv_n = tot.y > 0.f ? 1.f / tot.y : 0.f;
  if (dP != nullptr)
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
      const int64_t b = i / T;
      const int t = (int)(i - b * T);
      const float y = Y[b * ldy + t];
      dP[b * lddp + t] = isfinite(y) ? 2.f * (w ? w[b] : 1.f) * (tw ? tw[t] : 1.f) * (P[b * ldp + t] - y) * inv_n : 0.f;
    }
}

// ---- classification criteria: one cluster of kLossBlocks blocks ---------------------------------------------------
// Block r of the cluster owns the flattened range [r n / G, (r + 1) n / G) of the n items ((b, t) pairs); its (loss, count)
// partial comes from block_sum2, and every block adds the G partials in rank order through distributed shared memory, so all
// blocks hold the same totals (bit for bit) before the gradient pass.  No float atomics, no scratch memory, no host sync.
constexpr int kLossBlocks = 8;        // portable cluster size: 8 SMs share the transcendental work of a wide (10 k x 617) batch
constexpr int kLossThreads = 1024;

struct ItemRange {
  int64_t i0, i1;
};
__device__ __forceinline__ ItemRange cluster_item_range(int64_t n, unsigned rank) {
  return {n * (int64_t)rank / kLossBlocks, n * (int64_t)(rank + 1) / kLossBlocks};
}

// (b, t) of item i of a B x T grid, stepped by a fixed stride with one division per thread instead of one per item
struct ItemCursor {
  int64_t b, sb;
  int t, st, T;
  __device__ __forceinline__ ItemCursor(int64_t i, int64_t stride, int T_) : T(T_) {
    b = i / T;
    t = (int)(i - b * T);
    sb = stride / T;
    st = (int)(stride - sb * T);
  }
  __device__ __forceinline__ void next() {
    b += sb;
    t += st;
    if (t >= T) {
      t -= T;
      ++b;
    }
  }
};

// the cluster-wide totals of this block's (loss, count) partial
__device__ __forceinline__ float2 cluster_sum2(float l, float n) {
  namespace cg = cooperative_groups;
  __shared__ float2 s_part;
  cg::cluster_group cl = cg::this_cluster();
  const float2 part = block_sum2(l, n);
  if (threadIdx.x == 0) s_part = part;
  cl.sync();
  float2 tot = make_float2(0.f, 0.f);
  for (int k = 0; k < kLossBlocks; ++k) {             // rank order: the same sum in every block
    const float2 q = *cl.map_shared_rank(&s_part, k);
    tot.x += q.x;
    tot.y += q.y;
  }
  cl.sync();                                          // the partials stay mapped until every block has read them
  return tot;
}

__device__ __forceinline__ float sample_weight(const float* w, const float* tw, int64_t b, int t) {
  return (w ? w[b] : 1.f) * (tw ? tw[t] : 1.f);
}

// loss = sum w tw m [max(z, 0) - z y + log1p(exp(-|z|))] / sum m,  dP = w tw m (sigmoid(z) - y) / sum m
__global__ void __cluster_dims__(kLossBlocks, 1, 1) __launch_bounds__(kLossThreads, 1)
k_bce_loss(const float* __restrict__ P, int64_t ldp, const float* __restrict__ Y, int64_t ldy, const float* __restrict__ w,
           const float* __restrict__ tw, int64_t B, int T, float* __restrict__ loss, float* __restrict__ dP, int64_t lddp) {
  const int64_t n = B * (int64_t)T;
  const unsigned rank = cooperative_groups::this_cluster().block_rank();
  const ItemRange rg = cluster_item_range(n, rank);
  float l = 0.f, cnt = 0.f;
  ItemCursor it(rg.i0 + threadIdx.x, blockDim.x, T);
  for (int64_t i = rg.i0 + threadIdx.x; i < rg.i1; i += blockDim.x, it.next()) {
    const float y = Y[it.b * ldy + it.t];
    if (isfinite(y)) {
      const float z = P[it.b * ldp + it.t];
      const float L = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
      l = fmaf(sample_weight(w, tw, it.b, it.t), L, l);
      cnt += 1.f;
    }
  }
  const float2 tot = cluster_sum2(l, cnt);
  if (rank == 0 && threadIdx.x == 0) loss[0] = tot.y > 0.f ? tot.x / tot.y : 0.f;
  if (dP == nullptr) return;
  const float inv_n = tot.y > 0.f ? 1.f / tot.y : 0.f;
  it = ItemCursor(rg.i0 + threadIdx.x, blockDim.x, T);
  for (int64_t i = rg.i0 + threadIdx.x; i < rg.i1; i += blockDim.x, it.next()) {
    const float y = Y[it.b * ldy + it.t];
    float g = 0.f;
    if (isfinite(y)) {
      const float z = P[it.b * ldp + it.t];
      const float e = expf(-fabsf(z));
      const float tail = e / (1.f + e);                      // min(sigmoid(z), 1 - sigmoid(z)), without cancellation
      g = sample_weight(w, tw, it.b, it.t) * (z >= 0.f ? (1.f - y) - tail : tail - y) * inv_n;
    }
    dP[it.b * lddp + it.t] = g;
  }
}

// max and sum of exp(z - max) of the C logits z[0..C)
__device__ __forceinline__ float2 softmax_stats(const float* __restrict__ z, int C) {
  float mx = -INFINITY;
  for (int c = 0; c < C; ++c) mx = fmaxf(mx, z[c]);
  float s = 0.f;
  for (int c = 0; c < C; ++c) s += expf(z[c] - mx);
  return make_float2(mx, s);
}

// a finite target that is not a class id in [0, C) -> -1 (its loss is NaN: the sync-free stand-in for torch's raise)
__device__ __forceinline__ int class_of(float y, int C) {
  return (y >= 0.f && y < (float)C && y == floorf(y)) ? (int)y : -1;
}

// P is B x (T C), logits of task t in columns [t C, t C + C).  loss = sum w tw m [lse(z) - z_y] / sum m,
// dP = w tw m (softmax(z) - onehot(y)) / sum m
__global__ void __cluster_dims__(kLossBlocks, 1, 1) __launch_bounds__(kLossThreads, 1)
k_ce_loss(const float* __restrict__ P, int64_t ldp, const float* __restrict__ Y, int64_t ldy, const float* __restrict__ w,
          const float* __restrict__ tw, int64_t B, int T, int C, float* __restrict__ loss, float* __restrict__ dP,
          int64_t lddp) {
  const float kNaN = __int_as_float(0x7fc00000);
  const int64_t n = B * (int64_t)T;
  const unsigned rank = cooperative_groups::this_cluster().block_rank();
  const ItemRange rg = cluster_item_range(n, rank);
  float l = 0.f, cnt = 0.f;
  ItemCursor it(rg.i0 + threadIdx.x, blockDim.x, T);
  for (int64_t i = rg.i0 + threadIdx.x; i < rg.i1; i += blockDim.x, it.next()) {
    const float y = Y[it.b * ldy + it.t];
    if (isfinite(y)) {
      const float* z = P + it.b * ldp + (int64_t)it.t * C;
      const int k = class_of(y, C);
      const float2 ms = softmax_stats(z, C);
      const float L = k >= 0 ? (ms.x - z[k]) + logf(ms.y) : kNaN;     // lse - z_k, the large terms cancelled first
      l = fmaf(sample_weight(w, tw, it.b, it.t), L, l);
      cnt += 1.f;
    }
  }
  const float2 tot = cluster_sum2(l, cnt);
  if (rank == 0 && threadIdx.x == 0) loss[0] = tot.y > 0.f ? tot.x / tot.y : 0.f;
  if (dP == nullptr) return;
  const float inv_n = tot.y > 0.f ? 1.f / tot.y : 0.f;
  it = ItemCursor(rg.i0 + threadIdx.x, blockDim.x, T);
  for (int64_t i = rg.i0 + threadIdx.x; i < rg.i1; i += blockDim.x, it.next()) {
    const float y = Y[it.b * ldy + it.t];
    const float* z = P + it.b * ldp + (int64_t)it.t * C;
    float* g = dP + it.b * lddp + (int64_t)it.t * C;
    if (!isfinite(y)) {
      for (int c = 0; c < C; ++c) g[c] = 0.f;
      continue;
    }
    const int k = class_of(y, C);
    if (k < 0) {
      for (int c = 0; c < C; ++c) g[c] = kNaN;
      continue;
    }
    float mx = -INFINITY;
    for (int c = 0; c < C; ++c) mx = fmaxf(mx, z[c]);
    float s = 0.f, others = 0.f;
    for (int c = 0; c < C; ++c) {
      const float e = expf(z[c] - mx);
      s += e;
      others += c == k ? 0.f : e;
    }
    const float sw = sample_weight(w, tw, it.b, it.t) * inv_n / s;
    for (int c = 0; c < C; ++c)                               // softmax_k - 1 = -(sum of the other classes) / s
      g[c] = c == k ? -sw * others : sw * expf(z[c] - mx);
  }
}

// eval output: sigmoid (C == 1) or softmax over each group of C columns; one thread per (b, t)
__global__ void __launch_bounds__(256)
k_class_probs(const float* __restrict__ P, int64_t ldp, int64_t B, int T, int C, float* __restrict__ Q, int64_t ldq) {
  const int64_t n = B * (int64_t)T, stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  ItemCursor it(i0, stride, T);
  for (int64_t i = i0; i < n; i += stride, it.next()) {
    const float* z = P + it.b * ldp + (int64_t)it.t * C;
    float* q = Q + it.b * ldq + (int64_t)it.t * C;
    if (C == 1) {
      const float e = expf(-fabsf(z[0]));
      q[0] = z[0] >= 0.f ? 1.f / (1.f + e) : e / (1.f + e);
      continue;
    }
    const float2 ms = softmax_stats(z, C);
    for (int c = 0; c < C; ++c) q[c] = expf(z[c] - ms.x) / ms.y;
  }
}

// dP = dQ q (1 - q) (sigmoid) or q (dQ - <dQ, q>) per group (softmax)
__global__ void __launch_bounds__(256)
k_class_probs_bwd(const float* __restrict__ Q, int64_t ldq, const float* __restrict__ dQ, int64_t lddq, int64_t B, int T, int C,
                  float* __restrict__ dP, int64_t lddp) {
  const int64_t n = B * (int64_t)T, stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  ItemCursor it(i0, stride, T);
  for (int64_t i = i0; i < n; i += stride, it.next()) {
    const float* q = Q + it.b * ldq + (int64_t)it.t * C;
    const float* g = dQ + it.b * lddq + (int64_t)it.t * C;
    float* d = dP + it.b * lddp + (int64_t)it.t * C;
    if (C == 1) {
      d[0] = g[0] * q[0] * (1.f - q[0]);
      continue;
    }
    float dot = 0.f;
    for (int c = 0; c < C; ++c) dot = fmaf(g[c], q[c], dot);
    for (int c = 0; c < C; ++c) d[c] = q[c] * (g[c] - dot);
  }
}

}  // namespace head
}  // namespace dmpnn

using namespace dmpnn;

extern "C" int dmpnn_bn_train_fwd(const float* X, int64_t ldx, int64_t B, int64_t d, const float* gamma, const float* beta,
                                  float eps, float momentum, float* running_mean, float* running_var, float* Y, int64_t ldy,
                                  float* Xhat, int64_t ldh, float* save_mean, float* save_invstd, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DMPNN_CHECK_ARG(B > 0 && d > 0 && X && Y && Xhat && save_mean && save_invstd, "bn_train_fwd: bad args (B must be >= 1)");
  DMPNN_CHECK_ARG(ldx >= d && ldy >= d && ldh >= d, "bn_train_fwd: row strides too small");
  head::k_bn_train_fwd<<<(unsigned)((d + 31) / 32), head::kWarps * 32, 0, st>>>(X, ldx, B, (int)d, gamma, beta, eps, momentum,
                                                                              running_mean, running_var, Y, ldy, Xhat, ldh,
                                                                              save_mean, save_invstd);
  DMPNN_CHECK_LAUNCH("bn_train_fwd", 1);
  return 0;
}

extern "C" int dmpnn_bn_bwd(const float* dY, int64_t lddy, const float* Xhat, int64_t ldh, int64_t B, int64_t d,
                            const float* gamma, const float* invstd, float* dX, int64_t lddx, float* dgamma, float* dbeta,
                            void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DMPNN_CHECK_ARG(B > 0 && d > 0 && dY && Xhat && invstd && dX, "bn_bwd: bad args");
  DMPNN_CHECK_ARG(lddy >= d && ldh >= d && lddx >= d, "bn_bwd: row strides too small");
  head::k_bn_bwd<<<(unsigned)((d + 31) / 32), head::kWarps * 32, 0, st>>>(dY, lddy, Xhat, ldh, B, (int)d, gamma, invstd, dX, lddx,
                                                                        dgamma, dbeta);
  DMPNN_CHECK_LAUNCH("bn_bwd", 1);
  return 0;
}

extern "C" int dmpnn_mse_loss(const float* P, int64_t ldp, const float* Y, int64_t ldy, const float* weights,
                              const float* task_weights, int64_t B, int64_t T, float* loss, float* dP, int64_t lddp,
                              void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DMPNN_CHECK_ARG(B >= 0 && T > 0 && loss && (B == 0 || (P && Y)), "mse_loss: bad args");
  DMPNN_CHECK_ARG(ldp >= T && ldy >= T && (dP == nullptr || lddp >= T), "mse_loss: row strides too small");
  head::k_mse_loss<<<1, 1024, 0, st>>>(P, ldp, Y, ldy, weights, task_weights, B, (int)T, loss, dP, lddp);
  DMPNN_CHECK_LAUNCH("mse_loss", 1);
  return 0;
}

extern "C" int dmpnn_bce_loss(const float* P, int64_t ldp, const float* Y, int64_t ldy, const float* weights,
                              const float* task_weights, int64_t B, int64_t T, float* loss, float* dP, int64_t lddp,
                              void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DMPNN_CHECK_ARG(B >= 0 && T > 0 && T <= INT32_MAX && loss && (B == 0 || (P && Y)), "bce_loss: bad args");
  DMPNN_CHECK_ARG(ldp >= T && ldy >= T && (dP == nullptr || lddp >= T), "bce_loss: row strides too small");
  head::k_bce_loss<<<head::kLossBlocks, head::kLossThreads, 0, st>>>(P, ldp, Y, ldy, weights, task_weights, B, (int)T, loss,
                                                                     dP, lddp);
  DMPNN_CHECK_LAUNCH("bce_loss", 1);
  return 0;
}

extern "C" int dmpnn_ce_loss(const float* P, int64_t ldp, const float* Y, int64_t ldy, const float* weights,
                             const float* task_weights, int64_t B, int64_t T, int64_t C, float* loss, float* dP, int64_t lddp,
                             void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DMPNN_CHECK_ARG(B >= 0 && T > 0 && C > 0 && T * C <= INT32_MAX && loss && (B == 0 || (P && Y)), "ce_loss: bad args");
  DMPNN_CHECK_ARG(ldp >= T * C && ldy >= T && (dP == nullptr || lddp >= T * C), "ce_loss: row strides too small");
  head::k_ce_loss<<<head::kLossBlocks, head::kLossThreads, 0, st>>>(P, ldp, Y, ldy, weights, task_weights, B, (int)T, (int)C,
                                                                    loss, dP, lddp);
  DMPNN_CHECK_LAUNCH("ce_loss", 1);
  return 0;
}

static unsigned class_probs_grid(int64_t n) {
  const int64_t blocks = (n + 255) / 256;
  return (unsigned)(blocks < 1 ? 1 : blocks > 148 * 8 ? 148 * 8 : blocks);
}

extern "C" int dmpnn_class_probs(const float* P, int64_t ldp, int64_t B, int64_t T, int64_t C, float* Q, int64_t ldq,
                                 void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DMPNN_CHECK_ARG(B >= 0 && T > 0 && C > 0 && T * C <= INT32_MAX && (B == 0 || (P && Q)), "class_probs: bad args");
  DMPNN_CHECK_ARG(ldp >= T * C && ldq >= T * C, "class_probs: row strides too small");
  if (B == 0) return 0;
  head::k_class_probs<<<class_probs_grid(B * T), 256, 0, st>>>(P, ldp, B, (int)T, (int)C, Q, ldq);
  DMPNN_CHECK_LAUNCH("class_probs", 1);
  return 0;
}

extern "C" int dmpnn_class_probs_bwd(const float* Q, int64_t ldq, const float* dQ, int64_t lddq, int64_t B, int64_t T,
                                     int64_t C, float* dP, int64_t lddp, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  DMPNN_CHECK_ARG(B >= 0 && T > 0 && C > 0 && T * C <= INT32_MAX && (B == 0 || (Q && dQ && dP)), "class_probs_bwd: bad args");
  DMPNN_CHECK_ARG(ldq >= T * C && lddq >= T * C && lddp >= T * C, "class_probs_bwd: row strides too small");
  if (B == 0) return 0;
  head::k_class_probs_bwd<<<class_probs_grid(B * T), 256, 0, st>>>(Q, ldq, dQ, lddq, B, (int)T, (int)C, dP, lddp);
  DMPNN_CHECK_LAUNCH("class_probs_bwd", 1);
  return 0;
}
