// Textcat head (spacy.TextCatCNN / TextCatReduce / TextCatBOW / TextCatEnsemble) in two kernels.
//
// textcat_doc_kernel: one CTA per document.  Reads the doc's rows of the tok2vec output X from the
// padded-ragged layout (doc_starts / doc_lens on the device: no host lengths), pools them (mean and/or
// max, fp32), hashes the doc's n-grams from attrs[:, 0] and sums the W_bow rows, computes the logits,
// softmax / logistic / identity, d_logits = (scores - truth) * known / n_docs and the loss partial, then
// d_pooled = d_logits W and the doc's dX rows (mean: d / len; max: d * [x == max] / n_ties), and red.adds
// d_logits into the W_bow gradient rows its n-grams name.  Extra CTAs past the last doc zero the pad
// rows of dX.  textcat_dw_kernel: dW = d_logits^T pooled, db = column sums of d_logits and the loss, a
// reduction over documents (a chunk of docs per CTA, sized so the grid fills the GPU; one atomic per chunk
// and element).
// Upstream (models/textcat.py): unpad + index_add_ / scatter_reduce over the token matrix, a dense
// (262144, n_labels) zero-fill + index_add_ for the BOW gradient, a host-built truth array per step.
#include <math.h>

#include "common.cuh"
#include "kernels.h"
#include "launch.h"

namespace srb {

constexpr int kTcThreads = 256;
constexpr int kTcWarps = kTcThreads / 32;
constexpr int kRowBatch = 8;        // rows loaded per thread before they are reduced
constexpr int kDwLabels = 8;

__device__ __forceinline__ float ldw(const void* p, size_t i, int f32) {
  return f32 ? ((const float*)p)[i] : bf2f(((const __nv_bfloat16*)p)[i]);
}

// models/textcat.py::_ngram_features: key = ((id_t * 1000003 + id_t+1) * 1000003 + ...) with int64
// wrap-around, f = key ^ (key >> 31) (arithmetic shift), then a non-negative remainder.
__device__ __forceinline__ int64_t bow_feature(const int64_t* attrs, int n_attr, int row, int n, int64_t n_rows) {
  uint64_t key = (uint64_t)attrs[(size_t)row * n_attr];
  for (int j = 1; j < n; ++j) key = key * 1000003ull + (uint64_t)attrs[(size_t)(row + j) * n_attr];
  const int64_t k = (int64_t)key;
  const int64_t f = k ^ (k >> 31);
  const int64_t r = f % n_rows;
  return r < 0 ? r + n_rows : r;
}

__global__ void __launch_bounds__(kTcThreads) textcat_doc_kernel(TextcatArgs a) {
  pdl_prologue();
  __shared__ float s_pool[kTextcatMaxPool];     // pooled: [mean | max]
  __shared__ float s_dp[kTextcatMaxPool];       // d_pooled
  __shared__ int s_cnt[kTextcatMaxPool];        // rows that reach each column's max
  __shared__ float s_lg[kTextcatMaxLabels];     // logits, then d_logits
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int w = a.w, nL = a.nL;
  const int P = (a.use_mean + a.use_max) * w;
  __nv_bfloat16* dX = (__nv_bfloat16*)a.dX;
  const __nv_bfloat16* X = (const __nv_bfloat16*)a.X;

  if ((int)blockIdx.x >= a.B) {                  // pad rows of dX stay exactly zero
    const int nw = (gridDim.x - a.B) * kTcWarps;
    const __nv_bfloat16 z = f2bf(0.f);
    for (int r = (blockIdx.x - a.B) * kTcWarps + warp; r < a.Tp; r += nw)
      if (a.mask[r] == 0.f)
        for (int c = lane; c < w; c += 32) dX[(size_t)r * w + c] = z;
    return;
  }
  const int d = blockIdx.x;
  const int nd = a.n_docs_dev != nullptr ? *a.n_docs_dev : a.n_docs;
  const int start = a.doc_starts[d], len = a.doc_lens[d];

  if (d >= nd) {                                 // doc slot past the batch: contributes nothing
    for (int k = tid; k < P; k += kTcThreads) a.pooled[(size_t)d * P + k] = 0.f;
    for (int l = tid; l < nL; l += kTcThreads) {
      a.scores[(size_t)d * nL + l] = 0.f;
      a.d_logits[(size_t)d * nL + l] = 0.f;
    }
    if (tid == 0) a.loss_doc[d] = 0.f;
    if (dX != nullptr)
      for (int r = 0; r < len; ++r)
        for (int c = tid; c < w; c += kTcThreads) dX[(size_t)(start + r) * w + c] = f2bf(0.f);
    return;
  }

  // ---- pooling (fp32); a doc of length 0 pools to 0
  const int moff = a.use_mean ? w : 0;
  if (X != nullptr) {
    const float inv = len > 0 ? 1.0f / (float)len : 0.f;
    for (int c = tid; c < w; c += kTcThreads) {
      float sum = 0.f, mx = -INFINITY;
      int cnt = 0;
      const __nv_bfloat16* xc = X + (size_t)start * w + c;
      int r = 0;
      for (; r + kRowBatch <= len; r += kRowBatch) {       // independent loads in flight, then the reduction
        float x[kRowBatch];
#pragma unroll
        for (int j = 0; j < kRowBatch; ++j) x[j] = bf2f(xc[(size_t)(r + j) * w]);
#pragma unroll
        for (int j = 0; j < kRowBatch; ++j) {
          sum += x[j];
          if (x[j] > mx) { mx = x[j]; cnt = 1; } else if (x[j] == mx) { ++cnt; }
        }
      }
      for (; r < len; ++r) {
        const float x = bf2f(xc[(size_t)r * w]);
        sum += x;
        if (x > mx) { mx = x; cnt = 1; } else if (x == mx) { ++cnt; }
      }
      if (a.use_mean) s_pool[c] = sum * inv;
      if (a.use_max) { s_pool[moff + c] = len > 0 ? mx : 0.f; s_cnt[c] = cnt; }
    }
  }
  __syncthreads();
  for (int k = tid; k < P; k += kTcThreads) a.pooled[(size_t)d * P + k] = s_pool[k];

  // ---- logits = pooled W^T + b (+ b_bow): one warp per label
  for (int l = warp; l < nL; l += kTcWarps) {
    float acc = 0.f;
    if (a.W != nullptr)
      for (int k = lane; k < P; k += 32) acc += s_pool[k] * ldw(a.W, (size_t)l * P + k, a.W_f32);
    acc = warp_sum(acc);
    if (lane == 0) {
      if (a.b != nullptr) acc += ldw(a.b, l, a.b_f32);
      if (a.b_bow != nullptr) acc += ldw(a.b_bow, l, a.b_bow_f32);
      s_lg[l] = acc;
    }
  }
  __syncthreads();
  // ---- bag of n-grams: sum_f W_bow[f]
  if (a.W_bow != nullptr) {
    for (int n = 1; n <= a.ngram; ++n)
      for (int t = tid; t + n <= len; t += kTcThreads) {
        const int64_t f = bow_feature(a.attrs, a.n_attr, start + t, n, a.bow_rows);
        for (int l = 0; l < nL; ++l) atomicAdd(&s_lg[l], ldw(a.W_bow, (size_t)f * nL + l, a.W_bow_f32));
      }
    __syncthreads();
  }

  // ---- output layer, d_logits, loss (warp 0; nL <= 128 = 4 per lane)
  if (warp == 0) {
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int l = lane + 32 * j;
      v[j] = l < nL ? s_lg[l] : -INFINITY;
    }
    if (a.act == 0) {                            // softmax (exclusive classes)
      float mx = fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3]));
      mx = warp_max(mx);
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[j] = (lane + 32 * j) < nL ? expf(v[j] - mx) : 0.f;
        sum += v[j];
      }
      sum = warp_sum(sum);
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] /= sum;
    } else if (a.act == 1) {                     // logistic (multi-label)
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = 1.0f / (1.0f + expf(-v[j]));
    }
    const float inv_n = 1.0f / (float)max(nd, 1);
    float lsum = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int l = lane + 32 * j;
      if (l < nL) {
        const size_t i = (size_t)d * nL + l;
        const float diff = (v[j] - a.truths[i]) * a.known[i];
        const float dl = diff * inv_n;
        a.scores[i] = v[j];
        a.d_logits[i] = dl;
        s_lg[l] = dl;
        lsum += diff * diff;
      }
    }
    lsum = warp_sum(lsum);
    if (lane == 0) a.loss_doc[d] = lsum;
  }
  __syncthreads();

  // ---- BOW gradient: red.add d_logits into the rows this doc's n-grams name
  if (a.W_bow != nullptr && a.gW_bow != nullptr) {
    for (int n = 1; n <= a.ngram; ++n)
      for (int t = tid; t + n <= len; t += kTcThreads) {
        const int64_t f = bow_feature(a.attrs, a.n_attr, start + t, n, a.bow_rows);
        for (int l = 0; l < nL; ++l) {
          const float g = s_lg[l];
          if (g != 0.f) atomicAdd(&a.gW_bow[(size_t)f * nL + l], g);
        }
      }
  }

  // ---- d_pooled = d_logits W, then the doc's dX rows
  if (X == nullptr || a.W == nullptr) return;
  for (int k = tid; k < P; k += kTcThreads) {
    float acc = 0.f;
    for (int l = 0; l < nL; ++l) acc += s_lg[l] * ldw(a.W, (size_t)l * P + k, a.W_f32);
    s_dp[k] = acc;
  }
  __syncthreads();
  const float inv = len > 0 ? 1.0f / (float)len : 0.f;
  for (int c = tid; c < w; c += kTcThreads) {
    const float dm = a.use_mean ? s_dp[c] * inv : 0.f;
    float dmx = 0.f, mxv = 0.f;
    if (a.use_max) {
      dmx = s_dp[moff + c] / (float)max(s_cnt[c], 1);   // ties share the gradient
      mxv = s_pool[moff + c];
    }
    const size_t base = (size_t)start * w + c;
    if (!a.use_max) {
      const __nv_bfloat16 g = f2bf(dm);
      for (int r = 0; r < len; ++r) dX[base + (size_t)r * w] = g;
      continue;
    }
    int r = 0;
    for (; r + kRowBatch <= len; r += kRowBatch) {
      float x[kRowBatch];
#pragma unroll
      for (int j = 0; j < kRowBatch; ++j) x[j] = bf2f(X[base + (size_t)(r + j) * w]);
#pragma unroll
      for (int j = 0; j < kRowBatch; ++j) dX[base + (size_t)(r + j) * w] = f2bf(x[j] == mxv ? dm + dmx : dm);
    }
    for (; r < len; ++r) {
      const size_t i = base + (size_t)r * w;
      dX[i] = f2bf(bf2f(X[i]) == mxv ? dm + dmx : dm);
    }
  }
}

// dW[l, k] += sum_d d_logits[d, l] * pooled[d, k]; db[l] (+ db_bow[l]) += sum_d d_logits[d, l];
// loss = sum_d loss_doc[d] / (n_docs * n_labels).  Grid (ceil(P / 256), ceil(nL / 8), ceil(B / chunk)).
__global__ void __launch_bounds__(256) textcat_dw_kernel(TextcatArgs a, int chunk) {
  pdl_prologue();
  const int P = (a.use_mean + a.use_max) * a.w, nL = a.nL;
  const int k = blockIdx.x * 256 + threadIdx.x;
  const int l0 = blockIdx.y * kDwLabels;
  const int d0 = blockIdx.z * chunk, d1 = min(a.B, d0 + chunk);
  if (a.gW != nullptr && k < P) {
    float acc[kDwLabels];
#pragma unroll
    for (int j = 0; j < kDwLabels; ++j) acc[j] = 0.f;
    for (int d = d0; d < d1; ++d) {
      const float p = a.pooled[(size_t)d * P + k];
      const float* dl = a.d_logits + (size_t)d * nL + l0;
#pragma unroll
      for (int j = 0; j < kDwLabels; ++j)
        if (l0 + j < nL) acc[j] += dl[j] * p;
    }
#pragma unroll
    for (int j = 0; j < kDwLabels; ++j)
      if (l0 + j < nL && acc[j] != 0.f) atomicAdd(&a.gW[(size_t)(l0 + j) * P + k], acc[j]);
  }
  if (blockIdx.x == 0 && threadIdx.x < kDwLabels && l0 + (int)threadIdx.x < nL) {
    const int l = l0 + threadIdx.x;
    float s = 0.f;
    for (int d = d0; d < d1; ++d) s += a.d_logits[(size_t)d * nL + l];
    if (s != 0.f) {
      if (a.gb != nullptr) atomicAdd(&a.gb[l], s);
      if (a.gb_bow != nullptr) atomicAdd(&a.gb_bow[l], s);
    }
  }
  if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x >= 32 && threadIdx.x < 64) {
    const int lane = threadIdx.x & 31;
    float s = 0.f;
    for (int d = lane; d < a.B; d += 32) s += a.loss_doc[d];
    s = warp_sum(s);
    if (lane == 0) {
      const int nd = a.n_docs_dev != nullptr ? *a.n_docs_dev : a.n_docs;
      *a.loss = s / ((float)max(nd, 1) * (float)nL);
    }
  }
}

bool launch_textcat_head(const TextcatArgs& a, cudaStream_t s) {
  const int P = (a.use_mean + a.use_max) * a.w;
  if (a.nL < 1 || a.nL > kTextcatMaxLabels || P > kTextcatMaxPool || a.ngram > kTextcatMaxNgram) return false;
  if (a.B <= 0) return true;
  int pad_blocks = 0;
  if (a.dX != nullptr) {
    pad_blocks = (a.Tp + kTcWarps - 1) / kTcWarps;
    if (pad_blocks > 148) pad_blocks = 148;
  }
  launch_k(textcat_doc_kernel, dim3(a.B + pad_blocks), dim3(kTcThreads), 0, s, a);
  // doc chunk: about two CTAs per SM in all (short chunks keep the per-thread loop short; at least 4 docs
  // each so the atomics stay a small fraction of the work)
  const int gx = (P + 255) / 256 > 0 ? (P + 255) / 256 : 1, gy = (a.nL + kDwLabels - 1) / kDwLabels;
  int chunk = (int)(((int64_t)a.B * gx * gy + 295) / 296);
  if (chunk < 4) chunk = 4;
  launch_k(textcat_dw_kernel, dim3(gx, gy, (a.B + chunk - 1) / chunk), dim3(256), 0, s, a, chunk);
  return true;
}

}  // namespace srb
