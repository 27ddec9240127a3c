// Launcher API between the torch binding (bindings.cpp) and the .cu files.
// Raw pointers + stream only: the .cu files never include torch headers, so they
// compile in seconds and can be profiled/inspected (cuobjdump) in isolation.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "comm_launch.h"

namespace srb {

struct HashEmbedTables {
  const void* table[8];     // bf16 (n_rows[a], width)
  float* grad[8];           // fp32 (n_rows[a], width) for backward
  uint32_t n_rows[8];
  uint32_t seed[8];
  uint32_t column[8];
  int n_tables;
  int width;
  int n_attr;               // columns of the attrs array
};

// K1: fused hashing + 4-row gather-sum for all tables, written straight into the
// concat layout. out: bf16 (Tp, n_tables*width).
void launch_hash_embed_fwd(const int64_t* attrs, const float* mask, HashEmbedTables t, void* out, int Tp,
                           const GateArgs& gate, cudaStream_t s);
// K1 backward: dE_a[rows] += mask * dY[:, a-block]  (fp32 atomics).
void launch_hash_embed_bwd(const int64_t* attrs, const float* mask, HashEmbedTables t, const void* dY, int Tp,
                           cudaStream_t s);

// K2 epilogue (+K3 LayerNorm, K5 dropout/residual): Z is the raw GEMM output.
//   H = max_p(Z[:, o, p] + b[o, p]); xhat = (H - mu) * rstd; N = xhat*G + beta; D = N*dropmask
//   Y = mask * (X + D | D)
void launch_maxout_ln_fwd(const void* Z, const void* bias, const void* G, const void* beta, const void* X_res,
                          const float* mask, void* Y, uint8_t* which, void* xhat, float* rstd, int Tp, int nO,
                          int nP, float drop_p, uint64_t seed, const int64_t* seed_dev, cudaStream_t s);
// Backward of the same: produces dZ (bf16, routed to the winning piece), dY_masked
// is folded in; accumulates db (nO*nP), dG, dbeta (nO) in fp32.
void launch_maxout_ln_bwd(const void* dY, const void* xhat, const float* rstd, const void* G, const uint8_t* which,
                          const float* mask, void* dZ, float* db, float* dG, float* dbeta, int Tp, int nO, int nP,
                          float drop_p, uint64_t seed, const int64_t* seed_dev, int has_ln, cudaStream_t s);

// Vectorised fast paths (elementwise_fast.cu); return false when the shape is not covered.
bool try_launch_maxout_ln_fwd_vec(const void* Z, const void* bias, const void* G, const void* beta, const void* X_res,
                                  const float* mask, void* Y, uint8_t* which, void* xhat, float* rstd, int Tp, int nO,
                                  int nP, float drop_p, uint64_t seed, const int64_t* seed_dev, cudaStream_t s);
bool try_launch_maxout_ln_bwd_vec(const void* dY, const void* xhat, const float* rstd, const void* G,
                                  const uint8_t* which, const float* mask, void* dZ, float* db, float* dG,
                                  float* dbeta, int Tp, int nO, int nP, float drop_p, uint64_t seed,
                                  const int64_t* seed_dev, int has_ln, cudaStream_t s);
// K1 backward over ids sorted per table: keys/perm are (n_tables, R).
void launch_hash_embed_bwd_sorted(const int64_t* keys, const void* perm, bool perm_is_i32, const float* mask, HashEmbedTables t,
                                  const void* dY, int R, cudaStream_t s);

// K6 fused: logits GEMM + softmax + CE gradient (pitch ldd, zero-initialised by the caller) + loss + argmax
bool try_launch_linear_softmax_xent(const void* X, const void* W, const void* b, const int64_t* labels, void* d_out,
                                    int64_t* guesses, float* loss, int Tp, int w, int nC, int ldd, cudaStream_t s);

// out[c] += sum_t X[t, c]  (bf16 in, fp32 accumulate); false = shape not supported.
bool try_launch_colsum_bf16(const void* X, float* out, int T, int C, int ld, int n_valid, cudaStream_t s);
// dst (bf16, n elements) = src (fp32); src = 0   (n % 8 == 0)
void launch_f32_to_bf16_zero(float* src, void* dst, size_t n, cudaStream_t s);

// K4 helpers for the library-GEMM path: materialised window / its transpose-add.
void launch_seq2col(const void* X, void* Xw, int Tp, int nI, cudaStream_t s);
// dX = col2seq(dXw) (+ residual dY*mask)
void launch_col2seq_residual(const void* dXw, const void* dY, const float* mask, void* dX, int Tp, int nI,
                             int add_residual, cudaStream_t s);

// K6: row softmax + cross-entropy gradient + loss + argmax, logits fp32 or bf16 (Tp, nC).
// logits: fp32 (Tp, ldl) WITHOUT bias (tcgen05 GEMM output); read, then left zeroed
bool launch_softmax_xent_bias(float* logits, const void* b, const int64_t* labels, void* d_out, int64_t* guesses,
                              float* loss, int Tp, int nC, int ldl, int ldd, cudaStream_t s);
void launch_softmax_xent(const float* logits, const int64_t* labels, void* d_out /*bf16*/, int64_t* guesses,
                         float* loss, int Tp, int nC, cudaStream_t s);

// K8: multi-tensor Adam with per-tensor gradient clipping over one shard.
//   key_off/key_len: extents (elements, relative to shard start) of each owned key.
//   hyper: device float[8] = {lr, beta1, beta2, eps, grad_clip, l2, l2_is_wd, grad_scale}
//   step: device int32 update counter (read, not incremented here)
void launch_adam_sumsq(const float* g, const int32_t* blk_key, const int32_t* blk_off, const int64_t* key_off,
                       const int64_t* key_len, float* norms_sq, int n_blocks, const float* hyper, const float* w,
                       cudaStream_t s);
void launch_adam_update(float* g, float* w, float* m1, float* m2, void* w_out_bf16, const int32_t* blk_key,
                        const int32_t* blk_off, const int64_t* key_off, const int64_t* key_len,
                        const float* norms_sq, int n_blocks, const float* hyper, const int32_t* step,
                        cudaStream_t s);
constexpr int kAdamChunk = 4096;   // elements per block

// K7: BILUO transition loop, one warp per doc, whole batch in one launch.
struct BiluoArgs {
  const void* Yf;          // bf16 (Tp, nF*nOP)
  const void* pad;         // bf16 (nF, nOP)
  const void* b;           // bf16 (nOP)
  const void* Wu;          // bf16 (nA, nO)
  const void* bu;          // bf16 (nA)
  const int32_t* doc_starts;   // (B) padded-row index of first token
  const int32_t* doc_lens;     // (B)
  const int32_t* tok_off;      // (B) offset of the doc in unpadded token order
  const int32_t* gold;         // (T) gold action per token (-1 missing) or nullptr
  const float* inv_active;     // (max_len) 1 / #docs still active at step k
  int32_t* feats;              // (T, 3) rows
  uint8_t* which;              // (T, nO)
  void* hid;                   // bf16 (T, nO)
  void* d_scores;              // bf16 (T, ld_scores); columns >= nA stay zero
  int ld_scores;               // row pitch of d_scores (multiple of 128: feeds the tcgen05 GEMMs directly)
  int32_t* actions;            // (T)
  float* loss;                 // scalar accumulator
  int B, nO, nP, nA, nA_pad, n_labels, train;
  int teacher;                 // train only: advance by the oracle's action (when it names one) instead of the arg-max
};
void launch_biluo_steps(BiluoArgs a, cudaStream_t s);
// Scatter d_hid (T, nO) through `which` into dYf (Tp, nF*nOP) fp32, dpad (nF, nOP), db (nOP).
void launch_transition_scatter(const void* d_hid, const uint8_t* which, const int32_t* feats, float* dYf,
                               float* dpad, float* db, int S, int nF, int nO, int nP, cudaStream_t s);

// K7 (parser): arc-eager transition loop with dynamic oracle, one warp per doc.
struct ArcArgs {
  const void* Yf;              // bf16 (Tp, 8*nOP)
  const void* pad;             // bf16 (8, nOP)
  const void* b;               // bf16 (nOP)
  const void* Wu;              // bf16 (nA, nO)
  const void* bu;              // bf16 (nA)
  const int32_t* doc_starts;   // (B)
  const int32_t* doc_lens;     // (B)
  const int32_t* tok_off;      // (B) offset of the doc in unpadded token order
  const int32_t* step_off;     // (B) offset of the doc's step records (capacity 2*len each)
  const int32_t* gold_heads;   // (T) doc-relative gold head (self = root, -1 = missing) or nullptr
  const int32_t* gold_labels;  // (T) gold label or -1
  int32_t* feats;              // (S, 8)
  uint8_t* which;              // (S, nO)
  void* hid;                   // bf16 (S, nO)
  void* d_scores;              // bf16 (S, ld_scores); columns >= nA stay zero
  int ld_scores;
  int32_t* history;            // (S) chosen action per step (optional)
  int32_t* heads_out;          // (T) predicted head (doc-relative, root = self)
  int32_t* labels_out;         // (T) predicted label or -1
  int32_t* n_steps;            // (B)
  float* loss;
  float scale;                 // gradient scale per step (1 / #docs)
  int B, nO, nP, nA, nA_pad, train;
  int max_n;                   // longest doc of the batch (the launcher rounds it up to a multiple of 32)
  int teacher;                 // train only: advance by the first minimum-cost action instead of the arg-max
};
bool launch_arc_eager_steps(ArcArgs a, cudaStream_t s);
int arc_eager_max_doc_len(int nO, int nP, int nA);
// Textcat head (textcat_kernels.cu): pooling / bag of n-grams -> logits -> softmax | logistic | identity ->
// d_logits, loss, dX and every parameter gradient, for a whole batch in two launches.
constexpr int kTextcatMaxLabels = 128;
constexpr int kTextcatMaxPool = 1024;     // n_pool * width
constexpr int kTextcatMaxNgram = 8;
struct TextcatArgs {
  const void* X;               // bf16 (Tp, w) tok2vec output, or nullptr (bag of words only)
  const float* mask;           // (Tp) 1.0 on real tokens
  const int64_t* attrs;        // (Tp, n_attr); column 0 = NORM id (bag of words)
  const int32_t* doc_starts;   // (B)
  const int32_t* doc_lens;     // (B)
  const int32_t* n_docs_dev;   // real doc count on the device, or nullptr: n_docs
  const void* W;               // (nL, P) output layer or nullptr; P = (use_mean + use_max) * w
  const void* b;               // (nL) or nullptr
  const void* W_bow;           // (bow_rows, nL) or nullptr
  const void* b_bow;           // (nL) or nullptr
  const float* truths;         // (B, nL)
  const float* known;          // (B, nL)
  float* scores;               // (B, nL)
  float* pooled;               // (B, P) scratch
  float* d_logits;             // (B, nL) scratch
  float* loss_doc;             // (B) scratch
  float* loss;                 // scalar, written
  void* dX;                    // bf16 (Tp, w) or nullptr
  float* gW;                   // fp32 gradient accumulators (+=), or nullptr
  float* gb;
  float* gW_bow;
  float* gb_bow;
  int64_t bow_rows;
  int n_docs, B, Tp, w, n_attr, nL, use_mean, use_max;
  int act;                     // 0 softmax, 1 logistic, 2 none (no_output_layer)
  int ngram;
  int W_f32, b_f32, W_bow_f32, b_bow_f32;   // weight dtypes: 1 = fp32, 0 = bf16
};
// false: shape outside the kernels' range (labels, n_pool * width, ngram_size)
bool launch_textcat_head(const TextcatArgs& a, cudaStream_t s);
extern int g_pdl;                                      // launch.h
// words [0, n_zero) <- 0, [n_zero, n_zero + n_ones) <- 0xFFFFFFFF; both counts multiples of 4, p 16-byte aligned
void launch_bump_i64(int64_t* p, int64_t by, cudaStream_t s);
void launch_arena_init(void* p, size_t n_zero_words, size_t n_ones_words, cudaStream_t s);

}  // namespace srb
