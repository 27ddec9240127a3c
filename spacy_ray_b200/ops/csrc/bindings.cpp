// torch.ops.srb.* bindings: tensor checks + raw-pointer launchers (kernels.h).
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/types.h>

#include <vector>

#include "gemm.h"
#include "kernels.h"
#include "comm.h"

namespace {

using at::Tensor;

#define SRB_CHECK_CUDA(x) TORCH_CHECK((x).is_cuda() && (x).is_contiguous(), #x " must be a contiguous CUDA tensor")
#define SRB_CHECK_BF16(x) TORCH_CHECK((x).scalar_type() == at::kBFloat16, #x " must be bfloat16")

cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }
const void* optptr(const c10::optional<Tensor>& t) { return t.has_value() && t->defined() ? t->data_ptr() : nullptr; }

srb::HashEmbedTables make_tables(const std::vector<Tensor>& tables, const std::vector<int64_t>& seeds,
                                 const std::vector<int64_t>& columns, int n_attr) {
  TORCH_CHECK(tables.size() <= 8 && tables.size() == seeds.size() && tables.size() == columns.size());
  srb::HashEmbedTables t{};
  t.n_tables = (int)tables.size();
  t.width = (int)tables[0].size(1);
  t.n_attr = n_attr;
  TORCH_CHECK(t.width % 8 == 0, "HashEmbed width must be a multiple of 8");
  for (size_t a = 0; a < tables.size(); ++a) {
    t.n_rows[a] = (uint32_t)tables[a].size(0);
    t.seed[a] = (uint32_t)seeds[a];
    t.column[a] = (uint32_t)columns[a];
  }
  return t;
}

Tensor hash_embed_fwd(const Tensor& attrs, const Tensor& mask, std::vector<Tensor> tables, std::vector<int64_t> seeds,
                      std::vector<int64_t> columns, std::vector<int64_t> gate) {
  SRB_CHECK_CUDA(attrs); SRB_CHECK_CUDA(mask);
  TORCH_CHECK(attrs.scalar_type() == at::kLong && mask.scalar_type() == at::kFloat);
  c10::cuda::CUDAGuard guard(attrs.device());
  auto t = make_tables(tables, seeds, columns, (int)attrs.size(1));
  for (size_t a = 0; a < tables.size(); ++a) { SRB_CHECK_CUDA(tables[a]); SRB_CHECK_BF16(tables[a]); t.table[a] = tables[a].data_ptr(); }
  const int Tp = (int)attrs.size(0);
  Tensor out = at::empty({Tp, (int64_t)t.n_tables * t.width}, attrs.options().dtype(at::kBFloat16));
  srb::launch_hash_embed_fwd(attrs.data_ptr<int64_t>(), mask.data_ptr<float>(), t, out.data_ptr(), Tp,
                             srb::make_gate_args(gate.data(), gate.size()), cur_stream());
  return out;
}

void hash_embed_bwd(const Tensor& dY, const Tensor& attrs, const Tensor& mask, std::vector<Tensor> grads,
                    std::vector<int64_t> seeds, std::vector<int64_t> columns) {
  SRB_CHECK_CUDA(dY); SRB_CHECK_BF16(dY); SRB_CHECK_CUDA(attrs);
  c10::cuda::CUDAGuard guard(attrs.device());
  auto t = make_tables(grads, seeds, columns, (int)attrs.size(1));
  for (size_t a = 0; a < grads.size(); ++a) {
    SRB_CHECK_CUDA(grads[a]);
    TORCH_CHECK(grads[a].scalar_type() == at::kFloat, "table gradients must be fp32");
    t.grad[a] = grads[a].data_ptr<float>();
  }
  srb::launch_hash_embed_bwd(attrs.data_ptr<int64_t>(), mask.data_ptr<float>(), t, dY.data_ptr(), (int)attrs.size(0),
                             cur_stream());
}

void hash_embed_bwd_sorted(const Tensor& dY, const Tensor& keys, const Tensor& perm, const Tensor& mask,
                           std::vector<Tensor> grads, std::vector<int64_t> seeds, std::vector<int64_t> columns) {
  SRB_CHECK_CUDA(dY); SRB_CHECK_BF16(dY); SRB_CHECK_CUDA(keys); SRB_CHECK_CUDA(perm);
  // keys: the raw (R, n_attr) attribute array; perm: (n_tables, R) row order sorted per table
  TORCH_CHECK(keys.scalar_type() == at::kLong && keys.dim() == 2 && perm.is_contiguous() &&
              (perm.scalar_type() == at::kLong || perm.scalar_type() == at::kInt));
  TORCH_CHECK(perm.size(0) == (int64_t)grads.size() && perm.size(1) == keys.size(0) && grads[0].size(1) <= 512);
  c10::cuda::CUDAGuard guard(dY.device());
  auto t = make_tables(grads, seeds, columns, (int)keys.size(1));
  for (size_t a = 0; a < grads.size(); ++a) {
    SRB_CHECK_CUDA(grads[a]);
    TORCH_CHECK(grads[a].scalar_type() == at::kFloat, "table gradients must be fp32");
    t.grad[a] = grads[a].data_ptr<float>();
  }
  srb::launch_hash_embed_bwd_sorted(keys.data_ptr<int64_t>(), perm.data_ptr(), perm.scalar_type() == at::kInt,
                                    mask.data_ptr<float>(), t,
                                    dY.data_ptr(), (int)perm.size(1), cur_stream());
}

// out (C,) fp32 += column sums of X (T, C) bf16
void colsum_acc(const Tensor& X, Tensor out, int64_t n_valid) {
  TORCH_CHECK(X.is_cuda(), "X must be a CUDA tensor"); SRB_CHECK_BF16(X); SRB_CHECK_CUDA(out);   // X rows may be strided
  const int64_t nv = n_valid > 0 ? n_valid : X.size(1);
  TORCH_CHECK(X.dim() == 2 && X.stride(1) == 1 && out.scalar_type() == at::kFloat && out.is_contiguous() &&
              nv <= X.size(1) && out.numel() >= nv);
  c10::cuda::CUDAGuard guard(X.device());
  const bool ok = srb::try_launch_colsum_bf16(X.data_ptr(), out.data_ptr<float>(), (int)X.size(0), (int)X.size(1),
                                              (int)X.stride(0), (int)nv, cur_stream());
  TORCH_CHECK(ok, "colsum_acc: unsupported shape (C must be a multiple of 8, <= 2048)");
}

// out (bf16, same shape) = src; src = 0 (see launch_f32_to_bf16_zero)
Tensor f32_to_bf16_zero(Tensor src) {
  SRB_CHECK_CUDA(src);
  TORCH_CHECK(src.scalar_type() == at::kFloat && src.numel() % 8 == 0);
  c10::cuda::CUDAGuard guard(src.device());
  Tensor out = at::empty(src.sizes(), src.options().dtype(at::kBFloat16));
  srb::launch_f32_to_bf16_zero(src.data_ptr<float>(), out.data_ptr(), (size_t)src.numel(), cur_stream());
  return out;
}

std::vector<Tensor> maxout_ln_fwd(const Tensor& Z, const c10::optional<Tensor>& bias, const c10::optional<Tensor>& G,
                                  const c10::optional<Tensor>& beta, const c10::optional<Tensor>& Xres,
                                  const Tensor& mask, int64_t nO, int64_t nP, double drop_p, int64_t seed,
                                  const c10::optional<Tensor>& seed_dev) {
  SRB_CHECK_CUDA(Z); SRB_CHECK_BF16(Z);
  TORCH_CHECK(nO % 32 == 0 && nO <= 512 && (nO * nP) % 8 == 0, "maxout_ln: nO must be a multiple of 32, <= 512");
  TORCH_CHECK(Z.size(1) == nO * nP);
  c10::cuda::CUDAGuard guard(Z.device());
  const int Tp = (int)Z.size(0);
  auto bf = Z.options();
  Tensor Y = at::empty({Tp, nO}, bf);
  Tensor which = nP > 1 ? at::empty({Tp, nO}, bf.dtype(at::kByte)) : at::empty({0}, bf.dtype(at::kByte));
  const bool has_ln = G.has_value() && G->defined();
  Tensor xhat = has_ln ? at::empty({Tp, nO}, bf) : at::empty({0}, bf);
  Tensor rstd = has_ln ? at::empty({Tp}, bf.dtype(at::kFloat)) : at::empty({0}, bf.dtype(at::kFloat));
  srb::launch_maxout_ln_fwd(Z.data_ptr(), optptr(bias), optptr(G), optptr(beta), optptr(Xres), mask.data_ptr<float>(),
                            Y.data_ptr(), nP > 1 ? which.data_ptr<uint8_t>() : nullptr, has_ln ? xhat.data_ptr() : nullptr,
                            has_ln ? rstd.data_ptr<float>() : nullptr, Tp, (int)nO, (int)nP, (float)drop_p,
                            (uint64_t)seed, (const int64_t*)optptr(seed_dev), cur_stream());
  return {Y, which, xhat, rstd};
}

Tensor maxout_ln_bwd(const Tensor& dY, const c10::optional<Tensor>& xhat, const c10::optional<Tensor>& rstd,
                     const c10::optional<Tensor>& G, const Tensor& which, const Tensor& mask, int64_t nP,
                     double drop_p, int64_t seed, Tensor db, c10::optional<Tensor> dG, c10::optional<Tensor> dbeta,
                     const c10::optional<Tensor>& seed_dev) {
  SRB_CHECK_CUDA(dY); SRB_CHECK_BF16(dY);
  c10::cuda::CUDAGuard guard(dY.device());
  const int Tp = (int)dY.size(0), nO = (int)dY.size(1);
  const bool has_ln = G.has_value() && G->defined();
  Tensor dZ = at::empty({Tp, (int64_t)nO * nP}, dY.options());
  srb::launch_maxout_ln_bwd(dY.data_ptr(), optptr(xhat), has_ln ? rstd->data_ptr<float>() : nullptr, optptr(G),
                            which.data_ptr<uint8_t>(), mask.data_ptr<float>(), dZ.data_ptr(), db.data_ptr<float>(),
                            has_ln ? dG->data_ptr<float>() : nullptr, has_ln ? dbeta->data_ptr<float>() : nullptr,
                            Tp, nO, (int)nP, (float)drop_p, (uint64_t)seed, (const int64_t*)optptr(seed_dev),
                            has_ln ? 1 : 0, cur_stream());
  return dZ;
}

Tensor seq2col(const Tensor& X) {
  SRB_CHECK_CUDA(X); SRB_CHECK_BF16(X);
  TORCH_CHECK(X.size(1) % 8 == 0);
  c10::cuda::CUDAGuard guard(X.device());
  Tensor Xw = at::empty({X.size(0), X.size(1) * 3}, X.options());
  srb::launch_seq2col(X.data_ptr(), Xw.data_ptr(), (int)X.size(0), (int)X.size(1), cur_stream());
  return Xw;
}

Tensor col2seq_residual(const Tensor& dXw, const c10::optional<Tensor>& dY, const Tensor& mask) {
  SRB_CHECK_CUDA(dXw); SRB_CHECK_BF16(dXw);
  c10::cuda::CUDAGuard guard(dXw.device());
  const int Tp = (int)dXw.size(0), nI = (int)dXw.size(1) / 3;
  Tensor dX = at::empty({Tp, nI}, dXw.options());
  srb::launch_col2seq_residual(dXw.data_ptr(), optptr(dY), mask.data_ptr<float>(), dX.data_ptr(), Tp, nI,
                               dY.has_value() && dY->defined() ? 1 : 0, cur_stream());
  return dX;
}

std::vector<Tensor> softmax_xent(const Tensor& logits, const Tensor& labels) {
  SRB_CHECK_CUDA(logits); SRB_CHECK_CUDA(labels);
  TORCH_CHECK(logits.scalar_type() == at::kFloat && labels.scalar_type() == at::kLong);
  TORCH_CHECK(logits.size(1) <= 256, "softmax_xent: at most 256 classes");
  c10::cuda::CUDAGuard guard(logits.device());
  const int Tp = (int)logits.size(0), nC = (int)logits.size(1);
  Tensor d = at::empty({Tp, nC}, logits.options().dtype(at::kBFloat16));
  Tensor guesses = at::empty({Tp}, logits.options().dtype(at::kLong));
  Tensor loss = at::zeros({}, logits.options());
  srb::launch_softmax_xent(logits.data_ptr<float>(), labels.data_ptr<int64_t>(), d.data_ptr(),
                           guesses.data_ptr<int64_t>(), loss.data_ptr<float>(), Tp, nC, cur_stream());
  return {d, guesses, loss};
}

// A record arena: one allocation carved into typed views, initialised by ONE kernel of ours
// (zero part first, then the "-1" part) instead of one library fill per tensor.
struct Arena {
  std::vector<int64_t> off, bytes;
  int64_t zero_bytes = 0, total = 0;
  bool in_ones = false;
  static int64_t up16(int64_t n) { return (n + 15) / 16 * 16; }
  int add(int64_t nbytes, bool ones = false) {
    TORCH_CHECK(ones || !in_ones, "Arena: zero-initialised parts first");
    if (ones && !in_ones) { in_ones = true; zero_bytes = total; }
    off.push_back(total); bytes.push_back(nbytes);
    total += up16(nbytes);
    return (int)off.size() - 1;
  }
  Tensor buf;
  void alloc(const at::TensorOptions& o, cudaStream_t s) {
    if (!in_ones) zero_bytes = total;
    buf = at::empty({total}, o.dtype(at::kByte));
    if (total) srb::launch_arena_init(buf.data_ptr(), (size_t)zero_bytes / 4, (size_t)(total - zero_bytes) / 4, s);
  }
  Tensor view(int i, at::ScalarType dt, at::IntArrayRef shape) const {
    return buf.narrow(0, off[i], bytes[i]).view(dt).view(shape);
  }
};

// Tagger head in one kernel.  Returns {d (Tp, ldd) bf16 with ldd = 128-multiple and zeros past nC, guesses, loss};
// an empty list when the shape is outside the kernel's range (caller falls back to GEMM + softmax_xent).
std::vector<Tensor> linear_softmax_xent(const Tensor& X, const Tensor& W, const Tensor& b, const Tensor& labels) {
  SRB_CHECK_CUDA(X); SRB_CHECK_BF16(X); SRB_CHECK_CUDA(W); SRB_CHECK_BF16(W); SRB_CHECK_CUDA(b); SRB_CHECK_BF16(b);
  SRB_CHECK_CUDA(labels);
  TORCH_CHECK(labels.scalar_type() == at::kLong && X.dim() == 2 && W.dim() == 2 && W.size(1) == X.size(1));
  c10::cuda::CUDAGuard guard(X.device());
  const int Tp = (int)X.size(0), w = (int)X.size(1), nC = (int)W.size(0);
  const int64_t ldd = ((nC + 7) / 8 * 8 + 127) / 128 * 128;
  Arena ar;
  const int i_d = ar.add((int64_t)Tp * ldd * 2), i_loss = ar.add(4);
  ar.alloc(X.options(), cur_stream());
  Tensor d = ar.view(i_d, at::kBFloat16, {Tp, ldd});
  Tensor guesses = at::empty({Tp}, X.options().dtype(at::kLong));
  Tensor loss = ar.view(i_loss, at::kFloat, {});
  const bool ok = srb::try_launch_linear_softmax_xent(X.data_ptr(), W.data_ptr(), b.data_ptr(), labels.data_ptr<int64_t>(),
                                                      d.data_ptr(), guesses.data_ptr<int64_t>(), loss.data_ptr<float>(),
                                                      Tp, w, nC, (int)ldd, cur_stream());
  if (!ok) return {};
  return {d, guesses, loss};
}

// Second half of the tensor-core tagger head: logits (Tp, ldl) fp32 without bias -> {d (Tp, ldd) bf16, zeros past
// nC, guesses, loss}; `logits` is zeroed again on the way (persistent scratch of the caller).
std::vector<Tensor> softmax_xent_bias(Tensor logits, const Tensor& b, const Tensor& labels, int64_t nC) {
  SRB_CHECK_CUDA(logits); SRB_CHECK_CUDA(b); SRB_CHECK_BF16(b); SRB_CHECK_CUDA(labels);
  TORCH_CHECK(logits.scalar_type() == at::kFloat && logits.dim() == 2 && logits.stride(1) == 1 &&
              labels.scalar_type() == at::kLong && b.numel() >= nC && nC <= 128);
  c10::cuda::CUDAGuard guard(logits.device());
  const int Tp = (int)logits.size(0);
  const int64_t ldd = ((nC + 7) / 8 * 8 + 127) / 128 * 128;
  auto o = logits.options();
  Arena ar;
  const int i_d = ar.add((int64_t)Tp * ldd * 2), i_loss = ar.add(4);
  ar.alloc(o, cur_stream());
  Tensor d = ar.view(i_d, at::kBFloat16, {Tp, ldd});
  Tensor guesses = at::empty({Tp}, o.dtype(at::kLong));
  Tensor loss = ar.view(i_loss, at::kFloat, {});
  TORCH_CHECK(srb::launch_softmax_xent_bias(logits.data_ptr<float>(), b.data_ptr(), labels.data_ptr<int64_t>(),
                                            d.data_ptr(), guesses.data_ptr<int64_t>(), loss.data_ptr<float>(), Tp,
                                            (int)nC, (int)logits.stride(0), (int)ldd, cur_stream()),
              "softmax_xent_bias: unsupported class count");
  return {d, guesses, loss};
}

void adam_shard(Tensor g, Tensor w, Tensor m1, Tensor m2, c10::optional<Tensor> w_out, const Tensor& blk_key,
                const Tensor& blk_off, const Tensor& key_off, const Tensor& key_len, Tensor norms, const Tensor& hyper,
                const Tensor& step) {
  SRB_CHECK_CUDA(g); SRB_CHECK_CUDA(w);
  TORCH_CHECK(g.scalar_type() == at::kFloat && w.scalar_type() == at::kFloat);
  c10::cuda::CUDAGuard guard(g.device());
  const int nb = (int)blk_key.numel();
  auto s = cur_stream();
  cudaMemsetAsync(norms.data_ptr(), 0, norms.numel() * sizeof(float), s);
  srb::launch_adam_sumsq(g.data_ptr<float>(), blk_key.data_ptr<int32_t>(), blk_off.data_ptr<int32_t>(),
                         key_off.data_ptr<int64_t>(), key_len.data_ptr<int64_t>(), norms.data_ptr<float>(), nb,
                         hyper.data_ptr<float>(), w.data_ptr<float>(), s);
  srb::launch_adam_update(g.data_ptr<float>(), w.data_ptr<float>(), m1.data_ptr<float>(), m2.data_ptr<float>(),
                          w_out.has_value() && w_out->defined() ? w_out->data_ptr() : nullptr,
                          blk_key.data_ptr<int32_t>(), blk_off.data_ptr<int32_t>(), key_off.data_ptr<int64_t>(),
                          key_len.data_ptr<int64_t>(), norms.data_ptr<float>(), nb, hyper.data_ptr<float>(),
                          step.data_ptr<int32_t>(), s);
}

std::vector<Tensor> biluo_steps(const Tensor& Yf, const Tensor& pad, const Tensor& b, const Tensor& Wu,
                                const Tensor& bu, const Tensor& doc_starts, const Tensor& doc_lens,
                                const Tensor& tok_off, const c10::optional<Tensor>& gold, const Tensor& inv_active,
                                int64_t n_tokens, int64_t nO, int64_t nP, int64_t n_labels, bool train, bool teacher) {
  SRB_CHECK_CUDA(Yf); SRB_CHECK_BF16(Yf); SRB_CHECK_BF16(pad); SRB_CHECK_BF16(b); SRB_CHECK_BF16(Wu); SRB_CHECK_BF16(bu);
  TORCH_CHECK(nP == 2 && nO % 32 == 0 && (nO * nP) / 32 <= 8, "biluo_steps: hidden width/pieces not supported");
  c10::cuda::CUDAGuard guard(Yf.device());
  const int64_t nA = Wu.size(0);
  TORCH_CHECK(nA == 4 * n_labels + 1 && nA <= 256);
  const int64_t nA_pad = (nA + 7) / 8 * 8;
  auto o = Yf.options();
  const int64_t T = n_tokens;
  Tensor feats = at::empty({train ? T : 0, 3}, o.dtype(at::kInt));
  Tensor which = at::empty({train ? T : 0, nO}, o.dtype(at::kByte));
  const int64_t ldd = (nA_pad + 127) / 128 * 128;             // GEMM-friendly pitch (dWu / d_hid run on tcgen05)
  const int64_t Tr = train ? T : 0;
  Arena ar;                                                   // rows past the real token count stay zero
  const int i_hid = ar.add(Tr * nO * 2), i_ds = ar.add(Tr * ldd * 2), i_loss = ar.add(4);
  ar.alloc(o, cur_stream());                                  // (fixed-capacity batches under CUDA graphs)
  Tensor hid = ar.view(i_hid, at::kBFloat16, {Tr, nO});
  Tensor d_scores = ar.view(i_ds, at::kBFloat16, {Tr, ldd});
  Tensor actions = at::empty({T}, o.dtype(at::kInt));
  Tensor loss = ar.view(i_loss, at::kFloat, {});
  srb::BiluoArgs a{};
  a.Yf = Yf.data_ptr(); a.pad = pad.data_ptr(); a.b = b.data_ptr(); a.Wu = Wu.data_ptr(); a.bu = bu.data_ptr();
  a.doc_starts = doc_starts.data_ptr<int32_t>(); a.doc_lens = doc_lens.data_ptr<int32_t>();
  a.tok_off = tok_off.data_ptr<int32_t>();
  a.gold = gold.has_value() && gold->defined() ? gold->data_ptr<int32_t>() : nullptr;
  a.inv_active = inv_active.data_ptr<float>();
  a.feats = feats.data_ptr<int32_t>(); a.which = which.data_ptr<uint8_t>(); a.hid = hid.data_ptr();
  a.d_scores = d_scores.data_ptr(); a.actions = actions.data_ptr<int32_t>(); a.loss = loss.data_ptr<float>();
  a.B = (int)doc_lens.numel(); a.nO = (int)nO; a.nP = (int)nP; a.nA = (int)nA; a.nA_pad = (int)nA_pad; a.ld_scores = (int)ldd;
  a.n_labels = (int)n_labels; a.train = train ? 1 : 0; a.teacher = (train && teacher) ? 1 : 0;
  srb::launch_biluo_steps(a, cur_stream());
  return {feats, which, hid, d_scores, actions, loss};
}

std::vector<Tensor> arc_eager_steps(const Tensor& Yf, const Tensor& pad, const Tensor& b, const Tensor& Wu,
                                    const Tensor& bu, const Tensor& doc_starts, const Tensor& doc_lens,
                                    const Tensor& tok_off, const Tensor& step_off,
                                    const c10::optional<Tensor>& gold_heads, const c10::optional<Tensor>& gold_labels,
                                    int64_t n_tokens, int64_t n_steps_cap, int64_t nO, int64_t nP, double scale,
                                    bool train, bool teacher, int64_t max_len) {
  SRB_CHECK_CUDA(Yf); SRB_CHECK_BF16(Yf); SRB_CHECK_BF16(pad); SRB_CHECK_BF16(b); SRB_CHECK_BF16(Wu); SRB_CHECK_BF16(bu);
  c10::cuda::CUDAGuard guard(Yf.device());
  const int64_t nA = Wu.size(0);
  const int64_t nA_pad = (nA + 7) / 8 * 8;
  auto o = Yf.options();
  const int64_t S = train ? n_steps_cap : 0;
  // record slots past a doc's last step stay inert: zero gradient, piece 0, "missing" features
  const int64_t ldd = (nA_pad + 127) / 128 * 128;
  const int64_t Bn = doc_lens.numel();
  Arena ar;
  const int i_which = ar.add(S * nO), i_hid = ar.add(S * nO * 2), i_ds = ar.add(S * ldd * 2), i_ns = ar.add(Bn * 4),
            i_loss = ar.add(4), i_feats = ar.add(S * 8 * 4, true), i_hist = ar.add(n_steps_cap * 4, true);
  ar.alloc(o, cur_stream());
  Tensor feats = ar.view(i_feats, at::kInt, {S, 8});
  Tensor which = ar.view(i_which, at::kByte, {S, nO});
  Tensor hid = ar.view(i_hid, at::kBFloat16, {S, nO});
  Tensor d_scores = ar.view(i_ds, at::kBFloat16, {S, ldd});
  Tensor history = ar.view(i_hist, at::kInt, {n_steps_cap});
  Tensor heads = at::empty({n_tokens}, o.dtype(at::kInt));
  Tensor labels = at::empty({n_tokens}, o.dtype(at::kInt));
  Tensor n_steps = ar.view(i_ns, at::kInt, {Bn});
  Tensor loss = ar.view(i_loss, at::kFloat, {});
  srb::ArcArgs a{};
  a.Yf = Yf.data_ptr(); a.pad = pad.data_ptr(); a.b = b.data_ptr(); a.Wu = Wu.data_ptr(); a.bu = bu.data_ptr();
  a.doc_starts = doc_starts.data_ptr<int32_t>(); a.doc_lens = doc_lens.data_ptr<int32_t>();
  a.tok_off = tok_off.data_ptr<int32_t>(); a.step_off = step_off.data_ptr<int32_t>();
  const bool have_gold = gold_heads.has_value() && gold_heads->defined();
  a.gold_heads = have_gold ? gold_heads->data_ptr<int32_t>() : nullptr;
  a.gold_labels = have_gold ? gold_labels->data_ptr<int32_t>() : nullptr;
  a.feats = feats.data_ptr<int32_t>(); a.which = which.data_ptr<uint8_t>(); a.hid = hid.data_ptr();
  a.d_scores = d_scores.data_ptr(); a.history = history.data_ptr<int32_t>();
  a.heads_out = heads.data_ptr<int32_t>(); a.labels_out = labels.data_ptr<int32_t>();
  a.n_steps = n_steps.data_ptr<int32_t>(); a.loss = loss.data_ptr<float>();
  a.scale = (float)scale;
  a.teacher = (train && teacher) ? 1 : 0;
  a.max_n = (int)max_len;
  a.B = (int)doc_lens.numel(); a.nO = (int)nO; a.nP = (int)nP; a.nA = (int)nA; a.nA_pad = (int)nA_pad; a.ld_scores = (int)ldd;
  a.train = train ? 1 : 0;
  TORCH_CHECK(srb::launch_arc_eager_steps(a, cur_stream()), "arc_eager_steps: unsupported hidden width / pieces / #actions");
  return {feats, which, hid, d_scores, history, heads, labels, n_steps, loss};
}

void transition_scatter(const Tensor& d_hid, const Tensor& which, const Tensor& feats, Tensor dYf, Tensor dpad,
                        Tensor db, int64_t nF, int64_t nP) {
  SRB_CHECK_CUDA(d_hid); SRB_CHECK_BF16(d_hid);
  c10::cuda::CUDAGuard guard(d_hid.device());
  srb::launch_transition_scatter(d_hid.data_ptr(), which.data_ptr<uint8_t>(), feats.data_ptr<int32_t>(),
                                 dYf.data_ptr<float>(), dpad.data_ptr<float>(), db.data_ptr<float>(),
                                 (int)d_hid.size(0), (int)nF, (int)d_hid.size(1), (int)nP, cur_stream());
}

// Textcat head: {loss (scalar), scores (B, nL) fp32, dX (Tp, w) bf16 or empty, pooled, d_logits}.  Parameter
// gradients are ACCUMULATED into gW / gb / gW_bow / gb_bow (fp32; may be views of the flat gradient bucket).
int weight_is_f32(const c10::optional<Tensor>& t, const char* name) {
  if (!t.has_value() || !t->defined()) return 0;
  TORCH_CHECK(t->is_cuda() && t->is_contiguous(), name, " must be a contiguous CUDA tensor");
  TORCH_CHECK(t->scalar_type() == at::kFloat || t->scalar_type() == at::kBFloat16, name, " must be fp32 or bf16");
  return t->scalar_type() == at::kFloat ? 1 : 0;
}
float* grad_ptr(const c10::optional<Tensor>& t, int64_t numel, const char* name) {
  if (!t.has_value() || !t->defined()) return nullptr;
  TORCH_CHECK(t->is_cuda() && t->is_contiguous() && t->scalar_type() == at::kFloat && t->numel() == numel,
              name, " must be a contiguous fp32 CUDA tensor of ", numel, " elements");
  return t->data_ptr<float>();
}

std::vector<Tensor> textcat_head(const c10::optional<Tensor>& X, const Tensor& mask, const Tensor& attrs,
                                 const Tensor& doc_starts, const Tensor& doc_lens, const c10::optional<Tensor>& n_docs_dev,
                                 int64_t n_docs, const c10::optional<Tensor>& W, const c10::optional<Tensor>& b,
                                 const c10::optional<Tensor>& W_bow, const c10::optional<Tensor>& b_bow,
                                 const Tensor& truths, const Tensor& known, const c10::optional<Tensor>& gW,
                                 const c10::optional<Tensor>& gb, const c10::optional<Tensor>& gW_bow,
                                 const c10::optional<Tensor>& gb_bow, int64_t n_labels, bool use_mean, bool use_max,
                                 int64_t act, int64_t ngram) {
  SRB_CHECK_CUDA(mask); SRB_CHECK_CUDA(attrs); SRB_CHECK_CUDA(doc_starts); SRB_CHECK_CUDA(doc_lens);
  SRB_CHECK_CUDA(truths); SRB_CHECK_CUDA(known);
  TORCH_CHECK(mask.scalar_type() == at::kFloat && attrs.scalar_type() == at::kLong && attrs.dim() == 2 &&
              doc_starts.scalar_type() == at::kInt && doc_lens.scalar_type() == at::kInt);
  const int64_t B = doc_lens.numel(), nL = n_labels;
  TORCH_CHECK(truths.scalar_type() == at::kFloat && known.scalar_type() == at::kFloat &&
              truths.numel() == B * nL && known.numel() == B * nL, "truths / known must be fp32 (B, n_labels)");
  const bool has_x = X.has_value() && X->defined();
  const bool has_w = W.has_value() && W->defined();
  const bool has_bow = W_bow.has_value() && W_bow->defined();
  TORCH_CHECK(has_x == has_w, "textcat_head: X and W come together (the pooled branch)");
  TORCH_CHECK(has_x || has_bow, "textcat_head: nothing to compute");
  c10::cuda::CUDAGuard guard(attrs.device());
  srb::TextcatArgs a{};
  const int64_t Tp = attrs.size(0);
  const int64_t w = has_x ? X->size(1) : 0;
  if (has_x) {
    SRB_CHECK_CUDA(*X); SRB_CHECK_BF16(*X);
    TORCH_CHECK(X->size(0) == Tp && mask.numel() == Tp);
  }
  const int64_t P = (has_x ? (int64_t)use_mean + (int64_t)use_max : 0) * w;
  a.W_f32 = weight_is_f32(W, "W"); a.b_f32 = weight_is_f32(b, "b");
  a.W_bow_f32 = weight_is_f32(W_bow, "W_bow"); a.b_bow_f32 = weight_is_f32(b_bow, "b_bow");
  if (has_w) TORCH_CHECK(W->numel() == nL * P, "W must be (n_labels, n_pool * width)");
  if (has_bow) TORCH_CHECK(W_bow->dim() == 2 && W_bow->size(1) == nL, "W_bow must be (rows, n_labels)");
  if (n_docs_dev.has_value() && n_docs_dev->defined()) {
    TORCH_CHECK(n_docs_dev->is_cuda() && n_docs_dev->scalar_type() == at::kInt && n_docs_dev->numel() >= 1);
    a.n_docs_dev = n_docs_dev->data_ptr<int32_t>();
  }
  auto o = truths.options();
  Tensor loss = at::empty({}, o);
  Tensor scores = at::empty({B, nL}, o);
  Tensor pooled = at::empty({B, P}, o);
  Tensor d_logits = at::empty({B, nL}, o);
  Tensor loss_doc = at::empty({B}, o);
  Tensor dX = has_x ? at::empty({Tp, w}, X->options()) : at::empty({0}, o.dtype(at::kBFloat16));
  a.X = has_x ? X->data_ptr() : nullptr;
  a.mask = mask.data_ptr<float>(); a.attrs = attrs.data_ptr<int64_t>();
  a.doc_starts = doc_starts.data_ptr<int32_t>(); a.doc_lens = doc_lens.data_ptr<int32_t>();
  a.W = optptr(W); a.b = optptr(b); a.W_bow = optptr(W_bow); a.b_bow = optptr(b_bow);
  a.truths = truths.data_ptr<float>(); a.known = known.data_ptr<float>();
  a.scores = scores.data_ptr<float>(); a.pooled = pooled.data_ptr<float>(); a.d_logits = d_logits.data_ptr<float>();
  a.loss_doc = loss_doc.data_ptr<float>(); a.loss = loss.data_ptr<float>();
  a.dX = has_x ? dX.data_ptr() : nullptr;
  a.gW = grad_ptr(gW, nL * P, "gW"); a.gb = grad_ptr(gb, nL, "gb");
  a.gW_bow = has_bow ? grad_ptr(gW_bow, W_bow->numel(), "gW_bow") : nullptr;
  a.gb_bow = grad_ptr(gb_bow, nL, "gb_bow");
  a.bow_rows = has_bow ? W_bow->size(0) : 1;
  a.n_docs = (int)n_docs; a.B = (int)B; a.Tp = (int)Tp; a.w = (int)w; a.n_attr = (int)attrs.size(1); a.nL = (int)nL;
  a.use_mean = (has_x && use_mean) ? 1 : 0; a.use_max = (has_x && use_max) ? 1 : 0;
  a.act = (int)act; a.ngram = has_bow ? (int)ngram : 0;
  TORCH_CHECK(srb::launch_textcat_head(a, cur_stream()),
              "textcat_head: outside the kernels' range (labels <= ", srb::kTextcatMaxLabels, ", n_pool * width <= ",
              srb::kTextcatMaxPool, ", ngram_size <= ", srb::kTextcatMaxNgram, ")");
  return {loss, scores, dX, pooled, d_logits};
}

}  // namespace

TORCH_LIBRARY(srb, m) {
  m.def("hash_embed_fwd(Tensor attrs, Tensor mask, Tensor[] tables, int[] seeds, int[] columns, int[] gate) -> Tensor");
  m.def("hash_embed_bwd(Tensor dY, Tensor attrs, Tensor mask, Tensor[] grads, int[] seeds, int[] columns) -> ()");
  m.def("hash_embed_bwd_sorted(Tensor dY, Tensor keys, Tensor perm, Tensor mask, Tensor[] grads, int[] seeds, int[] columns) -> ()");
  m.def("colsum_acc(Tensor X, Tensor(a!) out, int n_valid) -> ()");
  m.def("f32_to_bf16_zero(Tensor(a!) src) -> Tensor");
  m.def("maxout_ln_fwd(Tensor Z, Tensor? bias, Tensor? G, Tensor? beta, Tensor? Xres, Tensor mask, int nO, int nP, float drop_p, int seed, Tensor? seed_dev) -> Tensor[]");
  m.def("maxout_ln_bwd(Tensor dY, Tensor? xhat, Tensor? rstd, Tensor? G, Tensor which, Tensor mask, int nP, float drop_p, int seed, Tensor db, Tensor? dG, Tensor? dbeta, Tensor? seed_dev) -> Tensor");
  m.def("seq2col(Tensor X) -> Tensor");
  m.def("col2seq_residual(Tensor dXw, Tensor? dY, Tensor mask) -> Tensor");
  m.def("softmax_xent(Tensor logits, Tensor labels) -> Tensor[]");
  m.def("linear_softmax_xent(Tensor X, Tensor W, Tensor b, Tensor labels) -> Tensor[]");
  m.def("softmax_xent_bias(Tensor(a!) logits, Tensor b, Tensor labels, int nC) -> Tensor[]");
  m.def("adam_shard(Tensor g, Tensor w, Tensor m1, Tensor m2, Tensor? w_out, Tensor blk_key, Tensor blk_off, Tensor key_off, Tensor key_len, Tensor norms, Tensor hyper, Tensor step) -> ()");
  m.def("biluo_steps(Tensor Yf, Tensor pad, Tensor b, Tensor Wu, Tensor bu, Tensor doc_starts, Tensor doc_lens, Tensor tok_off, Tensor? gold, Tensor inv_active, int n_tokens, int nO, int nP, int n_labels, bool train, bool teacher) -> Tensor[]");
  m.def("arc_eager_steps(Tensor Yf, Tensor pad, Tensor b, Tensor Wu, Tensor bu, Tensor doc_starts, Tensor doc_lens, Tensor tok_off, Tensor step_off, Tensor? gold_heads, Tensor? gold_labels, int n_tokens, int n_steps_cap, int nO, int nP, float scale, bool train, bool teacher, int max_len) -> Tensor[]");
  m.def("arc_eager_capacity(int nO, int nP, int nA) -> int", [](int64_t nO, int64_t nP, int64_t nA) -> int64_t {
    return (int64_t)srb::arc_eager_max_doc_len((int)nO, (int)nP, (int)nA);
  });
  // programmatic dependent launch switch (launch.h): returns the previous setting
  m.def("set_pdl(bool on) -> bool", [](bool on) -> bool {
    const bool was = srb::g_pdl != 0;
    srb::g_pdl = on ? 1 : 0;
    return was;
  });
  m.def("bump_i64(Tensor(a!) t, int by) -> ()", [](at::Tensor t, int64_t by) {
    TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kLong && t.numel() >= 1);
    c10::cuda::CUDAGuard guard(t.device());
    srb::launch_bump_i64(t.data_ptr<int64_t>(), by, at::cuda::getCurrentCUDAStream().stream());
  });
  m.def("transition_scatter(Tensor d_hid, Tensor which, Tensor feats, Tensor dYf, Tensor dpad, Tensor db, int nF, int nP) -> ()");
  m.def("textcat_head(Tensor? X, Tensor mask, Tensor attrs, Tensor doc_starts, Tensor doc_lens, Tensor? n_docs_dev, int n_docs, Tensor? W, Tensor? b, Tensor? W_bow, Tensor? b_bow, Tensor truths, Tensor known, Tensor? gW, Tensor? gb, Tensor? gW_bow, Tensor? gb_bow, int n_labels, bool use_mean, bool use_max, int act, int ngram) -> Tensor[]");
  srb::register_gemm_ops(m);
  srb::register_comm_ops(m);
}

TORCH_LIBRARY_IMPL(srb, CUDA, m) {
  m.impl("hash_embed_fwd", hash_embed_fwd);
  m.impl("hash_embed_bwd", hash_embed_bwd);
  m.impl("hash_embed_bwd_sorted", hash_embed_bwd_sorted);
  m.impl("colsum_acc", colsum_acc);
  m.impl("f32_to_bf16_zero", f32_to_bf16_zero);
  m.impl("maxout_ln_fwd", maxout_ln_fwd);
  m.impl("maxout_ln_bwd", maxout_ln_bwd);
  m.impl("seq2col", seq2col);
  m.impl("col2seq_residual", col2seq_residual);
  m.impl("softmax_xent", softmax_xent);
  m.impl("linear_softmax_xent", linear_softmax_xent);
  m.impl("softmax_xent_bias", softmax_xent_bias);
  m.impl("adam_shard", adam_shard);
  m.impl("biluo_steps", biluo_steps);
  m.impl("arc_eager_steps", arc_eager_steps);
  m.impl("transition_scatter", transition_scatter);
  m.impl("textcat_head", textcat_head);
  srb::register_gemm_impls(m);
  srb::register_comm_impls(m);
}
