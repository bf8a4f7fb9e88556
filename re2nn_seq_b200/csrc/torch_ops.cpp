// PyTorch custom-op registration: TORCH_LIBRARY(re2nn, ...) over the C-ABI of libre2nn_b200.so.
//
// This file holds NO arithmetic.  Each op checks its tensors (CUDA, contiguous, dtype), allocates the outputs and
// workspaces with ATen on the tensor's device, and calls the corresponding extern "C" entry point of
// include/re2nn_b200.h on torch's current CUDA stream; a non-zero return becomes a c10::Error (RuntimeError)
// carrying re2nn_last_error().  The op set is the one SURVEY.md section 8b proposes for the reference's modules
// (farnn/model_decompose_single.py:207-304, farnn/model_onehot.py:351-428, baselines/crf.py:48-260):
//   re2nn::ifst_decompose_forward, re2nn::ifst_onehot_forward, re2nn::label_scores, re2nn::argmax_decode,
//   re2nn::crf_viterbi, re2nn::crf_nll, re2nn::crf_nll_backward; beyond it re2nn::crf_nbest, re2nn::crf_marginals,
//   re2nn::crf_partial_nll, re2nn::crf_partial_nll_backward.
// Built by re2nn_seq_b200/build.py into re2nn_seq_b200/libre2nn_torch.so (links libre2nn_b200.so, rpath $ORIGIN).
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <ATen/ATen.h>

#include <tuple>

#include "../../include/re2nn_b200.h"

namespace {

using at::Tensor;
using c10::optional;

void* stream() { return (void*)at::cuda::getCurrentCUDAStream().stream(); }

void fail(int rc, const char* what) {
  if (rc != 0) {
    const char* msg = re2nn_last_error();
    TORCH_CHECK(false, "re2nn_b200 ", what, " failed: ", msg ? msg : "?");
  }
}
const float* f32(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), "re2nn_b200: ", name, " must be a CUDA tensor (there is no CPU path)");
  TORCH_CHECK(t.is_contiguous(), "re2nn_b200: ", name, " must be contiguous");
  TORCH_CHECK(t.scalar_type() == at::kFloat, "re2nn_b200: ", name, " must be float32");
  return t.data_ptr<float>();
}
const float* f32(const optional<Tensor>& t, const char* name) { return t.has_value() ? f32(*t, name) : nullptr; }
const int64_t* i64(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), "re2nn_b200: ", name, " must be a CUDA tensor (there is no CPU path)");
  TORCH_CHECK(t.is_contiguous(), "re2nn_b200: ", name, " must be contiguous");
  TORCH_CHECK(t.scalar_type() == at::kLong, "re2nn_b200: ", name, " must be int64");
  return t.data_ptr<int64_t>();
}
const int64_t* i64(const optional<Tensor>& t, const char* name) { return t.has_value() ? i64(*t, name) : nullptr; }
Tensor bytes(size_t n, const Tensor& like) { return at::empty({(int64_t)n}, like.options().dtype(at::kByte)); }

// model_decompose_single.py:236-261 (both recurrences, gates, nonlinearity, mask, un-reverse) -> alpha, beta  B x L x S
std::tuple<Tensor, Tensor> ifst_decompose_forward(const optional<Tensor>& x, const Tensor& lengths, const Tensor& vtab,
                                                  const optional<Tensor>& gtab, const Tensor& S1, const Tensor& S2,
                                                  const Tensor& W, const Tensor& o, const Tensor& h0, const Tensor& hT,
                                                  const optional<Tensor>& Wss1, const optional<Tensor>& Wss2, int64_t L,
                                                  int64_t Lpad, int64_t farnn, int64_t update_nonlinear, int64_t precision,
                                                  int64_t v_mode, bool full_pad, double sigmoid_exponent, bool max_semiring,
                                                  const optional<Tensor>& wprep) {
  c10::cuda::CUDAGuard guard(S1.device());
  const int64_t B = lengths.size(0), S = S1.size(0), R = S1.size(1);
  re2nn_recurrence_args a;
  memset(&a, 0, sizeof(a));
  a.B = (int)B; a.Lpad = (int)Lpad; a.L = (int)L; a.S = (int)S; a.R = (int)R; a.farnn = (int)farnn;
  a.update_nonlinear = (int)update_nonlinear; a.precision = (int)precision; a.v_mode = (int)v_mode;
  a.full_pad = full_pad ? 1 : 0; a.save_for_backward = 0; a.sigmoid_exponent = (float)sigmoid_exponent;
  Tensor alpha = at::empty({B, L, S}, S1.options()), beta = at::empty({B, L, S}, S1.options());
  a.x = i64(x, "x"); a.lengths = i64(lengths, "lengths");
  a.vtab = f32(vtab, "vtab"); a.gtab = f32(gtab, "gtab");
  a.S1 = f32(S1, "S1"); a.S2 = f32(S2, "S2"); a.W = f32(W, "wildcard_mat"); a.o = f32(o, "o");
  a.h0 = f32(h0, "h0"); a.hT = f32(hT, "hT"); a.Wss1 = f32(Wss1, "Wss1"); a.Wss2 = f32(Wss2, "Wss2");
  a.alpha = alpha.data_ptr<float>(); a.beta = beta.data_ptr<float>();
  if (wprep.has_value() && !max_semiring) {      // operand-format weight copies prepared by re2nn_decompose_weight_prep
    TORCH_CHECK(wprep->is_cuda() && wprep->is_contiguous(), "re2nn_b200: wprep must be a contiguous CUDA buffer");
    TORCH_CHECK((size_t)wprep->nbytes() >= re2nn_decompose_weight_prep_bytes(&a), "re2nn_b200: wprep buffer too small");
    a.wprep = wprep->data_ptr();
  }
  if (max_semiring) {
    Tensor ws = bytes(re2nn_decompose_max_workspace((int)S, (int)R), S1);
    a.ws = ws.data_ptr(); a.ws_bytes = (size_t)ws.numel();
    fail(re2nn_decompose_max_recurrence(&a, stream()), "decompose_max_recurrence");
    return {alpha, beta};
  }
  Tensor ws = bytes(re2nn_decompose_recurrence_workspace(&a), S1);
  a.ws = ws.data_ptr(); a.ws_bytes = (size_t)ws.numel();
  fail(re2nn_decompose_recurrence(&a, stream()), "decompose_recurrence");
  return {alpha, beta};
}

// model_onehot.py:366-415 (language is the pre-summed language + wildcard tensor) -> alpha, beta  B x L x S
std::tuple<Tensor, Tensor> ifst_onehot_forward(const Tensor& x, const Tensor& lengths, const Tensor& language_sum, const Tensor& o,
                                               const Tensor& h0, const Tensor& hT, int64_t L, int64_t update_nonlinear,
                                               bool max_semiring, bool full_pad) {
  c10::cuda::CUDAGuard guard(language_sum.device());
  const int64_t B = x.size(0), S = language_sum.size(1);
  re2nn_onehot_args a;
  memset(&a, 0, sizeof(a));
  a.B = (int)B; a.Lpad = (int)x.size(1); a.L = (int)L; a.S = (int)S;
  a.update_nonlinear = (int)update_nonlinear; a.max_semiring = max_semiring ? 1 : 0; a.full_pad = full_pad ? 1 : 0;
  Tensor alpha = at::zeros({B, L, S}, language_sum.options()), beta = at::zeros({B, L, S}, language_sum.options());
  a.x = i64(x, "x"); a.lengths = i64(lengths, "lengths");
  a.language = f32(language_sum, "language"); a.W = nullptr; a.o = f32(o, "o"); a.h0 = f32(h0, "h0"); a.hT = f32(hT, "hT");
  a.alpha = alpha.data_ptr<float>(); a.beta = beta.data_ptr<float>();
  fail(re2nn_onehot_recurrence(&a, stream()), "onehot_recurrence");
  return {alpha, beta};
}

// model_decompose_single.py:202-205,263-272 + priority.py:20-30 -> all_scores  B x L x C
Tensor label_scores(const Tensor& alpha, const Tensor& beta, const Tensor& lengths, const Tensor& C_mat,
                    const optional<Tensor>& priority_mat, const optional<Tensor>& priority_bias, bool full_pad,
                    int64_t precision) {
  c10::cuda::CUDAGuard guard(alpha.device());
  const int64_t B = alpha.size(0), L = alpha.size(1), S = alpha.size(2), C = C_mat.size(0);
  Tensor scores = at::empty({B, L, C}, alpha.options());
  Tensor ws = bytes(re2nn_label_scores_workspace((int)B, (int)L, (int)S, (int)C, (int)precision, priority_mat.has_value()), alpha);
  fail(re2nn_label_scores(f32(alpha, "alpha"), f32(beta, "beta"), i64(lengths, "lengths"), (int)B, (int)L, (int)S,
                          f32(C_mat, "C_mat"), (int)C, f32(priority_mat, "priority_mat"), f32(priority_bias, "priority_bias"),
                          full_pad ? 1 : 0, (int)precision, scores.data_ptr<float>(), ws.data_ptr(), (size_t)ws.numel(), stream()),
       "label_scores");
  return scores;
}

// model_decompose.py:363-367 / model_onehot.py:148-180: clamp, first-max argmax, remap -> (flat N, padded B x L)
std::tuple<Tensor, Tensor> argmax_decode(const Tensor& scores, const Tensor& lengths, const optional<Tensor>& offsets,
                                         int64_t n_flat, int64_t clamp_col, double threshold, int64_t o_idx, bool want_flat,
                                         bool want_padded, const optional<Tensor>& flat_out) {
  c10::cuda::CUDAGuard guard(scores.device());
  const int64_t B = scores.size(0), L = scores.size(1), C = scores.size(2);
  auto lo = scores.options().dtype(at::kLong);
  Tensor flat = want_flat ? (flat_out.has_value() ? *flat_out : at::empty({n_flat}, lo)) : at::empty({0}, lo);
  Tensor padded = want_padded ? at::empty({B, L}, lo) : at::empty({0}, lo);
  fail(re2nn_argmax_decode(f32(scores, "scores"), i64(lengths, "lengths"), i64(offsets, "offsets"), (int)B, (int)L, (int)C,
                           (int)clamp_col, (float)threshold, o_idx, want_flat ? flat.data_ptr<int64_t>() : nullptr,
                           want_padded ? padded.data_ptr<int64_t>() : nullptr, stream()),
       "argmax_decode");
  return {flat_out.has_value() ? at::empty({0}, lo) : flat, padded};      // a caller-provided buffer is not returned (no aliasing)
}

// crf.py:102-195 (+ decode()'s CRF branch, model_decompose.py:349-359) -> (flat N, padded B x L)
std::tuple<Tensor, Tensor> crf_viterbi(const Tensor& feats, const Tensor& transitions, const Tensor& lengths,
                                       const optional<Tensor>& offsets, int64_t n_flat, int64_t clamp_col, double threshold,
                                       int64_t o_idx, bool want_flat, bool want_padded, const optional<Tensor>& flat_out) {
  c10::cuda::CUDAGuard guard(feats.device());
  const int64_t B = feats.size(0), L = feats.size(1), T = feats.size(2);
  auto lo = feats.options().dtype(at::kLong);
  Tensor flat = want_flat ? (flat_out.has_value() ? *flat_out : at::empty({n_flat}, lo)) : at::empty({0}, lo);
  Tensor padded = want_padded ? at::empty({B, L}, lo) : at::empty({0}, lo);
  Tensor hist = at::empty({B * L * T}, feats.options());
  fail(re2nn_crf_viterbi(f32(feats, "feats"), f32(transitions, "transitions"), i64(lengths, "lengths"), i64(offsets, "offsets"),
                         (int)B, (int)L, (int)T, (int)clamp_col, (float)threshold, o_idx,
                         want_padded ? padded.data_ptr<int64_t>() : nullptr, want_flat ? flat.data_ptr<int64_t>() : nullptr,
                         hist.data_ptr<float>(), stream()),
       "crf_viterbi");
  return {flat_out.has_value() ? at::empty({0}, lo) : flat, padded};
}

// crf.py:48-99,202-260 -> (loss scalar, per-sequence B, saved partitions B x L x T or empty)
std::tuple<Tensor, Tensor, Tensor> crf_nll(const Tensor& feats, const Tensor& transitions, const Tensor& lengths,
                                           const Tensor& tags, bool save) {
  c10::cuda::CUDAGuard guard(feats.device());
  const int64_t B = feats.size(0), L = feats.size(1), T = feats.size(2);
  Tensor per_seq = at::empty({B}, feats.options()), loss = at::empty({}, feats.options());
  Tensor part = save ? at::empty({B, L, T}, feats.options()) : at::empty({0}, feats.options());
  fail(re2nn_crf_nll(f32(feats, "feats"), f32(transitions, "transitions"), i64(lengths, "lengths"), i64(tags, "tags"), (int)B,
                     (int)L, (int)tags.size(1), (int)T, per_seq.data_ptr<float>(), loss.data_ptr<float>(),
                     save ? part.data_ptr<float>() : nullptr, stream()),
       "crf_nll");
  return {loss, per_seq, part};
}

std::tuple<Tensor, Tensor> crf_nll_backward(const Tensor& feats, const Tensor& transitions, const Tensor& lengths,
                                            const Tensor& tags, const Tensor& part, const Tensor& gscale) {
  c10::cuda::CUDAGuard guard(feats.device());
  const int64_t B = feats.size(0), L = feats.size(1), T = feats.size(2);
  Tensor dfeats = at::empty_like(feats), dtrans = at::empty({T, T}, feats.options());
  fail(re2nn_crf_nll_backward(f32(feats, "feats"), f32(transitions, "transitions"), i64(lengths, "lengths"), i64(tags, "tags"),
                              f32(part, "part"), f32(gscale, "gscale"), (int)B, (int)L, (int)tags.size(1), (int)T,
                              dfeats.data_ptr<float>(), dtrans.data_ptr<float>(), stream()),
       "crf_nll_backward");
  return {dfeats, dtrans};
}

// allowed-tag mask B x L x T: bool or uint8, one byte per tag
const uint8_t* mask8(const Tensor& t, const Tensor& feats) {
  TORCH_CHECK(t.is_cuda(), "re2nn_b200: allowed must be a CUDA tensor (there is no CPU path)");
  TORCH_CHECK(t.is_contiguous(), "re2nn_b200: allowed must be contiguous");
  TORCH_CHECK(t.scalar_type() == at::kBool || t.scalar_type() == at::kByte, "re2nn_b200: allowed must be bool or uint8");
  TORCH_CHECK(t.sizes() == feats.sizes(), "re2nn_b200: allowed must have the shape of feats (B x L x T)");
  return reinterpret_cast<const uint8_t*>(t.data_ptr());
}

// partial-annotation loss -> (loss scalar, per-sequence B, free and constrained partitions B x L x T each, or empty)
std::tuple<Tensor, Tensor, Tensor, Tensor> crf_partial_nll(const Tensor& feats, const Tensor& transitions,
                                                           const Tensor& lengths, const Tensor& allowed, bool save) {
  c10::cuda::CUDAGuard guard(feats.device());
  const int64_t B = feats.size(0), L = feats.size(1), T = feats.size(2);
  Tensor per_seq = at::empty({B}, feats.options()), loss = at::empty({}, feats.options());
  Tensor part = save ? at::empty({B, L, T}, feats.options()) : at::empty({0}, feats.options());
  Tensor part_a = save ? at::empty({B, L, T}, feats.options()) : at::empty({0}, feats.options());
  fail(re2nn_crf_partial_nll(f32(feats, "feats"), f32(transitions, "transitions"), i64(lengths, "lengths"),
                             mask8(allowed, feats), (int)B, (int)L, (int)T, per_seq.data_ptr<float>(),
                             loss.data_ptr<float>(), save ? part.data_ptr<float>() : nullptr,
                             save ? part_a.data_ptr<float>() : nullptr, stream()),
       "crf_partial_nll");
  return {loss, per_seq, part, part_a};
}

std::tuple<Tensor, Tensor> crf_partial_nll_backward(const Tensor& feats, const Tensor& transitions, const Tensor& lengths,
                                                    const Tensor& allowed, const Tensor& part, const Tensor& part_allowed,
                                                    const Tensor& gscale) {
  c10::cuda::CUDAGuard guard(feats.device());
  const int64_t B = feats.size(0), L = feats.size(1), T = feats.size(2);
  Tensor dfeats = at::empty_like(feats), dtrans = at::empty({T, T}, feats.options());
  fail(re2nn_crf_partial_nll_backward(f32(feats, "feats"), f32(transitions, "transitions"), i64(lengths, "lengths"),
                                      mask8(allowed, feats), f32(part, "part"), f32(part_allowed, "part_allowed"),
                                      f32(gscale, "gscale"), (int)B, (int)L, (int)T, dfeats.data_ptr<float>(),
                                      dtrans.data_ptr<float>(), stream()),
       "crf_partial_nll_backward");
  return {dfeats, dtrans};
}

// NCRF++ CRF._viterbi_decode_nbest -> (paths B x L x K int64, scores B x K)
std::tuple<Tensor, Tensor> crf_nbest(const Tensor& feats, const Tensor& transitions, const Tensor& lengths, int64_t nbest) {
  c10::cuda::CUDAGuard guard(feats.device());
  const int64_t B = feats.size(0), L = feats.size(1), T = feats.size(2);
  Tensor paths = at::empty({B, L, nbest}, feats.options().dtype(at::kLong));
  Tensor scores = at::empty({B, nbest}, feats.options());
  const size_t need = re2nn_crf_nbest_workspace((int)B, (int)L, (int)T, (int)nbest);
  Tensor ws = bytes(need, feats);
  fail(re2nn_crf_nbest(f32(feats, "feats"), f32(transitions, "transitions"), i64(lengths, "lengths"), (int)B, (int)L, (int)T,
                       (int)nbest, paths.data_ptr<int64_t>(), scores.data_ptr<float>(), ws.data_ptr(), need, stream()),
       "crf_nbest");
  return {paths, scores};
}

// tag marginals P(y_t = j | x) -> (marginals B x L x T, log Z B)
std::tuple<Tensor, Tensor> crf_marginals(const Tensor& feats, const Tensor& transitions, const Tensor& lengths) {
  c10::cuda::CUDAGuard guard(feats.device());
  const int64_t B = feats.size(0), L = feats.size(1), T = feats.size(2);
  Tensor marg = at::empty({B, L, T}, feats.options()), log_z = at::empty({B}, feats.options());
  Tensor part = at::empty({B, L, T}, feats.options());
  fail(re2nn_crf_marginals(f32(feats, "feats"), f32(transitions, "transitions"), i64(lengths, "lengths"), (int)B, (int)L,
                           (int)T, marg.data_ptr<float>(), log_z.data_ptr<float>(), part.data_ptr<float>(), stream()),
       "crf_marginals");
  return {marg, log_z};
}

int64_t abi_version() { return re2nn_abi_version(); }

}  // namespace

TORCH_LIBRARY(re2nn, m) {
  m.def("ifst_decompose_forward(Tensor? x, Tensor lengths, Tensor vtab, Tensor? gtab, Tensor S1, Tensor S2, Tensor W, Tensor o, "
        "Tensor h0, Tensor hT, Tensor? Wss1, Tensor? Wss2, int L, int Lpad, int farnn, int update_nonlinear, int precision, "
        "int v_mode, bool full_pad, float sigmoid_exponent, bool max_semiring, Tensor? wprep) -> (Tensor, Tensor)");
  m.def("ifst_onehot_forward(Tensor x, Tensor lengths, Tensor language_sum, Tensor o, Tensor h0, Tensor hT, int L, "
        "int update_nonlinear, bool max_semiring, bool full_pad) -> (Tensor, Tensor)");
  m.def("label_scores(Tensor alpha, Tensor beta, Tensor lengths, Tensor C_mat, Tensor? priority_mat, Tensor? priority_bias, "
        "bool full_pad, int precision) -> Tensor");
  m.def("argmax_decode(Tensor scores, Tensor lengths, Tensor? offsets, int n_flat, int clamp_col, float threshold, int o_idx, "
        "bool want_flat, bool want_padded, Tensor(a!)? flat_out) -> (Tensor, Tensor)");
  m.def("crf_viterbi(Tensor feats, Tensor transitions, Tensor lengths, Tensor? offsets, int n_flat, int clamp_col, "
        "float threshold, int o_idx, bool want_flat, bool want_padded, Tensor(a!)? flat_out) -> (Tensor, Tensor)");
  m.def("crf_nll(Tensor feats, Tensor transitions, Tensor lengths, Tensor tags, bool save) -> (Tensor, Tensor, Tensor)");
  m.def("crf_nll_backward(Tensor feats, Tensor transitions, Tensor lengths, Tensor tags, Tensor part, Tensor gscale) -> "
        "(Tensor, Tensor)");
  m.def("crf_partial_nll(Tensor feats, Tensor transitions, Tensor lengths, Tensor allowed, bool save) -> "
        "(Tensor, Tensor, Tensor, Tensor)");
  m.def("crf_partial_nll_backward(Tensor feats, Tensor transitions, Tensor lengths, Tensor allowed, Tensor part, "
        "Tensor part_allowed, Tensor gscale) -> (Tensor, Tensor)");
  m.def("crf_nbest(Tensor feats, Tensor transitions, Tensor lengths, int nbest) -> (Tensor paths, Tensor scores)");
  m.def("crf_marginals(Tensor feats, Tensor transitions, Tensor lengths) -> (Tensor marginals, Tensor log_z)");
  m.def("abi_version() -> int", &abi_version);
}

TORCH_LIBRARY_IMPL(re2nn, CUDA, m) {
  m.impl("ifst_decompose_forward", &ifst_decompose_forward);
  m.impl("ifst_onehot_forward", &ifst_onehot_forward);
  m.impl("label_scores", &label_scores);
  m.impl("argmax_decode", &argmax_decode);
  m.impl("crf_viterbi", &crf_viterbi);
  m.impl("crf_nll", &crf_nll);
  m.impl("crf_nll_backward", &crf_nll_backward);
  m.impl("crf_partial_nll", &crf_partial_nll);
  m.impl("crf_partial_nll_backward", &crf_partial_nll_backward);
  m.impl("crf_nbest", &crf_nbest);
  m.impl("crf_marginals", &crf_marginals);
}
