/*
 * re2nn_b200.h — C-ABI of the B200-native RE2NN-SEQ transducer hot path.
 *
 * The reference (jeffchy/RE2NN-SEQ) is pure Python/PyTorch and has NO FFI / plugin / custom-op
 * interface (SURVEY.md §8b).  Its boundary for this path is the nn.Module surface of
 * src_seq/farnn/*.py and src_seq/baselines/crf.py.  Each entry point below replaces the torch-op
 * sequence of one reference method (cited file:line, relative to /root/reference/src_seq/) and is
 * what a ctypes binding added to those modules would call (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C, no torch types.  Every pointer is a DEVICE pointer unless the name ends in _host.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - float = fp32, indices/lengths/labels = int64 exactly as the reference holds them
 *     (data.py:205-207).  Row-major, innermost dimension contiguous.
 *   - return value: 0 on success, non-zero on error; re2nn_last_error() gives the message.
 *     Errors are reported, never abort()ed (reference raises Python exceptions).
 *   - no hidden global state: scratch memory is caller-provided (`ws`, size from *_workspace()).
 *
 * Index semantics (SURVEY.md §8a): for a sequence of n tokens, alpha[b,t,:] (t<n) is the forward
 * state after consuming tokens 0..t; beta[b,t,:] is the backward state after consuming tokens
 * n-1..t+1 (beta[b,n-1,:] = hT).  The i-FST score of position t uses exactly these two rows.
 */
#ifndef RE2NN_B200_H
#define RE2NN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RE2NN_ABI_VERSION 4

/* update_nonlinear / additional_nonlinear (model_decompose_single.py:184-191, model_decompose.py:228-237) */
enum { RE2NN_NL_NONE = 0, RE2NN_NL_RELU = 1, RE2NN_NL_TANH = 2, RE2NN_NL_RELUTANH = 3, RE2NN_NL_SIGMOID = 4 };
/* arithmetic used by the recurrence GEMMs */
enum {
  RE2NN_PREC_FP32 = 0,      /* fp32 FFMA on CUDA cores: bit-for-bit the reference's operand precision */
  RE2NN_PREC_BF16 = 1,      /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM */
  RE2NN_PREC_TF32X3 = 2,    /* tcgen05 kind::tf32, 3-term split (hi*hi + hi*lo + lo*hi): fp32-grade */
  RE2NN_PREC_FP16X3 = 3     /* tcgen05 kind::f16 on fp16 planes hi + 2^-11*lo (same 22-bit budget as TF32X3 at half
                               the operand bytes); operands must stay below 65504 in magnitude */
};
/* how the per-step rank factor v_t is addressed */
enum {
  RE2NN_V_TOKEN = 0,        /* v_t = vtab[x[b,t]]           (FARNN_S_D_W_I_S, token ids)          */
  RE2NN_V_DENSE = 1         /* v_t = vtab[b*Lpad + t]       (FARNN_S_SF, pre-computed B x L x R)  */
};

int re2nn_abi_version(void);
const char* re2nn_last_error(void);
/* 1 if the running device is sm_100 and the tcgen05 kernels were compiled in. */
int re2nn_has_tcgen05(void);

/* ---- in-library kernel timing (used by bench.py for the roofline line) --------------------------------
 * When enabled, every step-GEMM launch of re2nn_decompose_recurrence is bracketed by CUDA events on
 * its own stream.  re2nn_profile_read synchronises those events, returns the summed milliseconds and
 * launch counts per kernel class (0 = gate GEMM, 1 = GEMM1 + Q epilogue, 2 = GEMM2 + state epilogue,
 * 3 = resident recurrence kernel: all steps in one launch; both output arrays hold 4 entries)
 * and resets the counters. */
int re2nn_profile_enable(int on);
/* debug: install (or clear with NULL) a device buffer receiving 32 clock64 stamps per CTA of every
 * tcgen05 step-GEMM launch (entry, alive-check, setup, MMAs issued, prefetch issued, accumulator ready,
 * epilogue done, exit, then arrival time of the first 24 k-blocks); slot = 32 * (256 * launch index + linear CTA id)
 * for the first 256 launches after the call, so the buffer must hold 32 * 65536 entries. */
int re2nn_debug_set_tc_trace(unsigned long long* device_buf);
/* debug: per-launch timeline: buf[2*i], buf[2*i+1] = %globaltimer (ns) at entry / exit of CTA (0,0,0) of the i-th
 * tcgen05 step-GEMM launch since the call (up to 4096 launches); NULL clears. */
int re2nn_debug_set_tc_timeline(unsigned long long* device_buf);
/* debug / calibration: CTA-group size of the tcgen05 step GEMMs built after the call: 0 = the cost model
 * picks per GEMM shape (default), 1 = single-CTA tiles (128 x bn), 2 = CTA pairs (cta_group::2, 256 x bn). */
int re2nn_debug_set_tc_cta_group(int cta_group);
/* debug / calibration: 1 (default) = inference without gates runs the whole recurrence in one resident launch
 * (a CTA pair per 128-row tile iterates over all steps); 0 = one launch per step GEMM. */
int re2nn_debug_set_resident(int on);
/* debug / calibration: 1 (default) = the weight-gradient GEMMs (X^T Y over every (step, sequence) row) run on tcgen05 in
 * 3xTF32 with the operands transposed on the fly; 0 = the CUDA-core kernel. */
int re2nn_debug_set_tn_tc(int on);
/* debug / calibration: 1 (default) = the CRF backward sweep gives each sequence three warps (one transition row per
 * lane, named barriers between them) when the tag set has at most 96 entries; 0 = one warp per sequence. */
int re2nn_debug_set_crf_backward_split(int on);
int re2nn_profile_read(double* ms_out_host, int64_t* count_out_host);
/* Per-launch [start, end] of kernel class `cls` in ms relative to the earliest start of the class, for up to
 * `cap` launches recorded since the last clearing read.  The event pairs also work inside stream capture (they
 * become external event nodes; every graph replay re-records them), so the timed configuration itself -- CUDA
 * graph, forked chunk streams -- can be measured: pass clear = 0 to keep the pairs registered across replays.
 * re2nn_profile_count: launches currently registered for the class.  re2nn_profile_enabled: current switch. */
int re2nn_profile_intervals(int cls, double* start_ms_host, double* end_ms_host, int cap, int clear);
int re2nn_profile_count(int cls);
int re2nn_profile_enabled(void);

/* ---- stand-alone GEMM through the step-GEMM mainloops (unit-test / calibration entry) -------------------
 * C[M x N] = A[M x K] @ B[N x K]^T, A/B/C fp32 row-major.  precision selects the mainloop:
 * RE2NN_PREC_FP32 (CUDA cores), RE2NN_PREC_BF16 / RE2NN_PREC_TF32X3 (tcgen05; operands are first
 * converted into `ws`).  Not on the reference's path; it exists so the tensor-core mainloop can be
 * checked in isolation against a known product. */
size_t re2nn_gemm_nt_workspace(int precision, int M, int N, int K);
int re2nn_gemm_nt(int precision, const float* A, const float* B, int M, int N, int K, float* C, void* ws,
                  size_t ws_bytes, void* stream);

/* ---- stand-alone weight-gradient GEMM (unit-test / calibration entry) ---------------------------------
 * C[P x Q] = sum_m X0[m, :]^T Y0[m, :] (m < rows0) + sum_m X1[m, :]^T Y1[m, :] (m < rows1), every operand fp32
 * row-major with its own leading dimension (ldx >= P, ldy >= Q, any alignment); pair 1 is optional (X1 = NULL).
 * Y2 (optional, single pair only, leading dimension ldy0): the right operand is Y0 * Y2 element-wise.  mask_len
 * (optional, needs Y2): row m = b * mask_L + t only counts when t < mask_len[b], rows0 = B * mask_L; the pad rows of
 * Y0 / Y2 may hold anything, NaN and Inf included (this is the dC product of the decompose backward).
 * path: 0 = the kernel re2nn_decompose_backward picks for this shape (re2nn_gemm_tn_path), 1 = the CUDA-core split-K
 * kernel, 2 = tcgen05 in 3xTF32 (fails without an sm_100 device or when P or Q is below 16).  ws: at least
 * re2nn_gemm_tn_workspace(P, Q) bytes.  Deterministic: the same call gives the same bits.
 * re2nn_gemm_tn_path: 1 or 2, the kernel the backward takes for a P x Q product over `rows` summed rows (has_y2: the
 * dC layout; it takes the same path as a plain product). */
int re2nn_gemm_tn_path(int P, int Q, int64_t rows, int has_y2);
size_t re2nn_gemm_tn_workspace(int P, int Q);
int re2nn_gemm_tn(int path, int P, int Q, const float* X0, const float* Y0, int ldx0, int ldy0, int64_t rows0, const float* X1,
                  const float* Y1, int ldx1, int ldy1, int64_t rows1, const float* Y2, const int64_t* mask_len, int mask_L,
                  float* C, void* ws, size_t ws_bytes, void* stream);

/* ---- generalised token factor table ------------------------------------------------------------
 * table[r, :] = V_embed[r,:]*beta_vec + phi_add(E[r,:] @ G) * (1 - beta_vec)   for r in [0, rows)
 * replaces get_generalized_v_embed_vec (farnn/model_decompose.py:222-241) evaluated per token id;
 * hoisted out of the time loop because it only depends on the token (SURVEY.md §2.2 K8). */
int re2nn_token_table(const float* V_embed, const float* E, const float* G, const float* beta_vec,
                      int rows, int D, int R, int additional_nonlinear, float* table, void* stream);

/* ---- gate addend table --------------------------------------------------------------------------
 * gate[r, 0:S]  = vtab[r,:] @ Wrs1 + bs1 ;  gate[r, S:2S] = vtab[r,:] @ Wrs2 + bs2  (farnn==2)
 * the token-only part of zt/rt (farnn/model_decompose_single.py:147-150). */
int re2nn_gate_table(const float* vtab, int rows, int R, int S, int farnn,
                     const float* Wrs1, const float* bs1, const float* Wrs2, const float* bs2,
                     float* gate, void* stream);

/* ---- output-vector sum ------------------------------------------------------------------------------
 * o[s] = sum_c C_mat[c,s] (+ wildcard_vec[s] if wildcard_vec != NULL, i.e. local_loss_func != 'CE1');
 * model_decompose_single.py:231-234, model_onehot.py:367-370.  Deterministic column sum. */
int re2nn_output_vector_sum(const float* C_mat, int C, int S, const float* wildcard_vec, float* o,
                            void* stream);

/* ---- decompose i-FST recurrence, both directions ------------------------------------------------
 * replaces the L-step loop of FARNN_S_D_W_I_S.forward_local / FARNN_S_SF.forward and
 * get_forward_score (farnn/model_decompose_single.py:138-200, 236-261, 417-481, 511-534),
 * including reverse()/cat()/reverse() (utils.py:183-189): beta is written at un-reversed indices. */
typedef struct re2nn_recurrence_args {
  int32_t B, Lpad, L;          /* batch, row stride of x (tokens per row), steps to run (= max length) */
  int32_t S, R;                /* states (incl. additional_states), rank */
  int32_t farnn;               /* 0 plain, 1 update gate, 2 update+reset gates */
  int32_t update_nonlinear;    /* RE2NN_NL_* */
  int32_t precision;           /* RE2NN_PREC_* */
  int32_t v_mode;              /* RE2NN_V_* */
  int32_t full_pad;            /* 1: also compute pad positions exactly like the reference does */
  int32_t save_for_backward;   /* 1: fill the *_save slabs below for re2nn_decompose_backward (fp32 only) */
  float sigmoid_exponent;
  const int64_t* x;            /* B x Lpad token ids (RE2NN_V_TOKEN) or NULL */
  const int64_t* lengths;      /* B */
  const float* vtab;           /* rows x R  (token table or dense v) */
  const float* gtab;           /* rows x (S*farnn) gate addends, NULL if farnn==0 */
  const float* S1;             /* S x R */
  const float* S2;             /* S x R */
  const float* W;              /* S x S wildcard_mat */
  const float* o;              /* S  output_vector_sum (model_decompose_single.py:231-234) */
  const float* h0;             /* S */
  const float* hT;             /* S */
  const float* Wss1;           /* S x S (farnn>=1) */
  const float* Wss2;           /* S x S (farnn==2) */
  float* alpha;                /* B x L x S out */
  float* beta;                 /* B x L x S out */
  /* save_for_backward slabs, step-major [direction][step][B][.] fp32, zero for rows that are already finished: */
  float* hbar_save;            /* 2 x (L+1) x B x S  operand of step k (after reset gate / *o)          */
  float* hst_save;             /* 2 x (L+1) x B x S  state before step k                               */
  float* u_save;               /* 2 x L x B x R      hbar @ S1|S2 (before * v_t)                        */
  float* a_save;               /* 2 x L x B x S      pre-activation before * o / phi                    */
  float* zsave;                /* 2 x L x B x S      update gate (farnn>=1) or NULL                     */
  float* rsave;                /* 2 x L x B x S      reset gate (farnn==2) or NULL                      */
  void* ws;                    /* scratch, >= re2nn_decompose_recurrence_workspace() bytes */
  size_t ws_bytes;
  /* Fused label-score operand (optional; inference, farnn == 0, tensor-core precisions, per-step path).  When
   * non-NULL the backward direction runs first and the state epilogue of the FORWARD direction multiplies every
   * alpha element by the stored beta and writes the product in the precision's operand format
   * ((B*L) rows x operand_ld(S), split formats: second plane at B*L*ld elements) -- what re2nn_label_scores would
   * otherwise rebuild by re-reading alpha and beta (model_decompose_single.py:202-205,263-269).  alpha is then never
   * written and may be NULL; rows past the length are left untouched.  Feed the buffer to re2nn_label_scores_ab.
   * Size: re2nn_label_scores_ab_bytes().  Ignored (alpha / beta written as usual) when the call takes the resident
   * kernel: query re2nn_decompose_recurrence_fuses(). */
  void* ab_out;
  /* Operand-format copies of S1 / S2 / W / gate weights prepared once by re2nn_decompose_weight_prep (optional, tensor-
   * core precisions): when non-NULL the call skips its 6-8 conversion launches.  The caller keeps the buffer valid and
   * re-prepares it when a parameter changes. */
  const void* wprep;
} re2nn_recurrence_args;

size_t re2nn_decompose_recurrence_workspace(const re2nn_recurrence_args* a);
int re2nn_decompose_recurrence(const re2nn_recurrence_args* a, void* stream);
/* Number of kernels re2nn_decompose_recurrence launches for this argument block (inference without gates on the
 * tensor-core paths runs ALL steps in one resident kernel; otherwise 2-3 step GEMMs per step). */
int re2nn_decompose_recurrence_launches(const re2nn_recurrence_args* a);
/* Converted weight copies for `wprep` (only S, R, farnn, precision and the weight pointers of the block are read). */
size_t re2nn_decompose_weight_prep_bytes(const re2nn_recurrence_args* a);
int re2nn_decompose_weight_prep(const re2nn_recurrence_args* a, void* out, void* stream);
/* 1 when a call with these arguments (and a non-NULL ab_out) would write the fused (alpha*beta) operand. */
int re2nn_decompose_recurrence_fuses(const re2nn_recurrence_args* a);
/* 1 when the call would take the resident single-launch path (only precision, S, R, farnn and save_for_backward of
 * the block are read): callers use it to decide whether splitting a batch over streams pays off. */
int re2nn_decompose_recurrence_resident(const re2nn_recurrence_args* a);

/* Same recurrence under the max-product semiring (train_mode == 'max': model_decompose_single.py:159-166,
 * utils.py:192-195).  Takes the same argument block (precision ignored: fp32; save_for_backward must be 0);
 * ws >= re2nn_decompose_max_workspace(S, R) bytes.  Inference only. */
size_t re2nn_decompose_max_workspace(int S, int R);
int re2nn_decompose_max_recurrence(const re2nn_recurrence_args* a, void* stream);

/* ---- dense-transition semiring step (FST variants, max-product training) ----------------------------------
 * out[b,s] = (+|max)_j h[b,j] * T[b,j,s]  (transposed = 0)  or  (+|max)_j h[b,j] * T[b,s,j]  (transposed = 1);
 * replaces utils.py:192-199 `_matmul` (bmm) / `_maxmul` at the call sites that materialise one dense S x S
 * transition per sequence (farnn/model_onehot.py:96-103,274-290, model_decompose_independent.py:177-181,
 * model_decompose_single.py:159-166).  argmax_out (max semiring, optional, B x S int32): the FIRST source state
 * attaining the maximum, which is where torch.max(dim) routes the gradient. */
int re2nn_batched_vecmat(const float* h, const float* T, int B, int S, int transposed, int max_semiring,
                         float* out, int32_t* argmax_out, void* stream);

/* ---- decompose i-FST backward (BPTT through both directions + label scores) ---------------------------
 * replaces torch.autograd over forward_local (train_decompose.py:192).  Input: d loss / d all_scores.
 * Outputs: gradients of every parameter the reference trains (NULL pointer = not wanted).
 * fp32 data throughout.  On an sm_100 device the GEMMs of every BPTT step, the label-score GEMM and the long
 * weight-gradient products run on tcgen05 in 3xTF32 (fp32-grade products), the rest on CUDA cores in fp32.
 * Weight gradients are reduced deterministically (split-K partials + ordered sum), token-table scatter-adds use
 * float atomics. */
typedef struct re2nn_backward_args {
  int32_t B, Lpad, L, S, R, C;  /* C = columns of all_scores */
  int32_t farnn, update_nonlinear, v_mode, full_pad, ce1;
  int32_t table_rows;           /* rows of vtab (V+1, or B*Lpad in dense mode) */
  float sigmoid_exponent;
  const int64_t* x; const int64_t* lengths;
  const float* dscores;         /* B x L x C */
  const float* priority_mat;    /* C x C or NULL */
  /* forward inputs */
  const float *vtab, *S1, *S2, *W, *o, *h0, *hT, *Wss1, *Wss2, *Wrs1, *Wrs2, *C_mat;
  /* forward outputs / saves */
  const float *alpha, *beta, *hbar_save, *hst_save, *u_save, *a_save, *zsave, *rsave;
  /* gradients (fp32, overwritten) */
  float *dS1, *dS2, *dW, *dC, *d_o, *dh0, *dhT, *dWss1, *dWss2, *dWrs1, *dWrs2, *dbs1, *dbs2;
  float* dvtab;                 /* table_rows x R */
  void* ws; size_t ws_bytes;
  /* FST variants (model_decompose.py:373-456: the score is not (alpha*beta) @ C^T): when both are non-NULL the
   * gradients of the loss w.r.t. alpha / beta (B x L x S, exact zeros at rows past the length) are taken from here
   * and dscores / C_mat / priority_mat / dC are ignored -- the label-score stage is differentiated by the caller. */
  const float* dalpha_in; const float* dbeta_in;
} re2nn_backward_args;
/* debug / calibration: 1 (default) = the two GEMMs of every BPTT step run on the tensor cores in 3xTF32 when
 * tcgen05 is available, 0 = fp32 CUDA cores.  Changes the workspace size: set it before querying. */
int re2nn_debug_set_backward_tc(int on);
size_t re2nn_decompose_backward_workspace(const re2nn_backward_args* a);
int re2nn_decompose_backward(const re2nn_backward_args* a, void* stream);

/* token-table backward: dvtab -> dV_embed (rows x R), dbeta_vec (R), dG (D x R), dE (rows x D); NULL = skip.
 * (model_decompose.py:222-241 differentiated) */
size_t re2nn_token_table_backward_workspace(int rows, int D, int R);
int re2nn_token_table_backward(const float* dvtab, const float* V_embed, const float* E, const float* G,
                               const float* beta_vec, int rows, int D, int R, int additional_nonlinear,
                               float* dV_embed, float* dbeta_vec, float* dG, float* dE, void* ws,
                               size_t ws_bytes, void* stream);

/* ---- onehot i-FST recurrence, both directions ---------------------------------------------------
 * replaces FARNN_S_O_I_S.forward_score's recurrence (farnn/model_onehot.py:358-415):
 * T = language_tensor[x_t] + wildcard_mat is formed on the fly (no V x S x S temporary),
 * fwd h <- phi((h (.) T) * o), bwd h <- phi((h*o) (.) T^T), (.) = sum- or max-product (utils.py:192-199). */
typedef struct re2nn_onehot_args {
  int32_t B, Lpad, L, S;
  int32_t update_nonlinear;
  int32_t max_semiring;        /* train_mode == 'max' */
  int32_t full_pad;
  const int64_t* x;
  const int64_t* lengths;
  const float* language;       /* (V+1) x S x S; with W == NULL: the pre-summed language + W (re2nn_onehot_sum_tensor) */
  const float* W;              /* S x S, or NULL */
  const float* o;              /* S */
  const float* h0;
  const float* hT;
  float* alpha;                /* B x L x S */
  float* beta;                 /* B x L x S */
} re2nn_onehot_args;
int re2nn_onehot_recurrence(const re2nn_onehot_args* a, void* stream);
/* debug / calibration: CTAs one (sequence, direction) slice is spread over (thread-block cluster, transition rows
 * split, partial state vectors exchanged through distributed shared memory): 0 = pick by batch size, 1, 2, 4. */
int re2nn_debug_set_onehot_cluster(int nc);
/* out[v] = language[v] + W  (model_onehot.py:366 `sum_tensor`): the reference redoes this V*S*S add on every
 * forward; here it is done once per parameter version and the recurrence then streams a single tensor. */
int re2nn_onehot_sum_tensor(const float* language, const float* W, int V1, int S, float* out, void* stream);

/* ---- onehot i-FST backward (sum semiring) ----------------------------------------------------------------
 * replaces torch.autograd over FARNN_S_O_I_S.forward_score (train_onehot.py:179-181): the only trained
 * parameter of that module is language_tensor (model_onehot.py:326-340).  dalpha/dbeta: d loss / d states
 * (B x L x S, from re2nn_label_scores_backward); dlanguage ((V+1) x S x S) must be zero-initialised and
 * receives the scatter-added outer products (float atomics). */
typedef struct re2nn_onehot_backward_args {
  int32_t B, Lpad, L, S, update_nonlinear, full_pad;
  const int64_t* x; const int64_t* lengths;
  const float *language, *W, *o, *h0, *hT, *alpha, *beta, *dalpha, *dbeta;
  float* dlanguage;
} re2nn_onehot_backward_args;
int re2nn_onehot_backward(const re2nn_onehot_backward_args* a, void* stream);

/* d loss / d alpha, d loss / d beta from d loss / d scores:  dAB = dscores [@ P^T] @ C ; dalpha = dAB*beta,
 * dbeta = dAB*alpha (zero at pads).  ws: B*L*C floats when priority_mat != NULL. */
int re2nn_label_scores_backward(const float* dscores, const float* alpha, const float* beta,
                                const int64_t* lengths, int B, int L, int S, const float* C_mat, int C,
                                const float* priority_mat, int full_pad, float* dalpha, float* dbeta,
                                float* ws, void* stream);

/* ---- per-position label scores -------------------------------------------------------------------
 * scores[b,t,c] = sum_s C[c,s] * alpha[b,t,s] * beta[b,t,s]  for t < lengths[b] (all t if full_pad);
 * replaces get_final_score + its L-step loop (model_decompose_single.py:202-205,263-269;
 * model_onehot.py:346-349,417-426).  Optional PriorityLayer (priority.py:20-30) is applied when
 * priority_mat != NULL: scores <- scores @ priority_mat + priority_bias.  Rows past the length are
 * written as 0.  ws: re2nn_label_scores_workspace() bytes.  A precision outside RE2NN_PREC_* fails with
 * "unknown precision" before any CUDA call (so does re2nn_label_scores_ab). */
size_t re2nn_label_scores_workspace(int B, int L, int S, int C, int precision, int has_priority);
int re2nn_label_scores(const float* alpha, const float* beta, const int64_t* lengths,
                       int B, int L, int S, const float* C_mat, int C,
                       const float* priority_mat, const float* priority_bias, int full_pad,
                       int precision /* RE2NN_PREC_*: fp32 = CUDA cores, else tcgen05 */,
                       float* scores /* B x L x C */, void* ws, size_t ws_bytes, void* stream);

/* ---- argmax decode --------------------------------------------------------------------------------
 * replaces decode()'s non-CRF branch / local_decode / forward_RE (model_decompose.py:363-369,
 * model_onehot.py:148-180): optional clamp of column clamp_col to `threshold`, first-max argmax,
 * remap clamp_col -> o_idx.  clamp_col < 0 disables clamp+remap (local_loss_func != 'CE1').
 * flat_pred (N = sum lengths, batch-major; offsets = exclusive prefix sum of lengths) and/or
 * padded_pred (B x L, every position decoded) may be NULL. */
int re2nn_argmax_decode(const float* scores, const int64_t* lengths, const int64_t* offsets,
                        int B, int L, int C, int clamp_col, float threshold, int64_t o_idx,
                        int64_t* flat_pred, int64_t* padded_pred, void* stream);

/* Longest-first schedule of a batch in one launch (no reference counterpart: the reference computes every pad position
 * of model_decompose_single.py:236-249 and needs no order; here 128-row tiles stop at their own last step, so tiles of
 * similar length finish together).  order = the permutation torch.sort(lengths, descending=True, stable=True) returns,
 * offsets = exclusive prefix sums of the lengths in the caller's order (start of each sequence in the flattened
 * valid-only layout of utils.py:153-164), lengths_sorted / offsets_sorted = both gathered through `order`; all int64[B].
 * Single CTA: re2nn_length_order_supported(B, L) tells whether the call is in range (B <= 16384, lengths <= L < 256). */
int re2nn_length_order_supported(int B, int L);
int re2nn_length_order(const int64_t* lengths, int B, int L, int64_t* order, int64_t* lengths_sorted, int64_t* offsets,
                       int64_t* offsets_sorted, void* stream);
/* flat[offsets[b] + t] = padded[b, t] for t < lengths[b]: utils.py:153-164 `flatten` for int64 labels, without
 * the Python loop over the batch (padded rows have stride Lrow, the first L columns are considered). */
int re2nn_flatten_i64(const int64_t* padded, const int64_t* lengths, const int64_t* offsets, int B, int Lrow,
                      int L, int64_t* flat, void* stream);

/* Label scores from the fused operand written by re2nn_decompose_recurrence (ab_out): scores = ab @ C^T [@ P + b].
 * ws: re2nn_label_scores_workspace(..) bytes with the same arguments. */
size_t re2nn_label_scores_ab_bytes(int B, int L, int S, int precision);
int re2nn_label_scores_ab(const void* ab, int B, int L, int S, const float* C_mat, int C, const float* priority_mat,
                          const float* priority_bias, int precision, float* scores, void* ws, size_t ws_bytes,
                          void* stream);

/* ---- CRF Viterbi ------------------------------------------------------------------------------------
 * replaces CRF._viterbi_decode (baselines/crf.py:102-195) plus decode()'s CRF branch
 * (model_decompose.py:349-359).  feats B x L x T (T = tagset+2), transitions T x T.
 * padded_path reproduces the reference's B x L output bit for bit (pads 0, last column = final
 * pointer); flat_pred additionally applies the clamp_col -> o_idx remap.  Either may be NULL.
 * part_ws: B*L*T fp32 scratch (the partition history; back-pointers on the best path are recomputed from it).
 * Sequences of length 0 produce no tags (their padded row is zero); lengths are clamped to L. */
int re2nn_crf_viterbi(const float* feats, const float* transitions, const int64_t* lengths,
                      const int64_t* offsets, int B, int L, int T, int clamp_col, float threshold,
                      int64_t o_idx, int64_t* padded_path, int64_t* flat_pred, float* part_ws,
                      void* stream);

/* debug / calibration: sequences one warp of the Viterbi sweep decodes together (0 = pick by batch size; 1, 2). */
int re2nn_debug_set_viterbi_seqs(int ns);

/* ---- CRF negative log-likelihood ---------------------------------------------------------------------
 * replaces CRF.neg_log_likelihood_loss = _calculate_PZ - _score_sentence (baselines/crf.py:48-99,
 * 202-260).  per_seq[b] = logZ_b - gold_b ; *loss = sum_b per_seq[b] (deterministic reduction).
 * part_save (B x L x T, may be NULL) keeps the forward partitions for re2nn_crf_nll_backward. */
int re2nn_crf_nll(const float* feats, const float* transitions, const int64_t* lengths,
                  const int64_t* tags, int B, int L, int Ltags, int T, float* per_seq, float* loss,
                  float* part_save, void* stream);

/* d loss / d feats (B x L x T, zero at pads) and d loss / d transitions (T x T), scaled by *gscale
 * (device scalar, the upstream gradient).  T <= 225: a larger tag set returns an error ("tag set too large"),
 * since one sequence's T x T accumulator no longer fits in shared memory. */
int re2nn_crf_nll_backward(const float* feats, const float* transitions, const int64_t* lengths,
                           const int64_t* tags, const float* part_save, const float* gscale,
                           int B, int L, int Ltags, int T, float* dfeats, float* dtrans, void* stream);

/* ---- cross entropy over valid positions -----------------------------------------------------------------
 * nn.CrossEntropyLoss() mean over the N valid tokens (model_decompose.py:80, :289).
 * n_total: number of tokens the mean divides by (global count under data parallelism). */
int re2nn_ce_loss(const float* scores, const int64_t* lengths, const int64_t* labels, int B, int L,
                  int Llab, int C, int64_t n_total, float* per_pos /* B*L scratch */, float* loss,
                  void* stream);
int re2nn_ce_loss_backward(const float* scores, const int64_t* lengths, const int64_t* labels,
                           const float* gscale, int B, int L, int Llab, int C, int64_t n_total,
                           float* dscores, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RE2NN_B200_H */
