// Decompose i-FST recurrence driver, token/gate tables and label scores (C-ABI entry points).
// Reference: /root/reference/src_seq/farnn/model_decompose_single.py:138-269, model_decompose.py:222-241.
#include <stdarg.h>

#include <algorithm>
#include <memory>
#include <mutex>
#include <vector>

#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "recurrence_resident.cuh"

namespace re2nn {

thread_local char g_err[512] = "";
int set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}

// ---- workspace ----------------------------------------------------------------------------------
struct RecWs {
  int* tile_last[2];
  void* Q[2];
  void* Hbar[2][2];   // [parity][dir]
  void* Hst[2];
  float* H[2];
  float* Z[2];
  void* wprep;        // prepared (converted / concatenated) weights
  WeightPrep wp;
};

static size_t carve(const re2nn_recurrence_args& a, char* base, RecWs* ws) {
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  const int prec = a.precision;
  RecWs w;
  memset(&w, 0, sizeof(w));
  for (int z = 0; z < 2; ++z) {
    w.tile_last[z] = (int*)take((size_t)cdiv(a.B, 128) * sizeof(int));
    w.Q[z] = take(operand_bytes(prec, a.B, a.R));
    w.Hbar[0][z] = take(operand_bytes(prec, a.B, a.S));
    w.Hbar[1][z] = take(operand_bytes(prec, a.B, a.S));
    if (a.farnn >= 1) {
      w.Hst[z] = take(operand_bytes(prec, a.B, a.S));
      w.H[z] = (float*)take((size_t)a.B * a.S * 4);
      w.Z[z] = (float*)take((size_t)a.B * a.S * 4);
    }
  }
  if (a.wprep != nullptr && prec != RE2NN_PREC_FP32)      // converted weights supplied by the caller (cached per parameter version)
    weight_prep_carve(prec, a.S, a.R, a.farnn, (char*)a.wprep, &w.wp);
  else
    off += weight_prep_carve(prec, a.S, a.R, a.farnn, base ? base + off : nullptr, &w.wp);
  if (ws) *ws = w;
  return off;
}

// last step at which any row of a 128-row tile is alive: fwd k < n, bwd k < n-1  (one warp-reduced max per tile)
__global__ void __launch_bounds__(128) tile_last_kernel(const int64_t* __restrict__ len, int B, int* __restrict__ fwd,
                                                        int* __restrict__ bwd) {
  const int m = blockIdx.x * 128 + threadIdx.x;
  int n = m < B ? (int)len[m] : 0;
  n = __reduce_max_sync(0xffffffffu, n);
  __shared__ int sh[4];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    n = max(max(sh[0], sh[1]), max(sh[2], sh[3]));
    fwd[blockIdx.x] = n - 1;
    bwd[blockIdx.x] = n - 2;
  }
}

// ---- init: step "-1" ------------------------------------------------------------------------------
template <int PREC>
__global__ void rec_init_kernel(int B, int L, int S, int farnn, const int64_t* len, const float* h0, const float* hT,
                                const float* o, RecWs w, int ldh, size_t h_plane, float* beta, float* hst_save,
                                float* hbar_save) {
  const size_t total = (size_t)2 * B * S;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int s = (int)(i % S);
    size_t r = i / S;
    int m = (int)(r % B), z = (int)(r / B);
    float h = z == 0 ? h0[s] : hT[s];
    if (farnn >= 1) {
      w.H[z][(size_t)m * S + s] = h;
      OperandFmt<PREC>::store(w.Hst[z], (size_t)m * ldh + s, h_plane, h);
    }
    if (farnn <= 1) OperandFmt<PREC>::store(w.Hbar[0][z], (size_t)m * ldh + s, h_plane, z == 1 ? h * o[s] : h);
    if (hst_save) {   // training: slab 0 of direction z
      const size_t slab = (size_t)z * (L + 1) * B * S;
      hst_save[slab + (size_t)m * S + s] = h;
      if (farnn <= 1) hbar_save[slab + (size_t)m * S + s] = z == 1 ? h * o[s] : h;
    }
    if (z == 1) {
      int n = (int)len[m];
      if (n >= 1 && n <= L) beta[((size_t)m * L + (n - 1)) * S + s] = h;   // beta_n = hT
    }
  }
}

// ---- optional per-launch timing ------------------------------------------------------------------------
struct ProfPair { cudaEvent_t a, b; };
static bool g_resident_on = true;    // inference: run the whole recurrence in one resident launch (tensor-core precisions)
static bool g_prof_on = false;
static std::vector<ProfPair> g_prof_pool;        // all event pairs ever created
static std::vector<int> g_prof_used[4];          // indices into the pool, per kernel class (3 = resident recurrence)
static std::vector<char> g_prof_captured;        // per pool entry: recorded inside stream capture (external event nodes)
static size_t g_prof_next = 0;
static std::mutex g_prof_mu;

// Works inside stream capture too: the pair is recorded as EXTERNAL event nodes, so every replay of the captured
// graph re-records the same two events and re2nn_profile_intervals() reads the launch as it ran inside the graph.
static bool prof_capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  return cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive;
}
static cudaError_t prof_record(cudaEvent_t ev, cudaStream_t st) {
  if (prof_capturing(st)) return cudaEventRecordWithFlags(ev, st, cudaEventRecordExternal);
  return cudaEventRecord(ev, st);
}
static int prof_begin(int cls, cudaStream_t st) {
  if (!g_prof_on) return -1;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (g_prof_next == g_prof_pool.size()) {
    ProfPair p;
    if (cudaEventCreate(&p.a) != cudaSuccess || cudaEventCreate(&p.b) != cudaSuccess) return -1;
    g_prof_pool.push_back(p);
    g_prof_captured.push_back(0);
  }
  int idx = (int)g_prof_next++;
  g_prof_captured[idx] = prof_capturing(st) ? 1 : 0;
  g_prof_used[cls].push_back(idx);
  prof_record(g_prof_pool[idx].a, st);
  return idx;
}
static void prof_end(int idx, cudaStream_t st) {
  if (idx >= 0) prof_record(g_prof_pool[idx].b, st);
}

// Launches whose events are current: once a graph has been captured only its (re-recorded) pairs are; the eager
// and warm-up launches registered before the capture are stale.
static std::vector<int> prof_live(int cls) {
  std::vector<int> live;
  bool any_captured = false;
  for (int c = 0; c < 4; ++c)
    for (int idx : g_prof_used[c]) any_captured = any_captured || g_prof_captured[idx];
  for (int idx : g_prof_used[cls])
    if (!any_captured || g_prof_captured[idx]) live.push_back(idx);
  return live;
}

template <int PREC, class Epi>
static cudaError_t launch_gemm(int cls, const GemmProblem& prob, const Epi& epi, const TcLaunch* plan, cudaStream_t st) {
  const int pi = prof_begin(cls, st);
  cudaError_t e;
  if (PREC == RE2NN_PREC_FP32) e = launch_simt_gemm(prob, epi, ALoadPlain{}, st);
  else e = launch_tc_gemm<PREC>(epi, plan, st);
  prof_end(pi, st);
  return e;
}

// How a call runs, decided here only (the argument check and the public queries ask this function too):
//   resident: inference on a tensor-core precision whose S and R fit the resident kernel -- one launch for all steps;
//   fused:    otherwise inference without gates on a tensor-core precision, ab_out set, no full_pad -- one direction
//             at a time, the forward state epilogue writes (alpha * beta) in operand format;
//   per-step: two or three step-GEMM launches per step (fp32, training, and everything else).
enum class RecPath { kPerStep, kResident, kFused };
static RecPath rec_path(const re2nn_recurrence_args& a) {
  if (a.precision == RE2NN_PREC_FP32 || a.save_for_backward) return RecPath::kPerStep;
  const int planes = a.precision == RE2NN_PREC_BF16 ? 1 : 2;
  if (g_resident_on && resident_supported(planes, a.S, a.R, a.precision != RE2NN_PREC_BF16)) return RecPath::kResident;
  if (a.ab_out != nullptr && a.farnn == 0 && !a.full_pad) return RecPath::kFused;
  return RecPath::kPerStep;
}

// Compile-time (NL, FARNN) of the state epilogue EpiH: calls f(EpiSel<NL, FARNN>{}).  A configuration gets its own
// instantiation where it is common enough to pay for one; -1 reads the value from StepParams at run time.  The
// resident kernel sizes its epilogue warps by FARNN, so it compiles every FARNN; the fused path runs farnn == 0 only.
template <int NL_, int FARNN_> struct EpiSel { static constexpr int NL = NL_, FARNN = FARNN_; };
enum class EpiSet { kTrain, kInfer, kFused, kResident };
template <EpiSet SET, class F>
static cudaError_t with_state_epi(int farnn, int nl, F&& f) {
  constexpr int T = RE2NN_NL_TANH;
  const bool th = nl == T;
  if constexpr (SET == EpiSet::kTrain) {
    if (th && farnn == 0) return f(EpiSel<T, 0>{});
    if (th && farnn == 2) return f(EpiSel<T, 2>{});
    return f(EpiSel<-1, -1>{});
  } else if constexpr (SET == EpiSet::kFused) {
    return th ? f(EpiSel<T, 0>{}) : f(EpiSel<-1, 0>{});
  } else if constexpr (SET == EpiSet::kInfer) {
    if (farnn == 0) return th ? f(EpiSel<T, 0>{}) : f(EpiSel<-1, 0>{});
    if (th) return farnn == 1 ? f(EpiSel<T, 1>{}) : f(EpiSel<T, 2>{});
    return f(EpiSel<-1, -1>{});
  } else {
    if (farnn == 0) return th ? f(EpiSel<T, 0>{}) : f(EpiSel<-1, 0>{});
    if (farnn == 1) return th ? f(EpiSel<T, 1>{}) : f(EpiSel<-1, 1>{});
    return th ? f(EpiSel<T, 2>{}) : f(EpiSel<-1, 2>{});
  }
}

// Inference: one resident launch (a CTA pair per 128-row tile runs all steps; recurrence_resident.cuh)
template <int PREC>
static int run_resident(const re2nn_recurrence_args& a, const RecWs& w, StepParams p, const GemmProblem& g_gate,
                        const GemmProblem* g_1, const GemmProblem* g_2, cudaStream_t st) {
  constexpr int kPlanes = OperandFmt<PREC>::kPlanes;
  std::unique_ptr<ResidentLaunch> rl(new ResidentLaunch);
  memset(rl.get(), 0, sizeof(ResidentLaunch));
  const int bn1 = resident_part(a.R), bn2 = resident_part(a.S);
  // The TMEM accumulator truncates, so the summation order is part of the result: the parity-grade split formats
  // keep the order of the per-step path (Q @ S^T first, measured 2-4x closer to fp32 than W first on cfg4);
  // bf16 starts G2 with Hbar @ W, whose operands do not wait for this step's Q
  rl->q_first = PREC == RE2NN_PREC_BF16 ? 0 : 1;
  for (int par = 0; par < 2; ++par) {
    GemmProblem r2 = g_2[par];
    if (!rl->q_first)
      for (int z = 0; z < 2; ++z) {
        r2.seg[z][0] = g_2[par].seg[z][1];
        r2.seg[z][1] = g_2[par].seg[z][0];
      }
    if (int rc = tc_make_launch<PREC>(g_1[par], &rl->g1[par], bn1)) return rc;
    if (int rc = tc_make_launch<PREC>(r2, &rl->g2[par], bn2)) return rc;
  }
  if (a.farnn >= 1)
    if (int rc = tc_make_launch<PREC>(g_gate, &rl->gate, bn2)) return rc;
  rl->steps = a.L;
  rl->alias_tbuf = resident_alias(kPlanes, rl->q_first != 0) ? 1 : 0;
  rl->stage_bytes = resident_stage_bytes(kPlanes, a.S, a.R);
  rl->stages = resident_stages(kPlanes, a.S, a.R, rl->q_first != 0);
  for (int z = 0; z < 2; ++z) { p.Hbar_cur[z] = w.Hbar[0][z]; p.Hbar_next[z] = w.Hbar[1][z]; p.Z[z] = w.Z[z]; }
  const int pi = prof_begin(3, st);
  const cudaError_t e = with_state_epi<EpiSet::kResident>(a.farnn, a.update_nonlinear, [&](auto sel) {
    using E = decltype(sel);
    return launch_resident<PREC, E::NL, E::FARNN>(*rl, p, a.B, st);
  });
  prof_end(pi, st);
  RE2NN_CUDA(e);
  return 0;
}

// Fused label-score operand (ab_out): the backward direction first (beta complete), then the forward direction
// whose state epilogue writes alpha * beta in operand format -- alpha itself is never materialised and the
// (alpha, beta) re-read of re2nn_label_scores disappears.  Single-direction launches (ndir = 1, dir_base = z).
template <int PREC>
static int run_fused(const re2nn_recurrence_args& a, const RecWs& w, StepParams p, const GemmProblem* g_1,
                     const GemmProblem* g_2, cudaStream_t st) {
  p.AB = a.ab_out; p.ldab = p.ldh; p.ab_plane = (size_t)a.B * a.L * p.ldh; p.beta_in = a.beta;
  for (int z = 0; z < 2; ++z) { p.Z[z] = w.Z[z]; p.Rg[z] = nullptr; }
  std::unique_ptr<TcLaunch[]> plan(new TcLaunch[8]);       // [z][par][g1 | g2]
  GemmProblem g1d[2][2], g2d[2][2];
  for (int z = 0; z < 2; ++z)
    for (int par = 0; par < 2; ++par) {
      g1d[z][par] = g_1[par]; g1d[z][par].ndir = 1; g1d[z][par].seg[0][0] = g_1[par].seg[z][0];
      g2d[z][par] = g_2[par]; g2d[z][par].ndir = 1;
      g2d[z][par].seg[0][0] = g_2[par].seg[z][0]; g2d[z][par].seg[0][1] = g_2[par].seg[z][1];
      if (int rc = tc_make_launch<PREC>(g1d[z][par], &plan[(z * 2 + par) * 2])) return rc;
      if (int rc = tc_make_launch<PREC>(g2d[z][par], &plan[(z * 2 + par) * 2 + 1])) return rc;
    }
  for (int zi = 0; zi < 2; ++zi) {
    const int z = 1 - zi;                                    // backward direction first
    p.dir_base = z;
    for (int k = 0; k < a.L; ++k) {
      p.k = k;
      const int par = k & 1;
      for (int zz = 0; zz < 2; ++zz) { p.Hbar_cur[zz] = w.Hbar[par][zz]; p.Hbar_next[zz] = w.Hbar[par ^ 1][zz]; }
      RE2NN_CUDA((launch_gemm<PREC>(1, g1d[z][par], EpiQ<PREC>{p}, &plan[(z * 2 + par) * 2], st)));
      const TcLaunch* p2 = &plan[(z * 2 + par) * 2 + 1];
      RE2NN_CUDA(with_state_epi<EpiSet::kFused>(a.farnn, a.update_nonlinear, [&](auto sel) {
        using E = decltype(sel);
        if (z == 1) return launch_gemm<PREC>(2, g2d[z][par], EpiH<PREC, E::NL, E::FARNN>{p}, p2, st);
        return launch_gemm<PREC>(2, g2d[z][par], EpiH<PREC, E::NL, E::FARNN, false, true>{p}, p2, st);
      }));
    }
  }
  return 0;
}

// One launch per step GEMM: gate (farnn >= 1), G1, G2.  TRAIN: the epilogues also write the save slabs.
template <int PREC, bool TRAIN>
static int run_steps(const re2nn_recurrence_args& a, const RecWs& w, StepParams p, const GemmProblem& g_gate,
                     const GemmProblem* g_1, const GemmProblem* g_2, cudaStream_t st) {
  const int B = a.B, S = a.S, R = a.R, L = a.L;
  std::unique_ptr<TcLaunch[]> plan;      // tcgen05: [gate, g1[0], g1[1], g2[0], g2[1]]; none on CUDA cores
  if constexpr (PREC != RE2NN_PREC_FP32) {
    plan.reset(new TcLaunch[5]);
    if (a.farnn >= 1)
      if (int rc = tc_make_launch<PREC>(g_gate, &plan[0])) return rc;
    for (int par = 0; par < 2; ++par) {
      if (int rc = tc_make_launch<PREC>(g_1[par], &plan[1 + par])) return rc;
      if (int rc = tc_make_launch<PREC>(g_2[par], &plan[3 + par])) return rc;
    }
  }
  auto plan_of = [&](int i) -> const TcLaunch* { return plan ? &plan[i] : nullptr; };
  for (int k = 0; k < L; ++k) {
    p.k = k;
    const int par = k & 1;
    GemmProblem gg = g_gate, g1 = g_1[par], g2 = g_2[par];
    for (int z = 0; z < 2; ++z) {
      p.Hbar_cur[z] = w.Hbar[par][z];
      p.Hbar_next[z] = w.Hbar[par ^ 1][z];
      p.Z[z] = w.Z[z];
      p.Rg[z] = nullptr;
      if constexpr (TRAIN) {
        const size_t sS = (size_t)B * S, sR = (size_t)B * R;
        float* hb_k = a.hbar_save + ((size_t)z * (L + 1) + k) * sS;
        float* hs_k = a.hst_save + ((size_t)z * (L + 1) + k) * sS;
        p.HstNext[z] = hs_k + sS;
        p.Usave[z] = a.u_save + ((size_t)z * L + k) * sR;
        p.Asave[z] = a.a_save + ((size_t)z * L + k) * sS;
        if (a.farnn >= 1) p.Z[z] = a.zsave + ((size_t)z * L + k) * sS;
        p.Rg[z] = a.farnn == 2 ? a.rsave + ((size_t)z * L + k) * sS : nullptr;
        if (PREC == RE2NN_PREC_FP32) {
          // fp32: the operands themselves live in the step-major save slabs instead of the ping-pong buffers
          p.Hbar_cur[z] = hb_k;
          p.Hbar_next[z] = hb_k + sS;
          p.Hst[z] = hs_k + sS;
          gg.seg[z][0].A = hs_k;
          g1.seg[z][0].A = hb_k;
          g2.seg[z][1].A = hb_k;
        } else {
          // tensor cores: operands stay in their (ping-pong) operand-format buffers, the epilogues add fp32 copies
          p.HbarSaveNext[z] = hb_k + sS;
          p.HbarSaveCur[z] = hb_k;
        }
      }
    }
    if (a.farnn >= 1) RE2NN_CUDA((launch_gemm<PREC>(0, gg, EpiGate<PREC, TRAIN>{p}, plan_of(0), st)));
    RE2NN_CUDA((launch_gemm<PREC>(1, g1, EpiQ<PREC, TRAIN>{p}, plan_of(1 + par), st)));
    RE2NN_CUDA(with_state_epi<TRAIN ? EpiSet::kTrain : EpiSet::kInfer>(a.farnn, a.update_nonlinear, [&](auto sel) {
      using E = decltype(sel);
      return launch_gemm<PREC>(2, g2, EpiH<PREC, E::NL, E::FARNN, TRAIN>{p}, plan_of(3 + par), st);
    }));
  }
  return 0;
}

template <int PREC>
static int run_recurrence(const re2nn_recurrence_args& a, cudaStream_t st) {
  RecWs w;
  size_t need = carve(a, (char*)a.ws, &w);
  RE2NN_CHECK(a.ws && a.ws_bytes >= need, "decompose_recurrence: workspace too small (%zu < %zu)", a.ws_bytes, need);
  const int B = a.B, S = a.S, R = a.R, L = a.L;
  const int ldh = operand_ld(PREC, S), ldq = operand_ld(PREC, R);
  RE2NN_CHECK((size_t)B * (size_t)std::max(ldh, ldq) < ((size_t)1 << 31) && (size_t)B * L < ((size_t)1 << 31),
              "decompose_recurrence: batch too large for 32-bit row indexing (B=%d)", B);
  RE2NN_CHECK(PREC == RE2NN_PREC_FP32 || L < 32768, "decompose_recurrence: tensor-core paths keep output rows in 16 bits (L=%d)", L);
  const size_t h_plane = (size_t)B * ldh, q_plane = (size_t)B * ldq;

  if (a.wprep != nullptr && PREC != RE2NN_PREC_FP32) weight_prep_bind(w.wp, a.farnn);
  else if (int rc = weight_prep_run<PREC>(a, w.wp, st)) return rc;
  tile_last_kernel<<<cdiv(B, 128), 128, 0, st>>>(a.lengths, B, w.tile_last[0], w.tile_last[1]);
  RE2NN_LAUNCH_CHECK();
  {
    size_t total = (size_t)2 * B * S;
    int blocks = (int)((total + 255) / 256);
    if (blocks > sm_count() * 8) blocks = sm_count() * 8;
    rec_init_kernel<PREC><<<blocks, 256, 0, st>>>(B, L, S, a.farnn, a.lengths, a.h0, a.hT, a.o, w, ldh, h_plane, a.beta,
                                                  a.save_for_backward ? a.hst_save : nullptr,
                                                  a.save_for_backward ? a.hbar_save : nullptr);
    RE2NN_LAUNCH_CHECK();
  }

  // the three step GEMMs, per ping-pong parity of the Hbar operand
  GemmProblem g_gate, g_1[2], g_2[2];
  memset(&g_gate, 0, sizeof(g_gate));
  g_gate.M = B; g_gate.N = S * a.farnn; g_gate.nseg = 1; g_gate.ndir = 2;
  if (a.farnn >= 1)
    for (int z = 0; z < 2; ++z) g_gate.seg[z][0] = w.wp.seg_gate(w.Hst[z], ldh, h_plane);
  for (int par = 0; par < 2; ++par) {
    memset(&g_1[par], 0, sizeof(GemmProblem));
    memset(&g_2[par], 0, sizeof(GemmProblem));
    g_1[par].M = B; g_1[par].N = R; g_1[par].nseg = 1; g_1[par].ndir = 2;   // P = Hbar @ S1 | Hbar @ S2
    g_2[par].M = B; g_2[par].N = S; g_2[par].nseg = 2; g_2[par].ndir = 2;   // Q @ S2^T + Hbar @ W | Q @ S1^T + Hbar @ W^T
    for (int z = 0; z < 2; ++z) {
      g_1[par].seg[z][0] = w.wp.seg_g1(z, w.Hbar[par][z], ldh, h_plane);
      g_2[par].seg[z][0] = w.wp.seg_g2q(z, w.Q[z], ldq, q_plane);
      g_2[par].seg[z][1] = w.wp.seg_g2w(z, w.Hbar[par][z], ldh, h_plane);
    }
  }
  StepParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.Lpad = a.Lpad; p.L = L; p.S = S; p.R = R;
  p.farnn = a.farnn; p.nl = a.update_nonlinear; p.v_mode = a.v_mode; p.full_pad = a.full_pad;
  p.sig_k = a.sigmoid_exponent;
  p.x = a.x; p.len = a.lengths; p.tile_last[0] = w.tile_last[0]; p.tile_last[1] = w.tile_last[1]; p.vtab = a.vtab; p.gtab = a.gtab; p.ldg = S * a.farnn;
  p.o = a.o; p.hinit[0] = a.h0; p.hinit[1] = a.hT;
  p.ldq = ldq; p.q_plane = q_plane; p.ldh = ldh; p.h_plane = h_plane;
  p.out[0] = a.alpha; p.out[1] = a.beta;
  for (int z = 0; z < 2; ++z) { p.Q[z] = w.Q[z]; p.Hst[z] = w.Hst[z]; p.H[z] = w.H[z]; }

  if constexpr (PREC != RE2NN_PREC_FP32) {
    switch (rec_path(a)) {
      case RecPath::kResident: return run_resident<PREC>(a, w, p, g_gate, g_1, g_2, st);
      case RecPath::kFused: return run_fused<PREC>(a, w, p, g_1, g_2, st);
      case RecPath::kPerStep: break;
    }
  }
  if (a.save_for_backward) return run_steps<PREC, true>(a, w, p, g_gate, g_1, g_2, st);
  return run_steps<PREC, false>(a, w, p, g_gate, g_1, g_2, st);
}

// Calls f(std::integral_constant<int, PREC>{}) for a RE2NN_PREC_* value.  Any other value fails with "unknown
// precision" before a CUDA call.  check_tc: the tensor-core precisions first need an sm_100 device.
template <class F>
static int with_precision(const char* who, int precision, bool check_tc, F&& f) {
  if (precision < RE2NN_PREC_FP32 || precision > RE2NN_PREC_FP16X3)
    return set_error("%s: unknown precision %d", who, precision);
  RE2NN_CHECK(!check_tc || precision == RE2NN_PREC_FP32 || re2nn_has_tcgen05(), "%s: tcgen05 path needs an sm_100 device",
              who);
  switch (precision) {
    case RE2NN_PREC_FP32: return f(std::integral_constant<int, RE2NN_PREC_FP32>{});
    case RE2NN_PREC_BF16: return f(std::integral_constant<int, RE2NN_PREC_BF16>{});
    case RE2NN_PREC_TF32X3: return f(std::integral_constant<int, RE2NN_PREC_TF32X3>{});
    default: return f(std::integral_constant<int, RE2NN_PREC_FP16X3>{});
  }
}

}  // namespace re2nn

using namespace re2nn;

// (alpha * beta) in operand format for the tcgen05 score GEMM; rows past the length are zero.
// One warp per (sequence, position) row: the row index math happens once per warp, lanes sweep the S columns
// with 16-byte loads when the row pitch allows it.
template <int PREC>
__global__ void __launch_bounds__(256) ab_operand_kernel(const float* __restrict__ alpha, const float* __restrict__ beta,
                                                         const int64_t* __restrict__ len, int B, int L, int S, int ld,
                                                         int full_pad, void* __restrict__ dst, size_t plane) {
  const size_t m = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (m >= (size_t)B * L) return;
  const int b = (int)(m / L), t = (int)(m - (size_t)b * L);
  const bool valid = full_pad || t < (int)len[b];
  const size_t row = m * (size_t)ld;
  if (valid && (S & 3) == 0) {
    const float4* a4 = reinterpret_cast<const float4*>(alpha + m * S);
    const float4* b4 = reinterpret_cast<const float4*>(beta + m * S);
    for (int c = lane; c < (S >> 2); c += 32) {
      const float4 x = __ldg(a4 + c), y = __ldg(b4 + c);
      OperandFmt<PREC>::store4(dst, row + 4 * c, plane, make_float4(x.x * y.x, x.y * y.y, x.z * y.z, x.w * y.w));
    }
    for (int s = S + lane; s < ld; s += 32) OperandFmt<PREC>::store(dst, row + s, plane, 0.f);
  } else {
    for (int s = lane; s < ld; s += 32) {
      float v = 0.f;
      if (valid && s < S) v = __ldg(alpha + m * S + s) * __ldg(beta + m * S + s);
      OperandFmt<PREC>::store(dst, row + s, plane, v);
    }
  }
}

// fp32 row-major [N x K] -> K-major PREC operand (leading dimension operand_ld(PREC, K)) at dst
template <int PREC>
static cudaError_t to_operand(const float* src, size_t N, int K, void* dst, cudaStream_t st) {
  const int ld = operand_ld(PREC, K);
  convert_weight_kernel<PREC><<<(unsigned)((N * ld + 255) / 256), 256, 0, st>>>(src, (int)N, K, K, 0, dst, ld, N * ld, 0);
  return cudaGetLastError();
}

// C[M x N] = A_op @ B_op^T on tcgen05, both operands K-major PREC operands with leading dimension operand_ld(PREC, K)
template <int PREC>
static int gemm_nt_op(const void* A, const void* B, size_t M, int N, int K, float* C, cudaStream_t st) {
  const int ld = operand_ld(PREC, K);
  TcLaunch plan;
  if (int rc = tc_make_launch<PREC>(gemm_problem((int)M, N, GemmSeg{A, B, ld, ld, K, 1, M * ld, (size_t)N * ld}), &plan))
    return rc;
  RE2NN_CUDA((launch_tc_gemm<PREC>(EpiStore{C, N, nullptr}, &plan, st)));
  return 0;
}

// Label-score workspace: the raw scores ahead of a priority layer, then the operand-format copies of (alpha * beta)
// (unless the caller has them: ab_given) and of C_mat.
static size_t label_scores_bytes(int B, int L, int S, int C, int precision, bool has_priority, bool ab_given) {
  const size_t M = (size_t)B * L;
  size_t need = 256;
  if (has_priority) need += align_up(M * C * 4, 256);
  if (precision != RE2NN_PREC_FP32) need += operand_bytes(precision, ab_given ? 0 : M, S) + operand_bytes(precision, C, S);
  return need;
}

// scores = (alpha * beta) @ C^T [@ P + b], or from the fused operand `ab` when it is given (tensor-core precisions).
static int label_scores(const char* who, const void* ab, const float* alpha, const float* beta, const int64_t* lengths,
                        int B, int L, int S, const float* C_mat, int C, const float* priority_mat,
                        const float* priority_bias, int full_pad, int precision, float* scores, void* ws,
                        size_t ws_bytes, cudaStream_t st) {
  return with_precision(who, precision, true, [&](auto prec) -> int {
    constexpr int PREC = decltype(prec)::value;
    const size_t M = (size_t)B * L;
    const size_t need = label_scores_bytes(B, L, S, C, PREC, priority_mat != nullptr, ab != nullptr);
    RE2NN_CHECK(need <= 256 || (ws && ws_bytes >= need), "%s: workspace too small", who);
    float* raw = priority_mat ? (float*)ws : scores;       // the priority layer's input, at the head of the workspace
    char* wp = (char*)ws + (priority_mat ? align_up(M * C * 4, 256) : 0);
    if constexpr (PREC == RE2NN_PREC_FP32) {
      RE2NN_CUDA(launch_simt_gemm(gemm_problem((int)M, C, GemmSeg{alpha, C_mat, S, S, S, 1, 0, 0}), EpiStore{raw, C, nullptr},
                                  ALoadAlphaBeta{alpha, beta, lengths, L, full_pad}, st));
    } else {
      if (!ab) {
        const int ld = operand_ld(PREC, S);
        ab_operand_kernel<PREC><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(alpha, beta, lengths, B, L, S, ld, full_pad, wp,
                                                                          M * ld);
        RE2NN_LAUNCH_CHECK();
        ab = wp;
        wp += operand_bytes(PREC, M, S);
      }
      RE2NN_CUDA(to_operand<PREC>(C_mat, C, S, wp, st));
      if (int rc = gemm_nt_op<PREC>(ab, wp, M, C, S, raw, st)) return rc;
    }
    if (priority_mat)
      RE2NN_CUDA(launch_simt_gemm(gemm_problem((int)M, C, GemmSeg{raw, priority_mat, C, C, C, 0, 0, 0}),
                                  EpiStore{scores, C, priority_bias}, ALoadPlain{}, st));
    return 0;
  });
}

extern "C" {

int re2nn_abi_version(void) { return RE2NN_ABI_VERSION; }

int re2nn_debug_set_tc_trace(unsigned long long* device_buf) {
  RE2NN_CUDA(cudaMemcpyToSymbol(g_tc_trace, &device_buf, sizeof(device_buf)));
  g_tc_trace_launches = device_buf ? 0 : -1;
  return 0;
}

int re2nn_debug_set_tc_timeline(unsigned long long* device_buf) {
  unsigned int zero = 0;
  RE2NN_CUDA(cudaMemcpyToSymbol(g_tc_timeline_ctr, &zero, sizeof(zero)));
  RE2NN_CUDA(cudaMemcpyToSymbol(g_tc_timeline, &device_buf, sizeof(device_buf)));
  return 0;
}

int re2nn_debug_set_tc_cta_group(int cta_group) {
  RE2NN_CHECK(cta_group >= 0 && cta_group <= 2, "debug_set_tc_cta_group: expected 0, 1 or 2");
  g_tc_force_cg = cta_group;
  return 0;
}

int re2nn_debug_set_resident(int on) {
  g_resident_on = on != 0;
  return 0;
}

int re2nn_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
  return 0;
}

int re2nn_profile_read(double* ms_out_host, int64_t* count_out_host) {
  RE2NN_CHECK(ms_out_host && count_out_host, "profile_read: null output");
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int c = 0; c < 4; ++c) {
    double tot = 0.0;
    for (int idx : g_prof_used[c]) {
      float ms = 0.f;
      RE2NN_CUDA(cudaEventSynchronize(g_prof_pool[idx].b));
      RE2NN_CUDA(cudaEventElapsedTime(&ms, g_prof_pool[idx].a, g_prof_pool[idx].b));
      tot += ms;
    }
    ms_out_host[c] = tot;
    count_out_host[c] = (int64_t)g_prof_used[c].size();
    g_prof_used[c].clear();
  }
  g_prof_next = 0;
  return 0;
}
// Per-launch intervals of one kernel class since the last clearing read, in ms relative to the earliest start of
// that class (launches on forked streams overlap: the caller takes the union).  clear = 0 keeps the event pairs
// registered, which is what a captured graph needs: its replays re-record the same events.
int re2nn_profile_intervals(int cls, double* start_ms, double* end_ms, int cap, int clear) {
  RE2NN_CHECK(cls >= 0 && cls < 4 && start_ms && end_ms && cap >= 0, "profile_intervals: bad arguments");
  std::lock_guard<std::mutex> lk(g_prof_mu);
  const std::vector<int> used = prof_live(cls);
  const int n = (int)std::min<size_t>(used.size(), (size_t)cap);
  for (int i = 0; i < n; ++i) RE2NN_CUDA(cudaEventSynchronize(g_prof_pool[used[i]].b));
  int first = 0;
  for (int i = 1; i < n; ++i) {      // earliest start: the one no other start precedes
    float d = 0.f;
    RE2NN_CUDA(cudaEventElapsedTime(&d, g_prof_pool[used[first]].a, g_prof_pool[used[i]].a));
    if (d < 0.f) first = i;
  }
  for (int i = 0; i < n; ++i) {
    float s0 = 0.f, s1 = 0.f;
    RE2NN_CUDA(cudaEventElapsedTime(&s0, g_prof_pool[used[first]].a, g_prof_pool[used[i]].a));
    RE2NN_CUDA(cudaEventElapsedTime(&s1, g_prof_pool[used[first]].a, g_prof_pool[used[i]].b));
    start_ms[i] = s0;
    end_ms[i] = s1;
  }
  if (clear) {
    for (int c = 0; c < 4; ++c) g_prof_used[c].clear();
    g_prof_next = 0;
  }
  return 0;
}
int re2nn_profile_count(int cls) {
  if (cls < 0 || cls >= 4) return 0;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  return (int)prof_live(cls).size();
}
int re2nn_profile_enabled(void) { return g_prof_on ? 1 : 0; }
const char* re2nn_last_error(void) { return re2nn::g_err; }

size_t re2nn_decompose_recurrence_workspace(const re2nn_recurrence_args* a) {
  if (!a) return 0;
  return carve(*a, nullptr, nullptr);
}

int re2nn_decompose_recurrence_fuses(const re2nn_recurrence_args* a) {
  if (!a) return 0;
  re2nn_recurrence_args q = *a;
  q.ab_out = &q;                 // as if the caller asked for the operand
  return rec_path(q) == RecPath::kFused ? 1 : 0;
}

int re2nn_decompose_recurrence_resident(const re2nn_recurrence_args* a) {
  if (!a) return 0;
  return rec_path(*a) == RecPath::kResident ? 1 : 0;
}

size_t re2nn_decompose_weight_prep_bytes(const re2nn_recurrence_args* a) {
  if (!a || a->precision == RE2NN_PREC_FP32) return 0;
  return weight_prep_carve(a->precision, a->S, a->R, a->farnn, nullptr, nullptr);
}

int re2nn_decompose_weight_prep(const re2nn_recurrence_args* a, void* out, void* stream) {
  RE2NN_CHECK(a && out && a->S1 && a->S2 && a->W, "decompose_weight_prep: null tensor");
  RE2NN_CHECK(a->precision != RE2NN_PREC_FP32, "decompose_weight_prep: the fp32 path uses the parameters as they are");
  RE2NN_CHECK(a->farnn == 0 || a->Wss1, "decompose_weight_prep: farnn>=1 needs Wss1");
  RE2NN_CHECK(a->farnn < 2 || a->Wss2, "decompose_weight_prep: farnn==2 needs Wss2");
  // no device check: the conversion kernels run on any GPU
  return with_precision("decompose_weight_prep", a->precision, false, [&](auto prec) -> int {
    WeightPrep wp;
    weight_prep_carve(prec, a->S, a->R, a->farnn, (char*)out, &wp);
    return weight_prep_run<decltype(prec)::value>(*a, wp, (cudaStream_t)stream);
  });
}

int re2nn_decompose_recurrence_launches(const re2nn_recurrence_args* a) {
  if (!a) return -1;
  int n = 2;                                                     // tile_last + rec_init
  if (a->precision == RE2NN_PREC_FP32) {
    n += a->farnn == 2 ? 1 : 0;                                  // [Wss1 | Wss2] concat
  } else if (a->wprep == nullptr) {
    WeightConv convs[kMaxWeightConvs];                           // operand-format copies of the weights
    n += weight_convs(*a, WeightPrep{}, convs);
  }
  switch (rec_path(*a)) {
    case RecPath::kResident: return n + 1;
    case RecPath::kFused: return n + a->L * 4;                  // single-direction launches, two directions
    case RecPath::kPerStep: break;
  }
  return n + a->L * (2 + (a->farnn >= 1 ? 1 : 0));
}

int re2nn_decompose_recurrence(const re2nn_recurrence_args* a, void* stream) {
  RE2NN_CHECK(a != nullptr, "decompose_recurrence: null args");
  RE2NN_CHECK(a->B > 0 && a->L > 0 && a->S > 0 && a->R > 0, "decompose_recurrence: bad dims B=%d L=%d S=%d R=%d", a->B,
              a->L, a->S, a->R);
  RE2NN_CHECK(a->L <= a->Lpad, "decompose_recurrence: L (%d) > Lpad (%d)", a->L, a->Lpad);
  RE2NN_CHECK(a->farnn >= 0 && a->farnn <= 2, "decompose_recurrence: farnn must be 0, 1 or 2 (got %d)", a->farnn);
  RE2NN_CHECK(a->update_nonlinear >= RE2NN_NL_NONE && a->update_nonlinear <= RE2NN_NL_RELUTANH,
              "decompose_recurrence: unsupported update_nonlinear %d", a->update_nonlinear);
  RE2NN_CHECK(a->v_mode == RE2NN_V_DENSE || a->x != nullptr, "decompose_recurrence: token mode needs x");
  RE2NN_CHECK(a->lengths && a->vtab && a->S1 && a->S2 && a->W && a->o && a->h0 && a->hT && a->beta &&
                  (a->alpha || rec_path(*a) == RecPath::kFused),
              "decompose_recurrence: null tensor");
  RE2NN_CHECK(a->farnn == 0 || (a->gtab && a->Wss1), "decompose_recurrence: farnn>=1 needs gtab and Wss1");
  RE2NN_CHECK(a->farnn < 2 || a->Wss2, "decompose_recurrence: farnn==2 needs Wss2");
  if (a->save_for_backward) {
    RE2NN_CHECK(a->precision != RE2NN_PREC_BF16, "decompose_recurrence: training needs a parity-grade precision");
    RE2NN_CHECK(a->hbar_save && a->hst_save && a->u_save && a->a_save, "decompose_recurrence: missing save slabs");
    RE2NN_CHECK(a->farnn == 0 || a->zsave, "decompose_recurrence: farnn>=1 training needs zsave");
    RE2NN_CHECK(a->farnn < 2 || a->rsave, "decompose_recurrence: farnn==2 training needs rsave");
  }
  return with_precision("decompose_recurrence", a->precision, true, [&](auto prec) -> int {
    return run_recurrence<decltype(prec)::value>(*a, (cudaStream_t)stream);
  });
}

size_t re2nn_gemm_nt_workspace(int precision, int M, int N, int K) {
  if (precision == RE2NN_PREC_FP32) return 256;
  return operand_bytes(precision, M, K) + operand_bytes(precision, N, K) + 256;
}

int re2nn_gemm_nt(int precision, const float* A, const float* B, int M, int N, int K, float* C, void* ws,
                  size_t ws_bytes, void* stream) {
  RE2NN_CHECK(A && B && C && M > 0 && N > 0 && K > 0, "gemm_nt: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  return with_precision("gemm_nt", precision, true, [&](auto prec) -> int {
    constexpr int PREC = decltype(prec)::value;
    if constexpr (PREC == RE2NN_PREC_FP32) {
      RE2NN_CUDA(launch_simt_gemm(gemm_problem(M, N, GemmSeg{A, B, K, K, K, 1, 0, 0}), EpiStore{C, N, nullptr},
                                  ALoadPlain{}, st));
      return 0;
    } else {
      RE2NN_CHECK(ws && ws_bytes >= re2nn_gemm_nt_workspace(precision, M, N, K), "gemm_nt: workspace too small");
      void* Bo = (char*)ws + operand_bytes(PREC, M, K);
      RE2NN_CUDA(to_operand<PREC>(A, M, K, ws, st));
      RE2NN_CUDA(to_operand<PREC>(B, N, K, Bo, st));
      return gemm_nt_op<PREC>(ws, Bo, M, N, K, C, st);
    }
  });
}

int re2nn_token_table(const float* V_embed, const float* E, const float* G, const float* beta_vec, int rows, int D,
                      int R, int additional_nonlinear, float* table, void* stream) {
  RE2NN_CHECK(V_embed && E && G && beta_vec && table, "token_table: null tensor");
  RE2NN_CHECK(rows > 0 && D > 0 && R > 0, "token_table: bad dims");
  EpiTokenTable epi{table, V_embed, beta_vec, R, additional_nonlinear};
  RE2NN_CUDA(launch_simt_gemm(gemm_problem(rows, R, GemmSeg{E, G, D, R, D, 0, 0, 0}), epi, ALoadPlain{}, (cudaStream_t)stream));
  return 0;
}

int re2nn_gate_table(const float* vtab, int rows, int R, int S, int farnn, const float* Wrs1, const float* bs1,
                     const float* Wrs2, const float* bs2, float* gate, void* stream) {
  RE2NN_CHECK(farnn == 1 || farnn == 2, "gate_table: farnn must be 1 or 2");
  RE2NN_CHECK(vtab && Wrs1 && bs1 && gate && (farnn == 1 || (Wrs2 && bs2)), "gate_table: null tensor");
  const int ldg = S * farnn;
  for (int gi = 0; gi < farnn; ++gi) {
    const GemmProblem g = gemm_problem(rows, S, GemmSeg{vtab, gi == 0 ? Wrs1 : Wrs2, R, S, R, 0, 0, 0});
    EpiStore epi{gate + (size_t)gi * S, ldg, gi == 0 ? bs1 : bs2};
    RE2NN_CUDA(launch_simt_gemm(g, epi, ALoadPlain{}, (cudaStream_t)stream));
  }
  return 0;
}

size_t re2nn_label_scores_ab_bytes(int B, int L, int S, int precision) {
  if (precision == RE2NN_PREC_FP32) return 0;
  return operand_bytes(precision, (size_t)B * L, S);
}

int re2nn_label_scores_ab(const void* ab, int B, int L, int S, const float* C_mat, int C, const float* priority_mat,
                          const float* priority_bias, int precision, float* scores, void* ws, size_t ws_bytes,
                          void* stream) {
  RE2NN_CHECK(ab && C_mat && scores && B > 0 && L > 0 && S > 0 && C > 0, "label_scores_ab: bad arguments");
  RE2NN_CHECK(precision != RE2NN_PREC_FP32, "label_scores_ab: the fused operand exists for the tensor-core precisions only");
  return label_scores("label_scores_ab", ab, nullptr, nullptr, nullptr, B, L, S, C_mat, C, priority_mat, priority_bias, 0,
                      precision, scores, ws, ws_bytes, (cudaStream_t)stream);
}

size_t re2nn_label_scores_workspace(int B, int L, int S, int C, int precision, int has_priority) {
  return label_scores_bytes(B, L, S, C, precision, has_priority != 0, false);
}

int re2nn_label_scores(const float* alpha, const float* beta, const int64_t* lengths, int B, int L, int S,
                       const float* C_mat, int C, const float* priority_mat, const float* priority_bias, int full_pad,
                       int precision, float* scores, void* ws, size_t ws_bytes, void* stream) {
  RE2NN_CHECK(alpha && beta && lengths && C_mat && scores, "label_scores: null tensor");
  return label_scores("label_scores", nullptr, alpha, beta, lengths, B, L, S, C_mat, C, priority_mat, priority_bias,
                      full_pad, precision, scores, ws, ws_bytes, (cudaStream_t)stream);
}

}  // extern "C"

extern "C" int re2nn_has_tcgen05(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10;
}
