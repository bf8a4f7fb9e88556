// Hand-written backward of the decompose i-FST path (fp32): label scores -> BPTT through both
// recurrences (gates included) -> parameter gradients.  Replaces torch.autograd over
// FARNN_S_D_W_I_S.forward_local / FARNN_S_SF.forward
// (/root/reference/src_seq/farnn/model_decompose_single.py:138-269, train_decompose.py:192).
//
// Per step k = L-1 .. 0 (both directions in every launch):
//   E1   G = g + dOut ; gate blend grads ; d pre-activation ; DA[k]                    (elementwise)
//   GEMM dq  = DA[k] @ S2|S1
//   E2   DU[k] = dq*v ; Q[k] = u*v ; dvtab[token] += dq*u                               (elementwise)
//   GEMM dhb = DU[k] @ S1^T|S2^T + DA[k] @ W^T|W
//   E3   reset-gate grads ; g <- carry + dh~ ; o / h_init products                      (elementwise)
//   GEMM g  += [dz|dr] @ [Wss1|Wss2]^T                                                  (farnn >= 1)
// Without gates E3 of step k and E1 of step k-1 are one launch (bwd_e31_kernel), the step GEMMs run on tcgen05 in
// 3xTF32, and the elementwise kernels between them are launched with programmatic stream serialization like the GEMMs.
// After the sweep every weight gradient is ONE large transposed GEMM over all (step, sequence) rows
// (K = 2*L*B) -- on tcgen05 with the operands transposed on the fly (gemm_tn_tc.cuh), CUDA cores for short reductions --
// reduced deterministically (split-K partials + ordered sum); bias / vector gradients are deterministic column sums
// of the per-step slabs.
#include <algorithm>
#include <initializer_list>
#include <memory>

#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "gemm_tn_tc.cuh"

namespace re2nn {

// ---- epilogues local to the backward ---------------------------------------------------------------------
struct EpiStore2 {          // C_z = acc (per direction output pointers)
  float* C[2];
  int ldc;
  int accumulate;           // C += acc
  __device__ __forceinline__ EpiStore2 for_dir(int z) const { EpiStore2 e = *this; e.C[0] = C[z]; return e; }
  __device__ __forceinline__ bool tile_alive(int, int) const { return true; }
  __device__ __forceinline__ RowCtx row(int) const { return RowCtx{0, 0, true}; }
  __device__ __forceinline__ Col col(int) const { return Col{0.f, 0.f}; }
  __device__ __forceinline__ Pre prefetch(const RowCtx&, int m, int n) const {
    return Pre{accumulate ? C[0][(size_t)m * ldc + n] : 0.f, 0.f};
  }
  __device__ __forceinline__ float compute(const Col&, float acc, const Pre& pre) const { return acc + pre.a; }
  __device__ __forceinline__ void store(const Col&, const RowCtx&, int m, int n, float v, float, const Pre&) const {
    C[0][(size_t)m * ldc + n] = v;
  }
  __device__ __forceinline__ void apply(const Col&, const RowCtx&, int m, int n, float acc, const Pre& pre) const {
    C[0][(size_t)m * ldc + n] = acc + pre.a;
  }
};

// dAB = draw @ C ; dAlpha = dAB * beta ; dBeta = dAB * alpha  (valid rows only)
struct EpiDAB {
  const float* alpha; const float* beta; const int64_t* len;
  float* dalpha; float* dbeta;
  int L, S, full_pad;
  __device__ __forceinline__ EpiDAB for_dir(int) const { return *this; }
  __device__ __forceinline__ bool tile_alive(int, int) const { return true; }
  __device__ __forceinline__ RowCtx row(int m) const {
    int b = m / L, t = m - b * L;
    return RowCtx{0, (full_pad || t < (int)len[b]) ? 0 : -1, true};
  }
  __device__ __forceinline__ Col col(int) const { return Col{0.f, 0.f}; }
  __device__ __forceinline__ Pre prefetch(const RowCtx& r, int m, int n) const {
    if (r.orow < 0) return Pre{0.f, 0.f};
    size_t i = (size_t)m * S + n;
    return Pre{alpha[i], beta[i]};
  }
  __device__ __forceinline__ void apply(const Col&, const RowCtx& r, int m, int n, float acc, const Pre& pre) const {
    size_t i = (size_t)m * S + n;
    dalpha[i] = r.orow < 0 ? 0.f : acc * pre.b;
    dbeta[i] = r.orow < 0 ? 0.f : acc * pre.a;
  }
  // compute / store split of the tcgen05 epilogue (batches of rows: all arithmetic, then all stores)
  static constexpr bool kRows = false;
  __device__ __forceinline__ float compute(const Col&, float acc, const Pre&) const { return acc; }
  __device__ __forceinline__ void store(const Col& c, const RowCtx& r, int m, int n, float v, float, const Pre& pre) const {
    apply(c, r, m, n, v, pre);
  }
};

// ---- transposed ("TN") GEMM: C[P x Q] = sum over pairs, rows m:  X[m, p] * Y[m, q]  ---------------------------
// (TnPair / TnProblem: gemm_tn_tc.cuh, which holds the tcgen05 version of this kernel)

// The right operand as the CUDA-core kernel reads it: Y itself, or the masked Y * Y2 of a problem with Y2 (run_tn)
struct YLoadPlain {
  __device__ __forceinline__ float operator()(const TnPair& pr, size_t m, int q) const { return __ldg(pr.Y + m * pr.ldy + q); }
};
struct YLoadAlphaBeta {
  const float* beta; const int64_t* len; int L, full_pad;
  __device__ __forceinline__ float operator()(const TnPair& pr, size_t m, int q) const {
    int b = (int)(m / L), t = (int)(m - (size_t)b * L);
    if (!full_pad && t >= (int)len[b]) return 0.f;
    return __ldg(pr.Y + m * pr.ldy + q) * __ldg(beta + m * pr.ldy + q);
  }
};

constexpr int kTnSplit = 64;

template <class YLoad>
__global__ void __launch_bounds__(256) tn_gemm_kernel(const TnProblem prob, float* __restrict__ partial, const YLoad yload) {
  constexpr int BP = 64, BQ = 64, BK = 16;
  __shared__ __align__(16) float Xs[BK][BP + 4];
  __shared__ __align__(16) float Ys[BK][BQ + 4];
  const int p0 = blockIdx.x * BP, q0 = blockIdx.y * BQ, split = blockIdx.z;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int pi = 0; pi < prob.npairs; ++pi) {
    const TnPair pr = prob.pair[pi];
    const size_t chunk = (pr.rows + kTnSplit - 1) / kTnSplit;
    const size_t r0 = chunk * split, r1 = min(pr.rows, r0 + chunk);
    for (size_t m0 = r0; m0 < r1; m0 += BK) {
#pragma unroll
      for (int i = 0; i < (BP * BK) / 256; ++i) {
        int idx = tid + i * 256;
        int pp = idx & (BP - 1), kk = idx >> 6;
        float v = 0.f;
        if (m0 + kk < r1 && p0 + pp < prob.P) v = __ldg(pr.X + (m0 + kk) * pr.ldx + p0 + pp);
        Xs[kk][pp] = v;
      }
#pragma unroll
      for (int i = 0; i < (BQ * BK) / 256; ++i) {
        int idx = tid + i * 256;
        int qq = idx & (BQ - 1), kk = idx >> 6;
        float v = 0.f;
        if (m0 + kk < r1 && q0 + qq < prob.Q) v = yload(pr, m0 + kk, q0 + qq);
        Ys[kk][qq] = v;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        const float4 a = *reinterpret_cast<const float4*>(&Xs[kk][ty * 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Ys[kk][tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
  float* out = partial + (size_t)split * prob.P * prob.Q;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int pp = p0 + ty * 4 + i;
    if (pp >= prob.P) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int qq = q0 + tx * 4 + j;
      if (qq < prob.Q) out[(size_t)pp * prob.Q + qq] = acc[i][j];
    }
  }
}

// out[i] (+)= sum_s partial[s][i]   (ordered => deterministic)
__global__ void split_reduce_kernel(const float* __restrict__ partial, int nsplit, size_t n, float* __restrict__ out,
                                    int accumulate) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float acc = accumulate ? out[i] : 0.f;
    for (int s = 0; s < nsplit; ++s) acc += partial[(size_t)s * n + i];
    out[i] = acc;
  }
}

static bool g_tn_tc = true;      // long reductions on tcgen05 (gemm_tn_tc.cuh); re2nn_debug_set_tn_tc

enum { kTnPathCuda = 1, kTnPathTc = 2 };

// The kernel a weight-gradient product of P x Q over `rows` summed rows runs on: tcgen05 once the reduction is long
// enough to fill a pipeline per CTA, the CUDA-core kernel otherwise.
static int tn_path(int P, int Q, size_t rows) {
  if (g_tn_tc && re2nn_has_tcgen05() != 0 && rows >= 4096 && P >= 16 && Q >= 16) return kTnPathTc;
  return kTnPathCuda;
}

// out (+)= sum over pairs X^T Y.  path 0 = tn_path's choice; kTnPathTc requires tcgen05 and P, Q >= 16 (callers check).
// The partial buffer holds kTnSplit slices of P x Q.
static cudaError_t run_tn(const TnProblem& prob, float* partial, float* out, int accumulate, cudaStream_t st, int path = 0) {
  const size_t n = (size_t)prob.P * prob.Q;
  size_t rows = 0;
  for (int i = 0; i < prob.npairs; ++i) rows += prob.pair[i].rows;
  if (path == 0) path = tn_path(prob.P, prob.Q, rows);
  if (path == kTnPathTc) {
    // Consecutive row chunks of at most kTnSplit * kTnMaxKb k-blocks (shared by the pairs), so that no split of any
    // launch accumulates more than kTnMaxKb k-blocks; the later chunks add onto `out`.  Masked chunks start on a sequence.
    size_t crows = (size_t)kTnSplit * kTnMaxKb * kTnKBlock / prob.npairs, longest = 0;
    if (prob.mask_len != nullptr) crows = std::max<size_t>(crows / prob.mask_L, 1) * prob.mask_L;
    for (int i = 0; i < prob.npairs; ++i) longest = std::max(longest, prob.pair[i].rows);
    for (size_t c0 = 0; c0 == 0 || c0 < longest; c0 += crows) {
      TnProblem sub = prob;         // one chunk: the problem itself
      sub.npairs = 0;
      for (int i = 0; i < prob.npairs; ++i) {
        const TnPair& p = prob.pair[i];
        if (c0 > 0 && p.rows <= c0) continue;
        sub.pair[sub.npairs++] = TnPair{p.X + c0 * p.ldx, p.Y + c0 * p.ldy, p.ldx, p.ldy, std::min(p.rows - c0, crows)};
      }
      if (prob.Y2 != nullptr) sub.Y2 = prob.Y2 + c0 * prob.pair[0].ldy;     // Y2 goes with a single pair
      if (prob.mask_len != nullptr) sub.mask_len = prob.mask_len + c0 / prob.mask_L;
      const TnTcPlan pl = tn_tc_plan(sub, kTnSplit);
      if (cudaError_t e = launch_tn_tc(sub, partial, pl, st)) return e;
      split_reduce_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 1184), 256, 0, st>>>(partial, pl.nsplit, n, out,
                                                                                             c0 == 0 ? accumulate : 1);
      if (cudaError_t e = cudaGetLastError()) return e;
    }
    return cudaSuccess;
  }
  dim3 grid(cdiv(prob.P, 64), cdiv(prob.Q, 64), kTnSplit);
  if (prob.Y2 == nullptr) {
    tn_gemm_kernel<<<grid, 256, 0, st>>>(prob, partial, YLoadPlain{});
  } else {
    const bool masked = prob.mask_len != nullptr;
    const YLoadAlphaBeta yl{prob.Y2, prob.mask_len, masked ? prob.mask_L : 1, masked ? 0 : 1};
    tn_gemm_kernel<<<grid, 256, 0, st>>>(prob, partial, yl);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  split_reduce_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 1184), 256, 0, st>>>(partial, kTnSplit, n, out, accumulate);
  return cudaGetLastError();
}

// out = sum over `pairs` X^T Y (nothing when out is NULL)
static cudaError_t tn(float* out, int P, int Q, std::initializer_list<TnPair> pairs, float* partial, cudaStream_t st) {
  if (out == nullptr) return cudaSuccess;
  TnProblem t;
  memset(&t, 0, sizeof(t));
  t.P = P; t.Q = Q;
  for (const TnPair& p : pairs) t.pair[t.npairs++] = p;
  return run_tn(t, partial, out, 0, st);
}

// deterministic column sums: out[c] (+)= sum_r X[r, c].  grid (column blocks of 32, row splits): every CTA sums its
// contiguous row range for 32 columns (32 x 32 threads, fixed order); with more than one split the partials go to
// `part[split][c]` and colsum_finish_kernel adds them in split order, so the result does not depend on scheduling.
__global__ void __launch_bounds__(1024) colsum_rows_kernel(const float* __restrict__ X, size_t rows, int cols, int ld,
                                                           float* __restrict__ out, int accumulate,
                                                           float* __restrict__ part) {
  __shared__ float sh[32][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const size_t per = (rows + gridDim.y - 1) / gridDim.y;
  const size_t r0 = (size_t)blockIdx.y * per, r1 = r0 + per < rows ? r0 + per : rows;
  float acc = 0.f;
  if (c < cols)
    for (size_t r = r0 + threadIdx.y; r < r1; r += 32) acc += X[r * ld + c];
  sh[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float t = (part == nullptr && accumulate) ? out[c] : 0.f;
    for (int i = 0; i < 32; ++i) t += sh[i][threadIdx.x];
    if (part) part[(size_t)blockIdx.y * cols + c] = t;
    else out[c] = t;
  }
}
__global__ void colsum_finish_kernel(const float* __restrict__ part, int nsplit, int cols, float* __restrict__ out,
                                     int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float t = accumulate ? out[c] : 0.f;
  for (int i = 0; i < nsplit; ++i) t += part[(size_t)i * cols + c];
  out[c] = t;
}
// ws: optional scratch of at least 64 * cols floats; tall inputs are then split over up to 64 CTAs per column block
static cudaError_t colsum_rows(const float* X, size_t rows, int cols, int ld, float* out, int accumulate, cudaStream_t st,
                               float* ws = nullptr) {
  const int nsplit = ws ? (int)std::min<size_t>(64, (rows + 2047) / 2048) : 1;
  if (nsplit <= 1) {
    colsum_rows_kernel<<<dim3(cdiv(cols, 32), 1), dim3(32, 32), 0, st>>>(X, rows, cols, ld, out, accumulate, nullptr);
    return cudaGetLastError();
  }
  colsum_rows_kernel<<<dim3(cdiv(cols, 32), nsplit), dim3(32, 32), 0, st>>>(X, rows, cols, ld, out, accumulate, ws);
  colsum_finish_kernel<<<cdiv(cols, 256), 256, 0, st>>>(ws, nsplit, cols, out, accumulate);
  return cudaGetLastError();
}

// ---- per-step elementwise kernels ------------------------------------------------------------------------------
struct BwdCtx {
  int B, Lpad, L, S, R, k, farnn, nl, v_mode, full_pad;
  float kappa;
  const int64_t* x; const int64_t* len;
  const float *vtab, *o, *h0, *hT;
  const float *dalpha, *dbeta;                       // B x L x S
  const float *hst_save, *u_save, *a_save, *zsave, *rsave;
  float *g, *GA;                                     // 2 x B x S
  float *DA, *DZR, *DOprod, *Pinit;                  // slabs 2 x L x B x (S | S*farnn)
  float *DU, *Qs;                                    // slabs 2 x L x B x R
  float *DQ, *DHb;                                   // 2 x B x R, 2 x B x S
  float *dvtab, *dgtab;
  // tensor-core sweep: 3xTF32 operand-format copies of this step's DA / DU (A operands of the two step GEMMs)
  void* DAop[2]; void* DUop[2];
  void* DZop[2]; void* DRop[2];                      // farnn >= 1: dz / dr of this step (A operands of the gate GEMM)
  int ldS, ldR;
  size_t da_plane, du_plane;
  void* DrawOp; void* CmatOp;                        // tensor-core label-score backward: operand-format draw / C_mat^T
};

__device__ __forceinline__ size_t slab(const BwdCtx& c, int z, int k, int width) {
  return ((size_t)z * c.L + k) * c.B * width;
}
__device__ __forceinline__ size_t slab1(const BwdCtx& c, int z, int k, int width) {   // (L+1)-deep save slabs
  return ((size_t)z * (c.L + 1) + k) * c.B * width;
}

// Grid-stride loop over the (direction z, sequence b, column) elements of step c.k, columns fastest, with the row's
// step position: f(z, b, column, n = len[b], tpos, orow, alive).
template <class F>
__device__ __forceinline__ void for_each_elem(const BwdCtx& c, int width, const F& f) {
  const size_t total = (size_t)2 * c.B * width;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int col = (int)(i % width);
    const size_t rr = i / width;
    const int b = (int)(rr % c.B), z = (int)(rr / c.B);
    const int n = (int)c.len[b];
    int tpos, orow;
    bool alive;
    step_pos(z, c.k, n, c.full_pad, tpos, orow, alive);
    f(z, b, col, n, tpos, orow, alive);
  }
}

// E3 of element (z, b, s) at step c.k: DHb -> the carry g for step k-1 (GA + gB; GA = 0 without gates) and DOprod of the
// backward direction; with the reset gate also Pinit and the reset-gate gradient.  A row that is not alive gets zeros
// and keeps its carry (0 until the row's last live step).  Returns the carry.  kGates = true (bwd_e3_kernel): c.farnn
// decides, the carry is stored; false (bwd_e31_kernel): farnn = 0 is known, the gate branches are compiled out and the
// carry is stored only at k = 0, where it feeds dh0 / dhT.
template <bool kGates>
__device__ __forceinline__ float bwd_e3(const BwdCtx& c, int z, int b, int s, float on, bool alive) {
  const size_t e = (size_t)b * c.S + s;
  const size_t gi = (size_t)z * c.B * c.S + e;
  // formed where it is used: inside `z == 1` the index is uniform (fewer registers in bwd_e31_kernel)
  const auto sl = [&] { return slab(c, z, c.k, c.S) + e; };
  const int gw = c.S * c.farnn;
  const bool reset = kGates && c.farnn == 2;
  if (!alive) {
    const float g = c.g[gi];
    if (z == 1) c.DOprod[sl()] = 0.f;
    if (reset) {
      c.Pinit[sl()] = 0.f;
      c.DZR[slab(c, z, c.k, gw) + (size_t)b * gw + c.S + s] = 0.f;
      if (c.DRop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DRop[z], (size_t)b * c.ldS + s, c.da_plane, 0.f);
    }
    return g;
  }
  const float dhb = c.DHb[gi];
  const float hk = kGates ? c.hst_save[slab1(c, z, c.k, c.S) + e] : 0.f;   // without gates: loaded below, z = 1 only
  const float hinit = z == 0 ? c.h0[s] : c.hT[s];
  float rt = 1.f;
  if (reset) rt = c.rsave[sl()];
  const float htil = reset ? (1.f - rt) * hinit + rt * hk : hk;
  float dht = dhb;
  if (z == 1) {
    dht = dhb * on;
    c.DOprod[sl()] = dhb * (kGates ? htil : c.hst_save[slab1(c, z, c.k, c.S) + e]);
  }
  float gB = dht;
  if (reset) {
    gB = dht * rt;
    c.Pinit[sl()] = dht * (1.f - rt);
    const float drpre = dht * (hk - hinit) * rt * (1.f - rt) * c.kappa;
    c.DZR[slab(c, z, c.k, gw) + (size_t)b * gw + c.S + s] = drpre;
    if (c.DRop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DRop[z], (size_t)b * c.ldS + s, c.da_plane, drpre);
  }
  const float g = (kGates ? c.GA[gi] : 0.f) + gB;       // without gates: 0.f + gB, as GA + gB with GA = 0
  if (kGates || c.k == 0) c.g[gi] = g;
  return g;
}

__global__ void bwd_e1_kernel(const BwdCtx c) {
  for_each_elem(c, c.S, [&](int z, int b, int s, int, int, int orow, bool alive) {
    const size_t e = (size_t)b * c.S + s;
    const size_t sl = slab(c, z, c.k, c.S) + e;
    const int gw = c.S * c.farnn;
    if (!alive) {
      c.DA[sl] = 0.f;
      if (c.DAop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DAop[z], (size_t)b * c.ldS + s, c.da_plane, 0.f);
      if (z == 0) c.DOprod[sl] = 0.f;
      if (c.farnn >= 1) {
        c.DZR[slab(c, z, c.k, gw) + (size_t)b * gw + s] = 0.f;
        if (c.DZop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DZop[z], (size_t)b * c.ldS + s, c.da_plane, 0.f);
      }
      c.GA[(size_t)z * c.B * c.S + e] = 0.f;
      return;
    }
    const float* dout = z == 0 ? c.dalpha : c.dbeta;
    const float G = c.g[(size_t)z * c.B * c.S + e] + (orow >= 0 ? dout[((size_t)b * c.L + orow) * c.S + s] : 0.f);
    const float a = c.a_save[sl];
    const float on = c.o[s];
    const float hhat = apply_nl(z == 0 ? a * on : a, c.nl);
    float dhhat = G, gA = 0.f;
    if (c.farnn >= 1) {
      const float zt = c.zsave[sl];
      const float hk = c.hst_save[slab1(c, z, c.k, c.S) + e];
      dhhat = G * zt;
      gA = G * (1.f - zt);
      const float dzpre = G * (hhat - hk) * zt * (1.f - zt) * c.kappa;
      c.DZR[slab(c, z, c.k, gw) + (size_t)b * gw + s] = dzpre;
      if (c.DZop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DZop[z], (size_t)b * c.ldS + s, c.da_plane, dzpre);
    }
    const float dpre = dhhat * nl_grad_from_out(hhat, c.nl);
    const float da = z == 0 ? dpre * on : dpre;
    c.DA[sl] = da;
    if (z == 0) c.DOprod[sl] = dpre * a;
    if (c.DAop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DAop[z], (size_t)b * c.ldS + s, c.da_plane, da);
    c.GA[(size_t)z * c.B * c.S + e] = gA;
  });
}

// bwd_e2 / bwd_e31 sit between two tcgen05 step GEMMs 35 times per sweep: they are launched with programmatic stream
// serialization like the GEMMs, let the next GEMM begin its prologue (barrier init, TMEM allocation, descriptor
// prefetch) right away and wait for the previous GEMM's results themselves.
__global__ void bwd_e2_kernel(const BwdCtx c) {
  griddep_launch_dependents();
  griddep_wait();
  for_each_elem(c, c.R, [&](int z, int b, int r, int, int tpos, int, bool alive) {
    const size_t e = (size_t)b * c.R + r;
    const size_t sl = slab(c, z, c.k, c.R) + e;
    if (!alive) {
      c.DU[sl] = 0.f;
      c.Qs[sl] = 0.f;
      if (c.DUop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DUop[z], (size_t)b * c.ldR + r, c.du_plane, 0.f);
      return;
    }
    const size_t vrow = c.v_mode == RE2NN_V_TOKEN ? (size_t)c.x[(size_t)b * c.Lpad + tpos] : (size_t)b * c.Lpad + tpos;
    const float v = c.vtab[vrow * c.R + r];
    const float u = c.u_save[sl];
    const float dq = c.DQ[(size_t)z * c.B * c.R + e];
    c.DU[sl] = dq * v;
    if (c.DUop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DUop[z], (size_t)b * c.ldR + r, c.du_plane, dq * v);
    c.Qs[sl] = u * v;
    const float dv = dq * u;
    if (dv != 0.f) atomicAdd(c.dvtab + vrow * c.R + r, dv);
  });
}

__global__ void bwd_e3_kernel(const BwdCtx c) {
  for_each_elem(c, c.S, [&](int z, int b, int s, int, int, int, bool alive) {
    bwd_e3<true>(c, z, b, s, c.o[s], alive);
  });
}

// farnn = 0: E3 of step k and E1 of step k-1 touch the same element and nothing runs between them (no gate GEMM), so
// they are one launch: the carry g stays in a register, the GA / g round trip disappears.  Same arithmetic, same order.
__global__ void bwd_e31_kernel(const BwdCtx c) {
  griddep_launch_dependents();
  griddep_wait();
  for_each_elem(c, c.S, [&](int z, int b, int s, int n, int tpos, int orow, bool alive) {
    const float on = c.o[s];
    const float g = bwd_e3<false>(c, z, b, s, on, alive);
    if (c.k == 0) return;
    // ---- E1 of step k-1, without gates.  Written out here rather than shared with bwd_e1_kernel: a shared device
    // helper compiled to 30-32 registers for this kernel instead of 28.
    const int k1 = c.k - 1;
    step_pos(z, k1, n, c.full_pad, tpos, orow, alive);
    const size_t e = (size_t)b * c.S + s;
    const size_t sl = slab(c, z, k1, c.S) + e;
    if (!alive) {
      c.DA[sl] = 0.f;
      if (c.DAop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DAop[z], (size_t)b * c.ldS + s, c.da_plane, 0.f);
      if (z == 0) c.DOprod[sl] = 0.f;
      return;
    }
    const float* dout = z == 0 ? c.dalpha : c.dbeta;
    const float G = g + (orow >= 0 ? dout[((size_t)b * c.L + orow) * c.S + s] : 0.f);
    const float a = c.a_save[sl];
    const float hhat = apply_nl(z == 0 ? a * on : a, c.nl);
    const float dpre = G * nl_grad_from_out(hhat, c.nl);
    const float da = z == 0 ? dpre * on : dpre;
    c.DA[sl] = da;
    if (z == 0) c.DOprod[sl] = dpre * a;
    if (c.DAop[0]) OperandFmt<RE2NN_PREC_TF32X3>::store(c.DAop[z], (size_t)b * c.ldS + s, c.da_plane, da);
  });
}

// dgtab[token] += [dz | dr] of this step (after the gate slab is complete)
__global__ void bwd_gate_scatter_kernel(const BwdCtx c) {
  const int gw = c.S * c.farnn;
  for_each_elem(c, gw, [&](int z, int b, int col, int, int tpos, int, bool alive) {
    if (!alive) return;
    const float v = c.DZR[slab(c, z, c.k, gw) + (size_t)b * gw + col];
    if (v == 0.f) return;
    const size_t vrow = c.v_mode == RE2NN_V_TOKEN ? (size_t)c.x[(size_t)b * c.Lpad + tpos] : (size_t)b * c.Lpad + tpos;
    atomicAdd(c.dgtab + vrow * gw + col, v);
  });
}

// dhT += sum_b dbeta[b, n_b - 1, :]   (beta_n = hT is emitted directly)
__global__ void bwd_direct_hT_kernel(const float* __restrict__ dbeta, const int64_t* __restrict__ len, int B, int L,
                                     int S, float* __restrict__ dhT) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  float acc = dhT[s];
  for (int b = 0; b < B; ++b) {
    int n = (int)len[b];
    if (n >= 1 && n <= L) acc += dbeta[((size_t)b * L + (n - 1)) * S + s];
  }
  dhT[s] = acc;
}

// token table backward, elementwise part: gen = phi(E@G) arrives as the GEMM accumulator
struct EpiTokenBwd {
  const float* dvtab; const float* V_embed; const float* beta_vec;
  float* dV; float* dbeta_prod; float* dGpre;
  int R, nl;
  __device__ __forceinline__ EpiTokenBwd for_dir(int) const { return *this; }
  __device__ __forceinline__ bool tile_alive(int, int) const { return true; }
  __device__ __forceinline__ RowCtx row(int) const { return RowCtx{0, 0, true}; }
  __device__ __forceinline__ Col col(int n) const { return Col{__ldg(beta_vec + n), 0.f}; }
  __device__ __forceinline__ Pre prefetch(const RowCtx&, int m, int n) const {
    size_t i = (size_t)m * R + n;
    return Pre{dvtab[i], V_embed[i]};
  }
  __device__ __forceinline__ void apply(const Col& c, const RowCtx&, int m, int n, float acc, const Pre& pre) const {
    const size_t i = (size_t)m * R + n;
    const float gen = apply_nl(acc, nl);
    if (dV) dV[i] = pre.a * c.a;
    dbeta_prod[i] = pre.a * (pre.b - gen);
    dGpre[i] = pre.a * (1.f - c.a) * nl_grad_from_out(gen, nl);
  }
};

// The two GEMMs of every BPTT step (dq = DA @ S, dhbar = DU @ S^T + DA @ W^T) run on the tensor cores in 3xTF32
// (fp32-grade products, 8-bit exponent: safe for gradients of any magnitude) when tcgen05 is there.
static bool g_bwd_tc = true;
static bool bwd_uses_tc() { return g_bwd_tc && re2nn_has_tcgen05() != 0; }

static size_t bwd_carve(const re2nn_backward_args& a, char* base, BwdCtx* c, float** draw, float** partial,
                        float** dalpha, float** dbeta, WeightPrep* wp = nullptr) {
  size_t off = 0;
  auto take = [&](size_t floats) -> float* {
    float* p = base ? (float*)(base + off) : nullptr;
    off += align_up(floats * 4, 256);
    return p;
  };
  const size_t B = a.B, L = a.L, S = a.S, R = a.R, gw = (size_t)a.S * a.farnn;
  BwdCtx x;
  memset(&x, 0, sizeof(x));
  float* dA = take(B * L * S);
  float* dBt = take(B * L * S);
  x.g = take(2 * B * S);
  x.GA = take(2 * B * S);
  x.DA = take(2 * L * B * S);
  x.DOprod = take(2 * L * B * S);
  x.DU = take(2 * L * B * R);
  x.Qs = take(2 * L * B * R);
  x.DQ = take(2 * B * R);
  x.DHb = take(2 * B * S);
  if (a.farnn >= 1) {
    x.DZR = take(2 * L * B * gw);
    x.dgtab = take((size_t)a.table_rows * gw);
  }
  if (a.farnn == 2) x.Pinit = take(2 * L * B * S);
  float* dr = a.priority_mat ? take(B * L * (size_t)a.C) : nullptr;
  size_t pmax = std::max({S * R, S * S, (size_t)a.C * S, gw ? S * S : (size_t)0, gw ? R * S : (size_t)0});
  float* part = take((size_t)kTnSplit * pmax);
  if (bwd_uses_tc()) {
    constexpr int P = RE2NN_PREC_TF32X3;
    x.ldS = operand_ld(P, (int)S); x.ldR = operand_ld(P, (int)R);
    x.da_plane = B * x.ldS; x.du_plane = B * x.ldR;
    for (int z = 0; z < 2; ++z) {
      x.DAop[z] = take(operand_bytes(P, B, (int)S) / 4);
      x.DUop[z] = take(operand_bytes(P, B, (int)R) / 4);
    }
    if (a.C > 0) {        // label-score backward on tensor cores: draw (B*L x C) and C_mat^T (S x C) in operand format
      x.DrawOp = take(operand_bytes(P, B * L, a.C) / 4);
      x.CmatOp = take(operand_bytes(P, S, a.C) / 4);
    }
    for (int z = 0; z < 2 && a.farnn >= 1; ++z) {
      x.DZop[z] = take(operand_bytes(P, B, (int)S) / 4);
      if (a.farnn == 2) x.DRop[z] = take(operand_bytes(P, B, (int)S) / 4);
    }
    WeightPrep w;
    off += weight_prep_carve(P, (int)S, (int)R, 0, base ? base + off : nullptr, &w);
    if (a.farnn >= 1) {      // K-major copies of Wss1 / Wss2 themselves (the forward holds their transposes)
      w.buf[6] = take(operand_bytes(P, S, (int)S) / 4);
      if (a.farnn == 2) w.buf[7] = take(operand_bytes(P, S, (int)S) / 4);
    }
    if (wp) *wp = w;
  }
  if (c) *c = x;
  if (draw) *draw = dr;
  if (partial) *partial = part;
  if (dalpha) *dalpha = dA;
  if (dbeta) *dbeta = dBt;
  return off;
}

// launch with programmatic stream serialization (the kernel calls griddepcontrol itself)
static cudaError_t launch_pdl(void (*kernel)(BwdCtx), int grid, cudaStream_t st, const BwdCtx& c) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(256);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, c);
}

static int grid_for(size_t total) { return (int)std::min<size_t>((total + 255) / 256, (size_t)sm_count() * 16); }

// One GEMM of a BPTT step: on tcgen05 in 3xTF32 when it has a launch plan (whose tensor maps name the operand-format
// copies), else on CUDA cores over the fp32 operands of `g`.
static cudaError_t step_gemm(const GemmProblem& g, const EpiStore2& epi, const TcLaunch* tl, cudaStream_t st) {
  if (tl) return launch_tc_gemm<RE2NN_PREC_TF32X3>(epi, tl, st);
  return launch_simt_gemm(g, epi, ALoadPlain{}, st);
}

// Label-score backward: undo the priority layer (draw = dscores @ P^T into draw_ws; draw = dscores without one), then
// dAB = draw @ C_mat -> dalpha = dAB * beta, dbeta = dAB * alpha (EpiDAB).  Given operand-format buffers for draw and
// C_mat^T, the second GEMM runs on tcgen05 in 3xTF32: it is tiny (K = C), what matters is the coalesced epilogue over
// alpha / beta / dalpha / dbeta.  Without them it runs on CUDA cores.  draw_out (optional) receives draw.
static int label_scores_bwd(const float* dscores, const float* priority_mat, float* draw_ws, const float* C_mat, int C,
                            const EpiDAB& edab, int B, void* draw_op, void* cmat_op, cudaStream_t st,
                            const float** draw_out) {
  const int M = B * edab.L, S = edab.S;
  const float* draw = dscores;
  if (priority_mat) {
    RE2NN_CUDA(launch_simt_gemm(gemm_problem(M, C, GemmSeg{dscores, priority_mat, C, C, C, 1, 0, 0}),
                                EpiStore{draw_ws, C, nullptr}, ALoadPlain{}, st));
    draw = draw_ws;
  }
  if (draw_op) {
    constexpr int P = RE2NN_PREC_TF32X3;
    const int ldc = operand_ld(P, C);
    const size_t pa = (size_t)M * ldc, pb = (size_t)S * ldc;
    convert_weight_kernel<P><<<(unsigned)std::min<size_t>((pa + 255) / 256, (size_t)sm_count() * 32), 256, 0, st>>>(
        draw, M, C, C, 0, draw_op, ldc, pa, 0);
    RE2NN_LAUNCH_CHECK();
    convert_weight_kernel<P><<<(unsigned)((pb + 255) / 256), 256, 0, st>>>(C_mat, S, C, S, 1, cmat_op, ldc, pb, 0);
    RE2NN_LAUNCH_CHECK();
    std::unique_ptr<TcLaunch> tl(new TcLaunch);
    if (int rc = tc_make_launch<P>(gemm_problem(M, S, GemmSeg{draw_op, cmat_op, ldc, ldc, C, 1, pa, pb}), tl.get()))
      return rc;
    RE2NN_CUDA((launch_tc_gemm<P>(edab, tl.get(), st)));
  } else {
    RE2NN_CUDA(launch_simt_gemm(gemm_problem(M, S, GemmSeg{draw, C_mat, C, S, C, 0, 0, 0}), edab, ALoadPlain{}, st));
  }
  if (draw_out) *draw_out = draw;
  return 0;
}

static int run_backward(const re2nn_backward_args& a, cudaStream_t st) {
  BwdCtx c;
  float *draw_ws, *partial, *dalpha, *dbeta;
  WeightPrep wp;
  memset(&wp, 0, sizeof(wp));
  const bool tc = bwd_uses_tc();
  const size_t need = bwd_carve(a, (char*)a.ws, &c, &draw_ws, &partial, &dalpha, &dbeta, &wp);
  RE2NN_CHECK(a.ws && a.ws_bytes >= need, "decompose_backward: workspace too small (%zu < %zu)", a.ws_bytes, need);
  const int B = a.B, L = a.L, S = a.S, R = a.R, C = a.C, gw = a.S * a.farnn;
  const size_t M = (size_t)B * L;
  c.B = B; c.Lpad = a.Lpad; c.L = L; c.S = S; c.R = R; c.farnn = a.farnn; c.nl = a.update_nonlinear;
  c.v_mode = a.v_mode; c.full_pad = a.full_pad; c.kappa = a.sigmoid_exponent;
  c.x = a.x; c.len = a.lengths; c.vtab = a.vtab; c.o = a.o; c.h0 = a.h0; c.hT = a.hT;
  c.dalpha = dalpha; c.dbeta = dbeta;
  c.hst_save = a.hst_save; c.u_save = a.u_save; c.a_save = a.a_save; c.zsave = a.zsave; c.rsave = a.rsave;
  c.dvtab = a.dvtab;

  const bool direct = a.dalpha_in != nullptr && a.dbeta_in != nullptr;   // caller differentiated its own score stage
  if (direct) {
    c.dalpha = a.dalpha_in; c.dbeta = a.dbeta_in;
    dbeta = const_cast<float*>(a.dbeta_in);
  } else {
    // 1. dscores -> dAlpha, dBeta (on tcgen05 when the carve made operand-format buffers for it)
    const float* draw;
    if (int rc = label_scores_bwd(a.dscores, a.priority_mat, draw_ws, a.C_mat, C,
                                  EpiDAB{a.alpha, a.beta, a.lengths, dalpha, dbeta, L, S, a.full_pad}, B, c.DrawOp,
                                  c.CmatOp, st, &draw))
      return rc;
    // 2. dC = draw^T @ (alpha * beta) over the valid positions: run_tn forms the masked product from Y2 / mask_len
    if (a.dC) {
      TnProblem t;
      memset(&t, 0, sizeof(t));
      t.P = C; t.Q = S; t.npairs = 1;
      t.pair[0] = TnPair{draw, a.alpha, C, S, M};
      t.Y2 = a.beta;
      if (!a.full_pad) { t.mask_len = a.lengths; t.mask_L = L; }
      RE2NN_CUDA(run_tn(t, partial, a.dC, 0, st));
    }
  }
  // 3. sweep
  RE2NN_CUDA(cudaMemsetAsync(c.g, 0, (size_t)2 * B * S * 4, st));
  RE2NN_CUDA(cudaMemsetAsync(a.dvtab, 0, (size_t)a.table_rows * R * 4, st));
  if (a.farnn >= 1) RE2NN_CUDA(cudaMemsetAsync(c.dgtab, 0, (size_t)a.table_rows * gw * 4, st));
  std::unique_ptr<TcLaunch> tq, th, tg;      // launch plans of the three step GEMMs on tcgen05 (none: CUDA cores)
  if (tc) {
    // K-major operand-format copies of S1, S2, W (the same layouts the forward uses) + the tensor maps of the two
    // step GEMMs; the A operands are the per-step DAop / DUop buffers, rewritten every step
    constexpr int P = RE2NN_PREC_TF32X3;
    re2nn_recurrence_args ra;
    memset(&ra, 0, sizeof(ra));
    ra.S = S; ra.R = R; ra.farnn = 0; ra.S1 = a.S1; ra.S2 = a.S2; ra.W = a.W;
    if (int rc = weight_prep_run<P>(ra, wp, st)) return rc;
    GemmProblem gq, gh;
    memset(&gq, 0, sizeof(gq));
    memset(&gh, 0, sizeof(gh));
    gq.M = B; gq.N = R; gq.nseg = 1; gq.ndir = 2;
    gh.M = B; gh.N = S; gh.nseg = 2; gh.ndir = 2;
    for (int z = 0; z < 2; ++z) {
      gq.seg[z][0] = wp.seg_g1(1 - z, c.DAop[z], c.ldS, c.da_plane);      // DA @ S2 (fwd) | DA @ S1 (bwd)
      gh.seg[z][0] = wp.seg_g2q(1 - z, c.DUop[z], c.ldR, c.du_plane);     // DU @ S1^T (fwd) | DU @ S2^T (bwd)
      gh.seg[z][1] = wp.seg_g2w(1 - z, c.DAop[z], c.ldS, c.da_plane);     // DA @ W^T (fwd) | DA @ W (bwd)
    }
    tq.reset(new TcLaunch);
    th.reset(new TcLaunch);
    if (int rc = tc_make_launch<P>(gq, tq.get())) return rc;
    if (int rc = tc_make_launch<P>(gh, th.get())) return rc;
    if (a.farnn >= 1) {
      const size_t pl = (size_t)S * wp.ldS;
      const int blocks = (int)(((size_t)S * wp.ldS + 255) / 256);
      convert_weight_kernel<P><<<blocks, 256, 0, st>>>(a.Wss1, S, S, S, 0, wp.buf[6], wp.ldS, pl, 0);
      if (a.farnn == 2) convert_weight_kernel<P><<<blocks, 256, 0, st>>>(a.Wss2, S, S, S, 0, wp.buf[7], wp.ldS, pl, 0);
      RE2NN_LAUNCH_CHECK();
      GemmProblem gg;
      memset(&gg, 0, sizeof(gg));
      gg.M = B; gg.N = S; gg.nseg = a.farnn; gg.ndir = 2;
      for (int z = 0; z < 2; ++z) {
        gg.seg[z][0] = GemmSeg{c.DZop[z], wp.buf[6], c.ldS, wp.ldS, S, 1, c.da_plane, pl};
        if (a.farnn == 2) gg.seg[z][1] = GemmSeg{c.DRop[z], wp.buf[7], c.ldS, wp.ldS, S, 1, c.da_plane, pl};
      }
      tg.reset(new TcLaunch);
      if (int rc = tc_make_launch<P>(gg, tg.get())) return rc;
    }
  }
  GemmProblem g;
  for (int k = L - 1; k >= 0; --k) {
    c.k = k;
    if (k == L - 1 || a.farnn >= 1) {      // without gates E1 of the later steps rides in bwd_e31_kernel
      bwd_e1_kernel<<<grid_for((size_t)2 * B * S), 256, 0, st>>>(c);
      RE2NN_LAUNCH_CHECK();
    }
    // dq = DA[k] @ S2 (fwd) | S1 (bwd)
    memset(&g, 0, sizeof(g));
    g.M = B; g.N = R; g.nseg = 1; g.ndir = 2;
    for (int z = 0; z < 2; ++z)
      g.seg[z][0] = GemmSeg{c.DA + ((size_t)z * L + k) * B * S, z == 0 ? a.S2 : a.S1, S, R, S, 0, 0, 0};
    RE2NN_CUDA(step_gemm(g, EpiStore2{{c.DQ, c.DQ + (size_t)B * R}, R, 0}, tq.get(), st));
    RE2NN_CUDA(launch_pdl(bwd_e2_kernel, grid_for((size_t)2 * B * R), st, c));
    // dhb = DU[k] @ S1^T + DA[k] @ W^T (fwd) | DU[k] @ S2^T + DA[k] @ W (bwd)
    memset(&g, 0, sizeof(g));
    g.M = B; g.N = S; g.nseg = 2; g.ndir = 2;
    for (int z = 0; z < 2; ++z) {
      g.seg[z][0] = GemmSeg{c.DU + ((size_t)z * L + k) * B * R, z == 0 ? a.S1 : a.S2, R, R, R, 1, 0, 0};
      g.seg[z][1] = GemmSeg{c.DA + ((size_t)z * L + k) * B * S, a.W, S, S, S, z == 0 ? 1 : 0, 0, 0};
    }
    RE2NN_CUDA(step_gemm(g, EpiStore2{{c.DHb, c.DHb + (size_t)B * S}, S, 0}, th.get(), st));
    if (a.farnn == 0) RE2NN_CUDA(launch_pdl(bwd_e31_kernel, grid_for((size_t)2 * B * S), st, c));
    else {
      bwd_e3_kernel<<<grid_for((size_t)2 * B * S), 256, 0, st>>>(c);
      RE2NN_LAUNCH_CHECK();
    }
    if (a.farnn >= 1) {
      // g += [dz | dr] @ [Wss1 | Wss2]^T
      memset(&g, 0, sizeof(g));
      g.M = B; g.N = S; g.nseg = a.farnn; g.ndir = 2;
      for (int z = 0; z < 2; ++z) {
        const float* dzr = c.DZR + ((size_t)z * L + k) * B * gw;
        g.seg[z][0] = GemmSeg{dzr, a.Wss1, gw, S, S, 1, 0, 0};
        if (a.farnn == 2) g.seg[z][1] = GemmSeg{dzr + S, a.Wss2, gw, S, S, 1, 0, 0};
      }
      RE2NN_CUDA(step_gemm(g, EpiStore2{{c.g, c.g + (size_t)B * S}, S, 1}, tg.get(), st));
      bwd_gate_scatter_kernel<<<grid_for((size_t)2 * B * gw), 256, 0, st>>>(c);
      RE2NN_LAUNCH_CHECK();
    }
  }
  // 4. weight gradients: one transposed GEMM each over all (step, sequence) rows
  const size_t rows1 = (size_t)L * B;                    // per-direction slab rows
  const float* Hb0 = a.hbar_save;                        // (L+1)-deep slabs: direction stride (L+1)*B*S
  const float* Hb1 = a.hbar_save + (size_t)(L + 1) * B * S;
  const float *DA0 = c.DA, *DA1 = c.DA + rows1 * S, *DU0 = c.DU, *DU1 = c.DU + rows1 * R;
  const float *Q0 = c.Qs, *Q1 = c.Qs + rows1 * R;
  // dS1 = fwd hbar^T du + bwd da^T q ; dS2 = fwd da^T q + bwd hbar^T du ; dW = fwd hbar^T da + bwd da^T hbar
  RE2NN_CUDA(tn(a.dS1, S, R, {{Hb0, DU0, S, R, rows1}, {DA1, Q1, S, R, rows1}}, partial, st));
  RE2NN_CUDA(tn(a.dS2, S, R, {{DA0, Q0, S, R, rows1}, {Hb1, DU1, S, R, rows1}}, partial, st));
  RE2NN_CUDA(tn(a.dW, S, S, {{Hb0, DA0, S, S, rows1}, {DA1, Hb1, S, S, rows1}}, partial, st));
  if (a.farnn >= 1) {
    const float* Hs0 = a.hst_save;
    const float* Hs1 = a.hst_save + (size_t)(L + 1) * B * S;
    const float* Z0 = c.DZR;
    const float* Z1 = c.DZR + rows1 * gw;
    RE2NN_CUDA(tn(a.dWss1, S, S, {{Hs0, Z0, S, gw, rows1}, {Hs1, Z1, S, gw, rows1}}, partial, st));
    if (a.farnn == 2) RE2NN_CUDA(tn(a.dWss2, S, S, {{Hs0, Z0 + S, S, gw, rows1}, {Hs1, Z1 + S, S, gw, rows1}}, partial, st));
    // token-side gate parameters through the gate table: Wrs = vtab^T dgtab, bs = colsum(dgtab), dvtab += dgtab Wrs^T
    RE2NN_CUDA(tn(a.dWrs1, R, S, {{a.vtab, c.dgtab, R, gw, (size_t)a.table_rows}}, partial, st));
    if (a.farnn == 2) RE2NN_CUDA(tn(a.dWrs2, R, S, {{a.vtab, c.dgtab + S, R, gw, (size_t)a.table_rows}}, partial, st));
    if (a.dbs1) RE2NN_CUDA(colsum_rows(c.dgtab, a.table_rows, S, gw, a.dbs1, 0, st, partial));
    if (a.farnn == 2 && a.dbs2) RE2NN_CUDA(colsum_rows(c.dgtab + S, a.table_rows, S, gw, a.dbs2, 0, st, partial));
    memset(&g, 0, sizeof(g));
    g.M = a.table_rows; g.N = R; g.nseg = a.farnn; g.ndir = 1;
    g.seg[0][0] = GemmSeg{c.dgtab, a.Wrs1, gw, S, S, 1, 0, 0};
    if (a.farnn == 2) g.seg[0][1] = GemmSeg{c.dgtab + S, a.Wrs2, gw, S, S, 1, 0, 0};
    RE2NN_CUDA(launch_simt_gemm(g, EpiStore2{{a.dvtab, a.dvtab}, R, 1}, ALoadPlain{}, st));
  }
  // 5. vector gradients
  if (a.d_o) RE2NN_CUDA(colsum_rows(c.DOprod, (size_t)2 * rows1, S, S, a.d_o, 0, st, partial));
  if (a.dh0) {
    RE2NN_CUDA(colsum_rows(c.g, B, S, S, a.dh0, 0, st));
    if (a.farnn == 2) RE2NN_CUDA(colsum_rows(c.Pinit, rows1, S, S, a.dh0, 1, st, partial));
  }
  if (a.dhT) {
    RE2NN_CUDA(colsum_rows(c.g + (size_t)B * S, B, S, S, a.dhT, 0, st));
    if (a.farnn == 2) RE2NN_CUDA(colsum_rows(c.Pinit + rows1 * S, rows1, S, S, a.dhT, 1, st, partial));
    bwd_direct_hT_kernel<<<cdiv(S, 128), 128, 0, st>>>(dbeta, a.lengths, B, L, S, a.dhT);
    RE2NN_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace re2nn

using namespace re2nn;

extern "C" {

int re2nn_debug_set_backward_tc(int on) {
  g_bwd_tc = on != 0;
  return 0;
}

int re2nn_debug_set_tn_tc(int on) {
  g_tn_tc = on != 0;
  return 0;
}

int re2nn_gemm_tn_path(int P, int Q, int64_t rows, int has_y2) {
  (void)has_y2;                  // both kernels form Y * Y2 themselves: the dC layout takes the same path
  return tn_path(P, Q, rows > 0 ? (size_t)rows : 0);
}

size_t re2nn_gemm_tn_workspace(int P, int Q) {
  return P > 0 && Q > 0 ? align_up((size_t)kTnSplit * P * Q * 4, 256) : 0;
}

int re2nn_gemm_tn(int path, int P, int Q, const float* X0, const float* Y0, int ldx0, int ldy0, int64_t rows0, const float* X1,
                  const float* Y1, int ldx1, int ldy1, int64_t rows1, const float* Y2, const int64_t* mask_len, int mask_L,
                  float* C, void* ws, size_t ws_bytes, void* stream) {
  RE2NN_CHECK(path >= 0 && path <= 2, "gemm_tn: path must be 0, 1 or 2");
  RE2NN_CHECK(P > 0 && Q > 0 && X0 && Y0 && C && ldx0 >= P && ldy0 >= Q && rows0 >= 0, "gemm_tn: bad arguments");
  RE2NN_CHECK(!X1 || (Y1 && ldx1 >= P && ldy1 >= Q && rows1 >= 0), "gemm_tn: bad second pair");
  RE2NN_CHECK(!Y2 || (!X1 && Y2 != Y0), "gemm_tn: Y2 needs a single pair and must not alias Y0");
  RE2NN_CHECK(!mask_len || (Y2 && mask_L > 0 && rows0 % mask_L == 0), "gemm_tn: a mask needs Y2 and rows0 = B * mask_L");
  RE2NN_CHECK(ws && ws_bytes >= re2nn_gemm_tn_workspace(P, Q), "gemm_tn: workspace too small");
  RE2NN_CHECK(path != kTnPathTc || (re2nn_has_tcgen05() != 0 && P >= 16 && Q >= 16),
              "gemm_tn: the tcgen05 path needs an sm_100 device and P, Q >= 16");
  TnProblem t;
  memset(&t, 0, sizeof(t));
  t.P = P; t.Q = Q; t.npairs = X1 ? 2 : 1;
  t.pair[0] = TnPair{X0, Y0, ldx0, ldy0, (size_t)rows0};
  if (X1) t.pair[1] = TnPair{X1, Y1, ldx1, ldy1, (size_t)rows1};
  t.Y2 = Y2;
  t.mask_len = mask_len;
  t.mask_L = mask_len ? mask_L : 0;
  RE2NN_CUDA(run_tn(t, (float*)ws, C, 0, (cudaStream_t)stream, path));
  return 0;
}

size_t re2nn_decompose_backward_workspace(const re2nn_backward_args* a) {
  if (!a) return 0;
  return bwd_carve(*a, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

int re2nn_decompose_backward(const re2nn_backward_args* a, void* stream) {
  RE2NN_CHECK(a != nullptr, "decompose_backward: null args");
  RE2NN_CHECK(a->B > 0 && a->L > 0 && a->S > 0 && a->R > 0 && (a->C > 0 || (a->dalpha_in && a->dbeta_in)), "decompose_backward: bad dims");
  RE2NN_CHECK(a->farnn >= 0 && a->farnn <= 2, "decompose_backward: farnn must be 0, 1 or 2");
  const bool direct = a->dalpha_in && a->dbeta_in;
  RE2NN_CHECK((direct || (a->dscores && a->C_mat)) && a->lengths && a->vtab && a->S1 && a->S2 && a->W && a->o && a->h0 &&
                  a->hT && a->alpha && a->beta && a->hbar_save && a->hst_save && a->u_save && a->a_save && a->dvtab,
              "decompose_backward: null tensor");
  RE2NN_CHECK(a->v_mode == RE2NN_V_DENSE || a->x, "decompose_backward: token mode needs x");
  RE2NN_CHECK(a->farnn == 0 || (a->zsave && a->Wss1 && a->Wrs1), "decompose_backward: farnn>=1 needs gate tensors");
  RE2NN_CHECK(a->farnn < 2 || (a->rsave && a->Wss2 && a->Wrs2), "decompose_backward: farnn==2 needs reset-gate tensors");
  return run_backward(*a, (cudaStream_t)stream);
}

int re2nn_label_scores_backward(const float* dscores, const float* alpha, const float* beta, const int64_t* lengths,
                                int B, int L, int S, const float* C_mat, int C, const float* priority_mat,
                                int full_pad, float* dalpha, float* dbeta, float* ws, void* stream) {
  RE2NN_CHECK(dscores && alpha && beta && lengths && C_mat && dalpha && dbeta, "label_scores_backward: null tensor");
  RE2NN_CHECK(!priority_mat || ws, "label_scores_backward: priority needs a workspace");
  return label_scores_bwd(dscores, priority_mat, ws, C_mat, C, EpiDAB{alpha, beta, lengths, dalpha, dbeta, L, S, full_pad},
                          B, nullptr, nullptr, (cudaStream_t)stream, nullptr);
}

size_t re2nn_token_table_backward_workspace(int rows, int D, int R) {
  return align_up((size_t)rows * R * 4, 256) * 2 + align_up((size_t)kTnSplit * D * R * 4, 256) + 256;
}

int re2nn_token_table_backward(const float* dvtab, const float* V_embed, const float* E, const float* G,
                               const float* beta_vec, int rows, int D, int R, int additional_nonlinear,
                               float* dV_embed, float* dbeta_vec, float* dG, float* dE, void* ws, size_t ws_bytes,
                               void* stream) {
  RE2NN_CHECK(dvtab && V_embed && E && G && beta_vec && ws, "token_table_backward: null tensor");
  RE2NN_CHECK(ws_bytes >= re2nn_token_table_backward_workspace(rows, D, R), "token_table_backward: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)ws;
  float* dbeta_prod = (float*)w;
  w += align_up((size_t)rows * R * 4, 256);
  float* dGpre = (float*)w;
  w += align_up((size_t)rows * R * 4, 256);
  float* partial = (float*)w;
  RE2NN_CUDA(launch_simt_gemm(gemm_problem(rows, R, GemmSeg{E, G, D, R, D, 0, 0, 0}),
                              EpiTokenBwd{dvtab, V_embed, beta_vec, dV_embed, dbeta_prod, dGpre, R, additional_nonlinear},
                              ALoadPlain{}, st));
  if (dbeta_vec) RE2NN_CUDA(colsum_rows(dbeta_prod, rows, R, R, dbeta_vec, 0, st));
  RE2NN_CUDA(tn(dG, D, R, {{E, dGpre, D, R, (size_t)rows}}, partial, st));
  if (dE)
    RE2NN_CUDA(launch_simt_gemm(gemm_problem(rows, D, GemmSeg{dGpre, G, R, R, R, 1, 0, 0}), EpiStore{dE, D, nullptr},
                                ALoadPlain{}, st));
  return 0;
}

}  // extern "C"
