// Problem description shared by the CUDA-core (fp32) and tcgen05 GEMM mainloops, plus the fused
// epilogue functors of the decompose recurrence.  One "step GEMM" computes, for both directions z,
//     C_z[M x N] = sum_seg A_{z,seg}[M x K_seg] * B_{z,seg}[K_seg x N]
// and hands every accumulator element to an epilogue functor instead of writing C.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace re2nn {

constexpr int kMaxSeg = 3;

struct GemmSeg {
  const void* A;   // M x K operand, row-major, leading dimension lda (elements)
  const void* B;   // b_nk ? N x K (K contiguous) : K x N (N contiguous); leading dimension ldb
  int lda, ldb, K, b_nk;
  size_t a_plane, b_plane;   // TF32X3 only: element offset of the "lo" plane
};
struct GemmProblem {
  int M, N, nseg, ndir;
  GemmSeg seg[2][kMaxSeg];
};
// One direction, one segment: C[M x N] = A @ B as `s` lays them out.
inline GemmProblem gemm_problem(int M, int N, const GemmSeg& s) {
  GemmProblem g;
  memset(&g, 0, sizeof(g));
  g.M = M; g.N = N; g.nseg = 1; g.ndir = 1;
  g.seg[0][0] = s;
  return g;
}

// ---- operand formats ---------------------------------------------------------------------------
// FP32: float, ld = K.   BF16: __nv_bfloat16, ld = roundup(K, 8).   TF32X3: two float planes (hi, lo).
template <int PREC> struct OperandFmt;
template <> struct OperandFmt<RE2NN_PREC_FP32> {
  static constexpr int kElemBytes = 4, kPlanes = 1, kLdAlign = 1;
  __device__ static __forceinline__ void store16(void* base, size_t idx, size_t, const float (&v)[16]) {
#pragma unroll
    for (int j = 0; j < 16; ++j) ((float*)base)[idx + j] = v[j];
  }
  __device__ static __forceinline__ void store(void* base, size_t idx, size_t, float v) { ((float*)base)[idx] = v; }
  // conversion unconditional, stores predicated: keeps unrolled epilogue batches branch-free
  __device__ static __forceinline__ void store_if(bool on, void* base, size_t idx, size_t, float v) {
    if (on) ((float*)base)[idx] = v;
  }
  // four consecutive elements, idx % 4 == 0 and the row pitch 16-byte aligned
  __device__ static __forceinline__ void store4(void* base, size_t idx, size_t, float4 v) {
    *reinterpret_cast<float4*>((float*)base + idx) = v;
  }
};
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {      // a -> low half, b -> high half
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
template <> struct OperandFmt<RE2NN_PREC_BF16> {
  static constexpr int kElemBytes = 2, kPlanes = 1, kLdAlign = 8;
  // sixteen consecutive elements of one row, idx % 8 == 0 and 16-byte aligned rows: two 16-byte stores
  __device__ static __forceinline__ void store16(void* base, size_t idx, size_t, const float (&v)[16]) {
    uint4* d = reinterpret_cast<uint4*>((__nv_bfloat16*)base + idx);
    d[0] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    d[1] = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
  }
  __device__ static __forceinline__ void store(void* base, size_t idx, size_t, float v) {
    ((__nv_bfloat16*)base)[idx] = __float2bfloat16_rn(v);
  }
  __device__ static __forceinline__ void store_if(bool on, void* base, size_t idx, size_t, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    if (on) ((__nv_bfloat16*)base)[idx] = h;
  }
  __device__ static __forceinline__ void store4(void* base, size_t idx, size_t, float4 v) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&lo);
    u.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>((__nv_bfloat16*)base + idx) = u;
  }
};
__device__ __forceinline__ float tf32_hi(float v) {   // round-to-nearest onto the 10-bit tf32 mantissa
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
  return __uint_as_float(u);
}
template <> struct OperandFmt<RE2NN_PREC_TF32X3> {
  static constexpr int kElemBytes = 4, kPlanes = 2, kLdAlign = 4;
  __device__ static __forceinline__ void store16(void* base, size_t idx, size_t plane, const float (&v)[16]) {
    float4* dh = reinterpret_cast<float4*>((float*)base + idx);
    float4* dl = reinterpret_cast<float4*>((float*)base + idx + plane);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const float4 h = make_float4(tf32_hi(v[4 * g]), tf32_hi(v[4 * g + 1]), tf32_hi(v[4 * g + 2]), tf32_hi(v[4 * g + 3]));
      dh[g] = h;
      dl[g] = make_float4(tf32_hi(v[4 * g] - h.x), tf32_hi(v[4 * g + 1] - h.y), tf32_hi(v[4 * g + 2] - h.z),
                          tf32_hi(v[4 * g + 3] - h.w));
    }
  }
  __device__ static __forceinline__ void store(void* base, size_t idx, size_t plane, float v) {
    float hi = tf32_hi(v);
    ((float*)base)[idx] = hi;
    ((float*)base)[idx + plane] = tf32_hi(v - hi);
  }
  __device__ static __forceinline__ void store_if(bool on, void* base, size_t idx, size_t plane, float v) {
    const float hi = tf32_hi(v), lo = tf32_hi(v - hi);
    float* d = (float*)base + idx;
    if (on) d[0] = hi;
    if (on) d[plane] = lo;
  }
  __device__ static __forceinline__ void store4(void* base, size_t idx, size_t plane, float4 v) {
    float4 h = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
    float4 l = make_float4(tf32_hi(v.x - h.x), tf32_hi(v.y - h.y), tf32_hi(v.z - h.z), tf32_hi(v.w - h.w));
    *reinterpret_cast<float4*>((float*)base + idx) = h;
    *reinterpret_cast<float4*>((float*)base + idx + plane) = l;
  }
};
// fp16 split: v = hi + lo * 2^-11 with hi = fp16(v), lo = fp16((v - hi) * 2^11): 22 mantissa bits in 4 bytes.
// The residual is kept scaled so it stays a normal fp16 number; its products go to a second accumulator that
// the epilogue folds in with the 2^-11 factor.
constexpr float kFp16LoScale = 2048.f;
template <> struct OperandFmt<RE2NN_PREC_FP16X3> {
  static constexpr int kElemBytes = 2, kPlanes = 2, kLdAlign = 8;
  __device__ static __forceinline__ void store16(void* base, size_t idx, size_t plane, const float (&v)[16]) {
    uint32_t h[8], l[8];
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      h[g] = pack_f16x2(v[2 * g], v[2 * g + 1]);
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h[g]));
      l[g] = pack_f16x2((v[2 * g] - f.x) * kFp16LoScale, (v[2 * g + 1] - f.y) * kFp16LoScale);
    }
    uint4* dh = reinterpret_cast<uint4*>((__half*)base + idx);
    uint4* dl = reinterpret_cast<uint4*>((__half*)base + idx + plane);
    dh[0] = make_uint4(h[0], h[1], h[2], h[3]);
    dh[1] = make_uint4(h[4], h[5], h[6], h[7]);
    dl[0] = make_uint4(l[0], l[1], l[2], l[3]);
    dl[1] = make_uint4(l[4], l[5], l[6], l[7]);
  }
  __device__ static __forceinline__ void store(void* base, size_t idx, size_t plane, float v) {
    const __half hi = __float2half_rn(v);
    ((__half*)base)[idx] = hi;
    ((__half*)base)[idx + plane] = __float2half_rn((v - __half2float(hi)) * kFp16LoScale);
  }
  __device__ static __forceinline__ void store_if(bool on, void* base, size_t idx, size_t plane, float v) {
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn((v - __half2float(hi)) * kFp16LoScale);
    __half* d = (__half*)base + idx;
    if (on) d[0] = hi;
    if (on) d[plane] = lo;
  }
  __device__ static __forceinline__ void store4(void* base, size_t idx, size_t plane, float4 v) {
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
    const __half2 l0 = __floats2half2_rn((v.x - f0.x) * kFp16LoScale, (v.y - f0.y) * kFp16LoScale);
    const __half2 l1 = __floats2half2_rn((v.z - f1.x) * kFp16LoScale, (v.w - f1.y) * kFp16LoScale);
    uint2 uh, ul;
    uh.x = *reinterpret_cast<const uint32_t*>(&h0); uh.y = *reinterpret_cast<const uint32_t*>(&h1);
    ul.x = *reinterpret_cast<const uint32_t*>(&l0); ul.y = *reinterpret_cast<const uint32_t*>(&l1);
    *reinterpret_cast<uint2*>((__half*)base + idx) = uh;
    *reinterpret_cast<uint2*>((__half*)base + idx + plane) = ul;
  }
};
inline bool prec_is_16bit(int prec) { return prec == RE2NN_PREC_BF16 || prec == RE2NN_PREC_FP16X3; }
inline bool prec_is_split(int prec) { return prec == RE2NN_PREC_TF32X3 || prec == RE2NN_PREC_FP16X3; }
inline int operand_ld(int prec, int K) {
  int a = prec_is_16bit(prec) ? 8 : (prec == RE2NN_PREC_TF32X3 ? 4 : 1);
  return (K + a - 1) / a * a;
}
inline size_t operand_bytes(int prec, size_t rows, int K) {
  size_t ld = operand_ld(prec, K);
  size_t eb = prec_is_16bit(prec) ? 2 : 4;
  size_t planes = prec_is_split(prec) ? 2 : 1;
  return align_up(rows * ld * eb * planes, 256);
}

// ---- per-step parameters of the decompose recurrence -----------------------------------------
struct StepParams {
  int B, Lpad, L, S, R, k;
  int farnn, nl, v_mode, full_pad;
  float sig_k;
  const int64_t* x;
  const int64_t* len;
  const int* tile_last[2];   // per direction, per 128-row tile: last step at which a row of the tile is alive
  const float* vtab;
  const float* gtab;
  int ldg;
  const float* o;
  const float* hinit[2];
  void* Q[2];        int ldq;  size_t q_plane;    // operand format, B x R
  void* Hbar_next[2]; int ldh; size_t h_plane;    // operand format, B x S : A operand of the NEXT step (farnn<=1)
  void* Hbar_cur[2];                              // operand format: written by the gate epilogue (farnn==2)
  void* Hst[2];                                   // operand format: post-update state, A operand of the gate GEMM
  float* H[2];                                    // fp32 state B x S (farnn>=1)
  float* Z[2];                                    // fp32 update gate B x S (farnn>=1)
  float* Rg[2];                                   // optional save of reset gate
  float* out[2];                                  // alpha / beta : B x L x S
  float* Usave[2];                                // training: u = hbar @ S1|S2          (B x R slab of this step)
  float* Asave[2];                                // training: pre-activation a          (B x S slab of this step)
  float* HstNext[2];                              // training: state before step k+1     (B x S slab)
  float* HbarSaveNext[2];                         // training on tensor cores: fp32 copy of the next operand
  float* HbarSaveCur[2];                          // training on tensor cores, farnn==2: fp32 copy of this step's operand
  int dir;                                        // set by bind(): the direction this CTA works on
  int dir_base;                                   // single-direction launches: tile direction index z means z + dir_base
  void* AB; int ldab; size_t ab_plane;            // fused label-score operand (alpha * beta), (B*L) x ldab
  const float* beta_in;                           // beta as written by the backward direction (fused scoring)
  // Move direction z into slot 0 so the epilogue addresses plain members instead of indexing the constant bank with
  // a run-time z for every element.
  // bind(): run-time index into the by-value copy.  That keeps the copy in LOCAL memory (the epilogues re-load the
  // fields they use), which the register-starved kernels want: the plain inference epilogues of the resident kernel
  // (twelve epilogue warps, 128 registers) measured 8-10 % slower with the fields held in registers.
  __device__ __forceinline__ void bind(int zt) {
    const int z = zt + dir_base;
    dir = z;
    hinit[0] = hinit[z]; Q[0] = Q[z]; Hbar_next[0] = Hbar_next[z]; Hbar_cur[0] = Hbar_cur[z];
    Hst[0] = Hst[z]; H[0] = H[z]; Z[0] = Z[z]; Rg[0] = Rg[z]; out[0] = out[z];
    Usave[0] = Usave[z]; Asave[0] = Asave[z]; HstNext[0] = HstNext[z];
    HbarSaveNext[0] = HbarSaveNext[z]; HbarSaveCur[0] = HbarSaveCur[z];
  }
  // bind_const(): selects between CONSTANT indices, so the copy is scalarised into registers.  For the kernels with
  // registers to spare (eight epilogue warps: the gated recurrences): their epilogues touch most fields, and with
  // 225 KB of the SM given to shared memory there is next to no L1 left to catch local-memory loads.
  __device__ __forceinline__ void bind_const(int zt) {
    const bool one = (zt + dir_base) != 0;
    dir = one ? 1 : 0;
#define RE2NN_BIND(f) f[0] = one ? f[1] : f[0]
    RE2NN_BIND(hinit); RE2NN_BIND(Q); RE2NN_BIND(Hbar_next); RE2NN_BIND(Hbar_cur);
    RE2NN_BIND(Hst); RE2NN_BIND(H); RE2NN_BIND(Z); RE2NN_BIND(Rg); RE2NN_BIND(out);
    RE2NN_BIND(Usave); RE2NN_BIND(Asave); RE2NN_BIND(HstNext);
    RE2NN_BIND(HbarSaveNext); RE2NN_BIND(HbarSaveCur);
#undef RE2NN_BIND
  }
};

struct RowCtx {
  int vrow, orow;
  bool alive;
};

__device__ __forceinline__ RowCtx make_row(const StepParams& p, int z, int m) {
  RowCtx r;
  int n = (int)p.len[m];
  int tpos;
  step_pos(z, p.k, n, p.full_pad, tpos, r.orow, r.alive);
  r.vrow = p.v_mode == RE2NN_V_TOKEN ? (int)p.x[(size_t)m * p.Lpad + tpos] : m * p.Lpad + tpos;
  return r;
}

// is any row of 128-row tile `mt` still alive at this step?  (one load; every warp role can ask independently)
__device__ __forceinline__ bool tile_alive(const StepParams& p, int z, int mt) {
  return p.full_pad || p.k <= __ldg(p.tile_last[z + p.dir_base] + mt);
}

// Every epilogue functor is split so the mainloops can (a) hoist per-column constants, (b) put all of a
// tile's dependent global loads in flight at once (on the tcgen05 path before the accumulator is ready):
//   Col  col(z, n)                              per-column constants (o[n], bias[n], ...)
//   Pre  prefetch(row, z, m, n)                 loads only
//   void apply(col, row, z, m, n, acc, pre)     arithmetic + stores
// Index math is 32-bit wherever the host guarantees rows*ld < 2^31 (checked in run_recurrence).
struct Pre { float a, b; };
struct Col { float a, b; };

// E1: Q = (Hbar @ S1|S2) * v_t            (model_decompose_single.py:170-171 / 175-176)
// TRAIN: also keep what BPTT needs (fp32 step-major slabs; rows that are finished hold exact zeros)
template <int PREC, bool TRAIN = false> struct EpiQ {
  StepParams p;
  __device__ __forceinline__ EpiQ for_dir(int z) const { EpiQ e = *this; e.p.bind(z); return e; }
  __device__ __forceinline__ bool tile_alive(int z, int mt) const { return re2nn::tile_alive(p, z, mt); }
  __device__ __forceinline__ RowCtx row(int m) const { return make_row(p, p.dir, m); }
  __device__ __forceinline__ Col col(int) const { return Col{0.f, 0.f}; }
  __device__ __forceinline__ Pre prefetch(const RowCtx& r, int, int n) const {
    return Pre{__ldg(p.vtab + (size_t)((uint32_t)r.vrow * (uint32_t)p.R + (uint32_t)n)), 0.f};
  }
  __device__ __forceinline__ float compute(const Col&, float acc, const Pre& pre) const { return acc * pre.a; }
  __device__ __forceinline__ void apply(const Col& c, const RowCtx& r, int m, int n, float acc, const Pre& pre) const {
    store(c, r, m, n, compute(c, acc, pre), acc, pre);
  }
  // ---- quad form (tc_epilogue_quads): four consecutive columns nb .. nb+3 of row m per call -----------------------
  static constexpr bool kRows = !TRAIN && PREC != RE2NN_PREC_FP32;
  __device__ __forceinline__ bool rows_vec() const {       // 16-byte vector access to the gathered rows is legal
    return (p.R & 3) == 0 && (reinterpret_cast<uintptr_t>(p.vtab) & 15) == 0;
  }
  __device__ __forceinline__ float4 col4(int, int, bool) const { return make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ float4 pre4(const RowCtx& r, int, int nb, int ncols, bool vec) const {
    const float* src = p.vtab + (size_t)((uint32_t)r.vrow * (uint32_t)p.R + (uint32_t)nb);
    if (vec && ncols == 4) return __ldg(reinterpret_cast<const float4*>(src));
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ncols > 0) v.x = __ldg(src);
    if (ncols > 1) v.y = __ldg(src + 1);
    if (ncols > 2) v.z = __ldg(src + 2);
    if (ncols > 3) v.w = __ldg(src + 3);
    return v;
  }
  __device__ __forceinline__ void apply4(const RowCtx&, int m, int nb, int ncols, bool, float4 acc, float4 v, float4) const {
    const float4 q = make_float4(acc.x * v.x, acc.y * v.y, acc.z * v.z, acc.w * v.w);
    const size_t idx = (size_t)((uint32_t)m * (uint32_t)p.ldq + (uint32_t)nb);
    if (nb + 4 <= p.ldq) OperandFmt<PREC>::store4(p.Q[0], idx, p.q_plane, q);      // columns past R are K padding
    else {
      const float qa[4] = {q.x, q.y, q.z, q.w};
      for (int j = 0; j < ncols; ++j) OperandFmt<PREC>::store(p.Q[0], idx + j, p.q_plane, qa[j]);
    }
  }
  __device__ __forceinline__ void store(const Col&, const RowCtx& r, int m, int n, float q, float acc, const Pre&) const {
    OperandFmt<PREC>::store(p.Q[0], (uint32_t)m * (uint32_t)p.ldq + (uint32_t)n, p.q_plane, q);
    if constexpr (TRAIN) {
      const bool live = p.full_pad || r.orow >= 0;
      p.Usave[0][(uint32_t)m * (uint32_t)p.R + (uint32_t)n] = live ? acc : 0.f;
    }
  }
};

// E2: h_next = phi((Q @ S2^T + Hbar @ W) [* o]) ; gate blend ; write alpha/beta + next operands
// (model_decompose_single.py:172-173,177-199).  NL / FARNN >= 0 fix update_nonlinear / farnn at compile
// time (the hot configurations), -1 reads them from StepParams.
// FUSE (forward direction, farnn == 0, inference): instead of the alpha row write alpha * beta in operand format
// for the label-score GEMM (beta was completed by the backward direction, which ran first).
template <int PREC, int NL = -1, int FARNN = -1, bool TRAIN = false, bool FUSE = false> struct EpiH {
  // nonlinearity flavour: MUFU tanh for bf16 operands, branch-free few-ulp for the parity-grade tensor-core modes in
  // inference, libm where gradients are taken (training saves) and on the fp32 CUDA-core path
  static constexpr int kFast = PREC == RE2NN_PREC_BF16 ? 1 : ((PREC == RE2NN_PREC_FP32 || TRAIN) ? 0 : 2);
  StepParams p;
  __device__ __forceinline__ EpiH for_dir(int z) const { EpiH e = *this; e.p.bind(z); return e; }
  __device__ __forceinline__ bool tile_alive(int z, int mt) const { return re2nn::tile_alive(p, z, mt); }
  __device__ __forceinline__ RowCtx row(int m) const { return make_row(p, p.dir, m); }
  __device__ __forceinline__ int farnn() const { return FARNN >= 0 ? FARNN : p.farnn; }
  __device__ __forceinline__ int nl() const { return NL >= 0 ? NL : p.nl; }
  __device__ __forceinline__ Col col(int n) const { return Col{__ldg(p.o + n), 0.f}; }
  __device__ __forceinline__ Pre prefetch(const RowCtx& r, int m, int n) const {
    if (farnn() >= 1) {
      const uint32_t si = (uint32_t)m * (uint32_t)p.S + (uint32_t)n;
      return Pre{p.Z[0][si], p.H[0][si]};
    }
    if constexpr (FUSE)      // rows without an output read (and drop) their row 0
      return Pre{__ldg(p.beta_in + ((size_t)m * (uint32_t)p.L + (uint32_t)max(r.orow, 0)) * (uint32_t)p.S + (uint32_t)n), 0.f};
    return Pre{0.f, 0.f};
  }
  // ---- quad form (tc_epilogue_quads), plain recurrence only (no gates, no training saves) ---------------------------
  static constexpr bool kRows = !TRAIN && FARNN == 0 && PREC != RE2NN_PREC_FP32;
  __device__ __forceinline__ bool rows_vec() const {
    bool ok = (p.S & 3) == 0 && (reinterpret_cast<uintptr_t>(p.o) & 15) == 0;
    if (FUSE) ok = ok && (reinterpret_cast<uintptr_t>(p.beta_in) & 15) == 0;
    else ok = ok && (reinterpret_cast<uintptr_t>(p.out[0]) & 15) == 0;
    return ok;
  }
  __device__ __forceinline__ float4 col4(int nb, int ncols, bool vec) const {       // o[nb .. nb+3]
    if (vec && ncols == 4) return __ldg(reinterpret_cast<const float4*>(p.o + nb));
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ncols > 0) v.x = __ldg(p.o + nb);
    if (ncols > 1) v.y = __ldg(p.o + nb + 1);
    if (ncols > 2) v.z = __ldg(p.o + nb + 2);
    if (ncols > 3) v.w = __ldg(p.o + nb + 3);
    return v;
  }
  __device__ __forceinline__ float4 pre4(const RowCtx& r, int m, int nb, int ncols, bool vec) const {
    if constexpr (FUSE) {      // beta row of this position (rows without an output read and drop their row 0)
      const float* src = p.beta_in + ((size_t)m * (uint32_t)p.L + (uint32_t)max(r.orow, 0)) * (uint32_t)p.S + (uint32_t)nb;
      if (vec && ncols == 4) return __ldg(reinterpret_cast<const float4*>(src));
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ncols > 0) v.x = __ldg(src);
      if (ncols > 1) v.y = __ldg(src + 1);
      if (ncols > 2) v.z = __ldg(src + 2);
      if (ncols > 3) v.w = __ldg(src + 3);
      return v;
    }
    return make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __device__ __forceinline__ void apply4(const RowCtx& r, int m, int nb, int ncols, bool vec, float4 acc, float4 pre, float4 oc) const {
    float4 hn, nx;
    if (p.dir == 0) { acc.x *= oc.x; acc.y *= oc.y; acc.z *= oc.z; acc.w *= oc.w; }
    hn.x = apply_nl_t<kFast>(acc.x, nl()); hn.y = apply_nl_t<kFast>(acc.y, nl());
    hn.z = apply_nl_t<kFast>(acc.z, nl()); hn.w = apply_nl_t<kFast>(acc.w, nl());
    nx = hn;
    if (p.dir == 1) { nx.x *= oc.x; nx.y *= oc.y; nx.z *= oc.z; nx.w *= oc.w; }
    const size_t hidx = (size_t)((uint32_t)m * (uint32_t)p.ldh + (uint32_t)nb);
    if (nb + 4 <= p.ldh) OperandFmt<PREC>::store4(p.Hbar_next[0], hidx, p.h_plane, nx);      // columns past S are K padding
    else {
      const float na[4] = {nx.x, nx.y, nx.z, nx.w};
      for (int j = 0; j < ncols; ++j) OperandFmt<PREC>::store(p.Hbar_next[0], hidx + j, p.h_plane, na[j]);
    }
    if (r.orow < 0) return;
    const size_t orow = (size_t)m * (uint32_t)p.L + (uint32_t)r.orow;
    if constexpr (FUSE) {
      const float4 ab = make_float4(hn.x * pre.x, hn.y * pre.y, hn.z * pre.z, hn.w * pre.w);
      const size_t aidx = orow * (uint32_t)p.ldab + (uint32_t)nb;
      if (nb + 4 <= p.ldab) OperandFmt<PREC>::store4(p.AB, aidx, p.ab_plane, ab);
      else {
        const float aa[4] = {ab.x, ab.y, ab.z, ab.w};
        for (int j = 0; j < ncols; ++j) OperandFmt<PREC>::store(p.AB, aidx + j, p.ab_plane, aa[j]);
      }
    } else {
      float* dst = p.out[0] + orow * (uint32_t)p.S + (uint32_t)nb;
      if (vec && ncols == 4) *reinterpret_cast<float4*>(dst) = hn;
      else {
        const float ha[4] = {hn.x, hn.y, hn.z, hn.w};
        for (int j = 0; j < ncols; ++j) dst[j] = ha[j];
      }
    }
  }
  // compute() is pure arithmetic so a mainloop can evaluate a batch of rows back to back (independent MUFU
  // chains) before any store is issued; store() does the memory side.
  __device__ __forceinline__ float compute(const Col& c, float acc, const Pre& pre) const {
    float hn = p.dir == 0 ? acc * c.a : acc;
    hn = apply_nl_t<kFast>(hn, nl());
    if (farnn() >= 1) hn = (1.f - pre.a) * pre.b + pre.a * hn;
    return hn;
  }
  __device__ __forceinline__ void apply(const Col& c, const RowCtx& r, int m, int n, float acc, const Pre& pre) const {
    store(c, r, m, n, compute(c, acc, pre), acc, pre);
  }
  __device__ __forceinline__ void store(const Col& c, const RowCtx& r, int m, int n, float hnew, float acc, const Pre& pre) const {
    const uint32_t hi = (uint32_t)m * (uint32_t)p.ldh + (uint32_t)n;
    const uint32_t si = (uint32_t)m * (uint32_t)p.S + (uint32_t)n;
    if constexpr (TRAIN) {
      // note: with full_pad a live row may have no output row (backward direction, beta_0)
      const bool live = p.full_pad || r.orow >= 0;
      p.Asave[0][si] = live ? acc : 0.f;
      if (!live) hnew = 0.f;
      p.HstNext[0][si] = hnew;
      if constexpr (PREC != RE2NN_PREC_FP32) {     // fp32: the operand buffer already is the fp32 slab
        if (farnn() <= 1) p.HbarSaveNext[0][si] = p.dir == 1 ? hnew * c.a : hnew;
      }
    }
    if (farnn() >= 1) {
      p.H[0][si] = hnew;
      OperandFmt<PREC>::store(p.Hst[0], hi, p.h_plane, hnew);
    }
    if (farnn() <= 1) OperandFmt<PREC>::store(p.Hbar_next[0], hi, p.h_plane, p.dir == 1 ? hnew * c.a : hnew);
    // address unconditionally, store conditionally: keeps the 16-row batches of the tcgen05 epilogue branch-free
    if constexpr (FUSE) {
      const size_t row = (size_t)m * (uint32_t)p.L + (uint32_t)max(r.orow, 0);
      OperandFmt<PREC>::store_if(r.orow >= 0, p.AB, row * (uint32_t)p.ldab + (uint32_t)n, p.ab_plane, hnew * pre.a);
    } else {
      float* dst = p.out[0] + (size_t)((uint32_t)m * (uint32_t)p.L + (uint32_t)(r.orow & 0x7fffffff)) * (uint32_t)p.S + (uint32_t)n;
      if (r.orow >= 0) *dst = hnew;
    }
  }
};

// Epilogues whose prefetch() reads a COLD array (one touch per element, straight from HBM) ask the mainloop to pull
// the lines of a tile into L2 while its MMAs are still running.  Default: nothing to do.
template <class Epi> struct EpiL2Prefetch { static constexpr bool kOn = false; };
__device__ __forceinline__ void l2_prefetch(const void* ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }
template <int PREC, int NL, int FARNN, bool TRAIN> struct EpiL2Prefetch<EpiH<PREC, NL, FARNN, TRAIN, true>> {
  static constexpr bool kOn = true;
  // issue(e, row ctx, m, n): pull what prefetch() will read for the 32 columns starting at n of row m into L2
  __device__ static __forceinline__ void issue(const EpiH<PREC, NL, FARNN, TRAIN, true>& e, const RowCtx& r, int m, int n) {
    l2_prefetch(e.p.beta_in + ((size_t)m * (uint32_t)e.p.L + (uint32_t)max(r.orow, 0)) * (uint32_t)e.p.S + (uint32_t)n);
  }
};

// EG: zt / rt gates and the reset-blended operand (model_decompose_single.py:147-157)
// columns [0,S) = update gate pre-activation, [S,2S) = reset gate pre-activation (farnn==2)
template <int PREC, bool TRAIN = false> struct EpiGate {
  static constexpr bool kRows = false;
  static constexpr bool kFast = PREC == RE2NN_PREC_BF16;
  // inference on the split formats: few-ulp branch-free sigmoid; training keeps the exact one (its backward
  // differentiates the saved gate values, parity against the float64 oracle at 1e-4)
  static constexpr int kSig = PREC == RE2NN_PREC_BF16 ? 1 : ((PREC == RE2NN_PREC_FP32 || TRAIN) ? 0 : 2);
  StepParams p;
  __device__ __forceinline__ EpiGate for_dir(int z) const { EpiGate e = *this; e.p.bind(z); return e; }
  __device__ __forceinline__ bool tile_alive(int z, int mt) const { return re2nn::tile_alive(p, z, mt); }
  __device__ __forceinline__ RowCtx row(int m) const { return make_row(p, p.dir, m); }
  __device__ __forceinline__ Col col(int n) const {
    if (n < p.S) return Col{0.f, 0.f};
    return Col{__ldg(p.hinit[0] + (n - p.S)), __ldg(p.o + (n - p.S))};
  }
  __device__ __forceinline__ Pre prefetch(const RowCtx& r, int m, int n) const {
    Pre q{__ldg(p.gtab + (size_t)r.vrow * p.ldg + n), 0.f};
    if (n >= p.S) q.b = p.H[0][(uint32_t)m * (uint32_t)p.S + (uint32_t)(n - p.S)];
    return q;
  }
  __device__ __forceinline__ float compute(const Col&, float acc, const Pre& pre) const {
    return sigmoid_m<kSig>((acc + pre.a) * p.sig_k);
  }
  __device__ __forceinline__ void apply(const Col& c, const RowCtx& r, int m, int n, float acc, const Pre& pre) const {
    store(c, r, m, n, compute(c, acc, pre), acc, pre);
  }
  __device__ __forceinline__ void store(const Col& c, const RowCtx&, int m, int n, float g, float, const Pre& pre) const {
    // update-gate columns [0,S) store z; reset-gate columns [S,2S) store the blended operand.  Both forms are
    // evaluated and only the stores are predicated, so the unrolled 16-row batches of the tcgen05 epilogue stay
    // branch-free (the branchy form ran 3x slower).
    const bool is_r = n >= p.S;
    const uint32_t s = (uint32_t)(is_r ? n - p.S : n);
    const uint32_t si = (uint32_t)m * (uint32_t)p.S + s;
    if (!is_r) p.Z[0][si] = g;
    float hb = (1.f - g) * c.a + g * pre.b;
    if (p.dir == 1) hb *= c.b;
    OperandFmt<PREC>::store_if(is_r, p.Hbar_cur[0], (uint32_t)m * (uint32_t)p.ldh + s, p.h_plane, hb);
    if constexpr (TRAIN) {
      if (is_r) p.Rg[0][si] = g;
      if constexpr (PREC != RE2NN_PREC_FP32) {
        if (is_r) p.HbarSaveCur[0][si] = hb;
      }
    }
  }
};

// plain store epilogue (gate table, label scores, generic C = A*B [+ bias]); used off the step loop
struct EpiStore {
  static constexpr bool kRows = false;
  float* C;
  int ldc;
  const float* bias;      // per-column or NULL
  __device__ __forceinline__ EpiStore for_dir(int) const { return *this; }
  __device__ __forceinline__ bool tile_alive(int, int) const { return true; }
  __device__ __forceinline__ RowCtx row(int) const { return RowCtx{0, 0, true}; }
  __device__ __forceinline__ Col col(int n) const { return Col{bias ? __ldg(bias + n) : 0.f, 0.f}; }
  __device__ __forceinline__ Pre prefetch(const RowCtx&, int, int) const { return Pre{0.f, 0.f}; }
  __device__ __forceinline__ float compute(const Col& c, float acc, const Pre&) const { return acc + c.a; }
  __device__ __forceinline__ void apply(const Col& c, const RowCtx& r, int m, int n, float acc, const Pre& pre) const {
    store(c, r, m, n, compute(c, acc, pre), acc, pre);
  }
  __device__ __forceinline__ void store(const Col&, const RowCtx&, int m, int n, float v, float, const Pre&) const {
    C[(size_t)m * ldc + n] = v;
  }
};

// token table epilogue: table = V_embed*beta + phi(acc)*(1-beta)     (model_decompose.py:226-239)
struct EpiTokenTable {
  static constexpr bool kRows = false;
  float* table;
  const float* V_embed;
  const float* beta_vec;
  int R, nl;
  __device__ __forceinline__ EpiTokenTable for_dir(int) const { return *this; }
  __device__ __forceinline__ bool tile_alive(int, int) const { return true; }
  __device__ __forceinline__ RowCtx row(int) const { return RowCtx{0, 0, true}; }
  __device__ __forceinline__ Col col(int n) const { return Col{__ldg(beta_vec + n), 0.f}; }
  __device__ __forceinline__ Pre prefetch(const RowCtx&, int m, int n) const {
    return Pre{__ldg(V_embed + (size_t)m * R + n), 0.f};
  }
  __device__ __forceinline__ void apply(const Col& c, const RowCtx&, int m, int n, float acc, const Pre& pre) const {
    float g = apply_nl(acc, nl);
    table[(size_t)m * R + n] = pre.a * c.a + g * (1.f - c.a);
  }
};

}  // namespace re2nn
