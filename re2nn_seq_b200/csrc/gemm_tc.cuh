// Weight preparation for the step GEMMs + the tcgen05 (5th-gen tensor core) mainloop.
#pragma once
#include "gemm_common.cuh"

namespace re2nn {

// ---- prepared B operands ---------------------------------------------------------------------------
// FP32 path: the user's fp32 weights are used in place; only [Wss1 | Wss2] is concatenated.
// tcgen05 paths: every B operand is copied once per call into a K-major ([N][K], K contiguous,
// leading dimension padded for TMA) array of the operand format.
struct WeightPrep {
  int prec, S, R, farnn;
  int ldS, ldR;                 // operand leading dimensions for K = S / K = R
  const void* g1[2];            // GEMM1 B: fwd S1 (K=S,N=R) | bwd S2
  const void* g2q[2];           // GEMM2 seg0 B: fwd S2^T (K=R,N=S) | bwd S1^T
  const void* g2w[2];           // GEMM2 seg1 B: fwd W (K=S,N=S) | bwd W^T
  const void* gate;             // [Wss1 | Wss2] (K=S, N=S*farnn)
  void* buf[8];                 // owned storage (workspace slices)
  size_t pl_g1, pl_g2q, pl_ss, pl_gate;   // TF32X3 lo-plane offsets (elements) per buffer kind

  GemmSeg seg_g1(int z, const void* A, int lda, size_t ap) const {
    if (prec == RE2NN_PREC_FP32) return GemmSeg{A, g1[z], lda, R, S, 0, ap, 0};
    return GemmSeg{A, g1[z], lda, ldS, S, 1, ap, pl_g1};
  }
  GemmSeg seg_g2q(int z, const void* A, int lda, size_t ap) const {
    if (prec == RE2NN_PREC_FP32) return GemmSeg{A, g2q[z], lda, R, R, 1, ap, 0};
    return GemmSeg{A, g2q[z], lda, ldR, R, 1, ap, pl_g2q};
  }
  GemmSeg seg_g2w(int z, const void* A, int lda, size_t ap) const {
    if (prec == RE2NN_PREC_FP32) return GemmSeg{A, g2w[z], lda, S, S, z == 1 ? 1 : 0, ap, 0};
    return GemmSeg{A, g2w[z], lda, ldS, S, 1, ap, pl_ss};
  }
  GemmSeg seg_gate(const void* A, int lda, size_t ap) const {
    if (prec == RE2NN_PREC_FP32) return GemmSeg{A, gate, lda, S * farnn, S, 0, ap, 0};
    return GemmSeg{A, gate, lda, ldS, S, 1, ap, pl_gate};
  }
};

inline size_t weight_prep_carve(int prec, int S, int R, int farnn, char* base, WeightPrep* wp) {
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  WeightPrep w;
  memset(&w, 0, sizeof(w));
  w.prec = prec; w.S = S; w.R = R; w.farnn = farnn;
  w.ldS = operand_ld(prec, S); w.ldR = operand_ld(prec, R);
  if (prec == RE2NN_PREC_FP32) {
    if (farnn == 2) w.buf[0] = take((size_t)S * 2 * S * 4);
  } else {
    // buf0: S1^T-as-[R][ldS]  buf1: S2^T-as-[R][ldS]  (GEMM1, N=R rows, K=S)
    // buf2: S2-as-[S][ldR]    buf3: S1-as-[S][ldR]    (GEMM2 seg0, N=S rows, K=R)
    // buf4: W^T-as-[S][ldS]   buf5: W-as-[S][ldS]     (GEMM2 seg1)
    // buf6: [Wss1|Wss2]^T-as-[S*farnn][ldS]           (gate)
    w.pl_g1 = (size_t)R * w.ldS; w.pl_g2q = (size_t)S * w.ldR; w.pl_ss = (size_t)S * w.ldS;
    w.pl_gate = (size_t)S * farnn * w.ldS;
    w.buf[0] = take(operand_bytes(prec, R, S));
    w.buf[1] = take(operand_bytes(prec, R, S));
    w.buf[2] = take(operand_bytes(prec, S, R));
    w.buf[3] = take(operand_bytes(prec, S, R));
    w.buf[4] = take(operand_bytes(prec, S, S));
    w.buf[5] = take(operand_bytes(prec, S, S));
    if (farnn >= 1) w.buf[6] = take(operand_bytes(prec, (size_t)S * farnn, S));
  }
  if (wp) *wp = w;
  return off;
}

static __global__ void concat_gate_kernel(const float* Wss1, const float* Wss2, int S, float* Wg) {
  const int total = S * 2 * S;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int k = i / (2 * S), n = i - k * 2 * S;
    Wg[i] = n < S ? Wss1[(size_t)k * S + n] : Wss2[(size_t)k * S + (n - S)];
  }
}

// dst[n][k] (ld = ldk, operand format) = src(k, n); src is row-major [rows_src x cols_src];
// transpose==1: src is [K x N] (dst = src^T); transpose==0: src is [N x K] (dst = src).
template <int PREC>
__global__ void convert_weight_kernel(const float* src, int N, int K, int ld_src, int transpose, void* dst, int ldk,
                                      size_t plane, int n_off) {
  const size_t total = (size_t)N * ldk;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n = (int)(i / ldk), k = (int)(i % ldk);
    float v = 0.f;
    if (k < K) v = transpose ? src[(size_t)k * ld_src + n] : src[(size_t)n * ld_src + k];
    OperandFmt<PREC>::store(dst, (size_t)(n + n_off) * ldk + k, plane, v);
  }
}

// One operand-format copy of a weight: row n + n_off, column k of buf[buf] = src(k, n) (transpose) or src(n, k), src
// row-major with leading dimension ld_src; the copy's leading dimension is operand_ld(PREC, K).
struct WeightConv {
  const float* src;
  int N, K, ld_src, transpose, buf;
  size_t plane;
  int n_off;
};
constexpr int kMaxWeightConvs = 8;

// The copies the tensor-core paths make, in launch order (buffer layout: weight_prep_carve); returns how many.
inline int weight_convs(const re2nn_recurrence_args& a, const WeightPrep& w, WeightConv* out) {
  const int S = a.S, R = a.R;
  int n = 0;
  out[n++] = WeightConv{a.S1, R, S, R, 1, 0, w.pl_g1, 0};     // [R][S] = S1^T
  out[n++] = WeightConv{a.S2, R, S, R, 1, 1, w.pl_g1, 0};
  out[n++] = WeightConv{a.S2, S, R, R, 0, 2, w.pl_g2q, 0};    // [S][R] = S2
  out[n++] = WeightConv{a.S1, S, R, R, 0, 3, w.pl_g2q, 0};
  out[n++] = WeightConv{a.W, S, S, S, 1, 4, w.pl_ss, 0};      // fwd: B[k=s][n=j] = W[s][j] -> [n][k] = W^T
  out[n++] = WeightConv{a.W, S, S, S, 0, 5, w.pl_ss, 0};      // bwd: B[k][n] = W[n][k]   -> [n][k] = W
  if (a.farnn >= 1) out[n++] = WeightConv{a.Wss1, S, S, S, 1, 6, w.pl_gate, 0};
  if (a.farnn == 2) out[n++] = WeightConv{a.Wss2, S, S, S, 1, 6, w.pl_gate, S};
  return n;
}

// operand pointers of the tensor-core formats (the buffers hold the converted copies)
inline void weight_prep_bind(WeightPrep& w, int farnn) {
  w.g1[0] = w.buf[0]; w.g1[1] = w.buf[1];
  w.g2q[0] = w.buf[2]; w.g2q[1] = w.buf[3];
  w.g2w[0] = w.buf[4]; w.g2w[1] = w.buf[5];
  if (farnn >= 1) w.gate = w.buf[6];
}

template <int PREC>
inline int weight_prep_run(const re2nn_recurrence_args& a, WeightPrep& w, cudaStream_t st) {
  const int S = a.S;
  if (PREC == RE2NN_PREC_FP32) {
    w.g1[0] = a.S1; w.g1[1] = a.S2;
    w.g2q[0] = a.S2; w.g2q[1] = a.S1;
    w.g2w[0] = a.W; w.g2w[1] = a.W;
    if (a.farnn == 2) {
      concat_gate_kernel<<<cdiv(S * 2 * S, 256), 256, 0, st>>>(a.Wss1, a.Wss2, S, (float*)w.buf[0]);
      RE2NN_LAUNCH_CHECK();
      w.gate = w.buf[0];
    } else {
      w.gate = a.Wss1;
    }
    return 0;
  }
  WeightConv convs[kMaxWeightConvs];
  const int n = weight_convs(a, w, convs);
  for (int i = 0; i < n; ++i) {
    const WeightConv& c = convs[i];
    const int ldk = operand_ld(PREC, c.K);
    const int blocks = (int)(((size_t)c.N * ldk + 255) / 256);
    convert_weight_kernel<PREC><<<blocks, 256, 0, st>>>(c.src, c.N, c.K, c.ld_src, c.transpose, w.buf[c.buf], ldk,
                                                        c.plane, c.n_off);
    RE2NN_LAUNCH_CHECK();
  }
  weight_prep_bind(w, a.farnn);
  return 0;
}

}  // namespace re2nn

#include "gemm_tc_impl.cuh"
