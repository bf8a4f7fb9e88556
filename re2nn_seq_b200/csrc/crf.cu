// CRF forward algorithm / Viterbi / gold score, argmax decode and cross-entropy kernels.
// Reference: /root/reference/src_seq/baselines/crf.py:16-260, farnn/model_decompose.py:339-371,
//            farnn/model_onehot.py:148-180.
// One warp owns one sequence: the tag dimension (T = tagset+2, 75 for SNIPS) is spread over the
// lanes, the T x T transition matrix sits in shared memory (fp32, read conflict-free along "to"),
// the running partition is exchanged through a per-warp shared buffer.  Arithmetic order follows the
// reference exactly where it decides an argmax: cur = (feat_j + trans_ij) + part_i, strict ">" keeps
// the first maximal index like torch.max(dim).
//
// Kernel by tag-set width T = tagset + 2 (shared memory capped at kSmemLimit = 200 KB):
//   re2nn_crf_nll            3-32 crf_nll_exp_kernel<1>, 33-64 <2>, 65-96 <3>, 97-128 <4>, 129-153 <5>,
//                            154-218 crf_nll_kernel<true>, >= 219 crf_nll_kernel<false>
//   re2nn_crf_nll_backward   3-96 crf_nll_backward_exp3_kernel, 97-111 crf_nll_backward_exp_kernel,
//                            112-159 crf_nll_backward_kernel<true>, 160-225 <false>, >= 226 error "tag set too large"
//                            (re2nn_debug_set_crf_backward_split(0): 3-111 crf_nll_backward_exp_kernel)
//   re2nn_crf_viterbi        3-160 crf_viterbi_kernel<cdiv(T, 32), NS> (NS = 2 for large batches, else 1),
//                            161-216 crf_viterbi_kernel<0, 1>, >= 217 crf_viterbi_global_kernel
#include <algorithm>

#include "common.cuh"

namespace re2nn {

constexpr int kCrfWarps = 8;
constexpr int kCrfOverrun = 32 * 5;   // floats a register-blocked row sweep may read past the T x T table (ignored values)

__device__ __forceinline__ float clamped_feat(const float* f, int j, int clamp_col, float thr) {
  float v = __ldg(f + j);
  return (j == clamp_col) ? fminf(v, thr) : v;
}

// ---- Viterbi (crf.py:102-195) ----------------------------------------------------------------------------------
// The sweep is issue-bound (T^2 candidate scores per position), so it keeps only what the result needs:
//   forward:   part_t[j] = max_i ((feat_t[j] + trans[i][j]) + part_{t-1}[i])      -- the reference's rounding order,
//              maxima only (max is exact in any order): per four source tags one LDS.128 of the TRANSPOSED
//              transition table, four packed adds (add.f32x2) and two three-input maxima per target tag;
//              every part_t is written to a history buffer instead of back-pointers;
//   backtrace: only the pointers ON the best path are ever read (crf.py:189-192), so each one is recomputed from
//              the stored partition: argmax_i ((feat_t[ptr] + trans[i][ptr]) + part_{t-1}[i]) with the same
//              expression bit for bit and the first maximal index (torch.max) -- T operations per position
//              instead of a T^2 compare/select sweep.
__device__ __forceinline__ unsigned long long pack_f32x2(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ unsigned long long add_f32x2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ float max3_of(float m, unsigned long long v) {
  float a, b;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
  asm("max.f32 %0, %1, %2, %3;" : "=f"(m) : "f"(m), "f"(a), "f"(b));
  return m;
}
// row pitch of the transposed table: a multiple of 4 words whose quarter is odd, so the 16-byte reads of eight
// consecutive target tags fall into distinct bank groups
__host__ __device__ inline int viterbi_pitch(int T) {
  int q = (T + 3) / 4;
  if ((q & 1) == 0) ++q;
  return 4 * q;
}

// trans[i][j] as the Viterbi kernels hold it: the transposed shared-memory table of pitch Tq, or the row-major
// matrix in global memory
struct TransposedTrans {
  const float* p;
  int Tq;
  __device__ __forceinline__ float operator()(int i, int j) const { return p[j * Tq + i]; }
};
struct RowMajorTrans {
  const float* p;
  int T;
  __device__ __forceinline__ float operator()(int i, int j) const { return p[i * T + j]; }
};

// part_0[j] = feat_0[j] + trans[START][j]
template <class Tr>
__device__ __forceinline__ float viterbi_start(Tr tr, const float* f0, int j, int T, int clamp_col, float thr) {
  return clamped_feat(f0, j, clamp_col, thr) + tr(T - 2, j);
}

// Backtrace of sequence b (n tags) from its partition history hs, all lanes of the warp cooperating.  Each pointer on
// the best path is the first maximal source tag over i of (f + trans[i][j]) + part[i], or part[i] + trans[i][j] for
// the STOP step (crf.py:166-175, torch.max tie-break).
template <class Tr>
__device__ __forceinline__ void viterbi_backtrace(Tr tr, const float* fs, const float* hs, int n, int b, int L, int T,
                                                  int lane, int clamp_col, float thr, int64_t o_idx,
                                                  const int64_t* offsets, int64_t* padded, int64_t* flat) {
  if (n <= 0) {   // empty sequence: no tags; the padded row is all zeros like the reference's masked back-pointers
    if (padded)
      for (int t = lane; t < L; t += 32) padded[(size_t)b * L + t] = 0;
    return;
  }
  auto best_source = [&](const float* part, float f, int j, bool with_f) -> int {
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = lane; i < T; i += 32) {
      const float v = with_f ? (f + tr(i, j)) + part[i] : part[i] + tr(i, j);
      if (v > best) { best = v; bi = i; }
    }
    if (bi == 0x7fffffff) bi = lane;   // nothing above -inf in this lane: keep order so index 0 wins a full tie
    warp_argmax_first(best, bi);
    if (best == -INFINITY) bi = 0;
    return bi;
  };
  int ptr = best_source(hs + (size_t)(n - 1) * T, 0.f, T - 1, false);
  const int64_t off = offsets ? offsets[b] : 0;
  auto emit = [&](int t, int tag) {
    if (lane == 0) {
      if (padded) padded[(size_t)b * L + t] = tag;
      if (flat) flat[off + t] = (tag == clamp_col) ? o_idx : (int64_t)tag;
    }
  };
  if (padded && lane == 0) {   // reference leaves pads at 0 and the final pointer in the last column
    for (int t = n; t < L - 1; ++t) padded[(size_t)b * L + t] = 0;
    if (n < L) padded[(size_t)b * L + (L - 1)] = ptr;
  }
  emit(n - 1, ptr);
  for (int t = n - 1; t >= 1; --t) {
    ptr = best_source(hs + (size_t)(t - 1) * T, clamped_feat(fs + (size_t)t * T, ptr, clamp_col, thr), ptr, true);
    emit(t - 1, ptr);
  }
}

// dynamic smem: trT[T][Tq] (trT[j][i] = trans[i][j], source tags i >= T hold -inf), then kCrfWarps * NS * 2 * Tq
// partitions.  One warp sweeps NS neighbouring sequences together: every transition value read from shared memory
// (the binding resource once the compare/select sweep is gone: each candidate needs its own 4-byte trans[i][j])
// serves NS candidates.  (Measured dead end: sweeping the T % 32 targets of a nearly empty last slot -- T = 131: three --
// with the lanes along the source tags instead: the serial warp reductions cost what the slot saves, 3.02 vs 2.90 ms.)  The inference path hands over length-sorted batches, so the NS sequences end within a
// step or two of each other; a finished sequence keeps computing (unobserved) values and stops storing.
template <int NJ, int NS>
__global__ void __launch_bounds__(kCrfWarps * 32) crf_viterbi_kernel(
    const float* __restrict__ feats, const float* __restrict__ trans_g, const int64_t* __restrict__ len,
    const int64_t* __restrict__ offsets, int B, int L, int T, int clamp_col, float thr, int64_t o_idx,
    int64_t* __restrict__ padded, int64_t* __restrict__ flat, float* hist) {
  extern __shared__ __align__(16) float smem[];
  const int Tq = viterbi_pitch(T);
  float* trT = smem;
  float* s_part = smem + (size_t)T * Tq;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int e = threadIdx.x; e < T * Tq; e += blockDim.x) {
    const int j = e / Tq, i = e - j * Tq;
    trT[e] = i < T ? trans_g[i * T + j] : -INFINITY;
  }
  for (int e = threadIdx.x; e < kCrfWarps * NS * 2 * Tq; e += blockDim.x) s_part[e] = 0.f;   // pad source slots stay 0
  __syncthreads();
  const int b0 = (blockIdx.x * kCrfWarps + warp) * NS;
  if (b0 >= B) return;
  constexpr int NQ = NJ > 0 ? NJ : 1;
  int n[NS];
  int nmax = 0;
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    n[s] = b0 + s < B ? min((int)len[b0 + s], L) : 0;
    nmax = max(nmax, n[s]);
  }
  float* pa = s_part + warp * NS * 2 * Tq;      // [s][Tq] current, then [s][Tq] next
  float* pb = pa + NS * Tq;
  const size_t seq = (size_t)L * T;
  const float* fb = feats + (size_t)b0 * seq;
  float* hb = hist + (size_t)b0 * seq;
  const TransposedTrans tr{trT, Tq};

#pragma unroll
  for (int s = 0; s < NS; ++s) {
    if (n[s] > 0)
      for (int j = lane; j < T; j += 32) {
        const float v = viterbi_start(tr, fb + s * seq, j, T, clamp_col, thr);
        pa[s * Tq + j] = v;
        hb[s * seq + j] = v;
      }
  }
  __syncwarp();
  if (NJ > 0) {
    // lane owns target tags j = lane + 32 q; slots past T re-read the last row and drop the result
    const float* rowp[NQ];
    float fnext[NS][NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int j = min(lane + 32 * q, T - 1);
      rowp[q] = trT + j * Tq;
#pragma unroll
      for (int s = 0; s < NS; ++s) fnext[s][q] = n[s] > 1 ? clamped_feat(fb + s * seq + T, j, clamp_col, thr) : 0.f;
    }
    for (int t = 1; t < nmax; ++t) {
      unsigned long long ff[NS][NQ];
      float best[NS][NQ];
#pragma unroll
      for (int s = 0; s < NS; ++s)
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          ff[s][q] = pack_f32x2(fnext[s][q], fnext[s][q]);
          best[s][q] = -INFINITY;
        }
#pragma unroll
      for (int s = 0; s < NS; ++s)
        if (t + 1 < n[s]) {      // next position's features in flight during this sweep
#pragma unroll
          for (int q = 0; q < NQ; ++q)
            fnext[s][q] = clamped_feat(fb + s * seq + (size_t)(t + 1) * T, min(lane + 32 * q, T - 1), clamp_col, thr);
        }
#pragma unroll 1
      for (int i0 = 0; i0 < Tq; i0 += 4) {
        unsigned long long p01[NS], p23[NS];
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const float4 p4 = *reinterpret_cast<const float4*>(pa + s * Tq + i0);
          p01[s] = pack_f32x2(p4.x, p4.y);
          p23[s] = pack_f32x2(p4.z, p4.w);
        }
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          const float4 t4 = *reinterpret_cast<const float4*>(rowp[q] + i0);
          const unsigned long long t01 = pack_f32x2(t4.x, t4.y), t23 = pack_f32x2(t4.z, t4.w);
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            const unsigned long long v01 = add_f32x2(add_f32x2(ff[s][q], t01), p01[s]);
            const unsigned long long v23 = add_f32x2(add_f32x2(ff[s][q], t23), p23[s]);
            best[s][q] = max3_of(max3_of(best[s][q], v01), v23);
          }
        }
      }
#pragma unroll
      for (int s = 0; s < NS; ++s)
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          const int j = lane + 32 * q;
          if (j < T) {
            pb[s * Tq + j] = best[s][q];
            if (t < n[s]) hb[s * seq + (size_t)t * T + j] = best[s][q];
          }
        }
      __syncwarp();
      float* tmp = pa; pa = pb; pb = tmp;
    }
  } else {
    for (int t = 1; t < nmax; ++t) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        if (t >= n[s]) continue;
        const float* ft = fb + s * seq + (size_t)t * T;
        for (int j = lane; j < T; j += 32) {
          const float f = clamped_feat(ft, j, clamp_col, thr);
          const float* row = trT + j * Tq;
          float best = -INFINITY;
          for (int i = 0; i < T; ++i) best = fmaxf(best, (f + row[i]) + pa[s * Tq + i]);
          pb[s * Tq + j] = best;
          hb[s * seq + (size_t)t * T + j] = best;
        }
      }
      __syncwarp();
      float* tmp = pa; pa = pb; pb = tmp;
    }
  }
  __syncwarp();      // the history rows are read back by every lane
#pragma unroll 1
  for (int s = 0; s < NS && b0 + s < B; ++s)
    viterbi_backtrace(tr, fb + s * seq, hb + s * seq, n[s], b0 + s, L, T, lane, clamp_col, thr, o_idx, offsets, padded,
                      flat);
}

// transitions too large for shared memory: same algorithm straight from global memory
__global__ void __launch_bounds__(kCrfWarps * 32) crf_viterbi_global_kernel(
    const float* __restrict__ feats, const float* __restrict__ trans_g, const int64_t* __restrict__ len,
    const int64_t* __restrict__ offsets, int B, int L, int T, int clamp_col, float thr, int64_t o_idx,
    int64_t* __restrict__ padded, int64_t* __restrict__ flat, float* hist) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kCrfWarps + warp;
  if (b >= B) return;
  const int n = min((int)len[b], L);
  const RowMajorTrans tr{trans_g, T};
  const float* fb = feats + (size_t)b * L * T;
  float* hb = hist + (size_t)b * L * T;
  if (n > 0)
    for (int j = lane; j < T; j += 32) hb[j] = viterbi_start(tr, fb, j, T, clamp_col, thr);
  __syncwarp();
  for (int t = 1; t < n; ++t) {
    const float* pa = hb + (size_t)(t - 1) * T;
    for (int j = lane; j < T; j += 32) {
      const float f = clamped_feat(fb + (size_t)t * T, j, clamp_col, thr);
      float best = -INFINITY;
      for (int i = 0; i < T; ++i) best = fmaxf(best, (f + tr(i, j)) + pa[i]);
      hb[(size_t)t * T + j] = best;
    }
    __syncwarp();
  }
  viterbi_backtrace(tr, fb, hb, n, b, L, T, lane, clamp_col, thr, o_idx, offsets, padded, flat);
}

// ---- per-sequence pieces of the NLL kernels (crf.py:48-99, 202-251); tr is the row-major T x T matrix -------------
// logZ = LSE_i(trans[i][STOP] + part[i]) over the last partition, one warp
__device__ __forceinline__ float crf_log_z(const float* tr, const float* part, int T, int lane) {
  float m = -INFINITY;
  for (int i = lane; i < T; i += 32) m = fmaxf(m, tr[i * T + (T - 1)] + part[i]);
  m = warp_max(m);
  float s = 0.f;
  for (int i = lane; i < T; i += 32) s += expf((tr[i * T + (T - 1)] + part[i]) - m);
  s = warp_sum(s);
  return m + logf(s);
}

// per_seq = logZ - (score of the gold path of the n tags tg), one warp
__device__ __forceinline__ void crf_store_nll(const float* tr, const float* part, const float* fb, const int64_t* tg,
                                              int n, int T, int lane, float* per_seq) {
  const float logZ = crf_log_z(tr, part, T, lane);
  float g = 0.f;
  for (int t = lane; t < n; t += 32) {
    int cur = (int)tg[t];
    int prev = t == 0 ? T - 2 : (int)tg[t - 1];
    g += __ldg(fb + (size_t)t * T + cur) + tr[prev * T + cur];
  }
  g = warp_sum(g);
  if (lane == 0) {
    g += tr[(int)tg[n - 1] * T + (T - 1)];
    *per_seq = logZ - g;
  }
}

// exact log-domain LSE_i((f + trans[i][j]) + part[i]) of column j
__device__ __forceinline__ float crf_column_lse(const float* tr, const float* part, float f, int j, int T) {
  float m = -INFINITY;
  for (int i = 0; i < T; ++i) m = fmaxf(m, (f + tr[i * T + j]) + part[i]);
  float s = 0.f;
  for (int i = 0; i < T; ++i) s += expf(((f + tr[i * T + j]) + part[i]) - m);
  return m + logf(s);
}

// Exact log-domain backward row i (tri = trans[i][.]): returns beta_{t-1}[i] = LSE_j((trans[i][j] + feat_t[j]) +
// beta_t[j]) and adds the pairwise marginals gs * exp(pi + e_ij), pi = part_{t-1}[i] - logZ, to the accumulator row dwi.
__device__ __forceinline__ float crf_backward_row_exact(const float* tri, const float* ft, const float* beta, float pi,
                                                        float gs, float* dwi, int T) {
  float mx = -INFINITY;
  for (int j = 0; j < T; ++j) mx = fmaxf(mx, (tri[j] + __ldg(ft + j)) + beta[j]);
  float sm = 0.f;
  for (int j = 0; j < T; ++j) {
    const float e = (tri[j] + __ldg(ft + j)) + beta[j];
    sm += expf(e - mx);
    dwi[j] += gs * expf(pi + e);
  }
  return mx + logf(sm);
}

// Shared-memory tables of the scaled-exponential backward kernels, built by the whole CTA: tr = trans_g (T x T),
// rmax[i] = max_j trans[i][j] (-inf for T <= i < Tp), te[i * pitch + j] = exp(trans[i][j] - rmax[i]), 0 in the pad
// columns j >= T.  (crf_nll_exp_kernel keeps its column-maximum table inline: built through a shared function, its
// T <= 32 instantiation spilled 8 bytes.)
__device__ __forceinline__ void crf_exp_row_table(const float* trans_g, int T, int Tp, int pitch, float* tr, float* te,
                                                  float* rmax) {
  for (int i = threadIdx.x; i < T * T; i += blockDim.x) tr[i] = trans_g[i];
  __syncthreads();
  for (int i = threadIdx.x; i < Tp; i += blockDim.x) {
    float m = -INFINITY;
    if (i < T)
      for (int j = 0; j < T; ++j) m = fmaxf(m, tr[i * T + j]);
    rmax[i] = m;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < T * pitch; i += blockDim.x) {
    const int r = i / pitch, c = i - r * pitch;
    te[i] = c < T ? expf(tr[r * T + c] - rmax[r]) : 0.f;
  }
  __syncthreads();
}

// dfeats rows from..L-1 of one sequence are zero (pads; every row of an empty sequence); `stride` threads from `tid`
__device__ __forceinline__ void crf_zero_rows(float* df, int from, int L, int T, int tid, int stride) {
  for (int i = from * T + tid; i < L * T; i += stride) df[i] = 0.f;
}

// Sum of the CTA's nacc private dtrans accumulators (T x T at row pitch Tq) into dtrans, one atomicAdd per element
__device__ __forceinline__ void crf_fold_dtrans(const float* s_dtr, int nacc, int T, int Tq, float* dtrans) {
  __syncthreads();
  for (int i = threadIdx.x; i < T * T; i += blockDim.x) {
    const int r = i / T, c = i - r * T;
    float v = 0.f;
    for (int w = 0; w < nacc; ++w) v += s_dtr[(size_t)w * T * Tq + r * Tq + c];
    if (v != 0.f) atomicAdd(dtrans + i, v);
  }
}

// log-partition + gold score.  per_seq[b] = logZ_b - gold_b.   (crf.py:48-99, 202-251)
template <bool TS>
__global__ void __launch_bounds__(kCrfWarps * 32) crf_nll_kernel(
    const float* __restrict__ feats, const float* __restrict__ trans_g, const int64_t* __restrict__ len,
    const int64_t* __restrict__ tags, int B, int L, int Ltags, int T, float* __restrict__ per_seq,
    float* __restrict__ part_save) {
  extern __shared__ float smem[];
  const int Tp = (T + 31) & ~31;
  float* s_trans = smem;
  float* s_part = smem + (TS ? T * T : 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (TS) {
    for (int i = threadIdx.x; i < T * T; i += blockDim.x) s_trans[i] = trans_g[i];
    __syncthreads();
  }
  const float* tr = TS ? s_trans : trans_g;
  const int b = blockIdx.x * kCrfWarps + warp;
  if (b >= B) return;
  const int n = min((int)len[b], L);      // lengths past the row are clamped
  if (n <= 0) {                           // an empty sequence contributes nothing (the reference cannot express it)
    if (lane == 0) per_seq[b] = 0.f;
    return;
  }
  float* pa = s_part + warp * 2 * Tp;
  float* pb = pa + Tp;
  const float* fb = feats + (size_t)b * L * T;
  float* ps = part_save ? part_save + (size_t)b * L * T : nullptr;

  for (int j = lane; j < T; j += 32) {
    float v = __ldg(fb + j) + tr[(T - 2) * T + j];
    pa[j] = v;
    if (ps) ps[j] = v;
  }
  __syncwarp();
  for (int t = 1; t < n; ++t) {
    const float* ft = fb + (size_t)t * T;
    for (int j = lane; j < T; j += 32) {
      const float v = crf_column_lse(tr, pa, __ldg(ft + j), j, T);
      pb[j] = v;
      if (ps) ps[(size_t)t * T + j] = v;
    }
    __syncwarp();
    float* tmp = pa; pa = pb; pb = tmp;
  }
  crf_store_nll(tr, pa, fb, tags + (size_t)b * Ltags, n, T, lane, per_seq + b);
}

// Same log-partition in the scaled exponential domain: with M = max_i part[i] and cmax[j] = max_i trans[i][j]
//   LSE_i(part[i] + trans[i][j]) = M + cmax[j] + log sum_i exp(part[i] - M) * exp(trans[i][j] - cmax[j])
// so a step costs T exps and T*T FFMAs instead of 2*T*T exps (the log-domain kernel above spends ~1200 instructions
// per (t, j); this one ~100).  exp(trans - cmax) is tabulated once per CTA.  A column whose sum underflows (only
// reachable from states that are e^-87 below the best one, e.g. hard-constrained transitions) falls back to the
// exact two-pass form for that (t, j), so the result stays within fp32 rounding of the log-domain kernel.
// dynamic smem: trans T*T | exp table T*T | cmax Tp | per warp: part a, part b, E (3 * Tp)
template <int NJ>
__global__ void __launch_bounds__(kCrfWarps * 32) crf_nll_exp_kernel(
    const float* __restrict__ feats, const float* __restrict__ trans_g, const int64_t* __restrict__ len,
    const int64_t* __restrict__ tags, int B, int L, int Ltags, int T, float* __restrict__ per_seq,
    float* __restrict__ part_save) {
  extern __shared__ float smem[];
  const int Tp = (T + 31) & ~31;
  float* tr = smem;
  float* te = tr + T * T;
  float* cmax = te + T * T + kCrfOverrun;     // pad: the row-overrun reads of the sweep never touch live words
  float* s_part = cmax + Tp;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < T * T; i += blockDim.x) tr[i] = trans_g[i];
  __syncthreads();
  for (int j = threadIdx.x; j < Tp; j += blockDim.x) {
    float m = -INFINITY;
    if (j < T)
      for (int i = 0; i < T; ++i) m = fmaxf(m, tr[i * T + j]);
    cmax[j] = m;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < T * T; i += blockDim.x) te[i] = expf(tr[i] - cmax[i % T]);
  __syncthreads();
  const int b = blockIdx.x * kCrfWarps + warp;
  if (b >= B) return;
  const int n = min((int)len[b], L);      // lengths past the row are clamped
  if (n <= 0) {                           // an empty sequence contributes nothing (the reference cannot express it)
    if (lane == 0) per_seq[b] = 0.f;
    return;
  }
  float* pa = s_part + warp * 3 * Tp;
  float* pb = pa + Tp;
  float* E = pb + Tp;
  const float* fb = feats + (size_t)b * L * T;
  float* ps = part_save ? part_save + (size_t)b * L * T : nullptr;

  for (int j = lane; j < Tp; j += 32) {
    float v = -INFINITY;
    if (j < T) {
      v = __ldg(fb + j) + tr[(T - 2) * T + j];
      if (ps) ps[j] = v;
    }
    pa[j] = v;
  }
  __syncwarp();
  for (int t = 1; t < n; ++t) {
    const float* ft = fb + (size_t)t * T;
    float M = -INFINITY;
    for (int i = lane; i < T; i += 32) M = fmaxf(M, pa[i]);
    M = warp_max(M);
    for (int i = lane; i < Tp; i += 32) E[i] = i < T ? expf(pa[i] - M) : 0.f;
    __syncwarp();
    float acc[NJ];
#pragma unroll
    for (int q = 0; q < NJ; ++q) acc[q] = 0.f;
    // lanes whose last slot falls past T read (and ignore) the following shared-memory words
#pragma unroll 5
    for (int i = 0; i < T; ++i) {
      const float e = E[i];
      const float* tei = te + i * T + lane;
#pragma unroll
      for (int q = 0; q < NJ; ++q) acc[q] = fmaf(e, tei[32 * q], acc[q]);
    }
#pragma unroll
    for (int q = 0; q < NJ; ++q) {
      const int j = lane + 32 * q;
      if (j < T) {
        const float f = __ldg(ft + j);
        // a column whose sum underflows is evaluated exactly in the log domain
        const float v = acc[q] > 1e-30f ? ((M + cmax[j]) + f) + logf(acc[q]) : crf_column_lse(tr, pa, f, j, T);
        pb[j] = v;
        if (ps) ps[(size_t)t * T + j] = v;
      }
    }
    __syncwarp();
    float* tmp = pa; pa = pb; pb = tmp;
  }
  crf_store_nll(tr, pa, fb, tags + (size_t)b * Ltags, n, T, lane, per_seq + b);
}

// CRF backward: marginals by the backward recursion, reusing the saved forward partitions.
//   dfeats[b,t,j] = gs * (P(y_t=j) - [tag_t=j]);  dtrans[i,j] += gs * (sum_t P(y_{t-1}=i,y_t=j) - gold counts)
// Every warp owns a private T x T accumulator in shared memory (row pitch padded to an odd number of words:
// lanes own rows, so the pitch decides the bank) => plain read-modify-write, no shared atomics; the CTA folds
// its warps' copies together and issues one global atomicAdd per element.
template <bool TS>
__global__ void crf_nll_backward_kernel(
    const float* __restrict__ feats, const float* __restrict__ trans_g, const int64_t* __restrict__ len,
    const int64_t* __restrict__ tags, const float* __restrict__ part_save, const float* __restrict__ gscale, int B,
    int L, int Ltags, int T, float* __restrict__ dfeats, float* __restrict__ dtrans) {
  extern __shared__ float smem[];
  const int nw = blockDim.x >> 5;
  const int Tp = (T + 31) & ~31;
  const int Tq = T | 1;                          // odd pitch of the private accumulators
  float* s_trans = smem;                         // T*T (if TS)
  float* s_dtr = smem + (TS ? T * T : 0);        // nw * T * Tq
  float* s_beta = s_dtr + (size_t)nw * T * Tq;   // nw * 2 * Tp
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (TS)
    for (int i = threadIdx.x; i < T * T; i += blockDim.x) s_trans[i] = trans_g[i];
  for (int i = threadIdx.x; i < nw * T * Tq; i += blockDim.x) s_dtr[i] = 0.f;
  __syncthreads();
  const float* tr = TS ? s_trans : trans_g;
  const float gs = gscale ? *gscale : 1.f;
  float* dw = s_dtr + (size_t)warp * T * Tq;
  const int b = blockIdx.x * nw + warp;
  const int n = b < B ? min((int)len[b], L) : 0;
  float* df = dfeats + (size_t)b * L * T;
  if (n > 0) {
    float* ba = s_beta + warp * 2 * Tp;   // beta_t
    float* bb = ba + Tp;                  // beta_{t-1}
    const float* fb = feats + (size_t)b * L * T;
    const float* ps = part_save + (size_t)b * L * T;
    const int64_t* tg = tags + (size_t)b * Ltags;
    const float logZ = crf_log_z(tr, ps + (size_t)(n - 1) * T, T, lane);
    for (int i = lane; i < T; i += 32) ba[i] = tr[i * T + (T - 1)];   // beta_{n-1}[i] = trans[i][STOP]
    __syncwarp();
    for (int t = n - 1; t >= 0; --t) {
      const float* pt = ps + (size_t)t * T;
      const int gold = (int)tg[t];
      // unary marginal at t  (+ STOP column / START row of dtrans); lane owns j => distinct addresses
      for (int j = lane; j < T; j += 32) {
        const float d = gs * (expf(pt[j] + ba[j] - logZ) - (j == gold ? 1.f : 0.f));
        df[(size_t)t * T + j] = d;
        if (t == n - 1) dw[j * Tq + (T - 1)] += d;
      }
      __syncwarp();
      if (t == 0) {
        for (int j = lane; j < T; j += 32) dw[(T - 2) * Tq + j] += df[j];
        break;
      }
      // pairwise marginals (t-1 -> t) and beta_{t-1}; lane owns source rows i
      const float* pp = ps + (size_t)(t - 1) * T;
      const float* ft = fb + (size_t)t * T;
      const int gprev = (int)tg[t - 1];
      for (int i = lane; i < T; i += 32) {
        float* dwi = dw + i * Tq;
        bb[i] = crf_backward_row_exact(tr + i * T, ft, ba, pp[i] - logZ, gs, dwi, T);
        if (i == gprev) dwi[gold] -= gs;
      }
      __syncwarp();
      float* tmp = ba; ba = bb; bb = tmp;
    }
  }
  if (b < B) crf_zero_rows(df, max(n, 0), L, T, lane, 32);
  crf_fold_dtrans(s_dtr, nw, T, Tq, dtrans);
}

// CRF backward in the scaled exponential domain (see crf_nll_exp_kernel): with w_j = feat_t[j] + beta_t[j],
// Mw = max_j w_j, W_j = exp(w_j - Mw), rmax[i] = max_j trans[i][j] and the table exp(trans[i][j] - rmax[i]),
//   beta_{t-1}[i]    = rmax[i] + Mw + log S_i,   S_i = sum_j table[i][j] * W_j
//   P(y_{t-1}=i,y_t=j) = exp(part_{t-1}[i] - logZ + rmax[i] + Mw) * table[i][j] * W_j
// i.e. T exps, T logs and 2 T*T multiply-adds per step instead of 3 T*T exps.  A row whose S_i underflows is
// evaluated exactly in the log domain (same formulas as crf_nll_backward_kernel).
// dynamic smem: trans T*T | table T*T | rmax Tp | per warp: dtrans accumulator T*Tq, beta a / b, W (3 * Tp)
__global__ void crf_nll_backward_exp_kernel(
    const float* __restrict__ feats, const float* __restrict__ trans_g, const int64_t* __restrict__ len,
    const int64_t* __restrict__ tags, const float* __restrict__ part_save, const float* __restrict__ gscale, int B,
    int L, int Ltags, int T, float* __restrict__ dfeats, float* __restrict__ dtrans) {
  extern __shared__ float smem[];
  const int nw = blockDim.x >> 5;
  const int Tp = (T + 31) & ~31;
  const int Tq = T | 1;
  float* tr = smem;
  float* te = tr + T * T;
  float* rmax = te + T * T;
  float* s_dtr = rmax + Tp;
  float* s_vec = s_dtr + (size_t)nw * T * Tq;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < nw * T * Tq; i += blockDim.x) s_dtr[i] = 0.f;
  crf_exp_row_table(trans_g, T, Tp, T, tr, te, rmax);
  const float gs = gscale ? *gscale : 1.f;
  float* dw = s_dtr + (size_t)warp * T * Tq;
  const int b = blockIdx.x * nw + warp;
  const int n = b < B ? min((int)len[b], L) : 0;
  float* df = dfeats + (size_t)b * L * T;
  if (n > 0) {
    float* ba = s_vec + warp * 3 * Tp;   // beta_t
    float* bb = ba + Tp;                 // beta_{t-1}
    float* W = bb + Tp;
    const float* fb = feats + (size_t)b * L * T;
    const float* ps = part_save + (size_t)b * L * T;
    const int64_t* tg = tags + (size_t)b * Ltags;
    const float logZ = crf_log_z(tr, ps + (size_t)(n - 1) * T, T, lane);
    for (int i = lane; i < T; i += 32) ba[i] = tr[i * T + (T - 1)];
    __syncwarp();
    for (int t = n - 1; t >= 0; --t) {
      // The sweep is one dependent chain per sequence and every step used to pay three or four HBM round trips in
      // sequence (partition row, feature row, tags: nobody has touched them since the forward pass).  Pull the rows of
      // the NEXT step into L1 now; they arrive while this step's T x T loops run.
      if (t >= 1 && lane < 8) {
        const int part = (lane & 3) * 32;                       // a row is T floats: up to four 128-byte lines
        const float* row = lane < 4 ? fb + (size_t)(t - 1) * T : ps + (size_t)(t >= 2 ? t - 2 : 0) * T;
        if (part < T) asm volatile("prefetch.global.L1 [%0];" ::"l"(row + part));
      }
      const float* pt = ps + (size_t)t * T;
      const int gold = (int)tg[t];
      for (int j = lane; j < T; j += 32) {
        const float d = gs * (expf(pt[j] + ba[j] - logZ) - (j == gold ? 1.f : 0.f));
        df[(size_t)t * T + j] = d;
        if (t == n - 1) dw[j * Tq + (T - 1)] += d;
      }
      __syncwarp();
      if (t == 0) {
        for (int j = lane; j < T; j += 32) dw[(T - 2) * Tq + j] += df[j];
        break;
      }
      const float* pp = ps + (size_t)(t - 1) * T;
      const float* ft = fb + (size_t)t * T;
      const int gprev = (int)tg[t - 1];
      // W_j = exp(feat_t[j] + beta_t[j] - Mw)
      float Mw = -INFINITY;
      for (int j = lane; j < T; j += 32) Mw = fmaxf(Mw, __ldg(ft + j) + ba[j]);
      Mw = warp_max(Mw);
      for (int j = lane; j < T; j += 32) W[j] = expf((__ldg(ft + j) + ba[j]) - Mw);
      __syncwarp();
      for (int i = lane; i < T; i += 32) {
        const float* tei = te + i * T;
        float* dwi = dw + i * Tq;
        float S = 0.f;
        for (int j = 0; j < T; ++j) S = fmaf(tei[j], W[j], S);
        if (S > 1e-30f) {
          const float A = gs * expf(((pp[i] - logZ) + rmax[i]) + Mw);
          int j = 0;
          for (; j + 8 <= T; j += 8) {
            float d[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) d[q] = fmaf(A * tei[j + q], W[j + q], dwi[j + q]);
#pragma unroll
            for (int q = 0; q < 8; ++q) dwi[j + q] = d[q];
          }
          for (; j < T; ++j) dwi[j] = fmaf(A * tei[j], W[j], dwi[j]);
          bb[i] = (rmax[i] + Mw) + logf(S);
        } else {   // underflow: exact log-domain evaluation of this row
          bb[i] = crf_backward_row_exact(tr + i * T, ft, ba, pp[i] - logZ, gs, dwi, T);
        }
        if (i == gprev) dwi[gold] -= gs;
      }
      __syncwarp();
      float* tmp = ba; ba = bb; bb = tmp;
    }
  }
  if (b < B) crf_zero_rows(df, max(n, 0), L, T, lane, 32);
  crf_fold_dtrans(s_dtr, nw, T, Tq, dtrans);
}

// The same sweep with THREE warps per sequence (T <= 96): warp `part` of a sequence owns transition rows / tag columns
// part*32 + lane, so a lane has one row instead of three and the per-step chain is a third as long; the warps of a
// sequence meet at a named barrier twice per step (W complete; beta_{t-1} complete).  The sweep is latency-bound --
// one dependent chain per sequence, seven sequences per SM because of the T x T accumulators -- so the step latency is
// the kernel time.  Same arithmetic per element and the same left-to-right row sums as crf_nll_backward_exp_kernel.
// dynamic smem: trans T*T | table T*T | rmax Tp | per SEQUENCE: dtrans accumulator T*Tq, beta a / b, W (3 * Tp)
__global__ void crf_nll_backward_exp3_kernel(
    const float* __restrict__ feats, const float* __restrict__ trans_g, const int64_t* __restrict__ len,
    const int64_t* __restrict__ tags, const float* __restrict__ part_save, const float* __restrict__ gscale, int B,
    int L, int Ltags, int T, float* __restrict__ dfeats, float* __restrict__ dtrans) {
  extern __shared__ float smem[];
  const int nseq = (blockDim.x >> 5) / 3;
  const int Tp = (T + 31) & ~31;
  const int Tq = (T + 3) & ~3;         // row pitch of the table and of the accumulators: 16-byte rows, LDS.128 / STS.128
  float* tr = smem;                    // (a quarter-warp of consecutive rows at pitch 76 hits 32 distinct banks)
  float* te = tr + ((T * T + 3) & ~3);
  float* rmax = te + T * Tq;
  float* s_dtr = rmax + Tp;
  float* s_vec = s_dtr + (size_t)nseq * T * Tq;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < nseq * T * Tq; i += blockDim.x) s_dtr[i] = 0.f;
  for (int i = threadIdx.x; i < nseq * 3 * Tp; i += blockDim.x) s_vec[i] = 0.f;   // W pad entries stay 0
  crf_exp_row_table(trans_g, T, Tp, Tq, tr, te, rmax);      // pad columns of the table contribute exact zeros
  const float gs = gscale ? *gscale : 1.f;
  const int seq = warp / 3, part = warp - seq * 3;
  const int own = part * 32 + lane;            // the row / column this lane owns
  const bool has = own < T;
  const int tid96 = part * 32 + lane;          // index among the 96 threads of the sequence
  auto seq_sync = [&]() { asm volatile("bar.sync %0, 96;" ::"r"(seq + 1) : "memory"); };
  float* dw = s_dtr + (size_t)seq * T * Tq;
  const int b = blockIdx.x * nseq + seq;
  const int n = b < B ? min((int)len[b], L) : 0;
  float* df = dfeats + (size_t)b * L * T;
  if (n > 0) {       // uniform over the three warps of a sequence
    float* ba = s_vec + seq * 3 * Tp;    // beta_t
    float* bb = ba + Tp;                 // beta_{t-1}
    float* W = bb + Tp;
    const float* fb = feats + (size_t)b * L * T;
    const float* ps = part_save + (size_t)b * L * T;
    const int64_t* tg = tags + (size_t)b * Ltags;
    const float logZ = crf_log_z(tr, ps + (size_t)(n - 1) * T, T, lane);   // every warp for itself, same result
    if (has) ba[own] = tr[own * T + (T - 1)];
    seq_sync();
    const float4* tei4 = reinterpret_cast<const float4*>(te + (has ? own : 0) * Tq);
    float* dwi = dw + (has ? own : 0) * Tq;
    for (int t = n - 1; t >= 0; --t) {
      // rows of the NEXT step into L1 while this step's loops run (see crf_nll_backward_exp_kernel)
      if (t >= 1 && part == 0 && lane < 8) {
        const int seg = (lane & 3) * 32;
        const float* row = lane < 4 ? fb + (size_t)(t - 1) * T : ps + (size_t)(t >= 2 ? t - 2 : 0) * T;
        if (seg < T) asm volatile("prefetch.global.L1 [%0];" ::"l"(row + seg));
      }
      // every global value of the step is requested here, ahead of the barriers (the compiler cannot move a load
      // above a bar.sync): partition rows t and t-1, feature row t, the two tags
      const float* pt = ps + (size_t)t * T;
      const float* pp = ps + (size_t)(t >= 1 ? t - 1 : 0) * T;
      const float* ft = fb + (size_t)t * T;
      const int oc = has ? own : 0;
      const float ptv = pt[oc], ppv = pp[oc], ftv = __ldg(ft + oc);
      float ftm[3];
#pragma unroll
      for (int q = 0; q < 3; ++q) ftm[q] = lane + 32 * q < T ? __ldg(ft + lane + 32 * q) : 0.f;
      const int gold = (int)tg[t];
      const int gprev = (int)tg[t >= 1 ? t - 1 : 0];
      float d = 0.f;
      if (has) {
        d = gs * (expf(ptv + ba[own] - logZ) - (own == gold ? 1.f : 0.f));
        df[(size_t)t * T + own] = d;
        if (t == n - 1) dwi[T - 1] += d;
      }
      if (t == 0) {
        // row T-2 belongs to one warp of the sequence, but its sweep over that row ended at the barrier that closed
        // the previous step; every lane adds to its own column.  A one-token sequence (t == n-1 == 0) has just added
        // to column T-1 of every row, row T-2 included: order the two updates of that element.
        if (n == 1) seq_sync();
        if (has) dw[(T - 2) * Tq + own] += d;
        break;
      }
      // W_j = exp(feat_t[j] + beta_t[j] - Mw): the maximum by every warp for itself, W by column owners
      float Mw = -INFINITY;
#pragma unroll
      for (int q = 0; q < 3; ++q)
        if (lane + 32 * q < T) Mw = fmaxf(Mw, ftm[q] + ba[lane + 32 * q]);
      Mw = warp_max(Mw);
      if (has) W[own] = expf((ftv + ba[own]) - Mw);
      seq_sync();
      if (has) {
        // four tag pairs per shared-memory instruction (the sweep issues ~2.5 loads per FMA otherwise); the row sum keeps
        // its left-to-right order, the pad columns add exact zeros
        const float4* W4 = reinterpret_cast<const float4*>(W);
        float4* dwi4 = reinterpret_cast<float4*>(dwi);
        const int n4 = Tq >> 2;
        float S = 0.f;
#pragma unroll 4
        for (int j = 0; j < n4; ++j) {
          const float4 t = tei4[j], w = W4[j];
          S = fmaf(t.x, w.x, S);
          S = fmaf(t.y, w.y, S);
          S = fmaf(t.z, w.z, S);
          S = fmaf(t.w, w.w, S);
        }
        if (S > 1e-30f) {
          const float A = gs * expf(((ppv - logZ) + rmax[own]) + Mw);
          int j = 0;
          for (; j + 2 <= n4; j += 2) {     // all loads of a batch before its stores
            const float4 t0 = tei4[j], w0 = W4[j], t1 = tei4[j + 1], w1 = W4[j + 1];
            float4 d0 = dwi4[j], d1 = dwi4[j + 1];
            d0.x = fmaf(A * t0.x, w0.x, d0.x); d0.y = fmaf(A * t0.y, w0.y, d0.y);
            d0.z = fmaf(A * t0.z, w0.z, d0.z); d0.w = fmaf(A * t0.w, w0.w, d0.w);
            d1.x = fmaf(A * t1.x, w1.x, d1.x); d1.y = fmaf(A * t1.y, w1.y, d1.y);
            d1.z = fmaf(A * t1.z, w1.z, d1.z); d1.w = fmaf(A * t1.w, w1.w, d1.w);
            dwi4[j] = d0;
            dwi4[j + 1] = d1;
          }
          for (; j < n4; ++j) {
            const float4 t0 = tei4[j], w0 = W4[j];
            float4 d0 = dwi4[j];
            d0.x = fmaf(A * t0.x, w0.x, d0.x); d0.y = fmaf(A * t0.y, w0.y, d0.y);
            d0.z = fmaf(A * t0.z, w0.z, d0.z); d0.w = fmaf(A * t0.w, w0.w, d0.w);
            dwi4[j] = d0;
          }
          bb[own] = (rmax[own] + Mw) + logf(S);
        } else {                           // underflow: exact log-domain evaluation of this row
          bb[own] = crf_backward_row_exact(tr + own * T, ft, ba, ppv - logZ, gs, dwi, T);
        }
        if (own == gprev) dwi[gold] -= gs;
      }
      seq_sync();                          // beta_{t-1} complete, nobody reads beta_t / W any more
      float* tmp = ba; ba = bb; bb = tmp;
    }
  }
  if (b < B) crf_zero_rows(df, max(n, 0), L, T, tid96, 96);
  crf_fold_dtrans(s_dtr, nseq, T, Tq, dtrans);
}

// deterministic sum of n floats (double accumulation), scaled
__global__ void __launch_bounds__(1024) reduce_sum_kernel(const float* __restrict__ v, size_t n, double scale,
                                                          float* __restrict__ out) {
  __shared__ double sh[32];
  double acc = 0.0;
  for (size_t i = threadIdx.x; i < n; i += blockDim.x) acc += (double)v[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (threadIdx.x == 0) *out = (float)(acc * scale);
  }
}

// one warp per (b,t): clamp, first-max argmax, remap
__global__ void __launch_bounds__(256) argmax_decode_kernel(const float* __restrict__ scores,
                                                            const int64_t* __restrict__ len,
                                                            const int64_t* __restrict__ offsets, int B, int L, int C,
                                                            int clamp_col, float thr, int64_t o_idx,
                                                            int64_t* __restrict__ flat, int64_t* __restrict__ padded) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= B * L) return;
  const int b = gw / L, t = gw - b * L;
  const bool valid = t < (int)len[b];
  if (!valid && !padded) return;
  const float* s = scores + (size_t)gw * C;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int c = lane; c < C; c += 32) {
    float v = clamped_feat(s, c, clamp_col, thr);
    if (v > best) { best = v; bi = c; }
  }
  if (bi == 0x7fffffff) bi = lane;
  warp_argmax_first(best, bi);
  if (best == -INFINITY) bi = 0;
  if (lane == 0) {
    int64_t tag = (bi == clamp_col) ? o_idx : (int64_t)bi;
    if (padded) padded[gw] = tag;
    if (flat && valid) flat[offsets[b] + t] = tag;
  }
}

// per-position cross entropy: lse(scores) - scores[label]; 0 at pads
__global__ void __launch_bounds__(256) ce_pos_kernel(const float* __restrict__ scores, const int64_t* __restrict__ len,
                                                     const int64_t* __restrict__ labels, int B, int L, int Llab, int C,
                                                     float* __restrict__ per_pos) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= B * L) return;
  const int b = gw / L, t = gw - b * L;
  if (t >= (int)len[b]) {
    if (lane == 0) per_pos[gw] = 0.f;
    return;
  }
  const float* s = scores + (size_t)gw * C;
  float m = -INFINITY;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, __ldg(s + c));
  m = warp_max(m);
  float e = 0.f;
  for (int c = lane; c < C; c += 32) e += expf(__ldg(s + c) - m);
  e = warp_sum(e);
  if (lane == 0) per_pos[gw] = (m + logf(e)) - __ldg(s + (int)labels[(size_t)b * Llab + t]);
}

__global__ void __launch_bounds__(256) ce_backward_kernel(const float* __restrict__ scores,
                                                          const int64_t* __restrict__ len,
                                                          const int64_t* __restrict__ labels,
                                                          const float* __restrict__ gscale, int B, int L, int Llab,
                                                          int C, float inv_n, float* __restrict__ dscores) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= B * L) return;
  const int b = gw / L, t = gw - b * L;
  float* d = dscores + (size_t)gw * C;
  if (t >= (int)len[b]) {
    for (int c = lane; c < C; c += 32) d[c] = 0.f;
    return;
  }
  const float* s = scores + (size_t)gw * C;
  float m = -INFINITY;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, __ldg(s + c));
  m = warp_max(m);
  float e = 0.f;
  for (int c = lane; c < C; c += 32) e += expf(__ldg(s + c) - m);
  e = warp_sum(e);
  const float g = (gscale ? *gscale : 1.f) * inv_n;
  const int lab = (int)labels[(size_t)b * Llab + t];
  for (int c = lane; c < C; c += 32) d[c] = g * (expf(__ldg(s + c) - m) / e - (c == lab ? 1.f : 0.f));
}

__global__ void colsum_kernel(const float* __restrict__ Cm, int C, int S, const float* __restrict__ wv,
                              float* __restrict__ o) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  float acc = 0.f;
  for (int c = 0; c < C; ++c) acc += Cm[(size_t)c * S + s];   // same order as torch's sum over dim 0
  o[s] = wv ? acc + wv[s] : acc;
}

// flat[offsets[b] + t] = padded[b, t] for t < len[b]   (utils.py:153-164 flatten, without the boolean-mask sync)
__global__ void flatten_i64_kernel(const int64_t* __restrict__ padded, const int64_t* __restrict__ len,
                                   const int64_t* __restrict__ offsets, int B, int Lrow, int L, int64_t* __restrict__ flat) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)B * L) return;
  const int b = (int)(i / L), t = (int)(i - (long long)b * L);
  if (t < (int)len[b]) flat[offsets[b] + t] = padded[(size_t)b * Lrow + t];
}

// Longest-first schedule of a batch in ONE launch: stable descending counting sort of the lengths (the permutation
// torch.sort(lengths, descending=True, stable=True) returns), the exclusive offsets of the flattened valid-only layout
// in the caller's order, and both gathered through the permutation.  Replaces a cast, a radix sort, two scans and
// three gathers (ten tiny dependent launches, ~60 us on the critical path of every inference batch).  One CTA; keys
// (lengths) below kOrderBins; tiles of 1024 sequences: rank of a sequence = sequences with a larger key + earlier
// sequences with the same key (earlier tiles via `base`, earlier warps of the tile via `whist`, earlier lanes via match).
constexpr int kOrderBins = 256;
constexpr int kOrderMaxB = 16384;
__global__ void __launch_bounds__(1024) length_order_kernel(const int64_t* __restrict__ len, int B, int nbins,
                                                            int64_t* __restrict__ order, int64_t* __restrict__ len_sorted,
                                                            int64_t* __restrict__ offs, int64_t* __restrict__ offs_sorted) {
  __shared__ int base[kOrderBins];
  __shared__ int whist[32][kOrderBins];
  __shared__ int wtot[32];
  __shared__ int carry;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int k = tid; k < nbins; k += 1024) base[k] = 0;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int i = tid; i < B; i += 1024) atomicAdd(&base[min(max((int)len[i], 0), nbins - 1)], 1);
  __syncthreads();
  int above = 0;
  if (tid < nbins)
    for (int k = tid + 1; k < nbins; ++k) above += base[k];
  __syncthreads();
  if (tid < nbins) base[tid] = above;            // first output slot of key tid (descending order)
  for (int t0 = 0; t0 < B; t0 += 1024) {
    for (int e = tid; e < 32 * nbins; e += 1024) whist[e / nbins][e % nbins] = 0;
    __syncthreads();
    const int i = t0 + tid;
    const bool valid = i < B;
    const int n = valid ? (int)len[i] : 0;
    const int k = valid ? min(max(n, 0), nbins - 1) : -1;
    const unsigned same = __match_any_sync(0xffffffffu, k);
    const int intra = __popc(same & ((1u << lane) - 1u));
    if (valid && intra == 0) whist[warp][k] = __popc(same);
    int incl = valid ? max(n, 0) : 0;             // inclusive scan of the lengths over the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) wtot[warp] = incl;
    __syncthreads();
    if (valid) {
      int before = 0, wpre = 0;
      for (int w = 0; w < warp; ++w) {
        before += whist[w][k];
        wpre += wtot[w];
      }
      const int pos = base[k] + before + intra;
      const int64_t off = (int64_t)carry + wpre + (incl - max(n, 0));
      offs[i] = off;
      order[pos] = i;
      len_sorted[pos] = n;
      offs_sorted[pos] = off;
    }
    __syncthreads();
    if (tid < nbins) {
      int s = 0;
      for (int w = 0; w < 32; ++w) s += whist[w][tid];
      base[tid] += s;
    }
    if (tid == 0) {
      int s = 0;
      for (int w = 0; w < 32; ++w) s += wtot[w];
      carry += s;
    }
    __syncthreads();
  }
}

static const size_t kSmemLimit = 200 * 1024;
static bool g_crf_bwd_split = true;      // CRF backward: three warps per sequence when T <= 96 (re2nn_debug_set_crf_backward_split)
static int g_viterbi_ns = 0;             // sequences per Viterbi warp, 0 = by batch size (re2nn_debug_set_viterbi_seqs)

// One launch of a CRF kernel; `configured` is that kernel's dynamic shared-memory state (ensure_dynamic_smem).
template <class Kernel, class... Args>
static int crf_launch(Kernel kernel, int (&configured)[kMaxDevices], int grid, int block, size_t smem, cudaStream_t st,
                      Args... args) {
  RE2NN_CUDA(ensure_dynamic_smem(kernel, (int)smem, configured));
  kernel<<<grid, block, smem, st>>>(args...);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

}  // namespace re2nn

using namespace re2nn;

extern "C" {

int re2nn_output_vector_sum(const float* C_mat, int C, int S, const float* wildcard_vec, float* o, void* stream) {
  RE2NN_CHECK(C_mat && o && C > 0 && S > 0, "output_vector_sum: bad arguments");
  colsum_kernel<<<cdiv(S, 128), 128, 0, (cudaStream_t)stream>>>(C_mat, C, S, wildcard_vec, o);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

int re2nn_flatten_i64(const int64_t* padded, const int64_t* lengths, const int64_t* offsets, int B, int Lrow, int L,
                      int64_t* flat, void* stream) {
  RE2NN_CHECK(padded && lengths && offsets && flat && L <= Lrow, "flatten_i64: bad arguments");
  const long long n = (long long)B * L;
  flatten_i64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(padded, lengths, offsets, B, Lrow, L, flat);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

int re2nn_length_order_supported(int B, int L) { return (B > 0 && B <= kOrderMaxB && L >= 0 && L + 1 <= kOrderBins) ? 1 : 0; }

int re2nn_length_order(const int64_t* lengths, int B, int L, int64_t* order, int64_t* lengths_sorted, int64_t* offsets,
                       int64_t* offsets_sorted, void* stream) {
  RE2NN_CHECK(lengths && order && lengths_sorted && offsets && offsets_sorted, "length_order: null tensor");
  RE2NN_CHECK(re2nn_length_order_supported(B, L), "length_order: B = %d, L = %d outside the single-CTA range (B <= %d, L < %d)", B,
              L, kOrderMaxB, kOrderBins);
  length_order_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(lengths, B, L + 1, order, lengths_sorted, offsets, offsets_sorted);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

int re2nn_crf_viterbi(const float* feats, const float* transitions, const int64_t* lengths, const int64_t* offsets,
                      int B, int L, int T, int clamp_col, float threshold, int64_t o_idx, int64_t* padded_path,
                      int64_t* flat_pred, float* part_ws, void* stream) {
  RE2NN_CHECK(feats && transitions && lengths && part_ws, "crf_viterbi: null tensor");
  RE2NN_CHECK(B > 0 && L > 0 && T >= 3 && T <= 65535, "crf_viterbi: bad dims B=%d L=%d T=%d", B, L, T);
  RE2NN_CHECK(!flat_pred || offsets, "crf_viterbi: flat output needs offsets");
  using Kernel = decltype(&crf_viterbi_global_kernel);
  static const Kernel kernels[2][6] = {       // [NS - 1][NJ]
      {crf_viterbi_kernel<0, 1>, crf_viterbi_kernel<1, 1>, crf_viterbi_kernel<2, 1>, crf_viterbi_kernel<3, 1>,
       crf_viterbi_kernel<4, 1>, crf_viterbi_kernel<5, 1>},
      {nullptr, crf_viterbi_kernel<1, 2>, crf_viterbi_kernel<2, 2>, crf_viterbi_kernel<3, 2>, crf_viterbi_kernel<4, 2>,
       crf_viterbi_kernel<5, 2>}};
  static int configured[2][6][kMaxDevices];
  const int Tq = viterbi_pitch(T);
  const int nj = cdiv(T, 32) <= 5 ? cdiv(T, 32) : 0;
  // sequences per warp: two halve the shared-memory reads of the transition table per candidate (measured at T = 131,
  // B = 16384: 3.7 -> 2.9 ms; four run out of registers: 4.3 ms), as long as the batch still fills the machine with
  // warps (cfg2, B = 4096: one sequence per warp is fastest, 0.18 vs 0.20 ms)
  int ns = g_viterbi_ns ? g_viterbi_ns : (B >= sm_count() * kCrfWarps * 8 ? 2 : 1);
  if (nj == 0) ns = 1;
  const size_t smem = ((size_t)T * Tq + (size_t)kCrfWarps * ns * 2 * Tq) * 4;
  if (smem > kSmemLimit)      // no dynamic shared memory: ensure_dynamic_smem leaves `configured` alone
    return crf_launch(crf_viterbi_global_kernel, configured[0][0], cdiv(B, kCrfWarps), kCrfWarps * 32, 0,
                      (cudaStream_t)stream, feats, transitions, lengths, offsets, B, L, T, clamp_col, threshold, o_idx,
                      padded_path, flat_pred, part_ws);
  return crf_launch(kernels[ns - 1][nj], configured[ns - 1][nj], cdiv(B, kCrfWarps * ns), kCrfWarps * 32, smem,
                    (cudaStream_t)stream, feats, transitions, lengths, offsets, B, L, T, clamp_col, threshold, o_idx,
                    padded_path, flat_pred, part_ws);
}

int re2nn_debug_set_crf_backward_split(int on) {
  g_crf_bwd_split = on != 0;
  return 0;
}

int re2nn_debug_set_viterbi_seqs(int ns) {
  RE2NN_CHECK(ns == 0 || ns == 1 || ns == 2, "debug_set_viterbi_seqs: expected 0, 1 or 2");
  g_viterbi_ns = ns;
  return 0;
}

int re2nn_crf_nll(const float* feats, const float* transitions, const int64_t* lengths, const int64_t* tags, int B,
                  int L, int Ltags, int T, float* per_seq, float* loss, float* part_save, void* stream) {
  RE2NN_CHECK(feats && transitions && lengths && tags && per_seq, "crf_nll: null tensor");
  RE2NN_CHECK(B > 0 && L > 0 && T >= 3, "crf_nll: bad dims");
  using Kernel = decltype(&crf_nll_kernel<true>);
  static const Kernel kernels[7] = {crf_nll_exp_kernel<1>, crf_nll_exp_kernel<2>, crf_nll_exp_kernel<3>,
                                    crf_nll_exp_kernel<4>, crf_nll_exp_kernel<5>, crf_nll_kernel<true>,
                                    crf_nll_kernel<false>};
  static int configured[7][kMaxDevices];
  const int Tp = (T + 31) & ~31;
  const size_t part = (size_t)kCrfWarps * 2 * Tp * 4;
  const size_t with_tr = part + (size_t)T * T * 4;
  const size_t exp_smem = ((size_t)2 * T * T + kCrfOverrun + Tp + (size_t)kCrfWarps * 3 * Tp) * 4;
  int k;           // exp<cdiv(T, 32)>, then the log-domain kernel with / without the transitions in shared memory
  size_t smem;
  if (exp_smem <= kSmemLimit && T <= 160) {
    k = cdiv(T, 32) - 1;
    smem = exp_smem;
  } else if (with_tr <= kSmemLimit) {
    k = 5;
    smem = with_tr;
  } else {
    k = 6;
    smem = part;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = crf_launch(kernels[k], configured[k], cdiv(B, kCrfWarps), kCrfWarps * 32, smem, st, feats, transitions,
                          lengths, tags, B, L, Ltags, T, per_seq, part_save))
    return rc;
  if (loss) {
    reduce_sum_kernel<<<1, 1024, 0, st>>>(per_seq, (size_t)B, 1.0, loss);
    RE2NN_LAUNCH_CHECK();
  }
  return 0;
}

int re2nn_crf_nll_backward(const float* feats, const float* transitions, const int64_t* lengths, const int64_t* tags,
                           const float* part_save, const float* gscale, int B, int L, int Ltags, int T, float* dfeats,
                           float* dtrans, void* stream) {
  RE2NN_CHECK(feats && transitions && lengths && tags && part_save && dfeats && dtrans, "crf_nll_backward: null tensor");
  using Kernel = decltype(&crf_nll_backward_exp_kernel);
  static const Kernel kernels[4] = {crf_nll_backward_exp3_kernel, crf_nll_backward_exp_kernel,
                                    crf_nll_backward_kernel<true>, crf_nll_backward_kernel<false>};
  static int configured[4][kMaxDevices];
  const int Tp = (T + 31) & ~31, Tq = T | 1;
  const size_t tr_bytes = (size_t)T * T * 4;
  // one CTA per SM either way (the per-sequence accumulators fill the shared memory): the scaled-exponential kernels
  // take everything the SM has, so that e.g. B = 1024 at T = 74 is 147 CTAs of seven sequences = ONE wave instead of
  // 171 CTAs of six = two
  const size_t smem_all = 226 * 1024;
  const size_t pw = ((size_t)T * Tq + 3 * Tp) * 4;             // per sequence of the scaled-exponential kernels
  const size_t fixed = 2 * tr_bytes + (size_t)Tp * 4;
  int k, nseq, block;       // kernel, sequences per CTA, threads per CTA
  size_t smem;
  if (fixed + 2 * pw <= kSmemLimit && T <= 96 && g_crf_bwd_split) {   // three warps per sequence
    const int Tv = (T + 3) & ~3;                                         // 16-byte rows of the table and accumulators
    const size_t fixed3 = ((((size_t)T * T + 3) & ~(size_t)3) + (size_t)T * Tv + Tp) * 4;
    const size_t pw3 = ((size_t)T * Tv + 3 * Tp) * 4;
    k = 0;
    nseq = (int)std::min<size_t>(kCrfWarps, (smem_all - fixed3) / pw3);
    block = nseq * 96;
    smem = fixed3 + nseq * pw3;
  } else if (fixed + 2 * pw <= kSmemLimit) {        // transitions + table + at least two accumulators fit
    k = 1;
    nseq = (int)std::min<size_t>(kCrfWarps, (smem_all - fixed) / pw);
    block = nseq * 32;
    smem = fixed + nseq * pw;
  } else {   // log domain: as many warps as the accumulators allow, transitions in shared memory when they still fit
    const size_t per_warp = ((size_t)T * Tq + 2 * Tp) * 4;
    const bool ts = tr_bytes + per_warp <= kSmemLimit;
    nseq = (int)std::min<size_t>(kCrfWarps, (kSmemLimit - (ts ? tr_bytes : 0)) / per_warp);
    RE2NN_CHECK(nseq >= 1, "crf_nll_backward: tag set too large (T=%d)", T);
    k = ts ? 2 : 3;
    block = nseq * 32;
    smem = (ts ? tr_bytes : 0) + nseq * per_warp;
  }
  cudaStream_t st = (cudaStream_t)stream;
  RE2NN_CUDA(cudaMemsetAsync(dtrans, 0, tr_bytes, st));
  return crf_launch(kernels[k], configured[k], cdiv(B, nseq), block, smem, st, feats, transitions, lengths, tags,
                    part_save, gscale, B, L, Ltags, T, dfeats, dtrans);
}

int re2nn_argmax_decode(const float* scores, const int64_t* lengths, const int64_t* offsets, int B, int L, int C,
                        int clamp_col, float threshold, int64_t o_idx, int64_t* flat_pred, int64_t* padded_pred,
                        void* stream) {
  RE2NN_CHECK(scores && lengths, "argmax_decode: null tensor");
  RE2NN_CHECK(!flat_pred || offsets, "argmax_decode: flat output needs offsets");
  const long long threads = (long long)B * L * 32;
  argmax_decode_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      scores, lengths, offsets, B, L, C, clamp_col, threshold, o_idx, flat_pred, padded_pred);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

int re2nn_ce_loss(const float* scores, const int64_t* lengths, const int64_t* labels, int B, int L, int Llab, int C,
                  int64_t n_total, float* per_pos, float* loss, void* stream) {
  RE2NN_CHECK(scores && lengths && labels && per_pos && loss, "ce_loss: null tensor");
  RE2NN_CHECK(n_total > 0, "ce_loss: n_total must be positive");
  cudaStream_t st = (cudaStream_t)stream;
  const long long threads = (long long)B * L * 32;
  ce_pos_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(scores, lengths, labels, B, L, Llab, C, per_pos);
  RE2NN_LAUNCH_CHECK();
  reduce_sum_kernel<<<1, 1024, 0, st>>>(per_pos, (size_t)B * L, 1.0 / (double)n_total, loss);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

int re2nn_ce_loss_backward(const float* scores, const int64_t* lengths, const int64_t* labels, const float* gscale,
                           int B, int L, int Llab, int C, int64_t n_total, float* dscores, void* stream) {
  RE2NN_CHECK(scores && lengths && labels && dscores, "ce_loss_backward: null tensor");
  const long long threads = (long long)B * L * 32;
  ce_backward_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      scores, lengths, labels, gscale, B, L, Llab, C, 1.f / (float)n_total, dscores);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
