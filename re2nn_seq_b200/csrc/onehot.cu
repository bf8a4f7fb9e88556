// Onehot i-FST recurrence: h <- phi((h (.) T[x_t]) * o) / h <- phi((h*o) (.) T[x_t]^T), T = language[x_t] + W.
// Reference: /root/reference/src_seq/farnn/model_onehot.py:358-415 (FARNN_S_O_I_S.forward_score),
//            utils.py:192-199 (_matmul / _maxmul).
// HBM-bound: every (sequence, direction, step) streams one S x S fp32 slice of the language tensor
// exactly once.  One CTA owns one (sequence, direction) for all its steps and keeps the state vector
// in shared memory; rows of the slice are read as full 128-byte lines (lanes along the contiguous
// "to-state" index), W comes from L2.  language + W is formed on the fly in the reference's own
// rounding order, so no V x S x S temporary is ever written (K1 in SURVEY.md §2.2).
#include <algorithm>

#include "common.cuh"

namespace re2nn {

constexpr int kOhThreads = 512;
constexpr int kOhWarps = kOhThreads / 32;

// T[s][j] (+ W[s][j] unless the caller passes a pre-summed tensor, W == nullptr)
__device__ __forceinline__ float tw(const float* __restrict__ T, const float* __restrict__ W, size_t i) {
  return W ? __ldg(T + i) + __ldg(W + i) : __ldg(T + i);
}

__device__ __forceinline__ float4 tw4(const float* __restrict__ T, const float* __restrict__ W, size_t i) {
  float4 t = __ldg(reinterpret_cast<const float4*>(T + i));
  if (W) {
    const float4 w = __ldg(reinterpret_cast<const float4*>(W + i));
    t.x += w.x; t.y += w.y; t.z += w.z; t.w += w.w;
  }
  return t;
}

// sum[v][s][j] = language[v][s][j] + W[s][j]   (model_onehot.py:366, hoisted: once per parameter version)
__global__ void onehot_sum_kernel(const float* __restrict__ lang, const float* __restrict__ W, size_t n_slice,
                                  size_t total, float* __restrict__ out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    out[i] = lang[i] + W[i % n_slice];
}

template <bool MAXP>
__device__ __forceinline__ float comb(float acc, float h, float t) {
  return MAXP ? fmaxf(acc, h * t) : fmaf(h, t, acc);
}

template <bool MAXP>
__device__ __forceinline__ float4 comb4(float4 acc, float h, float4 t) {
  acc.x = comb<MAXP>(acc.x, h, t.x); acc.y = comb<MAXP>(acc.y, h, t.y);
  acc.z = comb<MAXP>(acc.z, h, t.z); acc.w = comb<MAXP>(acc.w, h, t.w);
  return acc;
}
template <bool MAXP>
__device__ __forceinline__ float dot4(float acc, float4 h, float4 t) {
  acc = comb<MAXP>(acc, h.x, t.x); acc = comb<MAXP>(acc, h.y, t.y);
  acc = comb<MAXP>(acc, h.z, t.z); acc = comb<MAXP>(acc, h.w, t.w);
  return acc;
}

// (Measured dead end: a cp.async.bulk pipeline that streams 16-row stages of the slices ahead of the recurrence -- the
// tokens are known up front -- through shared memory was 1.5-1.7x SLOWER than these direct 16-byte loads at every batch
// size, B = 32: 1.14 vs 0.68 ms; the per-stage mbarrier round trips cost more than the load latency they hide.)
// ---- cluster helpers: small batches (cfg1: B = 32 -> 64 (sequence, direction) slices for 148 SMs) spread every slice over
// a thread-block cluster.  The S x S transition slice of a step is split by ROWS over the CTAs of the cluster (each
// streams 1/nc of the bytes); the S-float partial results are exchanged through distributed shared memory with one
// cluster barrier per step (double-buffered exchange arrays), and every CTA keeps a full copy of the state.
__device__ __forceinline__ uint32_t oh_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t oh_cluster_size() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void oh_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float oh_ld_remote(const float* local, uint32_t rank) {
  uint32_t la = (uint32_t)__cvta_generic_to_shared(local), ra;
  float v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(la), "r"(rank));
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(ra) : "memory");
  return v;
}

template <bool MAXP>
__global__ void __launch_bounds__(kOhThreads) onehot_recurrence_kernel(const re2nn_onehot_args a, const int rows8) {
  extern __shared__ float smem[];
  const int S = a.S;
  float* h = smem;                 // S   current state (bwd: already multiplied by o)
  float* part = smem + S;          // kOhWarps * S partial results (fwd)
  float* xbuf = part + kOhWarps * S;   // 2 * S: this CTA's contribution to the cluster exchange, per step parity
  const int nc = (int)oh_cluster_size(), cr = (int)oh_cluster_rank();
  const int b = blockIdx.x / nc, z = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = (int)a.lengths[b];
  const float* __restrict__ W = a.W;
  const float* __restrict__ o = a.o;
  float* out = z == 0 ? a.alpha : a.beta;
  const float init = MAXP ? -INFINITY : 0.f;
  // 16-byte path: rows start 16-byte aligned when S % 4 == 0 (cudaMalloc bases are 256-byte aligned)
  const bool vec4 = (S & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.language) | reinterpret_cast<uintptr_t>(W)) & 15) == 0;
  // rows of the slice this CTA streams: [r0, r1)
  const int rows_per = (S + nc - 1) / nc;
  const int r0 = min(S, cr * rows_per), r1 = min(S, r0 + rows_per);

  for (int s = tid; s < S; s += kOhThreads) {
    float v = z == 0 ? a.h0[s] : a.hT[s];
    if (z == 1) {
      if (cr == 0 && n >= 1 && n <= a.L) out[((size_t)b * a.L + (n - 1)) * S + s] = v;   // beta_n = hT
      v *= o[s];
    }
    h[s] = v;
  }
  __syncthreads();

  for (int k = 0; k < a.L; ++k) {
    int tpos, orow;
    bool alive;
    step_pos(z, k, n, a.full_pad, tpos, orow, alive);
    if (!alive) break;   // uniform over the block AND over the cluster (same sequence, same direction)
    const int64_t tok = a.x[(size_t)b * a.Lpad + tpos];
    const float* __restrict__ T = a.language + (size_t)tok * S * S;
    float* xb = xbuf + (k & 1) * S;
    if (z == 0) {
      // out[j] = (+|max)_s h[s] * (T[s][j] + W[s][j]) over this CTA's rows s; warps stride over rows, lanes over columns
      if (vec4) {
        // 16-byte loads, four rows in flight per lane: a CTA is one (sequence, direction) slice, so at small batch the
        // bytes in flight per SM decide the speed (8 KB with scalar loads = ~9 GB/s per SM)
        for (int jb = 0; jb < S; jb += 128) {
          const int j = jb + 4 * lane;
          if (j < S) {
            float4 acc = make_float4(init, init, init, init);
            int s = r0 + warp;
            for (; rows8 && s + 7 * kOhWarps < r1; s += 8 * kOhWarps) {      // eight rows in flight per lane
              float4 t[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) t[u] = tw4(T, W, (size_t)(s + u * kOhWarps) * S + j);
#pragma unroll
              for (int u = 0; u < 8; ++u) acc = comb4<MAXP>(acc, h[s + u * kOhWarps], t[u]);
            }
            for (; s + 3 * kOhWarps < r1; s += 4 * kOhWarps) {
              const float4 t0 = tw4(T, W, (size_t)s * S + j);
              const float4 t1 = tw4(T, W, (size_t)(s + kOhWarps) * S + j);
              const float4 t2 = tw4(T, W, (size_t)(s + 2 * kOhWarps) * S + j);
              const float4 t3 = tw4(T, W, (size_t)(s + 3 * kOhWarps) * S + j);
              acc = comb4<MAXP>(acc, h[s], t0);
              acc = comb4<MAXP>(acc, h[s + kOhWarps], t1);
              acc = comb4<MAXP>(acc, h[s + 2 * kOhWarps], t2);
              acc = comb4<MAXP>(acc, h[s + 3 * kOhWarps], t3);
            }
            for (; s < r1; s += kOhWarps) acc = comb4<MAXP>(acc, h[s], tw4(T, W, (size_t)s * S + j));
            *reinterpret_cast<float4*>(part + warp * S + j) = acc;
          }
        }
      } else {
        for (int jb = 0; jb < S; jb += 32) {
          const int j = jb + lane;
          float acc = init;
          if (j < S) {
            int s = r0 + warp;
            for (; s + 3 * kOhWarps < r1; s += 4 * kOhWarps) {
              float t0 = tw(T, W, (size_t)s * S + j);
              float t1 = tw(T, W, (size_t)(s + kOhWarps) * S + j);
              float t2 = tw(T, W, (size_t)(s + 2 * kOhWarps) * S + j);
              float t3 = tw(T, W, (size_t)(s + 3 * kOhWarps) * S + j);
              acc = comb<MAXP>(acc, h[s], t0);
              acc = comb<MAXP>(acc, h[s + kOhWarps], t1);
              acc = comb<MAXP>(acc, h[s + 2 * kOhWarps], t2);
              acc = comb<MAXP>(acc, h[s + 3 * kOhWarps], t3);
            }
            for (; s < r1; s += kOhWarps) acc = comb<MAXP>(acc, h[s], tw(T, W, (size_t)s * S + j));
            part[warp * S + j] = acc;
          }
        }
      }
      __syncthreads();
      if (nc == 1) {
        for (int j = tid; j < S; j += kOhThreads) {
          float acc = init;
#pragma unroll
          for (int w = 0; w < kOhWarps; ++w) acc = MAXP ? fmaxf(acc, part[w * S + j]) : acc + part[w * S + j];
          float v = apply_nl(acc * o[j], a.update_nonlinear);
          h[j] = v;
          if (orow >= 0) out[((size_t)b * a.L + orow) * S + j] = v;
        }
        __syncthreads();
      } else {
        for (int j = tid; j < S; j += kOhThreads) {
          float acc = init;
#pragma unroll
          for (int w = 0; w < kOhWarps; ++w) acc = MAXP ? fmaxf(acc, part[w * S + j]) : acc + part[w * S + j];
          xb[j] = acc;                                  // this CTA's rows
        }
        oh_cluster_sync();
        for (int j = tid; j < S; j += kOhThreads) {
          float acc = init;
          for (int c = 0; c < nc; ++c) {                // fixed rank order: every CTA forms the same sum
            const float pv = oh_ld_remote(xb + j, (uint32_t)c);
            acc = MAXP ? fmaxf(acc, pv) : acc + pv;
          }
          float v = apply_nl(acc * o[j], a.update_nonlinear);
          h[j] = v;
          if (cr == 0 && orow >= 0) out[((size_t)b * a.L + orow) * S + j] = v;
        }
        __syncthreads();
      }
    } else {
      // out[s] = (+|max)_j h[j] * (T[s][j] + W[s][j]) for this CTA's rows s
      float* hn = part;   // S
      if (vec4) {
        // a warp takes two rows at a time, lanes take 4 columns per load
        for (int s = r0 + warp; s < r1; s += 2 * kOhWarps) {
          const int s1 = s + kOhWarps;
          const bool two = s1 < r1;
          const float* __restrict__ Tr0 = T + (size_t)s * S;
          const float* __restrict__ Tr1 = T + (size_t)(two ? s1 : s) * S;
          const float* __restrict__ Wr0 = W ? W + (size_t)s * S : nullptr;
          const float* __restrict__ Wr1 = W ? W + (size_t)(two ? s1 : s) * S : nullptr;
          float acc0 = init, acc1 = init;
          for (int j = 4 * lane; j < S; j += 256) {
            const bool more = j + 128 < S;
            const float4 a0 = tw4(Tr0, Wr0, j), b0 = tw4(Tr1, Wr1, j);
            const float4 a1 = more ? tw4(Tr0, Wr0, j + 128) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 b1 = more ? tw4(Tr1, Wr1, j + 128) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 hv = *reinterpret_cast<const float4*>(h + j);
            acc0 = dot4<MAXP>(acc0, hv, a0);
            acc1 = dot4<MAXP>(acc1, hv, b0);
            if (more) {
              const float4 hw = *reinterpret_cast<const float4*>(h + j + 128);
              acc0 = dot4<MAXP>(acc0, hw, a1);
              acc1 = dot4<MAXP>(acc1, hw, b1);
            }
          }
          acc0 = MAXP ? warp_max(acc0) : warp_sum(acc0);
          acc1 = MAXP ? warp_max(acc1) : warp_sum(acc1);
          if (lane == 0) {
            hn[s] = acc0;
            if (two) hn[s1] = acc1;
          }
        }
      } else {
        // one warp per row s, lanes along j
        for (int s = r0 + warp; s < r1; s += kOhWarps) {
          const float* __restrict__ Tr = T + (size_t)s * S;
          const float* __restrict__ Wr = W ? W + (size_t)s * S : nullptr;
          float acc = init;
          int j = lane;
          for (; j + 96 < S; j += 128) {
            float t0 = tw(Tr, Wr, j);
            float t1 = tw(Tr, Wr, j + 32);
            float t2 = tw(Tr, Wr, j + 64);
            float t3 = tw(Tr, Wr, j + 96);
            acc = comb<MAXP>(acc, h[j], t0);
            acc = comb<MAXP>(acc, h[j + 32], t1);
            acc = comb<MAXP>(acc, h[j + 64], t2);
            acc = comb<MAXP>(acc, h[j + 96], t3);
          }
          for (; j < S; j += 32) acc = comb<MAXP>(acc, h[j], tw(Tr, Wr, j));
          acc = MAXP ? warp_max(acc) : warp_sum(acc);
          if (lane == 0) hn[s] = acc;
        }
      }
      __syncthreads();
      if (nc == 1) {
        for (int s = tid; s < S; s += kOhThreads) {
          float v = apply_nl(hn[s], a.update_nonlinear);
          if (orow >= 0) out[((size_t)b * a.L + orow) * S + s] = v;
          h[s] = v * o[s];
        }
        __syncthreads();
      } else {
        for (int s = r0 + tid; s < r1; s += kOhThreads) xb[s] = hn[s];      // this CTA's rows are final
        oh_cluster_sync();
        for (int s = tid; s < S; s += kOhThreads) {
          const float raw = oh_ld_remote(xb + s, (uint32_t)min(nc - 1, s / rows_per));
          float v = apply_nl(raw, a.update_nonlinear);
          if (cr == 0 && orow >= 0) out[((size_t)b * a.L + orow) * S + s] = v;
          h[s] = v * o[s];
        }
        __syncthreads();
      }
    }
  }
  if (nc > 1) oh_cluster_sync();      // no CTA may retire while a peer still reads its exchange arrays
}

// Backward of the sum-semiring recurrence for one (sequence, direction): walks the steps in reverse, keeps the
// state gradient in shared memory, scatter-adds dT[x_t] += outer products and propagates g through T[x_t].
//   fwd: pre = (h_prev . T) * o, h = phi(pre):  dacc = G*phi'(h)*o ; dT[s][j] += h_prev[s]*dacc[j] ; g_prev[s] = sum_j T[s][j]*dacc[j]
//   bwd: pre = T . (h_prev*o),   h = phi(pre):  dacc = G*phi'(h)   ; dT[s][j] += dacc[s]*hh[j]     ; g_prev[j] = o[j]*sum_s dacc[s]*T[s][j]
// Under full_pad the backward direction's step n-1 (token 0) produces a state that feeds the pad steps but has no output
// row (step_pos: orow = -1); the forward keeps it in shared memory only, so this kernel recomputes it once (hb).
__global__ void __launch_bounds__(kOhThreads) onehot_backward_kernel(const re2nn_onehot_backward_args a) {
  extern __shared__ float smem[];
  const int S = a.S;
  float* g = smem;            // S   gradient w.r.t. the state produced by the current step
  float* dacc = smem + S;     // S
  float* hprev = smem + 2 * S;  // S   operand of the step (bwd: already * o)
  float* part = smem + 3 * S;   // kOhWarps * S
  float* hb = part + kOhWarps * S;  // S, full_pad only: bwd state after token 0
  const int b = blockIdx.x, z = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = (int)a.lengths[b];
  const float* __restrict__ W = a.W;
  const float* __restrict__ o = a.o;
  const float* states = z == 0 ? a.alpha : a.beta;
  const float* dstates = z == 0 ? a.dalpha : a.dbeta;
  if (z == 1 && a.full_pad && n >= 1) {
    // hb = phi(T[x_0] . (prev*o)), prev = beta row 0 (the state after token 1), or hT when n == 1
    for (int s = tid; s < S; s += kOhThreads) dacc[s] = (n >= 2 ? states[(size_t)b * a.L * S + s] : a.hT[s]) * o[s];
    __syncthreads();
    const float* __restrict__ T = a.language + (size_t)a.x[(size_t)b * a.Lpad] * S * S;
    for (int s = warp; s < S; s += kOhWarps) {
      float acc = 0.f;
      for (int j = lane; j < S; j += 32) acc = fmaf(dacc[j], tw(T, W, (size_t)s * S + j), acc);
      acc = warp_sum(acc);
      if (lane == 0) hb[s] = apply_nl(acc, a.update_nonlinear);
    }
  }
  for (int s = tid; s < S; s += kOhThreads) g[s] = 0.f;
  __syncthreads();
  for (int k = a.L - 1; k >= 0; --k) {
    int tpos, orow;
    bool alive;
    step_pos(z, k, n, a.full_pad, tpos, orow, alive);
    if (!alive) continue;     // block-uniform
    // state before this step: output row of step k-1, or the initial vector
    int tp2, oprev;
    bool al2;
    if (k > 0) step_pos(z, k - 1, n, a.full_pad, tp2, oprev, al2); else oprev = -1;
    const int64_t tok = a.x[(size_t)b * a.Lpad + tpos];
    const float* __restrict__ T = a.language + (size_t)tok * S * S;
    float* __restrict__ dT = a.dlanguage + (size_t)tok * S * S;
    // orow / oprev < 0 only for the state after token 0 of the bwd direction under full_pad: hb, no output gradient
    for (int s = tid; s < S; s += kOhThreads) {
      const float h = orow >= 0 ? states[((size_t)b * a.L + orow) * S + s] : hb[s];
      const float G = orow >= 0 ? g[s] + dstates[((size_t)b * a.L + orow) * S + s] : g[s];
      float d = G * nl_grad_from_out(h, a.update_nonlinear);
      if (z == 0) d *= o[s];
      dacc[s] = d;
      float hp = k == 0 ? (z == 0 ? a.h0[s] : a.hT[s]) : (oprev >= 0 ? states[((size_t)b * a.L + oprev) * S + s] : hb[s]);
      hprev[s] = z == 0 ? hp : hp * o[s];
    }
    __syncthreads();
    if (z == 0) {
      // rows s over warps, columns j over lanes: dT[s][j] += hprev[s]*dacc[j]; g_prev[s] = sum_j (T+W)[s][j]*dacc[j]
      for (int s = warp; s < S; s += kOhWarps) {
        const float hs = hprev[s];
        float acc = 0.f;
        for (int j = lane; j < S; j += 32) {
          const float dj = dacc[j];
          acc = fmaf(tw(T, W, (size_t)s * S + j), dj, acc);
          const float v = hs * dj;
          if (v != 0.f) atomicAdd(dT + (size_t)s * S + j, v);
        }
        acc = warp_sum(acc);
        if (lane == 0) part[s] = acc;
      }
      __syncthreads();
      for (int s = tid; s < S; s += kOhThreads) g[s] = part[s];
      __syncthreads();
    } else {
      // dT[s][j] += dacc[s]*hh[j]; g_prev[j] = o[j] * sum_s dacc[s]*(T+W)[s][j]: warps stride rows, lanes columns
      for (int jb = 0; jb < S; jb += 32) {
        const int j = jb + lane;
        float acc = 0.f;
        if (j < S) {
          const float hj = hprev[j];
          for (int s = warp; s < S; s += kOhWarps) {
            const float ds = dacc[s];
            acc = fmaf(tw(T, W, (size_t)s * S + j), ds, acc);
            const float v = ds * hj;
            if (v != 0.f) atomicAdd(dT + (size_t)s * S + j, v);
          }
          part[warp * S + j] = acc;
        }
      }
      __syncthreads();
      for (int j = tid; j < S; j += kOhThreads) {
        float acc = 0.f;
#pragma unroll
        for (int w = 0; w < kOhWarps; ++w) acc += part[w * S + j];
        g[j] = acc * o[j];
      }
      __syncthreads();
    }
  }
}

}  // namespace re2nn

using namespace re2nn;

extern "C" int re2nn_onehot_sum_tensor(const float* language, const float* W, int V1, int S, float* out, void* stream) {
  RE2NN_CHECK(language && W && out && V1 > 0 && S > 0, "onehot_sum_tensor: bad arguments");
  const size_t total = (size_t)V1 * S * S;
  onehot_sum_kernel<<<sm_count() * 16, 256, 0, (cudaStream_t)stream>>>(language, W, (size_t)S * S, total, out);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

extern "C" int re2nn_onehot_backward(const re2nn_onehot_backward_args* a, void* stream) {
  RE2NN_CHECK(a != nullptr, "onehot_backward: null args");
  RE2NN_CHECK(a->x && a->lengths && a->language && a->o && a->h0 && a->hT && a->alpha && a->beta &&
                  a->dalpha && a->dbeta && a->dlanguage, "onehot_backward: null tensor");
  // S <= 2964; under full_pad one more S-float buffer (the recomputed state after token 0): S <= 2816
  const size_t smem = (size_t)(3 + kOhWarps + (a->full_pad ? 1 : 0)) * a->S * sizeof(float);
  RE2NN_CHECK(smem <= 220 * 1024, "onehot_backward: S=%d too large%s", a->S, a->full_pad ? " under full_pad" : "");
  RE2NN_CUDA(cudaFuncSetAttribute(onehot_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  onehot_backward_kernel<<<dim3(a->B, 2), kOhThreads, smem, (cudaStream_t)stream>>>(*a);
  RE2NN_LAUNCH_CHECK();
  return 0;
}

static int g_onehot_cluster = 0;      // debug: 0 = pick by batch size; 1, 2, 4 = force the cluster size

extern "C" int re2nn_debug_set_onehot_cluster(int nc) {
  RE2NN_CHECK((nc & 7) == 0 || (nc & 7) == 1 || (nc & 7) == 2 || (nc & 7) == 4, "debug_set_onehot_cluster: expected 0, 1, 2 or 4 (+8: four instead of eight rows in flight)");
  g_onehot_cluster = nc;
  return 0;
}

extern "C" int re2nn_onehot_recurrence(const re2nn_onehot_args* a, void* stream) {
  RE2NN_CHECK(a != nullptr, "onehot_recurrence: null args");
  RE2NN_CHECK(a->B > 0 && a->L > 0 && a->S > 0 && a->L <= a->Lpad, "onehot_recurrence: bad dims");
  RE2NN_CHECK(a->x && a->lengths && a->language && a->o && a->h0 && a->hT && a->alpha && a->beta,
              "onehot_recurrence: null tensor");
  RE2NN_CHECK(a->update_nonlinear >= RE2NN_NL_NONE && a->update_nonlinear <= RE2NN_NL_RELUTANH,
              "onehot_recurrence: unsupported update_nonlinear %d", a->update_nonlinear);
  const size_t smem = (size_t)(3 + kOhWarps) * a->S * sizeof(float);
  RE2NN_CHECK(smem <= 220 * 1024, "onehot_recurrence: S=%d too large for the shared-memory state", a->S);
  cudaStream_t st = (cudaStream_t)stream;
  // cluster size: spread a (sequence, direction) slice over 2 / 4 CTAs while the batch alone cannot fill the machine
  int nc = g_onehot_cluster & 7;
  if (nc == 0) {
    // measured (tools/bench_onehot_cluster.py, cfg1 shapes): B = 32: 0.69 ms alone, 0.42 ms on CTA pairs, 0.37-0.53 ms
    // on clusters of four depending on the box; B = 64: pairs = single CTAs; B >= 128: single CTAs win
    nc = 2L * a->B * 2 <= sm_count() ? 2 : 1;
  }
  const int rows8 = (g_onehot_cluster & 8) ? 0 : 1;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(a->B * nc), 2);
  cfg.blockDim = dim3(kOhThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)nc;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (a->max_semiring) {
    static int configured[kMaxDevices];
    RE2NN_CUDA(ensure_dynamic_smem(onehot_recurrence_kernel<true>, (int)smem, configured));
    RE2NN_CUDA(cudaLaunchKernelEx(&cfg, onehot_recurrence_kernel<true>, *a, rows8));
  } else {
    static int configured[kMaxDevices];
    RE2NN_CUDA(ensure_dynamic_smem(onehot_recurrence_kernel<false>, (int)smem, configured));
    RE2NN_CUDA(cudaLaunchKernelEx(&cfg, onehot_recurrence_kernel<false>, *a, rows8));
  }
  RE2NN_LAUNCH_CHECK();
  return 0;
}
