// Weight-gradient ("TN") GEMM on tcgen05 in 3xTF32:  C[P x Q] = sum over pairs, rows m:  X[m, p] * Y[m, q].
//
// Both operands are row-major slabs whose ROWS are the reduction index (every (step, sequence) row of the BPTT
// sweep), i.e. M/N-major for the tensor core.  Instead of MN-major descriptors the loader warps transpose on the
// fly: they read 32 slab rows (coalesced, 128 B per warp request), split every value into its tf32 hi / lo parts and
// write 16-byte pieces (four consecutive reduction indices of one output row / column) straight into the K-major
// SWIZZLE_128B tile layout the MMA descriptors expect (the same layout TMA produces for the step GEMMs).  One
// elected thread issues hi*hi into the main accumulator and lo*hi + hi*lo into a second one (the cross terms are
// 2^-11 smaller, so the truncating TMEM accumulation sees a chain of K/8 additions instead of 3K/8 on the main sum).
// Split-K over the grid's z dimension, partials reduced in a fixed order by split_reduce_kernel: deterministic.
//
// Replaces the CUDA-core tn_gemm_kernel (backward.cu) where the reduction is long: at cfg3 the three weight
// gradients are 30 GFLOP, 1.05 ms on CUDA cores (20 % of the training step).
#pragma once
#include "gemm_tc_impl.cuh"

namespace re2nn {

struct TnPair { const float* X; const float* Y; int ldx, ldy; size_t rows; };
// Y2 (optional, single pair): the right operand is Y * Y2 element-wise (same layout as pair 0's Y), and with mask_len
// row m = b * mask_L + t only counts when t < mask_len[b] -- dC = draw^T (alpha * beta) over the valid positions
// without materialising the product (pad rows of alpha / beta are undefined, possibly NaN).  Both kernels form it.
struct TnProblem { int P, Q, npairs; TnPair pair[2]; const float* Y2; const int64_t* mask_len; int mask_L; };

constexpr int kTnLoaderWarps = 8;
// eight warps, all loaders (two per scheduler: 255 registers each -- a ninth warp for the MMAs capped everybody at 168
// and the two k-blocks of values a thread holds spilled); lane 0 of warp 0 also issues the MMAs, one k-block late, so
// it never waits for the other warps; warps 0..3 drain TMEM at the end
constexpr int kTnThreads = 32 * kTnLoaderWarps;
constexpr int kTnKBlock = 32;                                 // reduction rows per pipeline stage: 128 bytes of tf32
// k-blocks one split accumulates at most (1536 rows).  The TMEM accumulator truncates every add, so a split's error grows
// with its chain, fastest on same-sign data where every truncation pulls the same way.  Measured on a B200 (max-norm
// relative vs float64, uniform [0, 1) operands): 128 k-blocks per split 2.5-2.8e-5, a whole 2240-k-block reduction in
// one split 5.3e-4; signed data about a third of that.  48 keeps every product within the 2e-5 gradient bound of
// DESIGN.md section 2 and leaves every plan of the benchmarked cfg3 training step alone (its longest chain, dS1 / dS2,
// is 46 k-blocks).  tn_tc_plan adds splits and run_tn reduces longer products in consecutive chunks so that no split
// exceeds the cap.
constexpr int kTnMaxKb = 48;

// rows of pair `pr` that split `split` of `nsplit` reduces: whole k-blocks, so only a pair's last chunk has a ragged end
__host__ __device__ inline void tn_split_range(size_t rows, int split, int nsplit, size_t* r0, size_t* r1) {
  const size_t kb = (rows + kTnKBlock - 1) / kTnKBlock;
  const size_t per = (kb + nsplit - 1) / nsplit;
  const size_t a = per * split * kTnKBlock, b = a + per * kTnKBlock;
  *r0 = a < rows ? a : rows;
  *r1 = b < rows ? b : rows;
}

__global__ void __launch_bounds__(kTnThreads, 1) tn_tc_kernel(const TnProblem prob, float* __restrict__ partial, const int bn,
                                                              const int stages) {
  constexpr int kATile = 128 * 128;                          // one plane of the X^T tile: 128 output rows x 128 bytes
  const int b_tile = bn * 128;
  const uint32_t stage_bytes = 2u * (uint32_t)(kATile + b_tile);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = smem_u32(smem_raw);
  if ((base & 1023u) != 0) __trap();
  const uint32_t bars = base + (uint32_t)stages * stage_bytes;      // full[4], empty[4], done, tmem slot
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (4 + s); };
  const uint32_t done_bar = bars + 64, tmem_slot = bars + 72;
  volatile uint32_t* tmem_slot_p = (volatile uint32_t*)(smem_raw + (size_t)stages * stage_bytes + 72);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p0 = blockIdx.x * 128, q0 = blockIdx.y * bn, split = blockIdx.z, nsplit = gridDim.z;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < 4; ++s) {
      mbar_init(full_bar(s), kTnLoaderWarps);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(done_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_p;

  // k-blocks this CTA reduces (same count in every role)
  int nkb_total = 0;
  for (int pi = 0; pi < prob.npairs; ++pi) {
    size_t r0, r1;
    tn_split_range(prob.pair[pi].rows, split, nsplit, &r0, &r1);
    nkb_total += (int)((r1 - r0 + kTnKBlock - 1) / kTnKBlock);
  }

  // ---- MMAs of k-block `j` (lane 0 of warp 0) -----------------------------------------------------------------------
  const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(bn >> 3) << 17) | ((128u >> 4) << 24);
  auto issue_mma = [&](int j) {
    const int st = j % stages;
    mbar_wait(full_bar(st), (uint32_t)(j / stages) & 1u);
    tc_fence_after();
    const uint32_t acc_main = tmem_base, acc_cross = tmem_base + 256u;
    const uint32_t sa = base + (uint32_t)st * stage_bytes;
    const uint64_t dah = make_smem_desc(sa), dal = make_smem_desc(sa + kATile);
    const uint64_t dbh = make_smem_desc(sa + 2 * kATile), dbl = make_smem_desc(sa + 2 * kATile + b_tile);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t more = (j | k) != 0 ? 1u : 0u;
      tc_mma<true>(acc_main, dah + 2u * k, dbh + 2u * k, idesc, more);
      tc_mma<true>(acc_cross, dal + 2u * k, dbh + 2u * k, idesc, more);
      tc_mma<true>(acc_cross, dah + 2u * k, dbl + 2u * k, idesc, 1u);
    }
    tc_commit(empty_bar(st));
  };
  const bool issuer = warp == 0 && lane == 0;
  {
    // ---- loaders: slab rows -> tf32 hi / lo planes, transposed into the K-major swizzled tiles -----------------
    // a unit = (output row / column c, group kq of four consecutive reduction rows) -> one 16-byte piece per plane;
    // lanes walk c, so every global request is a contiguous row segment.  A thread owns the same 4 + up to 8 units in
    // every k-block: their global offsets and shared-memory offsets are computed once per pair (the first version
    // redid the index math per load and was instruction-bound: 2000 instructions per warp and k-block).  All loads of
    // a k-block are issued before the first value is used, and the loads of the NEXT k-block before this one is
    // converted: a warp always has a k-block of HBM requests in flight while it splits and stores.
    const int tl = threadIdx.x;                            // 0 .. 255
    constexpr int kYU = 8;                                 // Y units per thread: bn * 8 / 256 <= 8
    struct Blk { float x[4][4]; float y[kYU][4]; };
    // tf32 split with integer rounding (add half an ulp of the 10-bit mantissa, clear the 13 low bits): two instructions
    // per part where cvt.rna.tf32 expands to a dozen; same round-to-nearest result for finite values
    auto tf32r = [](float v) { return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u); };
    auto put = [&](uint8_t* tile, int tile_bytes, uint32_t off, const float (&v)[4]) {
      const float4 h = make_float4(tf32r(v[0]), tf32r(v[1]), tf32r(v[2]), tf32r(v[3]));
      const float4 l = make_float4(tf32r(v[0] - h.x), tf32r(v[1] - h.y), tf32r(v[2] - h.z), tf32r(v[3] - h.w));
      *reinterpret_cast<float4*>(tile + off) = h;
      *reinterpret_cast<float4*>(tile + tile_bytes + off) = l;
    };
    int it = 0;
    for (int pi = 0; pi < prob.npairs; ++pi) {
      const TnPair pr = pi == 0 ? prob.pair[0] : prob.pair[1];
      size_t r0, r1;
      tn_split_range(pr.rows, split, nsplit, &r0, &r1);
      if (r0 >= r1) continue;
      // Per unit: a running pointer to its first element of the current k-block and its shared-memory offset (low
      // bits: kq).  Columns past P / Q read the last valid column instead of being predicated off: they only feed
      // accumulator rows / columns that are never written out.
      const float* px[4];
      const float* py[kYU];
      uint32_t xs[4], ys[kYU];
      uint32_t yact = 0;
      const size_t ldx = pr.ldx, ldy = pr.ldy;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int u = tl + 256 * j, c = u & 127, kq = u >> 7;
        px[j] = pr.X + (r0 + 4 * kq) * ldx + min(p0 + c, prob.P - 1);
        xs[j] = ((uint32_t)c * 128u + (uint32_t)((kq ^ (c & 7)) << 4)) | (uint32_t)kq;
      }
#pragma unroll
      for (int j = 0; j < kYU; ++j) {
        const int u = min(tl + 256 * j, bn * 8 - 1);       // inactive units alias the last one (loads stay in bounds)
        const int kq = u / bn, c = u - kq * bn;
        py[j] = pr.Y + (r0 + 4 * kq) * ldy + min(q0 + c, prob.Q - 1);
        ys[j] = ((uint32_t)c * 128u + (uint32_t)((kq ^ (c & 7)) << 4)) | (uint32_t)kq;
        if (tl + 256 * j < bn * 8) yact |= 1u << j;        // warp-uniform: bn * 8 is a multiple of 128
      }
      // loads of the k-block the pointers stand on, then advance them
      const ptrdiff_t y2off = prob.Y2 != nullptr ? prob.Y2 - pr.Y : 0;
      auto load_blk = [&](Blk& b, size_t m0) {
        uint32_t rowmask = 0xffffffffu;                    // bit r: row m0 + r counts (every warp works it out for itself)
        if (prob.mask_len != nullptr) {
          const size_t m = m0 + lane;
          const size_t bb = m / (size_t)prob.mask_L;
          const bool ok = m < pr.rows && (int)(m - bb * prob.mask_L) < (int)__ldg(prob.mask_len + bb);
          rowmask = __ballot_sync(0xffffffffu, ok);
        }
        if (m0 + kTnKBlock <= r1) {                        // whole k-block (all but a pair's last one): no row checks
#pragma unroll
          for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int i = 0; i < 4; ++i) b.x[j][i] = __ldg(px[j] + i * ldx);
            px[j] += kTnKBlock * ldx;
          }
#pragma unroll
          for (int j = 0; j < kYU; ++j) {
            if (yact >> j & 1u) {
#pragma unroll
              for (int i = 0; i < 4; ++i) b.y[j][i] = __ldg(py[j] + i * ldy);
              if (y2off != 0) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const float w = __ldg(py[j] + y2off + i * ldy);
                  b.y[j][i] = (rowmask >> (4 * (ys[j] & 7u) + i) & 1u) ? b.y[j][i] * w : 0.f;
                }
              }
            }
            py[j] += kTnKBlock * ldy;
          }
        } else {
          const int left = (int)(r1 - m0);
#pragma unroll
          for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) b.x[j][i] = 4 * (int)(xs[j] & 7u) + i < left ? __ldg(px[j] + i * ldx) : 0.f;
#pragma unroll
          for (int j = 0; j < kYU; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i)
              b.y[j][i] = ((yact >> j & 1u) && 4 * (int)(ys[j] & 7u) + i < left)
                              ? ((rowmask >> (4 * (ys[j] & 7u) + i) & 1u)
                                     ? __ldg(py[j] + i * ldy) * (y2off != 0 ? __ldg(py[j] + y2off + i * ldy) : 1.f)
                                     : 0.f)
                              : 0.f;
        }
      };
      auto store_blk = [&](const Blk& b, uint8_t* sa) {
#pragma unroll
        for (int j = 0; j < 4; ++j) put(sa, kATile, xs[j] & ~15u, b.x[j]);
#pragma unroll
        for (int j = 0; j < kYU; ++j)
          if (yact >> j & 1u) put(sa + 2 * kATile, b_tile, ys[j] & ~15u, b.y[j]);
      };
      Blk cur, nxt;
      load_blk(cur, r0);
      for (size_t m0 = r0; m0 < r1; m0 += kTnKBlock, ++it) {
        const bool more = m0 + kTnKBlock < r1;
        if (more) load_blk(nxt, m0 + kTnKBlock);           // next k-block's loads in flight before this one is used
        // the previous k-block's MMAs go out now, so they run while this one is split and stored into the other stage
        // (issued after the store they left the tensor pipe idle for a whole store phase: 27 % of the warp samples sat
        // on the `empty` barrier)
        if (issuer && it >= 1) issue_mma(it - 1);
        const int st = it % stages;
        mbar_wait(empty_bar(st), ((uint32_t)(it / stages) & 1u) ^ 1u);
        store_blk(cur, smem_raw + (size_t)st * stage_bytes);
        // generic-proxy writes -> visible to the tensor core's (async proxy) reads.  Shared memory only: the unqualified
        // fence would also wait for the next k-block's global loads, which are in flight on purpose
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(full_bar(st)) : "memory");
        if (more) cur = nxt;
      }
    }
    if (issuer && nkb_total > 0) {
      issue_mma(nkb_total - 1);
      tc_commit(done_bar);
    }
    __syncwarp();
    // ---- drain: warps 0..3 own TMEM lane quarters 0..3 --------------------------------------------------------------
    if (warp < 4) {
      const int q = warp & 3;
      const int p = p0 + q * 32 + lane;
      float* out = partial + ((size_t)split * prob.P + (size_t)min(p, prob.P - 1)) * prob.Q;
      if (nkb_total > 0) {
        mbar_wait(done_bar, 0);
        tc_fence_after();
      }
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
      for (int c0 = 0; c0 < bn; c0 += 32) {
        uint32_t a[32], b[32];
        if (nkb_total > 0) {
          tmem_ld32(trow + (uint32_t)c0, a);
          tmem_ld32(trow + 256u + (uint32_t)c0, b);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) a[j] = b[j] = 0u;
        }
        if (p < prob.P) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int qq = q0 + c0 + j;
            if (c0 + j < bn && qq < prob.Q) out[qq] = __uint_as_float(a[j]) + __uint_as_float(b[j]);
          }
        }
      }
      tc_fence_before();
    }
  }
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// k-blocks the busiest split reduces when the problem is cut into `nsplit` splits (tn_split_range, summed over the pairs)
inline size_t tn_chain_kb(const TnProblem& prob, int nsplit) {
  size_t kb = 0;
  for (int pi = 0; pi < prob.npairs; ++pi) {
    const size_t k = (prob.pair[pi].rows + kTnKBlock - 1) / kTnKBlock;
    kb += (k + nsplit - 1) / nsplit;
  }
  return kb;
}

// tile width over Q, split count and pipeline depth of one problem: one split per SM the tiles leave free, more when a
// split would otherwise accumulate more than kTnMaxKb k-blocks (up to max_split)
struct TnTcPlan { int bn, nt, nsplit, stages, smem; };
static_assert(2 * 2 * (128 * 128 + 256 * 128) + 256 <= kTcSmemLimit, "tn_tc_kernel needs two pipeline stages at bn = 256");
inline TnTcPlan tn_tc_plan(const TnProblem& prob, int max_split) {
  TnTcPlan pl;
  pl.nt = cdiv(prob.Q, 256);
  pl.bn = ((cdiv(prob.Q, pl.nt) + 15) / 16) * 16;
  const int tiles = cdiv(prob.P, 128) * pl.nt;
  pl.nsplit = std::max(1, std::min(max_split, sm_count() / tiles));
  while (pl.nsplit < max_split && tn_chain_kb(prob, pl.nsplit) > (size_t)kTnMaxKb) ++pl.nsplit;
  const int stage_bytes = 2 * (128 * 128 + pl.bn * 128);
  pl.stages = std::min(4, (kTcSmemLimit - 256) / stage_bytes);
  pl.smem = pl.stages * stage_bytes + 256;
  return pl;
}

inline cudaError_t launch_tn_tc(const TnProblem& prob, float* partial, const TnTcPlan& pl, cudaStream_t st) {
  static int configured[kMaxDevices];
  if (cudaError_t e = ensure_dynamic_smem(tn_tc_kernel, pl.smem, configured)) return e;
  dim3 grid(cdiv(prob.P, 128), pl.nt, pl.nsplit);
  tn_tc_kernel<<<grid, kTnThreads, pl.smem, st>>>(prob, partial, pl.bn, pl.stages);
  return cudaGetLastError();
}

}  // namespace re2nn
