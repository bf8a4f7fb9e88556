// Resident decompose recurrence for inference (farnn = 0 / 1 / 2): ONE launch runs every step of both directions.
//
// The per-step launches of recurrence.cu are bound by what happens BETWEEN the GEMMs, not by the GEMMs: every
// step boundary is a grid-wide dependency (drain the epilogue stores, resolve the launch, refill the operand
// pipeline), although a sequence only ever depends on its own rows.  Here a cluster of two CTAs owns one
// 128-row tile of one direction for the whole recurrence (model_decompose_single.py:236-249 is a loop over
// steps of row-independent updates) and the only synchronisation left is between those two CTAs:
//
//   CTA j of the pair computes column part j of both GEMMs of every step
//     G0:  (farnn >= 1) update gate z = sigma(k (H @ Wss1 + gtab_z)), and for farnn = 2 in a second phase the reset
//          gate r and the blended operand Hbar = (1 - r) h_init + r H [* o]          (EpiGate; z never leaves the CTA)
//     G1:  Q[:, part j of R]  = (Hbar @ S1|S2) * v_t                      (EpiQ)
//     G2:  H'[:, part j of S] = phi((Hbar @ W + Q @ S2^T|S1^T) [* o])      (EpiH: alpha/beta rows + next Hbar operand)
//   through the same TMA -> swizzled smem -> tcgen05.mma -> TMEM -> fused-epilogue pipeline as tc_gemm_kernel.
//   Q and Hbar travel between the two CTAs through L2 (operand-format buffers, read back by TMA); an mbarrier
//   per CTA ("ready", one arrival per epilogue warp of both CTAs, remote arrives over DSMEM) tells the TMA
//   producer when the rows it is about to load have been published.  Weight (B) tiles never wait for that
//   barrier, and G2 starts with its Hbar @ W segment, whose operands are already there while the G1 epilogue
//   is still running.
//
// Pairs never talk to other pairs, so tiles of different length drift apart freely, dead steps
// (k > tile_last) are never executed, and with more tiles than SM pairs a pair simply takes the next tile.
#pragma once
#include "gemm_tc_impl.cuh"

namespace re2nn {

struct __align__(64) ResidentLaunch {
  TcLaunch g1[2], g2[2];     // per ping-pong parity of the Hbar operand; cg = 1, bn = the columns of ONE CTA
  TcLaunch gate;             // farnn >= 1: H @ [Wss1 | Wss2] (N = S * farnn), tiles of the G2 width
  int steps;                 // L
  int stage_bytes, stages;   // pipeline geometry (planes * (A tile 16 KB + widest B tile))
  int q_first;               // G2 segment order: 0 = [Hbar @ W, Q @ S^T] (W overlaps the G1 epilogue), 1 = [Q, W]
  int alias_tbuf;            // epilogue transpose buffers live in the A regions of the pipeline stages (q_first only)
};

constexpr int kResEpiWarps = 12;        // at most three epilogue warps per TMEM lane quarter (shared-memory sizing)
// epilogue warps actually launched: twelve leave 128 registers per thread, enough for the epilogues without gates
// only.  The gate epilogues spill at that budget, and with 225 KB of the SM given to shared memory the spill traffic
// misses L1 on every access, so the gated kernels run 8
__host__ __device__ constexpr int resident_epi_warps(int farnn) { return farnn == 0 ? 12 : 8; }
constexpr int kResThreads = 64 + 32 * kResEpiWarps;
constexpr int kResTbufBytes = kResEpiWarps * kTcTbufWords * 4;
constexpr int kResCtxBytes = kResEpiWarps * kTcCtxWords * 4;
constexpr int kResTbufPerStage = 7;     // 7 x 4608 B fit the 32 KB A region (two planes) of one stage
constexpr uint32_t kResCorrOff = 256;   // TMEM column of the second (residual) accumulator of the fp16 split

template <int PREC, int NL, int FARNN>
__global__ void __launch_bounds__(64 + 32 * resident_epi_warps(FARNN), 1) tc_resident_kernel(const __grid_constant__ ResidentLaunch RL,
                                                                    const StepParams p_in) {
  constexpr bool TF32 = PREC == RE2NN_PREC_TF32X3;
  constexpr int kPlanes = OperandFmt<PREC>::kPlanes;
  constexpr bool SPLIT = kPlanes == 2;
  constexpr bool TWOACC = PREC == RE2NN_PREC_FP16X3;
  constexpr int kpb = 128 / OperandFmt<PREC>::kElemBytes;
  constexpr int kATile = 128 * 128;
  constexpr int EW = resident_epi_warps(FARNN);

  const int crank = (int)cluster_ctarank();
  const int worker = (int)(blockIdx.x >> 1), nworkers = (int)(gridDim.x >> 1);
  const int M = p_in.B, S = p_in.S, R = p_in.R;
  const int m_tiles = (M + 127) / 128, total_tiles = 2 * m_tiles;
  const int stages = RL.stages;
  const uint32_t stage_bytes = (uint32_t)RL.stage_bytes;
  const uint32_t b_off = (uint32_t)(kPlanes * kATile);                    // B tiles follow the A planes
  const uint32_t b_plane = stage_bytes / kPlanes - (uint32_t)kATile;      // bytes of one B plane slot
  const int bn1 = RL.g1[0].bn, bn2 = RL.g2[0].bn;
  unsigned long long* trace = nullptr;
  if (g_tc_trace) trace = g_tc_trace + 32ull * blockIdx.x;
  if (threadIdx.x == 0) tc_stamp(trace, 0);

  extern __shared__ uint8_t smem_raw[];
  // no alignment slack: this kernel has no static shared memory, so the dynamic window starts 1024-aligned
  // (checked; the swizzled TMA / UMMA tiles need it) and every byte of the 227 KB goes to the pipeline
  const uint32_t base = smem_u32(smem_raw);
  if ((base & 1023u) != 0) __trap();
  uint8_t* gen_base = smem_raw;
  const uint32_t stage_region = (uint32_t)stages * stage_bytes;
  const uint32_t bars = base + stage_region;          // full[4], empty[4], tfull, tempty, ready, tmem slot
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (4 + s); };
  const uint32_t tfull_bar = bars + 64, tempty_bar = bars + 72, ready_bar = bars + 80, tmem_slot = bars + 88;
  volatile uint32_t* tmem_slot_p = (volatile uint32_t*)(gen_base + stage_region + 88);
  int* ctx_base = reinterpret_cast<int*>(gen_base + stage_region + 256);
  // Transpose buffers.  With q_first every A-tile load of a phase is issued after the `ready` barrier, i.e. after
  // every epilogue warp of this CTA is done with its buffer, and the next epilogue starts after all MMAs of the
  // phase have read the stages: the buffers can then live in the A regions of the stages (7 per 32 KB region)
  // and the whole 227 KB go to the operand pipeline.
  float* tbuf_base = reinterpret_cast<float*>(gen_base + stage_region + 256 + kResCtxBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int par = 0; par < 2; ++par)
      for (int z = 0; z < 2; ++z) {
        const TcSeg s1 = RL.g1[par].seg[z][0];
        tma_prefetch_desc(&RL.g1[par].maps[s1.a_map]);
        tma_prefetch_desc(&RL.g1[par].maps[s1.b_map]);
        for (int s = 0; s < 2; ++s) {
          const TcSeg s2 = RL.g2[par].seg[z][s];
          tma_prefetch_desc(&RL.g2[par].maps[s2.a_map]);
          tma_prefetch_desc(&RL.g2[par].maps[s2.b_map]);
        }
      }
    if (FARNN >= 1)
      for (int z = 0; z < 2; ++z) {
        tma_prefetch_desc(&RL.gate.maps[RL.gate.seg[z][0].a_map]);
        tma_prefetch_desc(&RL.gate.maps[RL.gate.seg[z][0].b_map]);
      }
    for (int s = 0; s < 4; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tfull_bar, 1);
    mbar_init(tempty_bar, EW);
    mbar_init(ready_bar, 2 * EW);       // the epilogue warps of both CTAs
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  cluster_sync_all();     // the peer's ready barrier must exist before anything arrives on it
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_p;
  if (threadIdx.x == 0) tc_stamp(trace, 2);

  // steps this tile runs: rows past their length are never observed (tile_last: last step any row is alive)
  auto nsteps = [&](int z, int mt) -> int {
    if (p_in.full_pad) return RL.steps;
    return min(RL.steps, __ldg(p_in.tile_last[z] + mt) + 1);
  };

  if (warp == 0) {
    // ---- TMA producer ------------------------------------------------------------------------------------
    int it = 0;
    uint32_t rdy = 0;
    bool first = true;
    // one segment of one GEMM: nkb k-blocks of A (128 rows at m0) and B (bn rows at n0)
    auto load_segment = [&](const TcLaunch& T, const TcSeg sg, int m0, int n0, int bn, bool wait_ready, int tslot) {
      const uint32_t bytes = (uint32_t)(kPlanes * (kATile + bn * 128));
      const int nkb = sg.kblocks;
      const int npre = wait_ready ? min(stages, nkb) : 0;
      auto issue_b = [&](int kb, int st, uint32_t ph) {
        mbar_wait(empty_bar(st), ph ^ 1);
        mbar_expect_tx(full_bar(st), bytes);
        const uint32_t sa = base + (uint32_t)st * stage_bytes;
        tma_load_2d(sa + b_off, &T.maps[sg.b_map], full_bar(st), kb * kpb, n0);
        if (SPLIT) tma_load_2d(sa + b_off + b_plane, &T.maps[sg.b_lo], full_bar(st), kb * kpb, n0);
      };
      // weight tiles do not depend on the other CTA: put them in flight before waiting for the rows
      for (int kb = 0; kb < npre; ++kb) issue_b(kb, (it + kb) % stages, (uint32_t)((it + kb) / stages) & 1u);
      if (wait_ready) {
        if (tslot >= 0) tc_stamp(trace, tslot);
        mbar_wait_cluster(ready_bar, rdy & 1u);
        if (tslot >= 0) tc_stamp(trace, tslot + 1);
        ++rdy;
        fence_proxy_async();       // the rows were written through the generic proxy, TMA reads through the async proxy
      }
      for (int kb = 0; kb < nkb; ++kb) {
        const int st = (it + kb) % stages;
        if (kb >= npre) issue_b(kb, st, (uint32_t)((it + kb) / stages) & 1u);
        const uint32_t sa = base + (uint32_t)st * stage_bytes;
        tma_load_2d(sa, &T.maps[sg.a_map], full_bar(st), kb * kpb, m0);
        if (SPLIT) tma_load_2d(sa + kATile, &T.maps[sg.a_lo], full_bar(st), kb * kpb, m0);
      }
      it += nkb;
    };
    for (int tile = worker; tile < total_tiles; tile += nworkers) {
      const int z = tile / m_tiles, mt = tile - z * m_tiles;
      const int ns = nsteps(z, mt);
      const int m0 = mt * 128;
      if (lane == 0) {
        for (int k = 0; k < ns; ++k) {
          const int par = k & 1;
          // every phase waits for the rows published by the previous phase (nothing to wait for at the very start)
          if (FARNN >= 1) {      // G0: A = H (operand format), z columns [0,S), then r columns [S,2S) of [Wss1 | Wss2]
            load_segment(RL.gate, RL.gate.seg[z][0], m0, crank * bn2, bn2, !first, -1);
            first = false;
            if (FARNN == 2) load_segment(RL.gate, RL.gate.seg[z][0], m0, S + crank * bn2, bn2, true, -1);
          }
          // G1: A = Hbar[par], published by the previous phase (or rec_init_kernel for the first)
          const bool tr = tile == worker && (k == 2 || k == 3);     // debug trace: one steady-state step
          const int tb = k == 2 ? 8 : 26;
          load_segment(RL.g1[par], RL.g1[par].seg[z][0], m0, crank * bn1, bn1, !first, tr ? tb : -1);
          if (tr && k == 2) tc_stamp(trace, 10);
          first = false;
          // G2: the Hbar[par] @ W segment has everything visible already; the Q @ S2^T|S1^T segment waits for
          // this step's G1 epilogues of both CTAs
          load_segment(RL.g2[par], RL.g2[par].seg[z][0], m0, crank * bn2, bn2, RL.q_first != 0, tr && k == 2 && RL.q_first ? 11 : -1);
          load_segment(RL.g2[par], RL.g2[par].seg[z][1], m0, crank * bn2, bn2, RL.q_first == 0, tr && k == 2 && !RL.q_first ? 11 : -1);
          if (tr && k == 2) tc_stamp(trace, 13);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---- MMA issuer ----------------------------------------------------------------------------------------
    const uint32_t fmt = TF32 ? 2u : (PREC == RE2NN_PREC_FP16X3 ? 0u : 1u);
    int it = 0;
    uint32_t acc = 0;
    auto mma_gemm = [&](int nkb, int bn, int tslot) {
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(bn >> 3) << 17) | ((128u >> 4) << 24);
      mbar_wait(tempty_bar, (acc & 1u) ^ 1u);     // the epilogue warps have drained the accumulator
      tc_fence_after();
      for (int j = 0; j < nkb; ++j, ++it) {
        const int st = it % stages;
        mbar_wait(full_bar(st), (uint32_t)(it / stages) & 1u);
        if (tslot >= 0 && j == 0) tc_stamp(trace, tslot);
        tc_fence_after();
        const uint32_t sa = base + (uint32_t)st * stage_bytes;
        const uint64_t da = make_smem_desc(sa), db = make_smem_desc(sa + b_off);
#pragma unroll
        for (int k = 0; k < 4; ++k) tc_mma<TF32>(tmem_base, da + 2u * k, db + 2u * k, idesc, (j | k) != 0 ? 1u : 0u);
        if (SPLIT) {
          const uint64_t dal = make_smem_desc(sa + kATile), dbl = make_smem_desc(sa + b_off + b_plane);
          const uint32_t acc_lo = TWOACC ? tmem_base + kResCorrOff : tmem_base;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            tc_mma<TF32>(acc_lo, dal + 2u * k, db + 2u * k, idesc, TWOACC ? ((j | k) != 0 ? 1u : 0u) : 1u);
            tc_mma<TF32>(acc_lo, da + 2u * k, dbl + 2u * k, idesc, 1u);
          }
        }
        tc_commit(empty_bar(st));
      }
      tc_commit(tfull_bar);
      if (tslot >= 0) tc_stamp(trace, tslot + 1);
      ++acc;
    };
    for (int tile = worker; tile < total_tiles; tile += nworkers) {
      const int z = tile / m_tiles, mt = tile - z * m_tiles;
      const int ns = nsteps(z, mt);
      if (lane == 0) {
        const int kb1 = RL.g1[0].seg[z][0].kblocks;
        const int kb2 = RL.g2[0].seg[z][0].kblocks + RL.g2[0].seg[z][1].kblocks;
        for (int k = 0; k < ns; ++k) {
          const bool tr = tile == worker && k == 2;
          if (FARNN >= 1) mma_gemm(RL.gate.seg[z][0].kblocks, bn2, -1);
          if (FARNN == 2) mma_gemm(RL.gate.seg[z][0].kblocks, bn2, -1);
          mma_gemm(kb1, bn1, tr ? 14 : -1);
          mma_gemm(kb2, bn2, tr ? 16 : -1);
        }
      }
      __syncwarp();
    }
  } else {
    // ---- epilogue warps: warp w may touch TMEM lanes 32*(w%4) .. +31 ------------------------------------------
    const int q = warp & 3, ew = warp - 2, half = ew >> 2;
    float* tbuf = RL.alias_tbuf ? reinterpret_cast<float*>(gen_base + (size_t)(ew / kResTbufPerStage) * stage_bytes) +
                                      (ew % kResTbufPerStage) * kTcTbufWords
                                : tbuf_base + ew * kTcTbufWords;
    int* ctx = ctx_base + ew * kTcCtxWords;
    const uint32_t tmem_rows = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t ready_mine = mapa_shared(ready_bar, (uint32_t)crank), ready_peer = mapa_shared(ready_bar, (uint32_t)(crank ^ 1));
    uint32_t acc = 0;
    // hand the accumulator back to the MMA warp, then publish this warp's rows to both TMA producers
    auto release_and_publish = [&]() {
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tempty_bar) : "memory");
        asm volatile("fence.acq_rel.cluster;" ::: "memory");      // one release for both arrives
        asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(ready_mine) : "memory");
        asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(ready_peer) : "memory");
      }
      ++acc;
    };
    for (int tile = worker; tile < total_tiles; tile += nworkers) {
      const int z = tile / m_tiles, mt = tile - z * m_tiles;
      const int ns = nsteps(z, mt);
      const int mrow0 = mt * 128 + q * 32;
      StepParams ps = p_in;
      void* hbar0;      // host: Hbar_cur = parity-0 buffer, Hbar_next = parity-1 buffer
      void* hbar1;
      if constexpr (EW == 12) {      // see StepParams::bind / bind_const
        hbar0 = p_in.Hbar_cur[z];
        hbar1 = p_in.Hbar_next[z];
        ps.bind(z);
      } else {
        hbar0 = z ? p_in.Hbar_cur[1] : p_in.Hbar_cur[0];
        hbar1 = z ? p_in.Hbar_next[1] : p_in.Hbar_next[0];
        ps.bind_const(z);
      }
      for (int k = 0; k < ns; ++k) {
        ps.k = k;
        ps.Hbar_cur[0] = (k & 1) ? hbar1 : hbar0;
        ps.Hbar_next[0] = (k & 1) ? hbar0 : hbar1;
        const EpiQ<PREC> e1{ps};
        {
          RowCtx mine{0, -1, false};
          if (mrow0 + lane < M) mine = e1.row(mrow0 + lane);
          ctx[lane] = mine.vrow;
          ctx[32 + lane] = mine.orow;
        }
        __syncwarp();
        const bool tr = tile == worker && k == 2 && ew == 0 && lane == 0;
        if constexpr (FARNN >= 1) {
          const EpiGate<PREC> eg{ps};
          tc_epilogue_chunks<TWOACC, EW / 4>(eg, M, S, mrow0, crank * bn2, bn2, tmem_rows, kResCorrOff, half, lane,
                                                       tbuf, ctx, tfull_bar, acc & 1u, nullptr);
          release_and_publish();
          if (FARNN == 2) {
            tc_epilogue_chunks<TWOACC, EW / 4>(eg, M, 2 * S, mrow0, S + crank * bn2, bn2, tmem_rows, kResCorrOff,
                                                         half, lane, tbuf, ctx, tfull_bar, acc & 1u, nullptr);
            release_and_publish();
          }
        }
        if constexpr (EpiHasRows<EpiQ<PREC>>::value)
          tc_epilogue_quads<TWOACC, EW / 4>(e1, M, R, mrow0, crank * bn1, bn1, tmem_rows, kResCorrOff, half, lane, tbuf, ctx,
                                            tfull_bar, acc & 1u);
        else
          tc_epilogue_chunks<TWOACC, EW / 4>(e1, M, R, mrow0, crank * bn1, bn1, tmem_rows, kResCorrOff, half, lane, tbuf, ctx,
                                             tfull_bar, acc & 1u, nullptr);
        if (tr) tc_stamp(trace, 18);
        release_and_publish();
        const EpiH<PREC, NL, FARNN> e2{ps};
        if constexpr (EpiHasRows<EpiH<PREC, NL, FARNN>>::value)
          tc_epilogue_quads<TWOACC, EW / 4>(e2, M, S, mrow0, crank * bn2, bn2, tmem_rows, kResCorrOff, half, lane, tbuf, ctx,
                                            tfull_bar, acc & 1u, tr ? trace : nullptr);
        else
          tc_epilogue_chunks<TWOACC, EW / 4>(e2, M, S, mrow0, crank * bn2, bn2, tmem_rows, kResCorrOff, half, lane, tbuf, ctx,
                                             tfull_bar, acc & 1u, tr ? trace : nullptr);
        if (tr) tc_stamp(trace, 19);
        release_and_publish();
        if (tr) tc_stamp(trace, 30);
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();     // the peer may still arrive on this CTA's barriers until it is done as well
  if (threadIdx.x == 0) tc_stamp(trace, 7);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

inline int resident_part(int n) { return ((cdiv(n, 2) + 15) / 16) * 16; }      // columns of one CTA of the pair
inline int resident_stage_bytes(int planes, int S, int R) {
  return planes * (128 * 128 + std::max(resident_part(S), resident_part(R)) * 128);
}
// transpose buffers inside the stages: needs the [Q, W] order (see the kernel) and two-plane A regions
inline bool resident_alias(int planes, bool q_first) { return q_first && planes == 2; }
inline int resident_stages(int planes, int S, int R, bool q_first) {
  const int fixed = 256 + kResCtxBytes + (resident_alias(planes, q_first) ? 0 : kResTbufBytes);
  return std::min(4, (kTcSmemLimit - fixed) / resident_stage_bytes(planes, S, R));
}
inline int resident_smem_bytes(int planes, int stages, int stage_bytes, bool q_first) {
  return stages * stage_bytes + 256 + kResCtxBytes + (resident_alias(planes, q_first) ? 0 : kResTbufBytes);
}
// Can the resident kernel run this problem?  Each CTA of a pair takes half of R and half of S as ONE MMA tile
// and needs a two-stage operand pipeline (and, when aliased, room for all transpose buffers in the A regions).
inline bool resident_supported(int planes, int S, int R, bool q_first) {
  const int st = resident_stages(planes, S, R, q_first);
  if (resident_alias(planes, q_first) && st * kResTbufPerStage < kResEpiWarps) return false;
  return resident_part(S) <= 256 && resident_part(R) <= 256 && st >= 2;
}

template <int PREC, int NL, int FARNN>
inline cudaError_t launch_resident(const ResidentLaunch& RL, const StepParams& p, int B, cudaStream_t st) {
  const int smem = resident_smem_bytes(OperandFmt<PREC>::kPlanes, RL.stages, RL.stage_bytes, RL.q_first != 0);
  static int configured[kMaxDevices];
  if (cudaError_t e = ensure_dynamic_smem(tc_resident_kernel<PREC, NL, FARNN>, smem, configured)) return e;
  const long tiles = 2L * cdiv(B, 128);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(std::min<long>(tiles, sm_count() / 2) * 2));   // one CTA pair per SM pair
  cfg.blockDim = dim3(64 + 32 * resident_epi_warps(FARNN));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, tc_resident_kernel<PREC, NL, FARNN>, RL, p);
}

}  // namespace re2nn
