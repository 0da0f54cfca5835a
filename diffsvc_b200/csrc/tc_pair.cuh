// tcgen05 cta_group::2 main loop for the WaveNet contractions: a CTA PAIR (two SMs of one TPC, a 2-CTA cluster
// along the frame axis) computes a 256-frame x BN-channel tile with M = 256 MMAs issued by the even CTA.
//
// Why (DESIGN.md 3.1): the single-CTA main loop is bound by shared-memory bandwidth (TMA fill + SS-mode operand
// fetch ~ 130 B/clk/SM), not by the tensor pipe.  In a pair each SM stages and feeds only HALF of the weight
// (B) tile -- the hardware shares B between the two tensor cores -- while the activation (A) tile stays private.
//
// 3-pass error-compensated product x*w ~= xh*wh + xh*wl + xl*wh with TWO MMAs per K-step and NO duplicated
// weight rows.  The tile's BN output channels are split in halves a | b (h = BN/2 rows each; for the gated conv
// a = the gate rows, b = the filter rows of the tile).  Per stage each CTA holds ONE weight block P of BN rows:
//
//     even CTA:  P = [ wh_a ; wl_b ]          odd CTA:  P = [ wh_b ; wl_a ]
//
//   MMA 1  A = xh, B = P       (N = 2*BN: BN rows from each CTA)  -> accumulator column blocks (h wide)
//                                                                     [ xh*wh_a | xh*wl_b | xh*wh_b | xh*wl_a ]
//   MMA 2  A = xl, B = P[0:h]  (N = BN:   h rows from each CTA)   -> blocks 0, 1  += [ xl*wh_a | xl*wh_b ]
//
//   channel j <  h :  D[j] + D[3h + j]   = (xh*wh_a + xl*wh_a) + xh*wl_a
//   channel j >= h :  D[j] + D[j + h]    = (xh*wl_b + xl*wh_b) + xh*wh_b
//
// Per K-stage and SM at BN = 64: TMA 32 KB (A hi, lo) + 8 KB (P) and operand reads 32 + 8 + 4 KB = 84 KB, against
// 104 KB in the single-CTA kernel.  Same three products per channel; the b half adds them in another order
// (results equal to fp32 rounding, not bit-identical, to the single-CTA kernels).
//
// BN = 256 (large batches): [wh ; wl] concatenated would be N = 512 > the 256-column MMA limit, so the pair runs the
// single-CTA tile's three N = 256 MMAs (xh*wh, xh*wl into a second accumulator, xl*wh) with each CTA holding the hi and
// lo rows of ITS half of the tile: 160 KB of shared-memory traffic per stage against 224 KB -- the loop becomes
// tensor-bound (1536 MMA cycles per stage) -- and the results are bit-identical to the single-CTA 256-wide tile.
//
// Barriers: full[s] lives in the EVEN CTA (both CTAs' TMA loads complete_tx on it: cta_group::2 loads addressed
// through mapa), empty[s] and the accumulator-ready barrier exist in both CTAs and are signalled by multicast
// tcgen05.commit.  Everything else (PDL, epilogue, tensor maps) is shared with tc_gemm.cuh.
#pragma once
#include "tc_gemm.cuh"

namespace dsvc {

template <int BN> struct TcPairCfg {
  static constexpr int H = BN / 2;
  static constexpr int P_TILE = BN * TC_BK * 2;              // BN rows x 128 B
  static constexpr int STAGE = 2 * TC_A_TILE + P_TILE;       // A_hi, A_lo, P
  static constexpr int STAGES = (BN == 64) ? 5 : (BN == 128 ? 4 : 3);   // 200 / 192 / 192 KB of operands in flight
  static constexpr int SMEM = STAGES * STAGE + 1024 /*align*/ + 256 /*barriers*/;
  static_assert(4 * 32 * (BN + 4) * 4 <= STAGES * STAGE, "epilogue staging must fit in the operand ring");
};

__device__ __forceinline__ uint32_t mapa_cluster(uint32_t local_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta_rank));
  return r;
}
// cta_group::2 tile loads: data into THIS CTA's shared memory, bytes counted on `bar` (a shared::cluster address,
// the even CTA's full barrier)
__device__ __forceinline__ void tma2_load_2d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma2_load_3d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on the barrier at this CTA-relative address in BOTH CTAs of the pair once the MMAs issued so far are done
__device__ __forceinline__ void umma2_commit_both(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// One CTA of a pair: ny is the channel-tile index of its tile (the block row of tc_pair_kernel, the role-adjusted row of
// tc_pair2_kernel).  The tensor maps are the kernel's __grid_constant__ parameters, passed by reference.
template <class Epi, int BN>
__device__ __forceinline__ void tc_pair_cta(const CUtensorMap& tmAh, const CUtensorMap& tmAl, const CUtensorMap& tmBh,
                                            const CUtensorMap& tmBl, const typename Epi::Params& ep, int T, int K, int N,
                                            int taps, int dil, const int2* __restrict__ tiles, int ny) {
  using Cfg = TcPairCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int H = Cfg::H;
  pdl_launch_dependents();
  int m0 = blockIdx.x * TC_BM, b = blockIdx.z;
  if (tiles != nullptr) {
    // ragged batch (TcTiles): the two CTAs of a pair take consecutive table entries -- any two frame tiles, of any
    // items: only the weight block is shared.  A pair of dead slots leaves; a dead slot next to a live one takes
    // part with an all-padding activation tile (first frame beyond T: the TMA unit zero-fills it).
    const int2 t = __ldg(tiles + blockIdx.x), tp = __ldg(tiles + (blockIdx.x ^ 1u));
    if (t.y < 0 && tp.y < 0) return;
    b = t.y < 0 ? tp.x : t.x;
    m0 = t.y < 0 ? ((T + TC_BM - 1) / TC_BM) * TC_BM : t.y;
  }
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * Cfg::STAGE;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * STAGES);
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 1);
  auto tile_a = [&](int s, int lo) { return smem_base + (uint32_t)s * Cfg::STAGE + (uint32_t)lo * TC_A_TILE; };
  auto tile_p = [&](int s) { return smem_base + (uint32_t)s * Cfg::STAGE + 2u * TC_A_TILE; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef DSVC_TIMELINE
  const long long tl0 = clock64();
  TL_ENTRY();
#endif
  const uint32_t rank = cluster_ctarank();       // 0 = even CTA (issues the MMAs), 1 = odd
  const int kblocks = K / TC_BK;
  const int total = taps * kblocks;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAl) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBl) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);        // used in the even CTA only: its producer's arrive.expect_tx
      mbar_init(empty_bar(s), 1);       // one multicast commit per use
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(2 * BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                   // the peer's barriers are initialised before anything can arrive on them
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  if (warp == 3) TL_MARK(0);

  // the even CTA's full barrier of stage s, as a shared::cluster address valid from either CTA
  auto full_bar_leader = [&](int s) { return mapa_cluster(full_bar(s), 0u); };

  // weight block P of pipeline iteration `it`: rows a (first half of the tile's channels) and rows b (second half)
  auto load_p = [&](int it, int s) {
    const int tap = it / kblocks, kb = it - tap * kblocks;
    if constexpr (BN == 256) {
      // N = 2*BN would exceed the 256-column MMA limit: wh and wl are multiplied by separate MMAs (below), so each CTA
      // simply holds ITS half of the tile's rows, hi block then lo block: P = [ wh_half (128 rows) ; wl_half (128 rows) ]
      int r0, r1;                                     // two 64-row boxes
      if constexpr (Epi::kPair) {                     // [128 gate | 128 filter] from two packed super-tiles
        const int sb = tap * N + ny * 256;
        r0 = sb + (rank == 0 ? 0 : 64); r1 = r0 + 128;
      } else {
        r0 = tap * N + ny * 256 + (int)rank * 128; r1 = r0 + 64;
      }
      const uint32_t bar = full_bar_leader(s);
      const uint32_t p = tile_p(s);
      tma2_load_2d(&tmBh, bar, p, kb * TC_BK, r0);
      tma2_load_2d(&tmBh, bar, p + 64u * 128u, kb * TC_BK, r1);
      tma2_load_2d(&tmBl, bar, p + 128u * 128u, kb * TC_BK, r0);
      tma2_load_2d(&tmBl, bar, p + 192u * 128u, kb * TC_BK, r1);
    } else {
    int ra, rb;
    if constexpr (Epi::kPair) {
      // gate|filter packing: a 128-row super-tile holds [64 gate rows | 64 filter rows]; a BN-wide tile takes
      // H gate rows and the matching H filter rows
      const int per = 128 / BN;                       // tiles per super-tile (BN = 64: 2, BN = 128: 1)
      ra = tap * N + (ny / per) * 128 + (ny % per) * H;
      rb = ra + 64;
    } else {
      ra = tap * N + ny * BN;
      rb = ra + H;
    }
    const uint32_t bar = full_bar_leader(s);
    const uint32_t p = tile_p(s);
    // even: [wh_a ; wl_b]    odd: [wh_b ; wl_a]
    tma2_load_2d(&tmBh, bar, p, kb * TC_BK, rank == 0 ? ra : rb);
    tma2_load_2d(&tmBl, bar, p + (uint32_t)H * 128u, kb * TC_BK, rank == 0 ? rb : ra);
    }
  };
  auto load_a = [&](int it, int s) {
    const int tap = it / kblocks, kb = it - tap * kblocks;
    const int frame = m0 + (tap - (taps >> 1)) * dil;
    const uint32_t bar = full_bar_leader(s);
    tma2_load_3d(&tmAh, bar, tile_a(s, 0), kb * TC_BK, frame, b);
    tma2_load_3d(&tmAl, bar, tile_a(s, 1), kb * TC_BK, frame, b);
  };

  if (warp == 0) {
    // ===== TMA producer, one per CTA: its own 128 activation rows and its own weight block =====
    constexpr uint32_t tx_pair = 2u * Cfg::STAGE;            // bytes both CTAs deliver per stage
    const int pre = total < STAGES ? total : STAGES;
    if (elect_one_sync()) {
      for (int it = 0; it < pre; ++it) {
        if (rank == 0) mbar_expect_tx(full_bar(it), tx_pair);
        load_p(it, it);
      }
    }
    __syncwarp();
    pdl_wait();                                               // activations were written by the previous kernel
    TL_GT(13);
    if (elect_one_sync()) {
      for (int it = 0; it < pre; ++it) load_a(it, it);
    }
    __syncwarp();
    for (int it = pre; it < total; ++it) {
      const int s = it % STAGES;
      const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
      mbar_wait(empty_bar(s), ph ^ 1u);                       // own copy: the multicast commit arrives in both CTAs
      if (elect_one_sync()) {
        if (rank == 0) mbar_expect_tx(full_bar(s), tx_pair);
        load_a(it, s);
        load_p(it, s);
      }
      __syncwarp();
    }
  } else if (warp == 1 && rank == 0) {
    // ===== MMA issuer: the even CTA, for both =====
    const uint32_t idesc_hi = umma_idesc_f16(2 * TC_BM, BN == 256 ? 256 : 2 * BN);
    const uint32_t idesc_lo = umma_idesc_f16(2 * TC_BM, BN);
    for (int it = 0; it < total; ++it) {
      const int s = it % STAGES;
      const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
      mbar_wait(full_bar(s), ph);
      if (it == 0) TL_MARK(1);
      tc_fence_after();
      if (elect_one_sync()) {
        const uint64_t ah = umma_desc_sw128(tile_a(s, 0)), al = umma_desc_sw128(tile_a(s, 1));
        const uint64_t pd = umma_desc_sw128(tile_p(s));
#pragma unroll
        for (int k4 = 0; k4 < TC_BK / 16; ++k4) {
          const uint64_t koff = (uint64_t)((k4 * 32) >> 4);
          const uint32_t acc = (it > 0 || k4 > 0) ? 1u : 0u;
          if constexpr (BN == 256) {
            // three N = 256 MMAs, xh*wl in its own accumulator (columns 256..511), like the single-CTA 256-wide tile
            const uint64_t pl = umma_desc_sw128(tile_p(s) + 128u * 128u);
            umma2_f16(tmem_base, ah + koff, pd + koff, idesc_lo, acc);
            umma2_f16(tmem_base + (uint32_t)BN, ah + koff, pl + koff, idesc_lo, acc);
            umma2_f16(tmem_base, al + koff, pd + koff, idesc_lo, 1u);
          } else {
            umma2_f16(tmem_base, ah + koff, pd + koff, idesc_hi, acc);
            umma2_f16(tmem_base, al + koff, pd + koff, idesc_lo, 1u);
          }
        }
        umma2_commit_both(empty_bar(s));
        if (it == total - 1) umma2_commit_both(tmem_full_bar);
      }
      __syncwarp();
    }
    TL_MARK(2);
  }
  pdl_wait();
#ifdef DSVC_TIMELINE
  tc_epilogue<Epi, BN>(ep, smem_raw, smem_base, tmem_base, tmem_full_bar, 0u, T, N, m0, ny, b, warp, lane, true, tl0, 0, BN == 256 ? 0 : H);
#else
  tc_epilogue<Epi, BN>(ep, smem_raw, smem_base, tmem_base, tmem_full_bar, 0u, T, N, m0, ny, b, warp, lane, true, BN == 256 ? 0 : H);
#endif
  if (warp == 4) TL_MARK(6);
  tc_fence_before();
  __syncthreads();
  TL_GT(14);
  cluster_sync_all();                   // both CTAs have drained their accumulator halves
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * BN) : "memory");
  }
}

// Channel tiles ny0 .. ny0 + gridDim.y - 1 of an N-wide contraction (ny0 > 0: the second half of the WaveNet
// out-projection, launched on its own after the last layer)
template <class Epi, int BN>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_pair_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
               const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
               const typename Epi::Params ep, int T, int K, int N, int taps, int dil, const int2* __restrict__ tiles, int ny0) {
#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ >= 1000)
  tc_pair_cta<Epi, BN>(tmAh, tmAl, tmBh, tmBl, ep, T, K, N, taps, dil, tiles, ny0 + (int)blockIdx.y);
#endif
}

// Two independent contractions of one frame range in one grid (dense layout, no tile table): block rows y < nA run
// role A (channel tiles 0 .. nA - 1 of its N), rows y >= nA role B (channel tiles nyB + y - nA of its N).  Each role has
// its own tensor maps, epilogue, K, taps and dilation; the branch is uniform per CTA pair.  Both roles keep the PDL
// protocol of the plain kernel (dependents released at entry, griddepcontrol.wait before the first activation load), so
// role B may read what the kernel two launches back wrote: the previous kernel completes only after its own wait.
template <class EpiA, class EpiB, int BN>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_pair2_kernel(const __grid_constant__ CUtensorMap aAh, const __grid_constant__ CUtensorMap aAl,
                const __grid_constant__ CUtensorMap aBh, const __grid_constant__ CUtensorMap aBl,
                const typename EpiA::Params epA, int KA, int NA, int tapsA, int dilA, int nA,
                const __grid_constant__ CUtensorMap bAh, const __grid_constant__ CUtensorMap bAl,
                const __grid_constant__ CUtensorMap bBh, const __grid_constant__ CUtensorMap bBl,
                const typename EpiB::Params epB, int KB, int NB, int tapsB, int dilB, int nyB, int T) {
#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ >= 1000)
  if ((int)blockIdx.y < nA) tc_pair_cta<EpiA, BN>(aAh, aAl, aBh, aBl, epA, T, KA, NA, tapsA, dilA, nullptr, (int)blockIdx.y);
  else tc_pair_cta<EpiB, BN>(bAh, bAl, bBh, bBl, epB, T, KB, NB, tapsB, dilB, nullptr, nyB + (int)blockIdx.y - nA);
#endif
}

// DSVC_TC_PAIR=0 keeps every contraction on the single-CTA kernels (read per call: tests switch it per handle)
inline bool tc_pair_enabled() {
  const char* e = getenv("DSVC_TC_PAIR");
  return !(e && atoi(e) == 0);
}

// frame tiles in pairs (an odd last one pairs with an empty tile): the grid's x extent of a dense layout
inline int tc_pair_frame_ctas(int T) { return 2 * ceil_div(ceil_div(T, TC_BM), 2); }

// cluster of two CTAs along x, programmatic dependent launch
struct TcPairLaunch {
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[2];
  TcPairLaunch(dim3 grid, int smem, cudaStream_t s) {
    cfg.gridDim = grid;
    cfg.blockDim = dim3(TC_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
  }
};

// the weight maps of a BN-wide pair tile: boxes of H rows (BN = 256: two 64-row boxes per half)
template <int BN> const CUtensorMap& tc_pair_bh(const TcGemmMaps& m) { return BN == 64 ? m.b32_hi : m.b64_hi; }
template <int BN> const CUtensorMap& tc_pair_bl(const TcGemmMaps& m) { return BN == 64 ? m.b32_lo : m.b64_lo; }

// channel tiles ny0 .. ny0 + n_ny - 1 (n_ny = 0: all N / BN)
template <class Epi, int BN>
int tc_pair_launch_bn(const TcGemmMaps& m, const typename Epi::Params& e, int B, int T, int K, int N, int taps, int dil,
                      cudaStream_t s, TcTiles tt = TcTiles{}, int ny0 = 0, int n_ny = 0) {
  DSVC_TRY((ensure_dyn_smem<tc_pair_kernel<Epi, BN>>(TcPairCfg<BN>::SMEM)));
  const int ny = n_ny > 0 ? n_ny : N / BN;
  DSVC_REQUIRE(ny0 >= 0 && ny0 + ny <= N / BN, "tc_pair_launch: channel tiles %d..%d of %d", ny0, ny0 + ny - 1, N / BN);
  // a ragged batch's table has an even slot count
  TcPairLaunch l(tt.tab ? dim3(tt.slots, ny, 1) : dim3(tc_pair_frame_ctas(T), ny, B), TcPairCfg<BN>::SMEM, s);
  DSVC_CUDA(cudaLaunchKernelEx(&l.cfg, tc_pair_kernel<Epi, BN>, m.a_hi, m.a_lo, tc_pair_bh<BN>(m), tc_pair_bl<BN>(m), e, T, K, N,
                               taps, dil, tt.tab, ny0));
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

// tc_pair2_kernel: role A = channel tiles 0 .. nA - 1 of (mA, NA), role B = tiles nyB .. nyB + nB - 1 of (mB, NB); one item
// of T frames or a dense batch of B
template <class EpiA, class EpiB, int BN>
int tc_pair2_launch_bn(const TcGemmMaps& mA, const typename EpiA::Params& eA, int KA, int NA, int tapsA, int dilA, int nA,
                       const TcGemmMaps& mB, const typename EpiB::Params& eB, int KB, int NB, int tapsB, int dilB, int nyB, int nB,
                       int B, int T, cudaStream_t s) {
  DSVC_TRY((ensure_dyn_smem<tc_pair2_kernel<EpiA, EpiB, BN>>(TcPairCfg<BN>::SMEM)));
  DSVC_REQUIRE(KA % TC_BK == 0 && KB % TC_BK == 0 && nA > 0 && nA <= NA / BN && nB > 0 && nyB >= 0 && nyB + nB <= NB / BN,
               "tc_pair2_launch: bad roles (K %d / %d, tiles %d of %d, %d..%d of %d)", KA, KB, nA, NA / BN, nyB, nyB + nB - 1, NB / BN);
  TcPairLaunch l(dim3(tc_pair_frame_ctas(T), nA + nB, B), TcPairCfg<BN>::SMEM, s);
  DSVC_CUDA(cudaLaunchKernelEx(&l.cfg, tc_pair2_kernel<EpiA, EpiB, BN>, mA.a_hi, mA.a_lo, tc_pair_bh<BN>(mA), tc_pair_bl<BN>(mA), eA,
                               KA, NA, tapsA, dilA, nA, mB.a_hi, mB.a_lo, tc_pair_bh<BN>(mB), tc_pair_bl<BN>(mB), eB, KB, NB,
                               tapsB, dilB, nyB, T));
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

// One contraction on the tensor cores: the CTA-pair kernel for the 64- and 128-wide tile classes of the 3-pass
// mode, the single-CTA kernel otherwise (1-pass "fast mode", the 256-wide tiles of large batches, odd widths).
template <class Epi>
int tc_launch(const TcGemmMaps& m, const typename Epi::Params& e, int B, int T, int K, int N, int taps, int dil, int passes,
              cudaStream_t s, TcTiles tt = TcTiles{}) {
  DSVC_REQUIRE(K % TC_BK == 0, "tc_launch: K=%d must be a multiple of %d", K, TC_BK);
  if (passes == 3 && tc_pair_enabled()) {
    const int bn = tc_pick_bn(B, T, N, tt.live);
    if (bn == 64 && N % 64 == 0) return tc_pair_launch_bn<Epi, 64>(m, e, B, T, K, N, taps, dil, s, tt);
    if (bn == 128 && N % 128 == 0) return tc_pair_launch_bn<Epi, 128>(m, e, B, T, K, N, taps, dil, s, tt);
    if (bn == 256 && N % 256 == 0) return tc_pair_launch_bn<Epi, 256>(m, e, B, T, K, N, taps, dil, s, tt);
  }
  return tc_launch_single<Epi>(m, e, B, T, K, N, taps, dil, passes, s, tt);
}

}  // namespace dsvc
