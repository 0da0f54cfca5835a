// Narrow ResBlock convolutions of the vocoder (C = Cin = Cout = 32 or 16; modules/nsf_hifigan/models.py:57-64) on
// tcgen05: weights-stationary, persistent over frame tiles, the dilated taps fed from ONE activation window.
//
//   D[frame][n] = sum_{tap} sum_{c < C} A[frame + (tap - taps/2) * dil][c] * W[tap][n][c]
//
// Why not the WaveNet main loop (a narrow-row instantiation of tc_pair.cuh ran these convs in between, DESIGN.md 3.1g):
// there a tap is a pipeline stage -- 20 KB of operands through TMA and shared memory for 192 MMA cycles -- and every
// 256-frame tile is a CTA launch; above ~275 mel frames that lost to the FFMA GEMM.  Here
//   * the conv's whole weight set ([wh ; wl] per tap: taps x 4 KB at C = 32) is loaded into shared memory ONCE per CTA,
//   * a tile's activations are loaded ONCE: a window of 192 rows (the 128 output frames +- 32: every tap of every
//     ResBlock1 conv, k <= 11 x dilation <= 5, reaches at most 25 rows out) or 256 rows (+- 64, for ResBlock2
//     dilations up to 12), hi and lo planes, 24 / 32 KB at C = 32 -- and each tap's
//     operand is that window at a row offset: the UMMA descriptor's start address moves by (tap - taps/2) * dil rows
//     (the swizzle XOR is a function of the absolute shared-memory address, so any row offset reads consistently);
//     rows outside [0, L) are zero-filled by the TMA unit = the conv's zero padding,
//   * a CTA loops over frame tiles (two windows in flight), and two CTAs share an SM (<= 111 KB / 64 TMEM columns
//     each: every 192-row case, and the 256-row window up to k = 7 at C = 32), so one CTA's epilogue overlaps the
//     other's MMAs without any role specialisation.
// Operand rows are C fp16 = 64 / 32 bytes: SWIZZLE_64B / 32B tiles (umma_desc_k<C>), K per tap = C = 2 / 1 MMA K-steps.
// The 3-pass product keeps its two-MMA form: xh * [wh ; wl] (N = 2C) and xl * wh (N = C) into accumulator columns
// [0, C) | [C, 2C).  Epilogue: the shared tc_epilogue / EpiVoc functor on a C-wide tile.
#pragma once
#include "tc_gemm.cuh"

namespace dsvc {

// The window is TC_BM output frames plus PAD rows either side; PAD >= (taps / 2) * dil of every conv it runs.
// Two instances: PAD 32 (192 rows; every ResBlock1 conv of the shipped configs) and PAD 64 (256 rows, the TMA box
// height limit; ResBlock2 dilations up to 12 at kernel 7 reach 36 rows).
constexpr int NW_PAD = 32;        // the 192-row window
constexpr int NW_PAD_WIDE = 64;   // the 256-row window
constexpr int nw_rows(int pad) { return TC_BM + 2 * pad; }

template <int C, int PAD> struct NarrowCfg {
  static constexpr int ROWS = nw_rows(PAD);                // window rows per tile
  static constexpr int ROWB = C * 2;                       // bytes per operand row
  static constexpr int W_TAP = 2 * C * ROWB;               // [wh ; wl] of one tap
  static constexpr int WIN = ROWS * ROWB;                  // one plane of one window
  static constexpr int SLAB = 4 * 32 * (C + 4) * 4;        // epilogue staging
  static constexpr int BARS = 128;
  static int smem(int taps) { return taps * W_TAP + 4 * WIN + BARS + SLAB + 1024; }
};

template <int C, int PAD>
__global__ void __launch_bounds__(TC_THREADS, 2)
tc_narrow_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                 const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
                 const EpiVoc::Params ep, int L, int taps, int dil, int tiles_per_item, int n_tiles) {
#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ >= 1000)
  using Cfg = NarrowCfg<C, PAD>;
  static_assert(C == 32 || C == 16, "narrow convs: 32 or 16 channels");
  static_assert(Cfg::ROWS <= 256, "a window is one TMA box: at most 256 rows");
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t win_base = smem_base + (uint32_t)taps * Cfg::W_TAP;
  const uint32_t bar_base = win_base + 4u * Cfg::WIN;
  const uint32_t slab_base = bar_base + Cfg::BARS;
  const uint32_t w_full = bar_base, acc_full = bar_base + 8u, tmem_slot = bar_base + 32u;
  auto a_full = [&](int i) { return bar_base + 16u + 8u * i; };
  auto w_tap = [&](int tap) { return smem_base + (uint32_t)tap * Cfg::W_TAP; };
  auto win = [&](int buf, int lo) { return win_base + (uint32_t)(2 * buf + lo) * Cfg::WIN; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stride = (int)gridDim.x;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAl) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBl) : "memory");
  }
  if (warp == 1 && lane == 0) {
    mbar_init(w_full, 1);
    mbar_init(acc_full, 1);
    mbar_init(a_full(0), 1);
    mbar_init(a_full(1), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(2 * C) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  auto load_window = [&](int t, int buf) {           // one elected lane: the window of frame tile t, both planes
    const int b = t / tiles_per_item, m0 = (t - b * tiles_per_item) * TC_BM;
    mbar_expect_tx(a_full(buf), 2u * Cfg::WIN);
    tma_load_3d(&tmAh, a_full(buf), win(buf, 0), 0, m0 - PAD, b);
    tma_load_3d(&tmAl, a_full(buf), win(buf, 1), 0, m0 - PAD, b);
  };

  if (warp == 0) {
    if (elect_one_sync()) {                           // the weights: constants, requested before the dependency wait
      mbar_expect_tx(w_full, (uint32_t)taps * Cfg::W_TAP);
      for (int tap = 0; tap < taps; ++tap) {
        tma_load_2d(&tmBh, w_full, w_tap(tap), 0, tap * C);
        tma_load_2d(&tmBl, w_full, w_tap(tap) + (uint32_t)C * Cfg::ROWB, 0, tap * C);
      }
    }
    __syncwarp();
    pdl_wait();                                       // the activation planes were written by the previous kernel
    if (elect_one_sync()) {
      for (int i = 0; i < 2; ++i) {
        const int t = (int)blockIdx.x + i * stride;
        if (t < n_tiles) load_window(t, i);
      }
    }
    __syncwarp();
  }
  pdl_wait();                                         // every warp: the epilogue reads tensors earlier kernels wrote

  const uint32_t idesc_hi = umma_idesc_f16(TC_BM, 2 * C);     // xh * [wh ; wl]
  const uint32_t idesc_lo = umma_idesc_f16(TC_BM, C);         // xl * wh
  int i = 0;
  for (int t = (int)blockIdx.x; t < n_tiles; t += stride, ++i) {
    const int buf = i & 1;
    const int b = t / tiles_per_item, m0 = (t - b * tiles_per_item) * TC_BM;
    if (warp == 1) {
      // ===== MMA issuer: every tap from the same window, at a row offset =====
      if (i == 0) mbar_wait(w_full, 0u);
      mbar_wait(a_full(buf), (uint32_t)(i >> 1) & 1u);
      tc_fence_after();
      if (elect_one_sync()) {
        for (int tap = 0; tap < taps; ++tap) {
          const uint32_t row = (uint32_t)(PAD + (tap - (taps >> 1)) * dil) * Cfg::ROWB;
          const uint64_t ah = umma_desc_k<C>(win(buf, 0) + row), al = umma_desc_k<C>(win(buf, 1) + row);
          const uint64_t wd = umma_desc_k<C>(w_tap(tap));
#pragma unroll
          for (int k4 = 0; k4 < C / 16; ++k4) {
            const uint64_t koff = (uint64_t)((k4 * 32) >> 4);
            umma_f16(tmem_base, ah + koff, wd + koff, idesc_hi, (tap > 0 || k4 > 0) ? 1u : 0u);
            umma_f16(tmem_base, al + koff, wd + koff, idesc_lo, 1u);
          }
        }
        umma_commit(acc_full);
      }
      __syncwarp();
    }
    tc_epilogue<EpiVoc, C>(ep, smem_raw, slab_base, tmem_base, acc_full, (uint32_t)i & 1u, L, C, m0, 0, b, warp, lane, true
#ifdef DSVC_TIMELINE
                           , 0ll, 0
#endif
    );
    tc_fence_before();
    __syncthreads();                                  // accumulator and slab are free; this tile's MMAs have read the window
    tc_fence_after();
    if (warp == 0) {
      const int t2 = t + 2 * stride;
      if (t2 < n_tiles && elect_one_sync()) load_window(t2, buf);
      __syncwarp();
    }
  }
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * C) : "memory");
  }
#endif
}

template <int C, int PAD>
int tc_narrow_launch(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl,
                     const EpiVoc::Params& e, int B, int L, int taps, int dil, cudaStream_t s) {
  DSVC_REQUIRE(taps >= 1 && taps < 64 && (taps / 2) * dil <= PAD,
               "narrow conv: %d taps x dilation %d reach beyond the %d-row window", taps, dil, nw_rows(PAD));
  const int smem = NarrowCfg<C, PAD>::smem(taps);
  DSVC_TRY((ensure_dyn_smem<tc_narrow_kernel<C, PAD>>(smem)));
  static const int sms = [] {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
  }();
  // resident CTAs per SM at this tap count: 2 up to ~113 KB of shared memory (every 192-row case, the 256-row
  // window up to k = 7 at C = 32), else 1 -- a persistent grid larger than what is resident only queues
  static std::atomic<int> occ_by_taps[64];
  int occ = occ_by_taps[taps].load(std::memory_order_relaxed);
  if (occ == 0) {
    DSVC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, tc_narrow_kernel<C, PAD>, TC_THREADS, smem));
    DSVC_REQUIRE(occ >= 1, "narrow conv: %d bytes of shared memory do not fit an SM", smem);
    occ = occ < 2 ? occ : 2;
    occ_by_taps[taps].store(occ, std::memory_order_relaxed);
  }
  const int per_item = ceil_div(L, TC_BM), n_tiles = per_item * B;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(n_tiles < occ * sms ? n_tiles : occ * sms, 1, 1);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DSVC_CUDA(cudaLaunchKernelEx(&cfg, tc_narrow_kernel<C, PAD>, ah, al, bh, bl, e, L, taps, dil, per_item, n_tiles));
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

}  // namespace dsvc
