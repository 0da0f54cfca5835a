// tcgen05 / TMA main loop for the WaveNet contractions (sm_100a only).
//
//   D[frame][n] = sum_{tap} sum_{k} A[b][frame + (tap - taps/2)*dil][k] * W[tap][n][k]     (taps odd)
//
// A: activation plane, channels-last fp16 (hi, lo) pair [B][T][K]  (K-major)
// W: weight matrix fp16 (hi, lo) pair [taps*N][K]                  (K-major)
// One CTA owns a 128-frame x BN-channel output tile (BN = 128, or 64 when the grid would otherwise
// leave most of the 148 SMs idle).  Operands are staged by TMA into 128B-swizzled shared memory (the
// shifted tap is just a different TMA frame coordinate; out-of-range frames are zero-filled by the TMA
// unit = the conv's zero padding), multiplied by tcgen05.mma (M=128, N=BN, K=16 per instruction, fp32
// accumulators in TMEM) and read back with tcgen05.ld by all 16 warps, which run the fused epilogue
// functor (epilogues.cuh) on a shared-memory transpose of the tile.
//
// fp32-class accuracy on fp16 tensor cores: x = xh + xl, w = wh + wl (each fp16), and
//   x*w ~= xh*wh + xl*wh + xh*wl      (3 MMAs into the same fp32 accumulator; the dropped xl*wl
//                                      term is ~2^-22 relative)
// `passes == 1` issues only xh*wh ("fast mode", outside the parity gate).
//
// Warp roles (512 threads): warp 0 lane 0 = TMA producer, warp 1 lane 0 = MMA issuer, warp 2 = TMEM
// allocator; all 16 warps then run the epilogue (TMEM lane quarter = warp % 4, BN/4 columns each).
//
// Launched with programmatic dependent launch: the prologue (barrier init, TMEM alloc, tensor-map
// prefetch, weight-tile TMA) overlaps the tail of the previous kernel; everything that reads data the
// previous kernel wrote sits behind griddepcontrol.wait.
#pragma once
#include <cuda.h>
#include <stdlib.h>
#include <cmath>

#include "common.cuh"
#include "epilogues.cuh"

namespace dsvc {

struct TcGemmMaps {
  CUtensorMap a_hi, a_lo;        // activation planes, box {64 ch, 128 frames, 1 item}
  CUtensorMap b_hi, b_lo;        // weights, box {64, 128 rows}   (BN = 128 tiles)
  CUtensorMap b32_hi, b32_lo;    // weights, box {64, 32 rows}    (BN = 64 tiles: two boxes per stage)
  CUtensorMap b64_hi, b64_lo;    // weights, box {64, 64 rows}    (BN = 256 gate|filter tiles: four boxes per stage)
};
struct TcMaps {
  TcGemmMaps in, skip, head;
  std::vector<TcGemmMaps> dil, out;
};

// Ragged batches: the frame tiles that hold at least one valid frame, as (item, first frame) entries; the grid's x
// axis indexes this table instead of (frame tile, item).  `slots` (the grid size: the dense tile count, so a captured
// graph does not depend on the lengths) >= `live`; the entries past `live` are (0, -1) and their CTAs exit at once.
struct TcTiles {
  const int2* tab = nullptr;
  int slots = 0, live = 0;
};

struct F16Pair {           // tcgen05 operand: fp16 hi/lo copies of a (power-of-two scaled) weight matrix
  DevBuf hi, lo;
  float inv_scale = 1.f;   // multiply the accumulator by this in the epilogue
};


struct PlaneBuf {
  DevBuf f32, hi, lo;
  Plane view(bool tc) const {
    Plane p;
    p.f32 = tc ? nullptr : f32.as<float>();
    p.hi = tc ? hi.as<__half>() : nullptr;
    p.lo = tc ? lo.as<__half>() : nullptr;
    return p;
  }
  int reserve(size_t elems, bool tc) {
    if (tc) {
      DSVC_TRY(hi.reserve(elems * sizeof(__half)));
      DSVC_TRY(lo.reserve(elems * sizeof(__half)));
    } else {
      DSVC_TRY(f32.reserve(elems * sizeof(float)));
    }
    return DSVC_OK;
  }
};


// fp16 hi/lo split of a weight matrix with a power-of-two pre-scale that moves the weights into
// fp16's normal range (hi + lo reproduces w * scale to ~2^-22).
static inline int make_f16_pair(F16Pair& out, const float* w, size_t n, cudaStream_t s) {
  float mx = 0.f;
  for (size_t i = 0; i < n; ++i) mx = std::max(mx, std::fabs(w[i]));
  float scale = 1.f;
  if (mx > 0.f) {
    int e;
    std::frexp(1024.0f / mx, &e);          // 1024/mx = m * 2^e, m in [0.5,1)
    scale = std::ldexp(1.0f, e - 1);        // largest power of two <= 1024/mx
  }
  std::vector<__half> hi(n), lo(n);
  for (size_t i = 0; i < n; ++i) {
    const float v = w[i] * scale;
    const __half h = __float2half_rn(v);
    hi[i] = h;
    lo[i] = __float2half_rn(v - __half2float(h));
  }
  out.inv_scale = 1.0f / scale;
  DSVC_TRY(out.hi.upload(hi.data(), n * sizeof(__half), s));
  DSVC_TRY(out.lo.upload(lo.data(), n * sizeof(__half), s));
  DSVC_CUDA(cudaStreamSynchronize(s));   // host vectors go out of scope
  return DSVC_OK;
}


constexpr int TC_BM = 128;
constexpr int TC_BK = 64;
constexpr int TC_THREADS = 512;
constexpr int TC_A_TILE = TC_BM * TC_BK * 2;   // 16 KB: one [128 rows][64 fp16] tile

template <int BN> struct TcCfg {
  static constexpr int B_TILE = BN * TC_BK * 2;
  static constexpr int STAGE = 2 * (TC_A_TILE + B_TILE);     // A_hi, A_lo, B_hi, B_lo
  static constexpr int STAGES = (BN == 64) ? 4 : (BN == 128 ? 3 : 2);   // 192 KB of operands in flight
  static constexpr int SMEM = STAGES * STAGE + 1024 /*align*/ + 128 /*barriers*/;
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
#ifdef DSVC_WATCHDOG   // debug builds: a lost arrive fails loudly instead of hanging the GPU
  const long long t0 = clock64();
#endif
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) break;
#ifdef DSVC_WATCHDOG
    if (clock64() - t0 > 4000000000ll) {   // ~2 s
      printf("libdsvc: mbarrier wait timed out (block %d,%d,%d thread %d)\n", blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x);
      __trap();
    }
#endif
  }
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// one lane of a converged warp (the compiler then emits straight-line uniform-datapath code for the
// TMA / MMA issue instead of per-instruction ELECT + BRA.U.ANY serialisation loops)
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, px;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: 8-row groups are 1024 B apart (SBO), LBO unused (=1)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);       // start address  [0,14)
  d |= (uint64_t)1 << 16;                        // leading byte offset (16 B units) [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset [32,46)
  d |= (uint64_t)1 << 46;                        // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
  return d;
}
// K-major operand tile whose rows are KB fp16 wide (KB = 64 / 32 / 16 -> SWIZZLE_128B / 64B / 32B, the narrow rows of the
// vocoder's 32- and 16-channel stages): 8-row groups are 8 * row bytes apart
template <int KB>
__device__ __forceinline__ uint64_t umma_desc_k(uint32_t saddr) {
  static_assert(KB == 64 || KB == 32 || KB == 16, "operand rows of 128, 64 or 32 bytes");
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((8 * KB * 2) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(KB == 64 ? 2 : (KB == 32 ? 4 : 6)) << 61;      // SWIZZLE_128B / 64B / 32B
  return d;
}
// kind::f16 instruction descriptor: D = f32, A = B = f16, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&r)[32]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(r);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
        "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]),
        "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]),
        "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&r)[16]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(r);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
        "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&r)[8]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(r);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
               : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&r)[4]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(r);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
template <int CW> __device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&r)[CW]);
template <> __device__ __forceinline__ void tmem_ld_cols<8>(uint32_t taddr, float (&r)[8]) { tmem_ld8(taddr, r); }
template <> __device__ __forceinline__ void tmem_ld_cols<4>(uint32_t taddr, float (&r)[4]) { tmem_ld4(taddr, r); }
template <> __device__ __forceinline__ void tmem_ld_cols<32>(uint32_t taddr, float (&r)[32]) { tmem_ld32(taddr, r); }
template <> __device__ __forceinline__ void tmem_ld_cols<16>(uint32_t taddr, float (&r)[16]) { tmem_ld16(taddr, r); }

// ---- optional per-CTA timeline (cycles since kernel entry), build with -DDSVC_TIMELINE ----------
#ifdef DSVC_TIMELINE
__device__ long long g_timeline[1024][16];
#define TL_MARK(slot) do { if (lane == 0) g_timeline[((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) & 1023][slot] = clock64() - tl0; } while (0)
// slot 15: %globaltimer (ns) at CTA entry -- the one clock all CTAs share: orders early (pre-launched) and late CTAs
#define TL_ENTRY() do { if (threadIdx.x == 0) { unsigned long long gt_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_)); \
  g_timeline[((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) & 1023][15] = (long long)gt_; } } while (0)
// %globaltimer (ns) into `slot` by thread 0 (the pair kernel: 13 = past griddepcontrol.wait, 14 = epilogue done)
#define TL_GT(slot) do { if (threadIdx.x == 0) { unsigned long long gt_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_)); \
  g_timeline[((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) & 1023][slot] = (long long)gt_; } } while (0)
#else
#define TL_MARK(slot) do { } while (0)
#define TL_ENTRY() do { } while (0)
#define TL_GT(slot) do { } while (0)
#endif

// ===== epilogue (all 16 warps): TMEM -> registers -> smem transpose -> fused functor -> global =====
// LEAN (the step kernel, whose epilogue warps have 96 registers): row inputs that were not loaded early come in batches of
// 4 rows instead of all 8 -- one more round of load latency, 40 registers less.
template <class Epi, int BN, bool LEAN = false>
__device__ __forceinline__ void tc_epilogue(const typename Epi::Params& ep, uint8_t* smem_raw, uint32_t smem_base,
                                            uint32_t tmem_base, uint32_t tmem_full_bar, uint32_t tmem_parity, int T, int N,
                                            int m0, int ny, int b, int warp, int lane, bool two_acc
#ifdef DSVC_TIMELINE
                                            , long long tl0, int tl_off = 0
#endif
                                            , int pair_h = 0   // tc_pair.cuh accumulator layout: channel j adds column j + (j < h ? 3h : h)
                                            , uint32_t acc_free_bar = 0   // tc_step.cuh: shared::cluster address of the barrier that hands the
                                                                          // accumulator back to the MMA issuer (one arrive per warp), 0: none
) {
#ifndef DSVC_TIMELINE
    constexpr int tl_off = 0;
    (void)tl_off;
#endif
    // ===== epilogue (all 16 warps): TMEM -> registers -> smem transpose -> fused functor -> global =====
    // tcgen05.ld hands each thread one accumulator ROW (a frame); a warp may only touch the TMEM lane
    // quarter (warp % 4).  Global tensors are channels-last, so the four warps of a quarter stage their
    // 32 x BN/4 blocks into one [32 rows][BN cols] shared-memory slab (the pipeline stages are free once
    // tmem_full fires), then each takes 8 rows with lane <-> 4 consecutive channels: every global access
    // of the functor is a contiguous warp transaction, and the transcendental-heavy gating runs on 16
    // warps instead of 4.
    constexpr int NCH = Epi::kPair ? BN / 8 : BN / 4;     // float4 chunks per row (pair: gate chunks)
    constexpr int NH = NCH > 32 ? NCH / 32 : 1;           // column passes (BN = 256 plain tiles: 2)
    constexpr int LPR = NCH / NH;                         // lanes per row
    constexpr int RPI = 32 / LPR;                         // rows per iteration
    constexpr int NIT = 8 / RPI;                          // iterations for this warp's 8 rows
    constexpr int CW = BN / 4;                            // columns staged by this warp
    const int q = warp & 3;                      // TMEM lane quarter = rows 32q .. 32q+31 of the tile
    const int cg = warp >> 2;                    // column group staged by this warp; also its row octet
    const int lc = lane % LPR, rsub = lane / LPR;
    const int row0 = q * 32 + cg * 8;            // first of this warp's 8 rows (tile-relative)
    auto col_of = [&](int h) {                   // this lane's 4 channels in column pass h
      const int ch = lc + h * LPR;
      return Epi::kPair ? ny * (BN / 2) + 4 * ch : ny * BN + 4 * ch;
    };
    // While the MMAs run: pull the rows this warp's epilogue will read into L2 (one request per 128-B line)
    EpiCol cc[NH];
#pragma unroll
    for (int h = 0; h < NH; ++h) {
      const int ncol = col_of(h);
      const bool col_ok = Epi::kPair ? true : (ncol < N);
      if (col_ok && (lc & 7) == 0) {
#pragma unroll
        for (int i = 0; i < NIT; ++i) {
          const int p = m0 + row0 + i * RPI + rsub;
          if (p < T) Epi::l2_prefetch(ep, b, p, ncol);
        }
      }
      cc[h] = EpiCol{};
      if (col_ok) cc[h] = Epi::col(ep, ncol);
    }
    // The per-row inputs (all written by EARLIER kernels: residual stream, skip sum, conditioner slab, sampler state)
    // are loaded into registers while the MMAs still run, not after the accumulator has been staged: their L2 latency
    // leaves the epilogue's critical path (measured, one clip: staged -> done 2200 -> 1700 cycles in the conv kernel,
    // 3100 -> 2400 in the out-projection, 394 -> 384 us per DDPM step; bit-identical results).  Only for the narrow
    // tiles (<= 4 row iterations per thread: <= 32 registers).  -DDSVC_NO_EPI_HOIST restores the late loads.
#ifndef DSVC_NO_EPI_HOIST
    constexpr bool kHoist = (NH * NIT <= 4);
#else
    constexpr bool kHoist = false;
#endif
    EpiPre hpre[kHoist ? NH * NIT : 1];
    if constexpr (kHoist) {
#pragma unroll
      for (int h = 0; h < NH; ++h) {
        const int ncol = col_of(h);
        const bool col_ok = Epi::kPair ? true : (ncol < N);
#pragma unroll
        for (int i = 0; i < NIT; ++i) {
          const int p = m0 + row0 + i * RPI + rsub;
          hpre[h * NIT + i] = EpiPre{};
          if (p < T && col_ok) hpre[h * NIT + i] = Epi::pre(ep, b, p, ncol);
        }
      }
    }
    if (warp == 4) TL_MARK(3 + tl_off);    // epilogue prefetch issued
    mbar_wait(tmem_full_bar, tmem_parity);
    if (warp == 4) TL_MARK(4 + tl_off);    // accumulator ready
    tc_fence_after();
    constexpr int STG_LD = BN + 4;               // padded row: conflict-free float4 writes
    float* slab = reinterpret_cast<float*>(smem_raw + (smem_base - smem_u32(smem_raw))) + (size_t)q * 32 * STG_LD;
    {
      constexpr int LW = CW > 32 ? 32 : CW;      // columns per tcgen05.ld
#pragma unroll
      for (int c0 = 0; c0 < CW; c0 += LW) {
        float v[LW];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * CW + c0);
        tmem_ld_cols<LW>(taddr, v);
        if (two_acc) {                           // 3-pass mode: add the xh*wl accumulator (columns BN..2BN)
          const uint32_t partner = pair_h == 0 ? (uint32_t)BN : (uint32_t)((cg * CW + c0) < pair_h ? 3 * pair_h : pair_h);
          constexpr int PW = (LEAN && LW > 16) ? 16 : LW;   // LEAN: in pieces of 16 columns (48, not 64, accumulator registers live)
#pragma unroll
          for (int c1 = 0; c1 < LW; c1 += PW) {
            float v2[PW];
            tmem_ld_cols<PW>(taddr + partner + (uint32_t)c1, v2);
#pragma unroll
            for (int j = 0; j < PW; ++j) v[c1 + j] += v2[j];
          }
        }
#pragma unroll
        for (int j = 0; j < LW / 4; ++j)
          *reinterpret_cast<float4*>(slab + lane * STG_LD + cg * CW + c0 + j * 4) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
    }
    if (acc_free_bar != 0) {
      // persistent kernels: this warp's tcgen05.ld's have completed (tcgen05.wait::ld above): the accumulator buffer may be
      // overwritten by the next tile's MMAs while the functor below still runs
      tc_fence_before();
      if (lane == 0) asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(acc_free_bar) : "memory");
    }
    asm volatile("bar.sync %0, 128;" ::"r"(q + 1) : "memory");   // the 4 warps of this quarter
    if (warp == 4) TL_MARK(5 + tl_off);    // staged to smem
    const float* stg = slab + (size_t)(cg * 8) * STG_LD;
#pragma unroll
    for (int h = 0; h < NH; ++h) {
      const int ncol = col_of(h);
      const bool col_ok = Epi::kPair ? true : (ncol < N);
      const int ch = lc + h * LPR;
      constexpr int RCH = (kHoist || !LEAN) ? NIT : (NIT > 4 ? 4 : NIT);
#pragma unroll
      for (int i0 = 0; i0 < NIT; i0 += RCH) {
      EpiPre pre[RCH];
#pragma unroll
      for (int ii = 0; ii < RCH; ++ii) {
        const int i = i0 + ii;
        const int p = m0 + row0 + i * RPI + rsub;
        if constexpr (kHoist) pre[ii] = hpre[h * NIT + i];
        else if (p < T && col_ok) pre[ii] = Epi::pre(ep, b, p, ncol);
      }
#pragma unroll
      for (int ii = 0; ii < RCH; ++ii) {
        const int i = i0 + ii;
        const int r = i * RPI + rsub;
        const int p = m0 + row0 + r;
        if constexpr (Epi::kPair) {
          const float4 gv = *reinterpret_cast<const float4*>(stg + r * STG_LD + 4 * ch);
          const float4 fv = *reinterpret_cast<const float4*>(stg + r * STG_LD + BN / 2 + 4 * ch);
          if (p < T) {
            const float gg[4] = {gv.x, gv.y, gv.z, gv.w};
            const float ff[4] = {fv.x, fv.y, fv.z, fv.w};
            Epi::apply_pair(ep, b, p, ncol, gg, ff, cc[h], pre[ii]);
          }
        } else {
          const float4 xv = *reinterpret_cast<const float4*>(stg + r * STG_LD + 4 * ch);
          if (p < T && col_ok) {
            const float vv[4] = {xv.x, xv.y, xv.z, xv.w};
            Epi::apply(ep, b, p, ncol, vv, cc[h], pre[ii]);
          }
        }
      }
      }
    }
    if (acc_free_bar != 0) asm volatile("bar.sync %0, 128;" ::"r"(q + 1) : "memory");   // the slab is staged again by the next tile
}

// ---- the kernel -----------------------------------------------------------------------------
template <class Epi, int BN>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
               const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
               const typename Epi::Params ep, int T, int K, int N, int taps, int dil, int passes, const int2* __restrict__ tiles) {
#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ >= 1000)
  using Cfg = TcCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  pdl_launch_dependents();                   // let the next kernel's prologue start early
  int m0 = blockIdx.x * TC_BM, b = blockIdx.z;
  if (tiles != nullptr) {                    // ragged batch: (item, first frame) of this CTA's tile; dead slots leave
    const int2 t = __ldg(tiles + blockIdx.x);
    if (t.y < 0) return;
    b = t.x; m0 = t.y;
  }
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B tiles need 1024 B alignment
  const uint32_t bar_base = smem_base + STAGES * Cfg::STAGE;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * STAGES);
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 1);
  // stage layout: [A_hi 16K][A_lo 16K][B_hi][B_lo]
  auto tile_a = [&](int s, int lo) { return smem_base + (uint32_t)s * Cfg::STAGE + (uint32_t)lo * TC_A_TILE; };
  auto tile_b = [&](int s, int lo) { return smem_base + (uint32_t)s * Cfg::STAGE + 2u * TC_A_TILE + (uint32_t)lo * Cfg::B_TILE; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef DSVC_TIMELINE
  const long long tl0 = clock64();
  TL_ENTRY();
#endif
  const int n0 = blockIdx.y * BN;
  const int kblocks = K / TC_BK;
  const int total = taps * kblocks;
  const bool three = passes == 3;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAh) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBh) : "memory");
    if (three) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAl) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBl) : "memory");
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(2 * BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  if (warp == 3) TL_MARK(0);   // setup done

  // weight tile(s) of pipeline iteration `it` into stage s (weights are constants: no dependency on
  // the previous kernel, so the first STAGES of them are requested before griddepcontrol.wait)
  auto load_b = [&](int it, int s) {
    const int tap = it / kblocks, kb = it - tap * kblocks;
    const int row = tap * N + n0;
    if constexpr (BN == 128) {
      tma_load_2d(&tmBh, full_bar(s), tile_b(s, 0), kb * TC_BK, row);
      if (three) tma_load_2d(&tmBl, full_bar(s), tile_b(s, 1), kb * TC_BK, row);
    } else if constexpr (BN == 256) {
      if constexpr (Epi::kPair) {
        // [128 gate | 128 filter] from two packed super-tiles [64 gate | 64 filter]: four 64-row boxes
        const int sb = tap * N + (int)blockIdx.y * 256;
        for (int lo = 0; lo < (three ? 2 : 1); ++lo) {
          const CUtensorMap* mp = lo ? &tmBl : &tmBh;
          tma_load_2d(mp, full_bar(s), tile_b(s, lo), kb * TC_BK, sb);                        // gate, super-tile 0
          tma_load_2d(mp, full_bar(s), tile_b(s, lo) + 64u * 128u, kb * TC_BK, sb + 128);     // gate, super-tile 1
          tma_load_2d(mp, full_bar(s), tile_b(s, lo) + 128u * 128u, kb * TC_BK, sb + 64);     // filter, super-tile 0
          tma_load_2d(mp, full_bar(s), tile_b(s, lo) + 192u * 128u, kb * TC_BK, sb + 192);    // filter, super-tile 1
        }
      } else {
        tma_load_2d(&tmBh, full_bar(s), tile_b(s, 0), kb * TC_BK, row);
        tma_load_2d(&tmBh, full_bar(s), tile_b(s, 0) + 128u * 128u, kb * TC_BK, row + 128);
        if (three) {
          tma_load_2d(&tmBl, full_bar(s), tile_b(s, 1), kb * TC_BK, row);
          tma_load_2d(&tmBl, full_bar(s), tile_b(s, 1) + 128u * 128u, kb * TC_BK, row + 128);
        }
      }
    } else {
      // two 32-row boxes.  Pair (gate|filter) tiles live in a 128-row super-tile packed as
      // [64 gate rows | 64 filter rows]: tile h of super-tile j takes gate rows 128j+32h and
      // filter rows 128j+64+32h.  Plain tiles take rows n0 and n0+32.
      const int r0 = Epi::kPair ? tap * N + (int)(blockIdx.y >> 1) * 128 + (int)(blockIdx.y & 1) * 32 : row;
      const int r1 = Epi::kPair ? r0 + 64 : row + 32;
      tma_load_2d(&tmBh, full_bar(s), tile_b(s, 0), kb * TC_BK, r0);
      tma_load_2d(&tmBh, full_bar(s), tile_b(s, 0) + 32u * 128u, kb * TC_BK, r1);
      if (three) {
        tma_load_2d(&tmBl, full_bar(s), tile_b(s, 1), kb * TC_BK, r0);
        tma_load_2d(&tmBl, full_bar(s), tile_b(s, 1) + 32u * 128u, kb * TC_BK, r1);
      }
    }
  };
  auto load_a = [&](int it, int s) {
    const int tap = it / kblocks, kb = it - tap * kblocks;
    const int frame = m0 + (tap - (taps >> 1)) * dil;   // centred odd kernel (taps = 1: the frame itself)
    tma_load_3d(&tmAh, full_bar(s), tile_a(s, 0), kb * TC_BK, frame, b);
    if (three) tma_load_3d(&tmAl, full_bar(s), tile_a(s, 1), kb * TC_BK, frame, b);
  };

  if (warp == 0) {
    // ===== TMA producer (whole warp in the loop, one elected lane issues) =====
    const uint32_t tx_bytes = three ? Cfg::STAGE : Cfg::STAGE / 2;
    const int pre = total < STAGES ? total : STAGES;
    if (elect_one_sync()) {
      for (int it = 0; it < pre; ++it) {        // stages are initially free: no empty-wait needed
        mbar_expect_tx(full_bar(it), tx_bytes);
        load_b(it, it);
      }
    }
    __syncwarp();
    pdl_wait();                                 // activations below were written by the previous kernel
    if (elect_one_sync()) {
      for (int it = 0; it < pre; ++it) load_a(it, it);
    }
    __syncwarp();
    for (int it = pre; it < total; ++it) {
      const int s = it % STAGES;
      const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
      mbar_wait(empty_bar(s), ph ^ 1u);
      if (elect_one_sync()) {
        mbar_expect_tx(full_bar(s), tx_bytes);
        load_a(it, s);
        load_b(it, s);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===== MMA issuer (whole warp in the loop, one elected lane issues) =====
    const uint32_t idesc = umma_idesc_f16(TC_BM, BN);
    const uint32_t idesc2 = umma_idesc_f16(TC_BM, BN == 256 ? 256 : 2 * BN);   // [wh ; wl] concatenated along N
    for (int it = 0; it < total; ++it) {
      const int s = it % STAGES;
      const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
      mbar_wait(full_bar(s), ph);
      if (it == 0) TL_MARK(1);            // first operands landed
      tc_fence_after();
      if (elect_one_sync()) {
        const uint64_t ah = umma_desc_sw128(tile_a(s, 0)), al = umma_desc_sw128(tile_a(s, 1));
        const uint64_t bh = umma_desc_sw128(tile_b(s, 0));
#pragma unroll
        for (int k4 = 0; k4 < TC_BK / 16; ++k4) {
          const uint64_t koff = (uint64_t)((k4 * 32) >> 4);   // +32 B per K=16 step inside the swizzled row
          const uint32_t acc = (it > 0 || k4 > 0) ? 1u : 0u;
          if (three && BN == 256) {
            // N = 2*BN would exceed the 256-column MMA limit: three N=256 MMAs, xh*wl in its own accumulator
            const uint64_t bl = umma_desc_sw128(tile_b(s, 1));
            umma_f16(tmem_base, ah + koff, bh + koff, idesc, acc);
            umma_f16(tmem_base + (uint32_t)BN, ah + koff, bl + koff, idesc, acc);
            umma_f16(tmem_base, al + koff, bh + koff, idesc, 1u);
          } else if (three) {
            // xh*[wh;wl] as ONE N=2*BN MMA (the lo weight tile follows the hi tile in smem) into
            // columns [0,BN) | [BN,2BN), then xl*wh into [0,BN): 2 operand-A reads per K-step, not 3
            umma_f16(tmem_base, ah + koff, bh + koff, idesc2, acc);
            umma_f16(tmem_base, al + koff, bh + koff, idesc, 1u);
          } else {
            umma_f16(tmem_base, ah + koff, bh + koff, idesc, acc);
          }
        }
        umma_commit(empty_bar(s));                         // frees the smem stage once these MMAs have read it
        if (it == total - 1) umma_commit(tmem_full_bar);   // accumulator complete
      }
      __syncwarp();
    }
    TL_MARK(2);                             // all MMAs issued
  }
  pdl_wait();   // every warp: the epilogue reads tensors the previous kernel wrote
#ifdef DSVC_TIMELINE
  tc_epilogue<Epi, BN>(ep, smem_raw, smem_base, tmem_base, tmem_full_bar, 0u, T, N, m0, (int)blockIdx.y, b, warp, lane, three, tl0);
#else
  tc_epilogue<Epi, BN>(ep, smem_raw, smem_base, tmem_base, tmem_full_bar, 0u, T, N, m0, (int)blockIdx.y, b, warp, lane, three);
#endif
  if (warp == 4) TL_MARK(6);               // epilogue done
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * BN) : "memory");
  }
#endif
}

// ---- host side ------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline int tc_encode_fn(PFN_encodeTiled* out) {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    DSVC_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !p) {
      set_error("cuTensorMapEncodeTiled is not available from the installed driver");
      return DSVC_ECUDA;
    }
    fn = (PFN_encodeTiled)p;
  }
  *out = fn;
  return DSVC_OK;
}

// activation plane [B][T][K] fp16, box = {64 channels, 128 frames, 1 item}
static inline CUtensorMapSwizzle tc_swizzle_of(int kb) {
  return kb == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (kb == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}
// (kb: fp16 elements per operand row -- 64, or 32 / 16 for the narrow vocoder stages whose K per tap is that small)
static inline int tc_make_a_map(CUtensorMap* m, const __half* base, int B, int T, int K, int box_rows = TC_BM, int kb = TC_BK) {
  PFN_encodeTiled enc;
  DSVC_TRY(tc_encode_fn(&enc));
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)T * K * 2};
  cuuint32_t box[3] = {(cuuint32_t)kb, (cuuint32_t)box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   tc_swizzle_of(kb), CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(A [%d][%d][%d]) failed: %d", B, T, K, (int)r); return DSVC_ECUDA; }
  return DSVC_OK;
}
// weight matrix [rows][K] fp16, box = {64, box_rows}
static inline int tc_make_b_map(CUtensorMap* m, const __half* base, int rows, int K, int box_rows, int kb = TC_BK) {
  PFN_encodeTiled enc;
  DSVC_TRY(tc_encode_fn(&enc));
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)kb, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   tc_swizzle_of(kb), CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(B [%d][%d]) failed: %d", rows, K, (int)r); return DSVC_ECUDA; }
  return DSVC_OK;
}

template <class Epi, int BN>
int tc_launch_bn(const TcGemmMaps& m, const typename Epi::Params& e, int B, int T, int K, int N, int taps, int dil, int passes,
                 cudaStream_t s, TcTiles tt = TcTiles{}) {
  DSVC_TRY((ensure_dyn_smem<tc_gemm_kernel<Epi, BN>>(TcCfg<BN>::SMEM)));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = tt.tab ? dim3(tt.slots, ceil_div(N, BN), 1) : dim3(ceil_div(T, TC_BM), ceil_div(N, BN), B);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = TcCfg<BN>::SMEM;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const bool b64 = (BN == 256) && Epi::kPair;
  const CUtensorMap& bh = (BN == 64) ? m.b32_hi : (b64 ? m.b64_hi : m.b_hi);
  const CUtensorMap& bl = (BN == 64) ? m.b32_lo : (b64 ? m.b64_lo : m.b_lo);
  DSVC_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<Epi, BN>, m.a_hi, m.a_lo, bh, bl, e, T, K, N, taps, dil, passes, tt.tab));
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

// DSVC_TC_BN=64|128|256 forces the tile width (read per call: the parity tests switch it per handle)
inline int tc_forced_bn() {
  const char* e = getenv("DSVC_TC_BN");
  return e ? atoi(e) : -1;
}

// Tile width: the one that minimises  waves x (time of one CTA of that width),  waves = ceil(CTAs / SMs).  Relative CTA
// times measured with the layer kernels on a B200 (profiles/r2a_pair_vs_single_ab.txt: one clip, 64-wide tiles, conv
// kernel 9.4 us; 8 clips, 256-wide tiles, one wave, 25.4 us; 128-wide tiles, two waves, 29.5 us):  64: 0.37,
// 128: 0.56, 256: 1.  One 10 s clip -> 64 (96 CTAs, one wave); 8 x 689 frames -> 256 (144 CTAs, one wave); a ragged batch
// whose live tiles just miss one wave of 256-wide tiles (e.g. 50 x 3 = 150 CTAs) -> 128 instead of two waves of 256.
// (mtiles: frame tiles that do work -- the live entries of a ragged batch's tile table, else B * ceil(T / 128))
inline int tc_pick_bn(int B, int T, int N, int live_tiles = 0) {
  const long long mtiles = live_tiles > 0 ? live_tiles : (long long)ceil_div(T, TC_BM) * B;
  const int forced = tc_forced_bn();
  if (forced == 64 && N % 64 == 0) return 64;
  if (forced == 256 && N % 256 == 0) return 256;
  if (forced == 128 || forced == 256 || forced == 64) return (N % 128 != 0 && N % 64 == 0) ? 64 : 128;
  if (N % 128 != 0 && N % 64 == 0) return 64;        // a 128-wide tile would be half empty
  static const int sms = [] {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
  }();
  const int widths[3] = {64, 128, 256};
  const double cost[3] = {0.37, 0.56, 1.0};
  int best = 128;
  double best_t = 1e30;
  for (int i = 0; i < 3; ++i) {
    if (N % widths[i] != 0) continue;
    const long long ctas = mtiles * (N / widths[i]);
    const double t = (double)((ctas + sms - 1) / sms) * cost[i];
    if (t < best_t - 1e-9) { best_t = t; best = widths[i]; }      // ties: the narrower tile (more SMs busy, shorter chain)
  }
  return best;
}
inline int tc_ctas_per_mtile(int B, int T, int N) { return ceil_div(N, tc_pick_bn(B, T, N)); }

template <class Epi>
int tc_launch_single(const TcGemmMaps& m, const typename Epi::Params& e, int B, int T, int K, int N, int taps, int dil, int passes,
                     cudaStream_t s, TcTiles tt = TcTiles{}) {
  DSVC_REQUIRE(K % TC_BK == 0, "tc_launch: K=%d must be a multiple of %d", K, TC_BK);
  const int bn = tc_pick_bn(B, T, N, tt.live);
  if (bn == 64) return tc_launch_bn<Epi, 64>(m, e, B, T, K, N, taps, dil, passes, s, tt);
  if (bn == 256) return tc_launch_bn<Epi, 256>(m, e, B, T, K, N, taps, dil, passes, s, tt);
  return tc_launch_bn<Epi, 128>(m, e, B, T, K, N, taps, dil, passes, s, tt);
}

}  // namespace dsvc
