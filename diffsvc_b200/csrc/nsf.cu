// NSF-HiFiGAN generator: harmonic-plus-noise source, transposed-conv upsampling, MRF residual blocks.
// Reference: modules/nsf_hifigan/models.py:148-387 (SineGen :148, SourceModuleHnNSF :277,
// ResBlock1 :33, ResBlock2 :73, effective Generator :325), called from network/vocoders/nsf_hifigan.py:36-72.
//
// Activations are channels-last fp32 [B][L][C]; every Conv1d / ConvTranspose1d is an implicit GEMM
// (simt_gemm.cuh) with the LeakyReLU fused into the operand load and bias / residual / MRF
// accumulation fused into the epilogue.
#include "common.cuh"
#include "epilogues.cuh"
#include "simt_gemm.cuh"
#include "tc_pair.cuh"
#include "tc_narrow.cuh"

#include <memory>

namespace dsvc {

// ---------------------------------------------------------------------------------------------
// source module (models.py:177-276, :310-323)
// ---------------------------------------------------------------------------------------------
// torch.cumsum on CPU accumulates float tensors in double and rounds every prefix to float
// (acc_type<float, false> = double).  f0 is piecewise constant over a hop (nearest upsampling,
// models.py:331,363), so prefix sums have closed forms per frame; all scans run in fp64.

struct SrcDims { int B, T, hop, dim; float sr; };

__device__ __forceinline__ float rad_of(float f0, int h, float sr) {
  // (f0 * (h+1) / sr) % 1   (models.py:252-257, :188)
  return fmodf(div_rn(mul_rn(f0, (float)(h + 1)), sr), 1.0f);
}

// Exclusive running sum over the frames of one (item, harmonic) sequence, in the reference's order (torch's CPU
// cumsum adds sequentially in double): a warp fetches 32 frame increments at a time and every lane replays the
// 32 dependent adds from shuffles -- same rounding as a serial loop, without a global-memory round trip per frame.
template <class Inc>
__device__ __forceinline__ void warp_serial_scan(int T, double* __restrict__ dst, Inc inc_of) {
  const int lane = threadIdx.x & 31;
  double s = 0.0;
  for (int f0i = 0; f0i < T; f0i += 32) {
    const int f = f0i + lane;
    const double inc = f < T ? inc_of(f) : 0.0;
    double mine = 0.0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const double v = __shfl_sync(0xffffffffu, inc, j);
      if (lane == j) mine = s;
      s += v;
    }
    if (f < T) dst[f] = mine;
  }
}

// pass 1: S1[b][h][f] = sum_{f' < f} hop * rad_{f'}  (double), E[b][h] = extra of the initial phase.  One warp per sequence.
__global__ void __launch_bounds__(32)
src_frames1_kernel(SrcDims d, const float* __restrict__ f0, const float* __restrict__ rand_ini,
                   unsigned long long seed, double* __restrict__ S1, double* __restrict__ E) {
  const int i = blockIdx.x;
  const int b = i / d.dim, h = i % d.dim;
  if (threadIdx.x == 0) {
    float ri = 0.f;
    if (h > 0) ri = rand_ini ? rand_ini[b * d.dim + h] : philox_uniform(seed, 0x72616e64u, (uint64_t)b * d.dim + h);
    const float r0 = rad_of(f0[(size_t)b * d.T], h, d.sr);
    E[i] = (double)add_rn(r0, ri) - (double)r0;          // rad[:,0,:] += rand_ini  (models.py:195)
  }
  const float* f0b = f0 + (size_t)b * d.T;
  warp_serial_scan(d.T, S1 + (size_t)i * d.T, [&](int f) { return (double)d.hop * (double)rad_of(f0b[f], h, d.sr); });
}

// wrap flag of sample (f, k): (cumsum % 1)[n] - (cumsum % 1)[n-1] < 0   (models.py:205-207)
__device__ __forceinline__ bool wrap_flag(double base, float rad, int f, int k) {
  if (f == 0 && k == 0) return false;                  // cumsum_shift[:, 0] stays 0
  const float c_now = (float)(base + (double)(k + 1) * (double)rad);
  const float c_prev = (float)(base + (double)k * (double)rad);
  return sub_rn(fmodf(c_now, 1.0f), fmodf(c_prev, 1.0f)) < 0.0f;
}

// block-wide inclusive scan of 0/1 flags (blockDim multiple of 32, <= 1024)
__device__ __forceinline__ int block_scan_flags(bool flag, int* smem, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const unsigned bal = __ballot_sync(0xffffffffu, flag);
  const int incl = __popc(bal & (0xffffffffu >> (31 - lane)));
  if (lane == 0) smem[warp] = __popc(bal);
  __syncthreads();
  int off = 0, tot = 0;
  for (int w = 0; w < nwarp; ++w) {
    const int c = smem[w];
    if (w < warp) off += c;
    tot += c;
  }
  __syncthreads();
  total = tot;
  return off + incl;
}

// pass 2: W[b][h][f] = number of wraps inside frame f
__global__ void src_wraps_kernel(SrcDims d, const float* __restrict__ f0, const double* __restrict__ S1,
                                 const double* __restrict__ E, int* __restrict__ W) {
  __shared__ int sm[32];
  const int f = blockIdx.x, b = blockIdx.y;
  const float f0v = f0[(size_t)b * d.T + f];
  for (int h = 0; h < d.dim; ++h) {
    const int i = b * d.dim + h;
    const float rad = rad_of(f0v, h, d.sr);
    const double base = E[i] + S1[(size_t)i * d.T + f];
    int cnt = 0;
    for (int k0 = 0; k0 < d.hop; k0 += blockDim.x) {
      const int k = k0 + threadIdx.x;
      const bool fl = (k < d.hop) && wrap_flag(base, rad, f, k);
      int tot;
      block_scan_flags(fl, sm, tot);
      cnt += tot;
    }
    if (threadIdx.x == 0) W[(size_t)i * d.T + f] = cnt;
  }
}

// pass 3: S2[b][h][f] = sum over earlier frames of (rad + shift)   (double).  One warp per sequence.
__global__ void __launch_bounds__(32)
src_frames2_kernel(SrcDims d, const float* __restrict__ f0, const int* __restrict__ W, double* __restrict__ S2) {
  const int i = blockIdx.x;
  const int b = i / d.dim, h = i % d.dim;
  const float* f0b = f0 + (size_t)b * d.T;
  const int* Wi = W + (size_t)i * d.T;
  warp_serial_scan(d.T, S2 + (size_t)i * d.T, [&](int f) {
    const float rad = rad_of(f0b[f], h, d.sr);
    const int w = Wi[f];
    return (double)(d.hop - w) * (double)rad + (double)w * (double)add_rn(rad, -1.0f);
  });
}

// pass 4: sines, uv, additive noise, harmonic merge Linear(dim -> 1) + tanh  -> har[b][n]
__global__ void src_synth_kernel(SrcDims d, const float* __restrict__ f0, const double* __restrict__ S1,
                                 const double* __restrict__ S2, const double* __restrict__ E,
                                 const float* __restrict__ sine_noise, unsigned long long seed,
                                 const float* __restrict__ lin_w, const float* __restrict__ lin_b,
                                 float* __restrict__ har) {
  __shared__ int sm[32];
  const int f = blockIdx.x, b = blockIdx.y;
  const float f0v = f0[(size_t)b * d.T + f];
  const float uv = f0v > 0.0f ? 1.0f : 0.0f;                         // _f02uv, voiced_threshold 0
  const float noise_amp = add_rn(mul_rn(uv, 0.003f), div_rn(mul_rn(sub_rn(1.0f, uv), 0.1f), 3.0f));   // :270
  const size_t L = (size_t)d.T * d.hop;
  for (int k0 = 0; k0 < d.hop; k0 += blockDim.x) {
    const int k = k0 + threadIdx.x;
    float accum = 0.f;
    for (int h = 0; h < d.dim; ++h) {
      const int i = b * d.dim + h;
      const float rad = rad_of(f0v, h, d.sr);
      const double base1 = E[i] + S1[(size_t)i * d.T + f];
      // wraps among samples k' <= k of this frame: earlier chunks + scan inside this chunk
      int before = 0;
      for (int kk0 = 0; kk0 < k0; kk0 += blockDim.x) {
        const int kk = kk0 + threadIdx.x;
        int tot;
        block_scan_flags(wrap_flag(base1, rad, f, kk), sm, tot);
        before += tot;
      }
      int tot;
      const bool fl = (k < d.hop) && wrap_flag(base1, rad, f, k);
      const int wk = before + block_scan_flags(fl, sm, tot);
      if (k < d.hop) {
        const double c2 = E[i] + S2[(size_t)i * d.T + f] + (double)(k + 1 - wk) * (double)rad +
                          (double)wk * (double)add_rn(rad, -1.0f);
        const float ph = mul_rn(mul_rn((float)c2, 2.0f), 3.14159265358979323846f);   // cumsum * 2 * np.pi
        const float sine = mul_rn(sinf(ph), 0.1f);                                   // * sine_amp
        const size_t n = (size_t)f * d.hop + k;
        const size_t nidx = ((size_t)b * L + n) * d.dim + h;
        const float nz = sine_noise ? __ldg(sine_noise + nidx) : philox_normal(seed, 0x73696e65u, nidx);
        const float sw = add_rn(mul_rn(sine, uv), mul_rn(noise_amp, nz));            // :275
        accum = fmaf(lin_w[h], sw, accum);
      }
    }
    if (k < d.hop) har[(size_t)b * L + (size_t)f * d.hop + k] = tanhf(accum + lin_b[0]);
  }
}

// ---------------------------------------------------------------------------------------------
// noise_convs[i](har_source) added to the upsampled stream (models.py:370-374)
//   x[b][p][co] += bias[co] + sum_j w[co][j] * har[b][p*s - pad + j]
// ---------------------------------------------------------------------------------------------
//   w is stored [K][Cout] (channel-contiguous: a warp's weight read is one line); a thread owns one channel and
//   NP consecutive positions so that every weight feeds NP FMAs.
constexpr int NOISE_PB = 32;   // positions per block
constexpr int NOISE_NP = 4;    // positions per thread
__global__ void __launch_bounds__(256)
noise_conv_add_kernel(const float* __restrict__ har, const float* __restrict__ wt, const float* __restrict__ bias,
                      float* __restrict__ x, int Lsrc, int Lout, int Cout, int K, int stride, int pad) {
  extern __shared__ float sh[];   // har window for the block's positions
  const int b = blockIdx.y;
  const int p0 = blockIdx.x * NOISE_PB;
  const int span = (NOISE_PB - 1) * stride + K;
  for (int i = threadIdx.x; i < span; i += blockDim.x) {
    const int n = p0 * stride - pad + i;
    sh[i] = (n >= 0 && n < Lsrc) ? har[(size_t)b * Lsrc + n] : 0.f;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < (NOISE_PB / NOISE_NP) * Cout; idx += blockDim.x) {
    const int pg = idx / Cout, co = idx % Cout;
    const int pl = pg * NOISE_NP;
    float acc[NOISE_NP];
#pragma unroll
    for (int q = 0; q < NOISE_NP; ++q) acc[q] = 0.f;
    for (int j = 0; j < K; ++j) {
      const float wv = __ldg(wt + (size_t)j * Cout + co);
#pragma unroll
      for (int q = 0; q < NOISE_NP; ++q) acc[q] = fmaf(wv, sh[(pl + q) * stride + j], acc[q]);
    }
    const float bv = bias[co];
#pragma unroll
    for (int q = 0; q < NOISE_NP; ++q) {
      const int p = p0 + pl + q;
      if (p < Lout) {
        const size_t o = ((size_t)b * Lout + p) * Cout + co;
        x[o] = add_rn(x[o], acc[q] + bv);
      }
    }
  }
}

// conv_post (Cout = 1, k = 7) on leaky_relu(x, 0.01) then tanh (models.py:383-385)
__global__ void conv_post_tanh_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                      float* __restrict__ wav, int L, int C, int K, float slope) {
  const int b = blockIdx.y;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= L) return;
  float acc = 0.f;
  const int pad = (K - 1) / 2;
  for (int j = 0; j < K; ++j) {
    const int q = n - pad + j;
    if (q < 0 || q >= L) continue;
    const float* xr = x + ((size_t)b * L + q) * C;
    const float* wr = w + (size_t)j * C;
    for (int c = 0; c < C; c += 4) {
      const float4 v = *reinterpret_cast<const float4*>(xr + c);
      const float4 ww = __ldg(reinterpret_cast<const float4*>(wr + c));
      acc = fmaf(lrelu_(v.x, slope), ww.x, acc);
      acc = fmaf(lrelu_(v.y, slope), ww.y, acc);
      acc = fmaf(lrelu_(v.z, slope), ww.z, acc);
      acc = fmaf(lrelu_(v.w, slope), ww.w, acc);
    }
  }
  wav[(size_t)b * L + n] = tanhf(acc + bias[0]);
}

// mel [B][T][M] * scale -> c   (c = 2.30259 * mel, nsf_hifigan.py:39)
__global__ void scale_kernel(const float* __restrict__ in, float* __restrict__ out, size_t n, float s) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = mul_rn(s, in[i]);
}

struct ConvW {
  DevBuf w, b;
  int Cin = 0, Cout = 0, K = 0;
  // tcgen05 path (ResBlock convs whose channel count tiles by 64): fp16 hi/lo weights [K][Cout][Cin] + their TMA maps
  bool tc = false;
  int kb = 0;                 // narrow convs (Cin = Cout = 32 / 16) on tcgen05 (tc_narrow.cuh): operand rows of Cin fp16
  int pad = NW_PAD;           // ... and the rows their activation window reaches either side of a tile
  F16Pair h16;
  CUtensorMap bh, bl, b32h, b32l, b64h, b64l;   // weight boxes of 128 / 32 / 64 rows (tc_gemm.cuh, tc_pair.cuh)
};

// x -> fp16 (hi, lo) planes of leaky_relu(x): the operand of the first conv of every ResBlock of a stage
__global__ void act_split_kernel(const float* __restrict__ x, __half* __restrict__ hi, __half* __restrict__ lo, size_t n4, float slope) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 v = reinterpret_cast<const float4*>(x)[i];
  const float y[4] = {lrelu_(v.x, slope), lrelu_(v.y, slope), lrelu_(v.z, slope), lrelu_(v.w, slope)};
  Plane pl{nullptr, hi, lo};
  plane_store4(pl, i * 4, y);
}

}  // namespace dsvc

using namespace dsvc;

struct NsfStageMaps {          // activation-plane TMA maps of one upsample stage (depend on B, T)
  bool tc = false;
  TcGemmMaps px, pa, pt;
};

struct dsvc_nsf {
  dsvc_nsf_config cfg;
  int resblock = 1;            // 1: ResBlock1 (convs1 / convs2 pairs), 2: ResBlock2 (two convs, c1 only)
  int hop = 1;
  bool tc_enabled = true;      // DSVC_NSF_MATH=fp32 forces the FFMA path everywhere
  int narrow_pad = NW_PAD;     // window half-height of tc_narrow.cuh for the 32- / 16-channel stages; 0 = FFMA GEMM
  PlaneBuf PX, PA, PT;         // leaky_relu'ed operand planes: stage input, ResBlock state, conv1 output
  std::vector<NsfStageMaps> smaps;
  int maps_B = 0, maps_T = 0;
  const void* maps_base = nullptr;
  DevBuf lin_w, lin_b;
  ConvW pre, post;
  std::vector<std::unique_ptr<ConvW>> ups, noise, c1, c2;
  std::vector<int> ups_taps;
  // workspace
  int B = 0, T = 0;
  DevBuf melc, har, S1, S2, E, W, bufA, bufU, bufT, bufR0, bufR1, bufS;
};

namespace dsvc {

// [Cout][Cin][K] (PyTorch Conv1d) -> [K][Cout][Cin]
static int upload_conv(ConvW& c, const float* w, const float* b, int Cout, int Cin, int K, cudaStream_t s, bool tc = false) {
  std::vector<float> r((size_t)K * Cout * Cin);
  for (int co = 0; co < Cout; ++co)
    for (int ci = 0; ci < Cin; ++ci)
      for (int k = 0; k < K; ++k) r[((size_t)k * Cout + co) * Cin + ci] = w[((size_t)co * Cin + ci) * K + k];
  c.Cin = Cin; c.Cout = Cout; c.K = K;
  DSVC_TRY(c.b.upload(b, (size_t)Cout * 4, s));
  c.tc = tc;
  if (tc && Cin < 64) {
    // narrow conv (tc_narrow.cuh): the whole [tap][Cout][Cin] set sits in shared memory, one box of Cout rows per tap
    DSVC_REQUIRE(Cin == Cout && (Cin == 32 || Cin == 16), "narrow tcgen05 conv needs Cin == Cout in {32, 16} (got %d -> %d)", Cin, Cout);
    c.kb = Cin;
    DSVC_TRY(c.w.upload(r.data(), r.size() * 4, s));     // the FFMA form too (DSVC_NSF_NARROW=0, pairs off)
    DSVC_TRY(make_f16_pair(c.h16, r.data(), r.size(), s));
    DSVC_TRY(tc_make_b_map(&c.b32h, c.h16.hi.as<__half>(), K * Cout, Cin, Cout, Cin));
    DSVC_TRY(tc_make_b_map(&c.b32l, c.h16.lo.as<__half>(), K * Cout, Cin, Cout, Cin));
    c.bh = c.b64h = c.b32h; c.bl = c.b64l = c.b32l;
  } else if (tc) {   // the tcgen05 path reads only the fp16 pair (same [tap][Cout][Cin] row order)
    DSVC_TRY(make_f16_pair(c.h16, r.data(), r.size(), s));
    DSVC_TRY(tc_make_b_map(&c.bh, c.h16.hi.as<__half>(), K * Cout, Cin, 128));
    DSVC_TRY(tc_make_b_map(&c.bl, c.h16.lo.as<__half>(), K * Cout, Cin, 128));
    DSVC_TRY(tc_make_b_map(&c.b32h, c.h16.hi.as<__half>(), K * Cout, Cin, 32));
    DSVC_TRY(tc_make_b_map(&c.b32l, c.h16.lo.as<__half>(), K * Cout, Cin, 32));
    DSVC_TRY(tc_make_b_map(&c.b64h, c.h16.hi.as<__half>(), K * Cout, Cin, 64));
    DSVC_TRY(tc_make_b_map(&c.b64l, c.h16.lo.as<__half>(), K * Cout, Cin, 64));
  } else {
    DSVC_TRY(c.w.upload(r.data(), r.size() * 4, s));
  }
  DSVC_CUDA(cudaStreamSynchronize(s));
  return DSVC_OK;
}

// ConvTranspose1d [Cin][Cout][K], stride u, padding (K-u)/2 -> per output phase r:
//   [r][i][Cout][Cin] = W[ci][co][k0 + i*u], k0 = (r + pad) % u, zero when k >= K
static int upload_convT(ConvW& c, int& taps, const float* w, const float* b, int Cin, int Cout, int K, int u, cudaStream_t s) {
  const int pad = (K - u) / 2;
  taps = (K + u - 1) / u;
  std::vector<float> r((size_t)u * taps * Cout * Cin, 0.f);
  for (int ph = 0; ph < u; ++ph) {
    const int k0 = (ph + pad) % u;
    for (int i = 0; i < taps; ++i) {
      const int k = k0 + i * u;
      if (k >= K) continue;
      for (int co = 0; co < Cout; ++co)
        for (int ci = 0; ci < Cin; ++ci)
          r[(((size_t)ph * taps + i) * Cout + co) * Cin + ci] = w[((size_t)ci * Cout + co) * K + k];
    }
  }
  c.Cin = Cin; c.Cout = Cout; c.K = K;
  DSVC_TRY(c.w.upload(r.data(), r.size() * 4, s));
  DSVC_TRY(c.b.upload(b, (size_t)Cout * 4, s));
  DSVC_CUDA(cudaStreamSynchronize(s));
  return DSVC_OK;
}

static int launch_affine(const ConvGemmParams& p, const EpiAffine::Params& e, cudaStream_t s) {
  if (p.Cout > 64) {
    const long long ctas = (long long)ceil_div(p.rows, 128) * ceil_div(p.Cout, 128) * p.B * (p.nphase > 1 ? p.nphase : 1);
    if (ctas >= 2 * 148) return launch_conv_gemm_tile<128, 128, 8, 8, EpiAffine>(p, e, s);
    return launch_conv_gemm_tile<64, 128, 4, 8, EpiAffine>(p, e, s);
  }
  if (p.Cout > 32) return launch_conv_gemm_tile<128, 64, 8, 4, EpiAffine>(p, e, s);
  if (p.Cout > 16) return launch_conv_gemm_tile<256, 32, 8, 4, EpiAffine>(p, e, s);
  return launch_conv_gemm_tile<256, 16, 4, 4, EpiAffine>(p, e, s);
}

// out[b][p][:] (+)= conv(lrelu(in)) + bias (+ res), dilation d, "same" padding
static int conv_same(const ConvW& c, const float* in, float* out, const float* res, int B, int L, int dil, float slope,
                     int accumulate, float div, cudaStream_t s) {
  ConvGemmParams p{};
  p.A = in; p.W = c.w.as<float>(); p.B = B; p.Lin = L; p.Cin = c.Cin; p.Cout = c.Cout; p.taps = c.K; p.rows = L;
  p.in_stride = 1; p.in_off = -((c.K * dil - dil) / 2); p.tap_step = dil; p.nphase = 1; p.tpad = 0; p.in_slope = slope;
  p.a_batch_stride = (long long)L * c.Cin;
  EpiAffine::Params e{};
  e.bias = c.b.as<float>(); e.res = res; e.out = out; e.Lout = L; e.Cout = c.Cout; e.accumulate = accumulate; e.div = div;
  e.act = EpiAffine::ACT_NONE;
  return launch_affine(p, e, s);
}

// the same convolution on the tcgen05 path: `in` are the TMA maps of the (already leaky_relu'ed) operand planes
static int conv_same_tc(const ConvW& c, const TcGemmMaps& in, EpiVoc::Params e, int B, int L, int dil, cudaStream_t s) {
  TcGemmMaps g = in;
  g.b_hi = c.bh; g.b_lo = c.bl; g.b32_hi = c.b32h; g.b32_lo = c.b32l; g.b64_hi = c.b64h; g.b64_lo = c.b64l;
  e.bias = c.b.as<float>(); e.Lout = L; e.Cout = c.Cout; e.wscale = c.h16.inv_scale;
  if (c.kb == 32 && c.pad == NW_PAD) return tc_narrow_launch<32, NW_PAD>(in.a_hi, in.a_lo, c.b32h, c.b32l, e, B, L, c.K, dil, s);
  if (c.kb == 16 && c.pad == NW_PAD) return tc_narrow_launch<16, NW_PAD>(in.a_hi, in.a_lo, c.b32h, c.b32l, e, B, L, c.K, dil, s);
  if (c.kb == 32) return tc_narrow_launch<32, NW_PAD_WIDE>(in.a_hi, in.a_lo, c.b32h, c.b32l, e, B, L, c.K, dil, s);
  if (c.kb == 16) return tc_narrow_launch<16, NW_PAD_WIDE>(in.a_hi, in.a_lo, c.b32h, c.b32l, e, B, L, c.K, dil, s);
  return tc_launch<EpiVoc>(g, e, B, L, c.Cin, c.Cout, c.K, dil, 3, s);
}

// The 32- / 16-channel stages run on the weights-stationary narrow kernel (tc_narrow.cuh); DSVC_NSF_NARROW=0 keeps them
// on the FFMA GEMM (their weights are kept in both forms).
static bool nsf_tc_channels(const dsvc_nsf* h, int ch) {
  if (ch % 64 == 0) return true;
  return (ch == 32 || ch == 16) && h->narrow_pad > 0;
}
// ... when every ResBlock conv's taps stay inside the kernel's activation window (k/2 * dilation <= pad rows): the
// 192-row window (pad 32) when it fits; for ResBlock2 generators the 256-row one (pad 64) next.  ResBlock1 generators
// that reach past 32 rows stay on FFMA.  Returns the pad, 0 for the FFMA GEMM.
static int nsf_narrow_pad(const dsvc_nsf_config& cfg, int resblock) {
  const char* e = getenv("DSVC_NSF_NARROW");
  if (e && atoi(e) == 0) return 0;
  int reach = 0;
  for (int j = 0; j < cfg.num_kernels; ++j)
    for (int m = 0; m < cfg.num_dilations; ++m)
      reach = std::max(reach, (cfg.resblock_kernel_sizes[j] / 2) * std::max(1, cfg.resblock_dilation_sizes[j][m]));
  if (reach <= NW_PAD) return NW_PAD;
  if (resblock == 2 && reach <= NW_PAD_WIDE) return NW_PAD_WIDE;
  return 0;
}

// (re)build the activation-plane maps for a (B, T) shape
static int nsf_build_maps(dsvc_nsf* h, int B, int T) {
  const dsvc_nsf_config& cfg = h->cfg;
  if (h->maps_B == B && h->maps_T == T && h->maps_base == h->PX.hi.p) return DSVC_OK;
  h->smaps.assign(cfg.num_upsamples, NsfStageMaps{});
  int len = T, ch = cfg.upsample_initial_channel;
  for (int i = 0; i < cfg.num_upsamples; ++i) {
    len *= cfg.upsample_rates[i];
    ch >>= 1;
    NsfStageMaps& m = h->smaps[i];
    m.tc = h->tc_enabled && nsf_tc_channels(h, ch);
    if (!m.tc) continue;
    // narrow stages: operand rows of `ch` fp16 and one 192- / 256-row window per tile (tc_narrow.cuh); else [128 x 64] tiles
    const int kb = ch < 64 ? ch : TC_BK, box_rows = ch < 64 ? nw_rows(h->narrow_pad) : TC_BM;
    auto planes = [&](TcGemmMaps& g, const PlaneBuf& pb) -> int {
      DSVC_TRY(tc_make_a_map(&g.a_hi, pb.hi.as<__half>(), B, len, ch, box_rows, kb));
      DSVC_TRY(tc_make_a_map(&g.a_lo, pb.lo.as<__half>(), B, len, ch, box_rows, kb));
      return DSVC_OK;
    };
    DSVC_TRY(planes(m.px, h->PX));
    DSVC_TRY(planes(m.pa, h->PA));
    DSVC_TRY(planes(m.pt, h->PT));
  }
  h->maps_B = B; h->maps_T = T; h->maps_base = h->PX.hi.p;
  return DSVC_OK;
}

// MRF of ResBlock2 generators (models.py:86-91): per kernel j, x1 = c0(lrelu(xu)) + xu, xs (+)= c1(lrelu(x1)) + x1,
// the last j divides by num_kernels.  On tcgen05, conv 0 reads PX (lrelu(xu), written once per stage) and its epilogue
// writes x1 and the planes of lrelu(x1) to PA, which conv 1 reads.  On the FFMA GEMM the LeakyReLU is on the operand load.
static int nsf_mrf_resblock2(dsvc_nsf* h, int i, const float* xu, float* xs, int B, int lout, cudaStream_t s) {
  const dsvc_nsf_config& cfg = h->cfg;
  const int nk = cfg.num_kernels, C = h->c1[i * nk * 2]->Cout;
  float* x1 = h->bufR0.as<float>();
  const NsfStageMaps& sm = h->smaps[i];
  if (sm.tc) {
    const size_t n4 = (size_t)B * lout * C / 4;
    act_split_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(xu, h->PX.hi.as<__half>(), h->PX.lo.as<__half>(), n4, 0.1f);
    DSVC_LAUNCH_CHECK();
  }
  for (int j = 0; j < nk; ++j) {
    const ConvW& c0 = *h->c1[(i * nk + j) * 2];
    const ConvW& c1 = *h->c1[(i * nk + j) * 2 + 1];
    const int d0 = cfg.resblock_dilation_sizes[j][0], d1 = cfg.resblock_dilation_sizes[j][1];
    const int acc = j > 0 ? 1 : 0;
    const float div = (j + 1 == nk) ? (float)nk : 1.0f;
    if (sm.tc) {
      EpiVoc::Params e0{};
      e0.res = xu; e0.out = x1; e0.act = h->PA.view(true); e0.div = 1.0f; e0.slope = 0.1f;
      DSVC_TRY(conv_same_tc(c0, sm.px, e0, B, lout, d0, s));
      EpiVoc::Params e1{};
      e1.res = x1; e1.out = xs; e1.accumulate = acc; e1.div = div; e1.slope = 0.1f;
      DSVC_TRY(conv_same_tc(c1, sm.pa, e1, B, lout, d1, s));
    } else {
      DSVC_TRY(conv_same(c0, xu, x1, xu, B, lout, d0, 0.1f, 0, 1.0f, s));
      DSVC_TRY(conv_same(c1, x1, xs, x1, B, lout, d1, 0.1f, acc, div, s));
    }
  }
  return DSVC_OK;
}

}  // namespace dsvc

extern "C" {

int dsvc_nsf_create(dsvc_nsf_t** out, const dsvc_nsf_config* cfg, const dsvc_nsf_weights* w, void* stream) {
  return dsvc_nsf_create_ex(out, cfg, 1, w, stream);
}

int dsvc_nsf_create_ex(dsvc_nsf_t** out, const dsvc_nsf_config* cfg, int32_t resblock, const dsvc_nsf_weights* w,
                       void* stream) {
  DSVC_REQUIRE(out && cfg && w, "dsvc_nsf_create: null argument");
  DSVC_TRY(require_device());
  DSVC_REQUIRE(resblock == 1 || resblock == 2, "resblock %d: expected 1 (ResBlock1) or 2 (ResBlock2)", resblock);
  DSVC_REQUIRE(resblock == 1 || (cfg->num_dilations == 2 && !w->convs2_w && !w->convs2_b),
               "ResBlock2 takes exactly two convs per block (num_dilations 2, got %d) in convs1_*, and convs2_* NULL",
               cfg->num_dilations);
  DSVC_REQUIRE(cfg->num_upsamples >= 1 && cfg->num_upsamples <= DSVC_NSF_MAX_STAGES, "num_upsamples %d out of range", cfg->num_upsamples);
  DSVC_REQUIRE(cfg->num_kernels >= 1 && cfg->num_kernels <= DSVC_NSF_MAX_KERNELS, "num_kernels %d out of range", cfg->num_kernels);
  DSVC_REQUIRE(cfg->num_dilations >= 1 && cfg->num_dilations <= DSVC_NSF_MAX_DILATIONS, "num_dilations %d out of range", cfg->num_dilations);
  DSVC_REQUIRE(cfg->harmonic_num >= 0 && cfg->harmonic_num < 32, "harmonic_num out of range");
  cudaStream_t s = (cudaStream_t)stream;
  std::unique_ptr<dsvc_nsf> h(new dsvc_nsf());
  h->cfg = *cfg;
  h->resblock = resblock;
  {
    const char* ev = getenv("DSVC_NSF_MATH");
    h->tc_enabled = !(ev && strcmp(ev, "fp32") == 0);
    h->narrow_pad = nsf_narrow_pad(*cfg, resblock);
  }
  const int ns = cfg->num_upsamples, nk = cfg->num_kernels, nd = cfg->num_dilations, dim = cfg->harmonic_num + 1;
  int ch = cfg->upsample_initial_channel;
  h->hop = 1;
  for (int i = 0; i < ns; ++i) {
    const int u = cfg->upsample_rates[i], K = cfg->upsample_kernel_sizes[i];
    DSVC_REQUIRE(u >= 1 && K >= u && (K - u) % 2 == 0, "stage %d: unsupported ConvTranspose1d k=%d stride=%d", i, K, u);
    DSVC_REQUIRE((ch >> 1) % 4 == 0, "stage %d: output channels %d must be a multiple of 4", i, ch >> 1);
    h->hop *= u;
    ch >>= 1;
  }
  DSVC_REQUIRE(cfg->num_mels % 4 == 0 || true, "num_mels");
  if (cfg->has_source) {
    DSVC_REQUIRE(w->source_linear_w && w->source_linear_b && w->noise_convs_w && w->noise_convs_b, "has_source without source weights");
    DSVC_TRY(h->lin_w.upload(w->source_linear_w, (size_t)dim * 4, s));
    DSVC_TRY(h->lin_b.upload(w->source_linear_b, 4, s));
  }
  DSVC_TRY(upload_conv(h->pre, w->conv_pre_w, w->conv_pre_b, cfg->upsample_initial_channel, cfg->num_mels, 7, s));
  ch = cfg->upsample_initial_channel;
  int rest = h->hop;
  for (int i = 0; i < ns; ++i) {
    const int u = cfg->upsample_rates[i], K = cfg->upsample_kernel_sizes[i];
    const int cin = ch, cout = ch >> 1;
    rest /= u;   // prod(rates[i+1:])
    h->ups.emplace_back(new ConvW());
    int taps = 0;
    DSVC_TRY(upload_convT(*h->ups[i], taps, w->ups_w[i], w->ups_b[i], cin, cout, K, u, s));
    h->ups_taps.push_back(taps);
    h->noise.emplace_back(new ConvW());
    const int Kn = (i + 1 < ns) ? 2 * rest : 1;
    h->noise[i]->Cin = 1; h->noise[i]->Cout = cout; h->noise[i]->K = Kn;
    if (cfg->has_source) {
      std::vector<float> wt((size_t)Kn * cout);     // [cout][1][Kn] -> [Kn][cout]
      for (int co = 0; co < cout; ++co)
        for (int j = 0; j < Kn; ++j) wt[(size_t)j * cout + co] = w->noise_convs_w[i][(size_t)co * Kn + j];
      DSVC_TRY(h->noise[i]->w.upload(wt.data(), wt.size() * 4, s));
      DSVC_CUDA(cudaStreamSynchronize(s));
      DSVC_TRY(h->noise[i]->b.upload(w->noise_convs_b[i], (size_t)cout * 4, s));
    }
    for (int j = 0; j < nk; ++j)
      for (int m = 0; m < nd; ++m) {
        const int idx = (i * nk + j) * nd + m;
        const int k = cfg->resblock_kernel_sizes[j];
        DSVC_REQUIRE(k % 2 == 1, "resblock kernel size %d must be odd", k);
        h->c1.emplace_back(new ConvW());
        const bool tc = h->tc_enabled && nsf_tc_channels(h.get(), cout);
        DSVC_TRY(upload_conv(*h->c1[idx], w->convs1_w[idx], w->convs1_b[idx], cout, cout, k, s, tc));
        h->c1[idx]->pad = h->narrow_pad;
        if (resblock == 2) continue;                   // ResBlock2: resblocks.{i*nk+j}.convs.{m} only
        h->c2.emplace_back(new ConvW());
        DSVC_TRY(upload_conv(*h->c2[idx], w->convs2_w[idx], w->convs2_b[idx], cout, cout, k, s, tc));
        h->c2[idx]->pad = h->narrow_pad;
      }
    ch = cout;
  }
  {  // conv_post [1][ch][7] -> [7][ch]
    std::vector<float> r((size_t)7 * ch);
    for (int c = 0; c < ch; ++c)
      for (int k = 0; k < 7; ++k) r[(size_t)k * ch + c] = w->conv_post_w[(size_t)c * 7 + k];
    h->post.Cin = ch; h->post.Cout = 1; h->post.K = 7;
    DSVC_TRY(h->post.w.upload(r.data(), r.size() * 4, s));
    DSVC_TRY(h->post.b.upload(w->conv_post_b, 4, s));
  }
  DSVC_CUDA(cudaStreamSynchronize(s));
  *out = h.release();
  return DSVC_OK;
}

void dsvc_nsf_destroy(dsvc_nsf_t* h) { delete h; }

int dsvc_nsf_forward(dsvc_nsf_t* h, const float* mel, const float* f0, const float* rand_ini, const float* sine_noise,
                     uint64_t seed, float mel_scale, float* wav, int32_t B, int32_t T, void* stream) {
  DSVC_REQUIRE(h && mel && wav, "dsvc_nsf_forward: null argument");
  DSVC_REQUIRE(!f0 || h->cfg.has_source, "dsvc_nsf_forward: f0 given but the generator was created without source weights");
  DSVC_REQUIRE(B > 0 && T > 0, "dsvc_nsf_forward: B and T must be positive");
  cudaStream_t s = (cudaStream_t)stream;
  const dsvc_nsf_config& cfg = h->cfg;
  const int ns = cfg.num_upsamples, nk = cfg.num_kernels, nd = cfg.num_dilations, dim = cfg.harmonic_num + 1;
  const int hop = h->hop;
  const size_t L = (size_t)T * hop;
  DSVC_REQUIRE(L * (size_t)B < (1ull << 31), "waveform too long for 32-bit row indexing");

  // workspace (grow-only)
  size_t maxact = (size_t)T * cfg.upsample_initial_channel;
  {
    size_t len = T;
    int ch = cfg.upsample_initial_channel;
    for (int i = 0; i < ns; ++i) { len *= cfg.upsample_rates[i]; ch >>= 1; maxact = std::max(maxact, len * ch); }
  }
  maxact *= B;
  {
    size_t len = T, tcact = 0;
    int ch = cfg.upsample_initial_channel;
    for (int i = 0; i < ns; ++i) {
      len *= cfg.upsample_rates[i]; ch >>= 1;
      if (h->tc_enabled && nsf_tc_channels(h, ch)) tcact = std::max(tcact, len * ch * (size_t)B);
    }
    if (tcact) {
      DSVC_TRY(h->PX.reserve(tcact, true));
      DSVC_TRY(h->PA.reserve(tcact, true));
      DSVC_TRY(h->PT.reserve(tcact, true));
    }
    DSVC_TRY(nsf_build_maps(h, B, T));
  }
  DSVC_TRY(h->melc.reserve((size_t)B * T * cfg.num_mels * 4));
  DSVC_TRY(h->har.reserve((size_t)B * L * 4));
  DSVC_TRY(h->S1.reserve((size_t)B * dim * T * 8));
  DSVC_TRY(h->S2.reserve((size_t)B * dim * T * 8));
  DSVC_TRY(h->E.reserve((size_t)B * dim * 8));
  DSVC_TRY(h->W.reserve((size_t)B * dim * T * 4));
  DSVC_TRY(h->bufA.reserve(maxact * 4));
  DSVC_TRY(h->bufU.reserve(maxact * 4));
  DSVC_TRY(h->bufT.reserve(maxact * 4));
  DSVC_TRY(h->bufR0.reserve(maxact * 4));
  DSVC_TRY(h->bufR1.reserve(maxact * 4));
  DSVC_TRY(h->bufS.reserve(maxact * 4));

  // ---- V0 harmonic source (skipped without f0, like the reference's `if f0 is not None`) ----
  if (f0) {
    SrcDims d{B, T, hop, dim, (float)cfg.sampling_rate};
    const int nseq = B * dim;
    src_frames1_kernel<<<nseq, 32, 0, s>>>(d, f0, rand_ini, seed, h->S1.as<double>(), h->E.as<double>());
    DSVC_LAUNCH_CHECK();
    const int bt = std::min(512, ceil_div(hop, 32) * 32);
    src_wraps_kernel<<<dim3(T, B), bt, 0, s>>>(d, f0, h->S1.as<double>(), h->E.as<double>(), h->W.as<int>());
    DSVC_LAUNCH_CHECK();
    src_frames2_kernel<<<nseq, 32, 0, s>>>(d, f0, h->W.as<int>(), h->S2.as<double>());
    DSVC_LAUNCH_CHECK();
    src_synth_kernel<<<dim3(T, B), bt, 0, s>>>(d, f0, h->S1.as<double>(), h->S2.as<double>(), h->E.as<double>(), sine_noise,
                                               seed, h->lin_w.as<float>(), h->lin_b.as<float>(), h->har.as<float>());
    DSVC_LAUNCH_CHECK();
  }
  // ---- V1 conv_pre on c = mel_scale * mel ----
  {
    const size_t n = (size_t)B * T * cfg.num_mels;
    scale_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(mel, h->melc.as<float>(), n, mel_scale);
    DSVC_LAUNCH_CHECK();
    DSVC_TRY(conv_same(h->pre, h->melc.as<float>(), h->bufA.as<float>(), nullptr, B, T, 1, 1.0f, 0, 1.0f, s));
  }
  // ---- V2/V3 upsample stages ----
  float* x = h->bufA.as<float>();   // stage input
  float* xs = h->bufS.as<float>();
  int len = T, rest = hop;
  for (int i = 0; i < ns; ++i) {
    const int u = cfg.upsample_rates[i], K = cfg.upsample_kernel_sizes[i];
    const ConvW& up = *h->ups[i];
    const int lout = len * u;
    rest /= u;
    float* xu = h->bufU.as<float>();
    {  // x = ups[i](leaky_relu(x, 0.1))
      ConvGemmParams p{};
      p.A = x; p.W = up.w.as<float>(); p.B = B; p.Lin = len; p.Cin = up.Cin; p.Cout = up.Cout; p.taps = h->ups_taps[i];
      p.rows = len; p.in_stride = 1; p.in_off = 0; p.tap_step = -1; p.nphase = u; p.tpad = (K - u) / 2; p.in_slope = 0.1f;
      p.a_batch_stride = (long long)len * up.Cin;
      EpiAffine::Params e{};
      e.bias = up.b.as<float>(); e.res = nullptr; e.out = xu; e.Lout = lout; e.Cout = up.Cout; e.accumulate = 0; e.div = 1.0f;
      e.act = EpiAffine::ACT_NONE;
      if (u == 1) { p.nphase = 1; p.in_off = p.tpad; }
      DSVC_TRY(launch_affine(p, e, s));
    }
    if (f0) {  // x = x + noise_convs[i](har_source)
      const ConvW& nc = *h->noise[i];
      const int stride = (i + 1 < ns) ? rest : 1, pad = (i + 1 < ns) ? rest / 2 : 0;
      const size_t shbytes = (size_t)((NOISE_PB - 1) * stride + nc.K) * 4;
      noise_conv_add_kernel<<<dim3(ceil_div(lout, NOISE_PB), B), 256, shbytes, s>>>(
          h->har.as<float>(), nc.w.as<float>(), nc.b.as<float>(), xu, (int)L, lout, nc.Cout, nc.K, stride, pad);
      DSVC_LAUNCH_CHECK();
    }
    // MRF: xs = sum_j ResBlock1_j(xu) / num_kernels
    if (h->resblock == 2) {
      DSVC_TRY(nsf_mrf_resblock2(h, i, xu, xs, B, lout, s));
    } else if (h->smaps[i].tc) {
      // tcgen05 path: every conv reads fp16 (hi, lo) planes of leaky_relu(.) written by the producing epilogue
      const NsfStageMaps& sm = h->smaps[i];
      const size_t n4 = (size_t)B * lout * up.Cout / 4;
      act_split_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(xu, h->PX.hi.as<__half>(), h->PX.lo.as<__half>(), n4, 0.1f);
      DSVC_LAUNCH_CHECK();
      for (int j = 0; j < nk; ++j) {
        const float* cur = xu;
        const TcGemmMaps* in = &sm.px;
        for (int m = 0; m < nd; ++m) {
          const int idx = (i * nk + j) * nd + m;
          const int dil = cfg.resblock_dilation_sizes[j][m];
          EpiVoc::Params e1{};
          e1.act = h->PT.view(true); e1.div = 1.0f; e1.slope = 0.1f;
          DSVC_TRY(conv_same_tc(*h->c1[idx], *in, e1, B, lout, dil, s));
          EpiVoc::Params e2{};
          e2.res = cur; e2.slope = 0.1f;
          if (m + 1 < nd) {
            float* nxt = (m % 2 == 0) ? h->bufR0.as<float>() : h->bufR1.as<float>();
            e2.out = nxt; e2.act = h->PA.view(true); e2.div = 1.0f;
            DSVC_TRY(conv_same_tc(*h->c2[idx], sm.pt, e2, B, lout, 1, s));
            cur = nxt;
            in = &sm.pa;
          } else {
            e2.out = xs; e2.accumulate = j > 0 ? 1 : 0; e2.div = (j + 1 == nk) ? (float)nk : 1.0f;
            DSVC_TRY(conv_same_tc(*h->c2[idx], sm.pt, e2, B, lout, 1, s));
          }
        }
      }
    } else
    for (int j = 0; j < nk; ++j) {
      const float* cur = xu;
      for (int m = 0; m < nd; ++m) {
        const int idx = (i * nk + j) * nd + m;
        const int dil = cfg.resblock_dilation_sizes[j][m];
        DSVC_TRY(conv_same(*h->c1[idx], cur, h->bufT.as<float>(), nullptr, B, lout, dil, 0.1f, 0, 1.0f, s));
        const bool last = (m + 1 == nd);
        if (!last) {
          float* nxt = (m % 2 == 0) ? h->bufR0.as<float>() : h->bufR1.as<float>();
          DSVC_TRY(conv_same(*h->c2[idx], h->bufT.as<float>(), nxt, cur, B, lout, 1, 0.1f, 0, 1.0f, s));
          cur = nxt;
        } else {
          DSVC_TRY(conv_same(*h->c2[idx], h->bufT.as<float>(), xs, cur, B, lout, 1, 0.1f, j > 0 ? 1 : 0,
                             (j + 1 == nk) ? (float)nk : 1.0f, s));
        }
      }
    }
    // next stage reads xs; swap roles of bufA / bufS
    float* t = x; x = xs; xs = t;
    len = lout;
  }
  // ---- V4 conv_post + tanh (default leaky_relu slope 0.01, models.py:383) ----
  DSVC_REQUIRE(h->post.Cin % 4 == 0, "last stage channels must be a multiple of 4");
  conv_post_tanh_kernel<<<dim3(ceil_div(len, 256), B), 256, 0, s>>>(x, h->post.w.as<float>(), h->post.b.as<float>(), wav, len,
                                                                  h->post.Cin, 7, 0.01f);
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

}  // extern "C"
