// DiffNet denoiser + DDPM / PLMS samplers: host orchestration, weight repacking, small kernels.
// Reference: network/diff/net.py:58-135, network/diff/diffusion.py:146-198,269-278.
#include "common.cuh"
#include "epilogues.cuh"
#include "simt_gemm.cuh"
#include "tc_pair.cuh"
#include "tc_splitk.cuh"
#include "tc_layer.cuh"
#include "tc_step.cuh"

#include <algorithm>
#include <climits>
#include <cmath>
#include <memory>

namespace dsvc {

// ---------------------------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------------------------

// [B][R][Cc] (Cc contiguous, rows ldi apart) -> [B][Cc][R] (rows ldo apart) tiled transpose, optional operand-plane copy
// of the output.  ldi / ldo > the logical width: the mel axis of the tensor-core path's internal state, padded to Mp
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, Plane pl, int R, int Cc, int ldi, int ldo) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const float* ib = in + (size_t)b * R * ldi;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < Cc) ? ib[(size_t)r * ldi + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < Cc && r < R) {
      const float v = tile[threadIdx.x][i];
      const size_t idx = ((size_t)b * Cc + c) * ldo + r;
      if (out) out[idx] = v;
      if (pl.f32) pl.f32[idx] = v;
      if (pl.hi) {
        __half h, l;
        split_f16(v, h, l);
        pl.hi[idx] = h;
        pl.lo[idx] = l;
      }
    }
  }
}

// Packed ragged batch: the caller's [B][Cc][uT] tensor -> rows of the packed frame axis [Tp][ldo] (padding rows: zeros),
// optional operand-plane copy.  Consecutive packed rows are consecutive frames of one item, so both sides coalesce.
__global__ void pack_rows_kernel(const float* __restrict__ in, float* __restrict__ out, Plane pl, const int2* __restrict__ rowmap,
                                 int Tp, int Cc, int uT, int ldo) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.y * 32, r0 = blockIdx.x * 32;
  {
    const int r = r0 + threadIdx.x;
    const int2 m = r < Tp ? __ldg(rowmap + r) : make_int2(-1, 0);
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int c = c0 + i;
      tile[i][threadIdx.x] = (m.x >= 0 && c < Cc) ? in[((size_t)m.x * Cc + c) * uT + m.y] : 0.f;
    }
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    if (r < Tp && c < Cc) {
      const float v = tile[threadIdx.x][i];
      const size_t idx = (size_t)r * ldo + c;
      if (out) out[idx] = v;
      if (pl.f32) pl.f32[idx] = v;
      if (pl.hi) {
        __half h, l;
        split_f16(v, h, l);
        pl.hi[idx] = h;
        pl.lo[idx] = l;
      }
    }
  }
}

// the way back: rows of the packed axis [Tp][ldi] -> the live frames of the caller's [B][Cc][uT] tensor (frames at or
// beyond an item's length keep what the caller passed in)
__global__ void unpack_rows_kernel(const float* __restrict__ in, float* __restrict__ out, const int2* __restrict__ rowmap,
                                   int Tp, int Cc, int uT, int ldi) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.y * 32, r0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < Tp && c < Cc) ? in[(size_t)r * ldi + c] : 0.f;
  }
  __syncthreads();
  const int r = r0 + threadIdx.x;
  const int2 m = r < Tp ? __ldg(rowmap + r) : make_int2(-1, 0);
  if (m.x < 0) return;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i;
    if (c < Cc) out[((size_t)m.x * Cc + c) * uT + m.y] = tile[threadIdx.x][i];
  }
}

// conditioning encoder (fs2.py:94-154 no_fs2 path): one block per (frame, item)
__global__ void cond_encode_kernel(const float* __restrict__ hubert, const long long* __restrict__ mel2ph,
                                   const float* __restrict__ f0, const float* __restrict__ emb, int Th, int T, int H,
                                   int f0_bin, float mel_min, float mel_max, float* __restrict__ out,
                                   float* __restrict__ f0_denorm) {
  const int t = blockIdx.x, b = blockIdx.y;
  const long long idx = mel2ph[(size_t)b * T + t];
  const bool live = idx > 0;
  // denorm_f0 (pitch_norm 'log'): 2 ** f0, zeroed on padding (pitch_utils.py:66-67,74-75)
  const float den = live ? exp2f(f0[(size_t)b * T + t]) : 0.0f;
  // f0_to_coarse (pitch_utils.py:17-31)
  float m = mul_rn(1127.0f, logf(add_rn(1.0f, div_rn(den, 700.0f))));
  if (m > 0.0f) m = add_rn(div_rn(mul_rn(sub_rn(m, mel_min), (float)(f0_bin - 2)), sub_rn(mel_max, mel_min)), 1.0f);
  if (m <= 1.0f) m = 1.0f;
  if (m > (float)(f0_bin - 1)) m = (float)(f0_bin - 1);
  const int pitch = (int)(long long)(m + 0.5f);
  if (threadIdx.x == 0) f0_denorm[(size_t)b * T + t] = den;
  const float* hrow = live ? hubert + ((size_t)b * Th + (size_t)(idx - 1)) * H : nullptr;
  const float* erow = emb + (size_t)pitch * H;
  float* orow = out + ((size_t)b * T + t) * H;
  for (int h = threadIdx.x; h < H; h += blockDim.x) orow[h] = live ? add_rn(hrow[h], erow[h]) : 0.0f;
}

__global__ void set_state_kernel(StepState* st, int t, int interval, unsigned long long seed, const float* noise) {
  st->seed = seed;
  st->noise = noise;
  st->t = t;
  st->t_prev = max(t - interval, 0);
  st->interval = interval;
  st->step = 0;
  st->n_hist = 0;
  st->head = 0;
}

// end-of-step bookkeeping: t -= interval, history ring advances (PLMS)
__global__ void advance_state_kernel(StepState* st, int plms) {
  const int dec = st->interval;
  const int t = st->t - dec;
  st->t = t;
  st->t_prev = max(t - dec, 0);
  st->step += 1;
  if (plms) {
    st->n_hist = min(st->n_hist + 1, 3);
    st->head = (st->head + 1) & 3;
  }
}

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
}  // namespace dsvc

using namespace dsvc;

struct dsvc_diffnet {
  dsvc_diffnet_config cfg;
  bool tc = false;       // tcgen05 path
  int passes = 3;
  int Mp = 0;            // row stride of the mel axis inside the library (XS, hist, XIN, h_in / h_head / b_head): mel_bins
                         // rounded up to a whole 64-wide K block / tile on the tcgen05 path, mel_bins on the FFMA path
  // fp32 weights (GEMM layouts: [taps][Cout][Cin])
  DevBuf w_in, b_in, w_dil, w_cond, b_cond, w_out, b_out, w_skip, b_skip, w_head, b_head;
  DevBuf dtab;           // [Tn][L][C]
  // tcgen05 operands
  F16Pair h_in, h_skip, h_head;
  std::vector<std::unique_ptr<F16Pair>> h_dil, h_out;
  // schedule
  DevBuf c_recip, c_recipm1, c_coef1, c_coef2, c_logvar, c_acp;
  bool have_schedule = false;
  // workspace
  int B = 0, Tmax = 0;   // the layout the kernels run on: the caller's, or (1, Tp) for a packed batch
  int uB = 0, uT = 0;    // the caller's batch size and Tmax (what x / cond / noise / eval outputs are laid out in)
  DevBuf rowmap;         // packed batch: [Tp] (item, frame) per row, (-1, 0) = padding row
  bool packed = false;
  bool prepared = false;
  DevBuf X, S, XS, hist, CP, cond_cl, lengths, state;
  PlaneBuf Y, Z, SP, R, XIN;
  PlaneBuf Y2;           // fused-layer mode (tc_layer.cuh): conv-input plane of the odd layers (Y holds the even ones)
  PlaneBuf Z2;           // deferred-skip schedule: gated-activation plane of the odd layers (Z holds the even ones)
  bool skip_defer = false;   // layer l's skip half runs in layer l+1's conv kernel (enqueue_layer_conv); set in prepare
  bool pingpong = false; // Y / Y2 alternate by layer parity: a layer's out-proj never overwrites the plane its conv reads
  int fused_usable = 0;  // how many clusters of 2C/64 CTAs of tc_layer_kernel fit the device at once (probed in prepare; 0: none)
  TcMaps maps;           // TMA descriptors of the tcgen05 path (rebuilt in prepare)
  DevBuf tile_tab;       // ragged batches: (item, first frame) of every frame tile with a valid frame, dead slots (0,-1) behind
  int tile_slots = 0, tile_live = 0;   // 0 slots: dense grid (all items full length)
  DevBuf step_flags;     // step kernel (tc_step.cuh): [2][n_ft][32] dependency counters + the launch sequence word
  int step_bn = 0;       // slot width of the step kernel for this (B, Tmax), 0: per-layer kernels
  int step_pairs = 0;    // its grid: resident CTA pairs (each owns ceil(slots / pairs) slots)
  DevBuf sk_slab;        // split-K partial tiles [B][m_tiles][n_tiles][3][128][128] fp32 (tc_splitk.cuh)
  int num_sms = 148;
  // CUDA graphs of one sampler step
  cudaGraphExec_t g_ddpm = nullptr, g_plms = nullptr;
  cudaGraphExec_t g_ddpm_x = nullptr;  // DDPM_UNROLL consecutive steps in one graph: the programmatic (PDL) edges then run on
                                       // across the step boundary, which a graph launch boundary serialises
  uint64_t g_ddpm_x_nodes = 0;
  cudaStream_t cap_stream = nullptr;   // private stream used only to record graphs (the caller's may be the
                                       // legacy default stream, which cannot be captured)
  uint64_t g_ddpm_nodes = 0, g_plms_nodes = 0;   // kernels per replay of each graph
  bool g_ddpm_valid = false, g_plms_valid = false;

  ~dsvc_diffnet() {
    if (g_ddpm) cudaGraphExecDestroy(g_ddpm);
    if (g_ddpm_x) cudaGraphExecDestroy(g_ddpm_x);
    if (g_plms) cudaGraphExecDestroy(g_plms);
    if (cap_stream) cudaStreamDestroy(cap_stream);
  }
};

namespace dsvc {

static TcTiles tiles_of(const dsvc_diffnet* h) {
  TcTiles t;
  if (h->tile_slots > 0) { t.tab = h->tile_tab.as<int2>(); t.slots = h->tile_slots; t.live = h->tile_live; }
  return t;
}

static int upload_f(DevBuf& b, const std::vector<float>& v, cudaStream_t s) {
  return b.upload(v.data(), v.size() * sizeof(float), s);
}

static int gemm_affine(const float* A, const float* W, const float* bias, float* out, int rows, int Cin, int Cout,
                       int act, cudaStream_t s) {
  ConvGemmParams p{};
  p.A = A; p.W = W; p.B = 1; p.Lin = rows; p.Cin = Cin; p.Cout = Cout; p.taps = 1; p.rows = rows;
  p.in_stride = 1; p.in_off = 0; p.tap_step = 0; p.nphase = 1; p.tpad = 0; p.in_slope = 1.0f;
  p.a_batch_stride = (long long)rows * Cin;
  EpiAffine::Params e{};
  e.bias = bias; e.res = nullptr; e.out = out; e.Lout = rows; e.Cout = Cout; e.accumulate = 0; e.div = 1.0f; e.act = act;
  return launch_conv_gemm_tile<64, 128, 4, 8, EpiAffine>(p, e, s);
}

static int build(dsvc_diffnet* h, const dsvc_diffnet_weights* w, cudaStream_t s) {
  const int M = h->cfg.mel_bins, C = h->cfg.residual_channels, H = h->cfg.encoder_hidden, L = h->cfg.residual_layers;
  const int Tn = h->cfg.num_timesteps;
  DSVC_TRY(h->w_in.upload(w->input_projection_w, (size_t)C * M * 4, s));
  DSVC_TRY(h->b_in.upload(w->input_projection_b, (size_t)C * 4, s));
  DSVC_TRY(h->w_skip.upload(w->skip_projection_w, (size_t)C * C * 4, s));
  DSVC_TRY(h->b_skip.upload(w->skip_projection_b, (size_t)C * 4, s));
  DSVC_TRY(h->w_head.upload(w->output_projection_w, (size_t)M * C * 4, s));
  // the head bias is read as float4 at every column of the (padded) head tile: [Mp], zeros past M
  const int Mp = h->Mp;
  std::vector<float> bh((size_t)Mp, 0.f);
  memcpy(bh.data(), w->output_projection_b, (size_t)M * 4);
  DSVC_TRY(upload_f(h->b_head, bh, s));

  // dilated convs: [2C][C][3] -> [L][tap][2C paired][C]; pairing puts, in every 128-column tile,
  // 64 gate rows next to their 64 filter rows so one CTA/thread owns both halves of the gate.
  std::vector<float> wd((size_t)L * 3 * 2 * C * C), wc((size_t)L * 2 * C * H), bc((size_t)L * 2 * C),
      wo((size_t)L * 2 * C * C), bo((size_t)L * 2 * C);
  for (int l = 0; l < L; ++l) {
    const float* src = w->dilated_conv_w[l];
    for (int j = 0; j < 3; ++j)
      for (int pn = 0; pn < 2 * C; ++pn) {
        const int tile = pn / 128, within = pn % 128;
        const int orig = within < 64 ? tile * 64 + within : C + tile * 64 + (within - 64);
        float* dst = &wd[(((size_t)l * 3 + j) * 2 * C + pn) * C];
        for (int ci = 0; ci < C; ++ci) dst[ci] = src[((size_t)orig * C + ci) * 3 + j];
      }
    memcpy(&wc[(size_t)l * 2 * C * H], w->conditioner_proj_w[l], (size_t)2 * C * H * 4);
    for (int n = 0; n < 2 * C; ++n) bc[(size_t)l * 2 * C + n] = w->conditioner_proj_b[l][n] + w->dilated_conv_b[l][n];
    memcpy(&wo[(size_t)l * 2 * C * C], w->output_proj_w[l], (size_t)2 * C * C * 4);
    memcpy(&bo[(size_t)l * 2 * C], w->output_proj_b[l], (size_t)2 * C * 4);
  }
  DSVC_TRY(upload_f(h->w_cond, wc, s));
  DSVC_TRY(upload_f(h->b_cond, bc, s));
  DSVC_TRY(upload_f(h->b_out, bo, s));
  if (!h->tc) {
    DSVC_TRY(upload_f(h->w_dil, wd, s));
    DSVC_TRY(upload_f(h->w_out, wo, s));
  } else {
    // mel axis padded to Mp: input projection [C][Mp] with zero columns past M, head [Mp][C] with zero rows past M
    // (zeros leave the max-abs, so the power-of-two pre-scale, unchanged)
    std::vector<float> win((size_t)C * Mp, 0.f), whd((size_t)Mp * C, 0.f);
    for (int c = 0; c < C; ++c) memcpy(&win[(size_t)c * Mp], w->input_projection_w + (size_t)c * M, (size_t)M * 4);
    memcpy(whd.data(), w->output_projection_w, (size_t)M * C * 4);
    DSVC_TRY(make_f16_pair(h->h_in, win.data(), win.size(), s));
    DSVC_TRY(make_f16_pair(h->h_skip, w->skip_projection_w, (size_t)C * C, s));
    DSVC_TRY(make_f16_pair(h->h_head, whd.data(), whd.size(), s));
    for (int l = 0; l < L; ++l) {
      h->h_dil.emplace_back(new F16Pair());
      h->h_out.emplace_back(new F16Pair());
      DSVC_TRY(make_f16_pair(*h->h_dil[l], &wd[(size_t)l * 3 * 2 * C * C], (size_t)3 * 2 * C * C, s));
      DSVC_TRY(make_f16_pair(*h->h_out[l], &wo[(size_t)l * 2 * C * C], (size_t)2 * C * C, s));
    }
  }

  // step table D[t][l][:] = diffusion_projection_l(mlp(sinusoid(t)))  (net.py:124-125, :67)
  DevBuf basis, w0, b0, w2, b2, wp, bp, t1, t2;
  std::vector<float> wpv((size_t)L * C * C), bpv((size_t)L * C);
  for (int l = 0; l < L; ++l) {
    memcpy(&wpv[(size_t)l * C * C], w->diffusion_proj_w[l], (size_t)C * C * 4);
    memcpy(&bpv[(size_t)l * C], w->diffusion_proj_b[l], (size_t)C * 4);
  }
  DSVC_TRY(basis.upload(w->step_basis, (size_t)Tn * C * 4, s));
  DSVC_TRY(w0.upload(w->mlp0_w, (size_t)4 * C * C * 4, s));
  DSVC_TRY(b0.upload(w->mlp0_b, (size_t)4 * C * 4, s));
  DSVC_TRY(w2.upload(w->mlp2_w, (size_t)4 * C * C * 4, s));
  DSVC_TRY(b2.upload(w->mlp2_b, (size_t)C * 4, s));
  DSVC_TRY(upload_f(wp, wpv, s));
  DSVC_TRY(upload_f(bp, bpv, s));
  DSVC_TRY(t1.reserve((size_t)Tn * 4 * C * 4));
  DSVC_TRY(t2.reserve((size_t)Tn * C * 4));
  DSVC_TRY(h->dtab.reserve((size_t)Tn * L * C * 4));
  DSVC_TRY(gemm_affine(basis.as<float>(), w0.as<float>(), b0.as<float>(), t1.as<float>(), Tn, C, 4 * C, EpiAffine::ACT_MISH, s));
  DSVC_TRY(gemm_affine(t1.as<float>(), w2.as<float>(), b2.as<float>(), t2.as<float>(), Tn, 4 * C, C, EpiAffine::ACT_NONE, s));
  DSVC_TRY(gemm_affine(t2.as<float>(), wp.as<float>(), bp.as<float>(), h->dtab.as<float>(), Tn, C, L * C, EpiAffine::ACT_NONE, s));
  DSVC_CUDA(cudaStreamSynchronize(s));   // temporaries are freed on return
  return DSVC_OK;
}

// the gated-activation plane layer l writes: Z, or with the deferred skip Z / Z2 by layer parity -- layer l+1's conv kernel
// writes its own while the skip CTAs of layer l still read layer l's
static const PlaneBuf& zplane(const dsvc_diffnet* h, int l) { return (h->skip_defer && (l & 1)) ? h->Z2 : h->Z; }

// TMA descriptors of every contraction of the tcgen05 path (depend on B, Tmax and the workspace)
static int tc_build_maps(dsvc_diffnet* h) {
  const int Mp = h->Mp, C = h->cfg.residual_channels, L = h->cfg.residual_layers;
  const int B = h->B, T = h->Tmax;
  auto gemm = [&](TcGemmMaps& g, const PlaneBuf& a, int K, const F16Pair& w, int rows) -> int {
    DSVC_TRY(tc_make_a_map(&g.a_hi, a.hi.as<__half>(), B, T, K));
    DSVC_TRY(tc_make_a_map(&g.a_lo, a.lo.as<__half>(), B, T, K));
    DSVC_TRY(tc_make_b_map(&g.b_hi, w.hi.as<__half>(), rows, K, 128));
    DSVC_TRY(tc_make_b_map(&g.b_lo, w.lo.as<__half>(), rows, K, 128));
    DSVC_TRY(tc_make_b_map(&g.b32_hi, w.hi.as<__half>(), rows, K, 32));
    DSVC_TRY(tc_make_b_map(&g.b32_lo, w.lo.as<__half>(), rows, K, 32));
    DSVC_TRY(tc_make_b_map(&g.b64_hi, w.hi.as<__half>(), rows, K, 64));
    DSVC_TRY(tc_make_b_map(&g.b64_lo, w.lo.as<__half>(), rows, K, 64));
    return DSVC_OK;
  };
  DSVC_TRY(gemm(h->maps.in, h->XIN, Mp, h->h_in, C));
  DSVC_TRY(gemm(h->maps.skip, h->SP, C, h->h_skip, C));
  DSVC_TRY(gemm(h->maps.head, h->R, C, h->h_head, Mp));
  h->maps.dil.resize(L);
  h->maps.out.resize(L);
  for (int l = 0; l < L; ++l) {
    const PlaneBuf& yin = (h->pingpong && (l & 1)) ? h->Y2 : h->Y;
    DSVC_TRY(gemm(h->maps.dil[l], yin, C, *h->h_dil[l], 3 * 2 * C));
    DSVC_TRY(gemm(h->maps.out[l], zplane(h, l), C, *h->h_out[l], 2 * C));
  }
  return DSVC_OK;
}

// ---- one denoiser evaluation: enqueue all kernels on `s` --------------------------------------
struct HeadArgs {
  int mode = HEAD_EVAL;
  float* out = nullptr;
  int tsel = 0;   // 0: step table row st->t, 1: st->t_prev (second eval of the first PLMS iteration)
};

static ConvGemmParams base_params(const float* A, const float* W, int B, int T, int Cin, int Cout, int taps, int dil) {
  ConvGemmParams p{};
  p.A = A; p.W = W; p.B = B; p.Lin = T; p.Cin = Cin; p.Cout = Cout; p.taps = taps; p.rows = T;
  p.in_stride = 1; p.in_off = (taps == 3) ? -dil : 0; p.tap_step = dil; p.nphase = 1; p.tpad = 0; p.in_slope = 1.0f;
  p.a_batch_stride = (long long)T * Cin;
  return p;
}

template <class Epi>
static int launch_fp32(const dsvc_diffnet* h, const ConvGemmParams& p, const typename Epi::Params& e, cudaStream_t s) {
  // 64-row tiles when the 128-row grid would leave most of the 148 SMs idle
  const long long ctas128 = (long long)ceil_div(p.rows, 128) * ceil_div(p.Cout, 128) * p.B;
  if (ctas128 >= 2 * 148) return launch_conv_gemm_tile<128, 128, 8, 8, Epi>(p, e, s);
  return launch_conv_gemm_tile<64, 128, 4, 8, Epi>(p, e, s);
}

// ---- epilogue parameter blocks of the 2L+3 contractions of one evaluation ---------------------
static EpiInProj::Params mk_inproj(const dsvc_diffnet* h, int tsel) {
  EpiInProj::Params e{};
  e.bias = h->b_in.as<float>(); e.dtab = h->dtab.as<float>(); e.st = h->state.as<StepState>(); e.lengths = h->lengths.as<int>();
  e.X = h->X.as<float>(); e.Y = h->Y.view(h->tc); e.Tmax = h->Tmax; e.C = h->cfg.residual_channels; e.L = h->cfg.residual_layers;
  e.tsel = tsel; e.wscale = h->tc ? h->h_in.inv_scale : 1.f;
  e.rowmap = h->packed ? h->rowmap.as<int2>() : nullptr;
  return e;
}
static EpiGate::Params mk_gate(const dsvc_diffnet* h, int l) {
  const int C = h->cfg.residual_channels;
  EpiGate::Params e{};
  e.CP = h->CP.as<float>() + (size_t)l * h->B * h->Tmax * 2 * C; e.Z = zplane(h, l).view(h->tc); e.Tmax = h->Tmax; e.C = C;
  e.fast = h->tc ? 1 : 0; e.wscale = h->tc ? h->h_dil[l]->inv_scale : 1.f;
  return e;
}
static EpiOutProj::Params mk_outproj(const dsvc_diffnet* h, int l, int tsel) {
  const int C = h->cfg.residual_channels;
  EpiOutProj::Params e{};
  e.bias = h->b_out.as<float>() + (size_t)l * 2 * C; e.dtab = h->dtab.as<float>(); e.st = h->state.as<StepState>();
  e.lengths = h->lengths.as<int>(); e.X = h->X.as<float>(); e.S = h->S.as<float>(); e.SP = h->SP.view(h->tc);
  e.Y = ((h->pingpong && ((l + 1) & 1)) ? h->Y2 : h->Y).view(h->tc);   // the plane layer l+1's conv reads
  e.Tmax = h->Tmax; e.C = C; e.L = h->cfg.residual_layers; e.layer = l; e.tsel = tsel; e.fast = h->tc ? 1 : 0;
  e.wscale = h->tc ? h->h_out[l]->inv_scale : 1.f;
  e.rowmap = h->packed ? h->rowmap.as<int2>() : nullptr;
  return e;
}
static EpiSkipProj::Params mk_skip(const dsvc_diffnet* h) {
  EpiSkipProj::Params e{};
  e.bias = h->b_skip.as<float>(); e.R = h->R.view(h->tc); e.Tmax = h->Tmax; e.C = h->cfg.residual_channels;
  e.wscale = h->tc ? h->h_skip.inv_scale : 1.f;
  return e;
}
static EpiHead::Params mk_head(const dsvc_diffnet* h, const HeadArgs& ha) {
  EpiHead::Params e{};
  e.bias = h->b_head.as<float>(); e.st = h->state.as<StepState>(); e.mode = ha.mode; e.B = h->B; e.Tmax = h->Tmax;
  e.M = h->cfg.mel_bins; e.Mp = h->Mp; e.out = ha.out; e.xs = h->XS.as<float>(); e.XIN = h->XIN.view(h->tc);
  e.c_recip = h->c_recip.as<float>(); e.c_recipm1 = h->c_recipm1.as<float>(); e.c_coef1 = h->c_coef1.as<float>();
  e.c_coef2 = h->c_coef2.as<float>(); e.c_logvar = h->c_logvar.as<float>();
  e.alphas_cumprod = h->c_acp.as<float>(); e.hist = h->hist.as<float>();
  e.wscale = h->tc ? h->h_head.inv_scale : 1.f;
  e.rowmap = h->packed ? h->rowmap.as<int2>() : nullptr; e.uB = h->uB; e.uT = h->uT;
  return e;
}

// K0: input projection + ReLU
static int enqueue_inproj(dsvc_diffnet* h, int tsel, cudaStream_t s) {
  const int M = h->cfg.mel_bins, C = h->cfg.residual_channels;
  const EpiInProj::Params e = mk_inproj(h, tsel);
  if (h->tc) return tc_launch<EpiInProj>(h->maps.in, e, h->B, h->Tmax, h->Mp, C, 1, 0, h->passes, s, tiles_of(h));
  return launch_fp32<EpiInProj>(h, base_params(h->XIN.f32.as<float>(), h->w_in.as<float>(), h->B, h->Tmax, M, C, 1, 0), e, s);
}

// K3a: dilated conv + hoisted conditioner + gate -> Z.  With the deferred skip (skip_defer_pick) the same grid also runs
// the skip half of layer l-1's output projection: 64-wide out-projection tiles C/64 .. 2C/64-1, in block rows behind the
// conv's 2C/64.  Nothing in layer l waits for them: they read Z_{l-1} and S, written two launches back.
static int enqueue_layer_conv(dsvc_diffnet* h, int l, int tsel, cudaStream_t s) {
  const int C = h->cfg.residual_channels, B = h->B, T = h->Tmax;
  const int dil = 1 << (l % h->cfg.dilation_cycle_length);
  const EpiGate::Params e = mk_gate(h, l);
  if (h->tc) {
    const TcGemmMaps& m = h->maps.dil[l];
    if (h->skip_defer && l > 0)
      return tc_pair2_launch_bn<EpiGate, EpiOutProj, 64>(m, e, C, 2 * C, 3, dil, 2 * C / 64, h->maps.out[l - 1],
                                                          mk_outproj(h, l - 1, tsel), C, 2 * C, 1, 0, C / 64, C / 64, B, T, s);
    // grids that leave SMs idle (one clip): one tap per CTA in a 3-CTA cluster, reduced through an L2 slab
    // (measured, 43 frames: CTA pairs 295 us per step, split-K + pairs 316, split-K + single-CTA kernels 328 -- so the
    //  split is automatic only next to the single-CTA kernels, and on request: DSVC_SPLITK >= 1)
    const char* skv = getenv("DSVC_SPLITK");
    const bool sk_wanted = (skv && atoi(skv) >= 1) || !tc_pair_enabled();
    if (h->passes == 3 && sk_wanted && h->tile_slots == 0 && h->sk_slab.bytes >= tc_splitk_slab_bytes(B, T, 2 * C) &&
        tc_splitk_eligible(B, T, 2 * C, 3, h->num_sms))
      return tc_splitk_launch<EpiGate>(m, e, h->sk_slab.as<float>(), B, T, C, 2 * C, dil, s);
    return tc_launch<EpiGate>(m, e, B, T, C, 2 * C, 3, dil, h->passes, s, tiles_of(h));
  }
  const float* W = h->w_dil.as<float>() + (size_t)l * 3 * 2 * C * C;
  return launch_fp32<EpiGate>(h, base_params(h->Y.f32.as<float>(), W, B, T, C, 2 * C, 3, dil), e, s);
}

// K3b: output projection + residual + skip.  With the deferred skip: the residual half alone (out-projection tiles
// 0 .. C/64-1, the same 64-wide tiles and functor as the whole projection)
static int enqueue_layer_out(dsvc_diffnet* h, int l, int tsel, cudaStream_t s) {
  const int C = h->cfg.residual_channels, B = h->B, T = h->Tmax;
  const EpiOutProj::Params e = mk_outproj(h, l, tsel);
  if (h->skip_defer) return tc_pair_launch_bn<EpiOutProj, 64>(h->maps.out[l], e, B, T, C, 2 * C, 1, 0, s, TcTiles{}, 0, C / 64);
  if (h->tc) return tc_launch<EpiOutProj>(h->maps.out[l], e, B, T, C, 2 * C, 1, 0, h->passes, s, tiles_of(h));
  const float* W = h->w_out.as<float>() + (size_t)l * 2 * C * C;
  return launch_fp32<EpiOutProj>(h, base_params(h->Z.f32.as<float>(), W, B, T, C, 2 * C, 1, 0), e, s);
}

// the deferred skip half of the last layer (there is no next conv kernel to carry it): S / sqrt(L) -> SP
static int enqueue_layer_skip(dsvc_diffnet* h, int l, int tsel, cudaStream_t s) {
  const int C = h->cfg.residual_channels;
  return tc_pair_launch_bn<EpiOutProj, 64>(h->maps.out[l], mk_outproj(h, l, tsel), h->B, h->Tmax, C, 2 * C, 1, 0, s, TcTiles{},
                                          C / 64, C / 64);
}

// K3a + K3b as one kernel (tc_layer.cuh): a cluster of 2C/64 CTAs per frame tile, cluster barrier between the conv
// and the output projection.
static int enqueue_layer_fused(dsvc_diffnet* h, int l, int tsel, cudaStream_t s) {
  const int dil = 1 << (l % h->cfg.dilation_cycle_length);
  const TcGemmMaps* next = l + 1 < h->cfg.residual_layers ? &h->maps.dil[l + 1] : nullptr;
  return tc_layer_launch(h->maps.dil[l], h->maps.out[l], next, mk_gate(h, l), mk_outproj(h, l, tsel), h->B, h->Tmax,
                         h->cfg.residual_channels, dil, h->passes, s);
}

static bool fused_layers(const dsvc_diffnet* h) {
  if (h->tile_slots > 0) return false;     // ragged batches run from the tile table
  if (!(h->tc && h->pingpong && h->fused_usable >= 1 &&
        tc_layer_shape_ok(h->B, h->Tmax, h->cfg.residual_channels))) return false;
  // automatic mode: only while every frame tile's cluster is resident at once (a second wave of clusters doubles the layer)
  return tc_layer_env() >= 2 || (long long)ceil_div(h->Tmax, TC_BM) * h->B <= h->fused_usable;
}

// The whole evaluation as ONE launch (tc_step.cuh): phase table, tensor maps and epilogue parameter blocks of the 2L+3
// contractions in one kernel parameter.
static int enqueue_eval_step(dsvc_diffnet* h, const HeadArgs& ha, cudaStream_t s) {
  const int M = h->cfg.mel_bins, C = h->cfg.residual_channels, L = h->cfg.residual_layers;
  const int bn = h->step_bn;
  static thread_local StepPlan plan;            // ~22 KB: not on the stack
  auto put = [&](int at, const TcGemmMaps& g, bool a_side) {
    if (a_side) { plan.maps[at] = g.a_hi; plan.maps[at + 1] = g.a_lo; }
    else if (bn == 64) { plan.maps[at] = g.b32_hi; plan.maps[at + 1] = g.b32_lo; }
    else { plan.maps[at] = g.b64_hi; plan.maps[at + 1] = g.b64_lo; }
  };
  put(STEP_MAP_XIN, h->maps.in, true);  put(STEP_MAP_IN, h->maps.in, false);
  put(STEP_MAP_SP, h->maps.skip, true); put(STEP_MAP_SKIP, h->maps.skip, false);
  put(STEP_MAP_R, h->maps.head, true);  put(STEP_MAP_HEAD, h->maps.head, false);
  put(STEP_MAP_Y, h->maps.dil[0], true); put(STEP_MAP_Z, h->maps.out[0], true);
  plan.maps[4] = plan.maps[2]; plan.maps[5] = plan.maps[3];      // (slots of a second conv-input plane: unused)
  for (int l = 0; l < L; ++l) {
    put(STEP_MAP_LAYER0 + 4 * l, h->maps.dil[l], false);
    put(STEP_MAP_LAYER0 + 4 * l + 2, h->maps.out[l], false);
  }
  plan.n_maps = STEP_MAP_LAYER0 + 4 * L;
  plan.in = mk_inproj(h, ha.tsel);
  plan.skip = mk_skip(h);
  plan.head = mk_head(h, ha);
  int np = 0, done = 0;
  auto phase = [&](int kind, int K, int taps, int dil, int N, int n_tiles, int a_map, int b_map, int epi) {
    StepPhase& p = plan.phase[np++];
    p.kind = kind; p.K = K; p.taps = taps; p.dil = dil; p.N = N; p.n_tiles = n_tiles; p.a_map = a_map; p.b_map = b_map;
    p.expect = STEP_SIGNALS * done; p.epi = epi;
    done += n_tiles;
  };
  phase(STEP_IN, M, 1, 0, C, C / bn, STEP_MAP_XIN, STEP_MAP_IN, 0);
  for (int l = 0; l < L; ++l) {
    plan.gate[l] = mk_gate(h, l);
    plan.out[l] = mk_outproj(h, l, ha.tsel);
    phase(STEP_GATE, C, 3, 1 << (l % h->cfg.dilation_cycle_length), 2 * C, 2 * C / bn, STEP_MAP_Y, STEP_MAP_LAYER0 + 4 * l, l);
    phase(STEP_OUT, C, 1, 0, 2 * C, 2 * C / bn, STEP_MAP_Z, STEP_MAP_LAYER0 + 4 * l + 2, l);
  }
  phase(STEP_SKIP, C, 1, 0, C, C / bn, STEP_MAP_SP, STEP_MAP_SKIP, 0);
  phase(STEP_HEAD, C, 1, 0, M, M / bn, STEP_MAP_R, STEP_MAP_HEAD, 0);
  plan.n_phases = np;
  plan.final = STEP_SIGNALS * done;
  plan.n_ft = ceil_div(h->Tmax, 2 * TC_BM);
  plan.n_slots = 2 * C / bn;
  plan.T = h->Tmax;
  plan.flags = h->step_flags.as<unsigned>();
  plan.seq = plan.flags + (size_t)2 * plan.n_ft * 32;
  return bn == 64 ? tc_step_launch<64>(plan, h->step_pairs, s) : tc_step_launch<128>(plan, h->step_pairs, s);
}

// Slot width of the step kernel for the prepared shape, 0 when it does not apply: the tensor-core 3-pass path on CTA
// pairs, one item on the frame axis (a single clip or a packed batch), every channel count a multiple of the width, and
// all (frame tile, channel tile) pairs resident at once.
static int step_pick_bn(dsvc_diffnet* h) {
  const int M = h->cfg.mel_bins, C = h->cfg.residual_channels, L = h->cfg.residual_layers;
  if (!(h->tc && h->passes == 3 && tc_pair_enabled() && tc_step_enabled())) return 0;
  if (h->B != 1 || h->tile_slots > 0 || L > STEP_MAXL || h->pingpong) return 0;
  if (tc_forced_bn() > 0) return 0;               // a forced tile width means the per-layer kernels (tests of the tile classes)
  const int n_ft = ceil_div(h->Tmax, 2 * TC_BM);
  static int cap64 = -1, cap128 = -1;
  if (cap64 < 0) { int a = 0, b = 0; if (tc_step_max_pairs<64>(&a) != DSVC_OK || tc_step_max_pairs<128>(&b) != DSVC_OK) return 0; cap64 = a; cap128 = b; }
  // one clip (latency): 64-wide slots, one per pair.  Batches (throughput): 128-wide slots, two or more per pair --
  // the pair works on one slot while the other's hand-over is in flight.
  const char* sb = getenv("DSVC_STEP_BN");
  const int want = sb ? atoi(sb) : 0;
  if (want != 128 && M % 64 == 0 && C % 64 == 0 && cap64 > 0 && (n_ft * (2 * C / 64) <= cap64 || want == 64)) {
    const int S = n_ft * (2 * C / 64), R = ceil_div(S, cap64);
    h->step_pairs = ceil_div(S, R);
    return 64;
  }
  if (M % 128 == 0 && C % 128 == 0 && cap128 > 0) {
    const int S = n_ft * (2 * C / 128), R = ceil_div(S, cap128);
    h->step_pairs = ceil_div(S, R);
    return 128;
  }
  return 0;
}

// Deferred skip (DESIGN.md 3.1d): every layer kernel pre-launches whole.  The 64-wide out-projection of one clip is
// 2C/64 x frame-tile CTAs like the conv, and with ~206 KB of shared memory per CTA the two grids do not fit the SMs
// together, so half of each grid could only enter as the previous kernel drained.  Its skip half is read by nobody until
// the skip projection: it moves into the next layer's conv grid, and what stays between two convs is the residual half
// (C/64 tiles).  Conv + residual CTAs then fit the SMs at once.  Same tiles, same functors, same order of the skip sums:
// bit-identical to the layer-by-layer schedule.  Only the CTA-pair path with 64-wide tiles on a dense grid takes it;
// DSVC_SKIP_DEFER=0 keeps the layer-by-layer schedule (read when the handle is prepared).
static bool skip_defer_pick(const dsvc_diffnet* h) {
  const char* e = getenv("DSVC_SKIP_DEFER");
  if (e && atoi(e) == 0) return false;
  const char* skv = getenv("DSVC_SPLITK");
  if (skv && atoi(skv) >= 1) return false;
  const int C = h->cfg.residual_channels;
  if (!(h->tc && h->passes == 3 && tc_pair_enabled()) || h->tile_slots > 0 || h->step_bn > 0 || fused_layers(h)) return false;
  if (C % 64 != 0 || tc_pick_bn(h->B, h->Tmax, 2 * C) != 64) return false;
  const long long ft = (long long)tc_pair_frame_ctas(h->Tmax) * h->B;
  return ft * (2 * C / 64) + ft * (C / 64) <= h->num_sms;
}

// one denoiser evaluation: enqueue all kernels on `s`
static int enqueue_eval(dsvc_diffnet* h, const HeadArgs& ha, cudaStream_t s) {
  const int M = h->cfg.mel_bins, C = h->cfg.residual_channels, L = h->cfg.residual_layers;
  const int B = h->B, T = h->Tmax;
  if (h->step_bn > 0) return enqueue_eval_step(h, ha, s);
  DSVC_TRY(enqueue_inproj(h, ha.tsel, s));
  for (int l = 0; l < L; ++l) {
    if (fused_layers(h)) {
      DSVC_TRY(enqueue_layer_fused(h, l, ha.tsel, s));
      continue;
    }
    DSVC_TRY(enqueue_layer_conv(h, l, ha.tsel, s));
    // deferred skip: the last layer's residual output x' is read by nobody (skip projection and head read SP / R / XS)
    if (!h->skip_defer || l + 1 < L) DSVC_TRY(enqueue_layer_out(h, l, ha.tsel, s));
  }
  if (h->skip_defer) DSVC_TRY(enqueue_layer_skip(h, L - 1, ha.tsel, s));
  {  // K4a skip_projection + ReLU
    const EpiSkipProj::Params e = mk_skip(h);
    if (h->tc) DSVC_TRY(tc_launch<EpiSkipProj>(h->maps.skip, e, B, T, C, C, 1, 0, h->passes, s, tiles_of(h)));
    else DSVC_TRY(launch_fp32<EpiSkipProj>(h, base_params(h->SP.f32.as<float>(), h->w_skip.as<float>(), B, T, C, C, 1, 0), e, s));
  }
  {  // K4b output_projection + sampler update
    const EpiHead::Params e = mk_head(h, ha);
    if (h->tc) DSVC_TRY(tc_launch<EpiHead>(h->maps.head, e, B, T, C, h->Mp, 1, 0, h->passes, s, tiles_of(h)));
    else DSVC_TRY(launch_fp32<EpiHead>(h, base_params(h->R.f32.as<float>(), h->w_head.as<float>(), B, T, C, M, 1, 0), e, s));
  }
  return DSVC_OK;
}

static int load_x(dsvc_diffnet* h, const float* spec, cudaStream_t s) {
  // [B][M][T] -> XS [B][T][Mp] (+ operand plane of input_projection); the pad columns M..Mp-1 are not written
  const int M = h->cfg.mel_bins, Mp = h->Mp;
  dim3 grid(ceil_div(h->Tmax, 32), ceil_div(M, 32), h->B), block(32, 8);
  if (h->packed)
    pack_rows_kernel<<<grid, block, 0, s>>>(spec, h->XS.as<float>(), h->XIN.view(h->tc), h->rowmap.as<int2>(), h->Tmax, M, h->uT, Mp);
  else
  transpose_kernel<<<grid, block, 0, s>>>(spec, h->XS.as<float>(), h->XIN.view(h->tc), M, h->Tmax, h->Tmax, Mp);
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

static int store_x(dsvc_diffnet* h, float* x, cudaStream_t s) {
  const int M = h->cfg.mel_bins, Mp = h->Mp;
  Plane none{nullptr, nullptr, nullptr};
  dim3 grid(ceil_div(M, 32), ceil_div(h->Tmax, 32), h->B), block(32, 8);
  if (h->packed)
    unpack_rows_kernel<<<dim3(ceil_div(h->Tmax, 32), ceil_div(M, 32)), block, 0, s>>>(h->XS.as<float>(), x, h->rowmap.as<int2>(), h->Tmax, M, h->uT, Mp);
  else
  transpose_kernel<<<grid, block, 0, s>>>(h->XS.as<float>(), x, none, h->Tmax, M, Mp, h->Tmax);
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

// capture `body` (which enqueues on s) into an executable graph
template <class F>
static int capture_graph(dsvc_diffnet* h, cudaGraphExec_t* exec, uint64_t* nodes, F body) {
  if (*exec) { cudaGraphExecDestroy(*exec); *exec = nullptr; }
  const uint64_t before = g_launches.load(std::memory_order_relaxed);
  if (!h->cap_stream) DSVC_CUDA(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
  cudaStream_t s = h->cap_stream;
  cudaGraph_t g = nullptr;
  DSVC_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  int r = body(s);
  // recording is not launching: the kernels recorded here are counted per replay (dsvc_launch_count)
  *nodes = g_launches.load(std::memory_order_relaxed) - before;
  g_launches.fetch_sub(*nodes, std::memory_order_relaxed);
  cudaError_t ce = cudaStreamEndCapture(s, &g);
  if (r != DSVC_OK) { if (g) cudaGraphDestroy(g); return r; }
  DSVC_CUDA(ce);
  ce = cudaGraphInstantiate(exec, g, 0);
  cudaGraphDestroy(g);
  DSVC_CUDA(ce);
  return DSVC_OK;
}

}  // namespace dsvc

// ---------------------------------------------------------------------------------------------
// C-ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int dsvc_diffnet_create(dsvc_diffnet_t** out, const dsvc_diffnet_config* cfg, const dsvc_diffnet_weights* w, void* stream) {
  DSVC_REQUIRE(out && cfg && w, "dsvc_diffnet_create: null argument");
  DSVC_TRY(require_device());
  const int M = cfg->mel_bins, C = cfg->residual_channels, H = cfg->encoder_hidden, L = cfg->residual_layers;
  DSVC_REQUIRE(M > 0 && C > 0 && H > 0 && L > 0 && cfg->num_timesteps > 0 && cfg->dilation_cycle_length > 0,
               "dsvc_diffnet_create: non-positive dimension");
  DSVC_REQUIRE(C % 64 == 0, "residual_channels must be a multiple of 64 (got %d)", C);
  DSVC_REQUIRE(M % 4 == 0 && H % 4 == 0, "mel_bins and encoder_hidden must be multiples of 4");
  DSVC_REQUIRE(cfg->math == DSVC_MATH_TC3F16 || cfg->math == DSVC_MATH_FP32 || cfg->math == DSVC_MATH_TC1F16,
               "unknown math mode %d", cfg->math);
  if (cfg->math != DSVC_MATH_FP32)
    DSVC_REQUIRE(C % 128 == 0, "tensor-core math needs residual_channels %% 128 == 0 (got C=%d); use DSVC_MATH_FP32", C);
  dsvc_diffnet* h = new dsvc_diffnet();
  h->cfg = *cfg;
  h->tc = cfg->math != DSVC_MATH_FP32;
  h->passes = cfg->math == DSVC_MATH_TC1F16 ? 1 : 3;
  h->Mp = h->tc ? 64 * ceil_div(M, 64) : M;
  h->pingpong = h->tc && tc_layer_env() > 0;     // fused-layer mode needs the conv-input plane double-buffered
  int r = build(h, w, (cudaStream_t)stream);
  if (r != DSVC_OK) { delete h; return r; }
  *out = h;
  return DSVC_OK;
}

void dsvc_diffnet_destroy(dsvc_diffnet_t* h) { delete h; }

int dsvc_diffnet_set_schedule(dsvc_diffnet_t* h, const float* recip, const float* recipm1, const float* coef1,
                              const float* coef2, const float* logvar, const float* acp) {
  DSVC_REQUIRE(h && recip && recipm1 && coef1 && coef2 && logvar && acp, "dsvc_diffnet_set_schedule: null argument");
  const size_t n = (size_t)h->cfg.num_timesteps * 4;
  DSVC_TRY(h->c_recip.upload(recip, n, 0));
  DSVC_TRY(h->c_recipm1.upload(recipm1, n, 0));
  DSVC_TRY(h->c_coef1.upload(coef1, n, 0));
  DSVC_TRY(h->c_coef2.upload(coef2, n, 0));
  DSVC_TRY(h->c_logvar.upload(logvar, n, 0));
  DSVC_TRY(h->c_acp.upload(acp, n, 0));
  DSVC_CUDA(cudaStreamSynchronize(0));
  h->have_schedule = true;
  return DSVC_OK;
}

int dsvc_diffnet_prepare(dsvc_diffnet_t* h, int32_t B, int32_t Tmax, const int32_t* lengths, const float* cond, void* stream) {
  DSVC_REQUIRE(h && cond, "dsvc_diffnet_prepare: null argument");
  DSVC_REQUIRE(B > 0 && Tmax > 0, "dsvc_diffnet_prepare: B and Tmax must be positive");
  cudaStream_t s = (cudaStream_t)stream;
  const int M = h->cfg.mel_bins, C = h->cfg.residual_channels, H = h->cfg.encoder_hidden, L = h->cfg.residual_layers;
  const bool tc = h->tc;
  std::vector<int> len(B, Tmax);
  if (lengths)
    for (int b = 0; b < B; ++b) {
      DSVC_REQUIRE(lengths[b] >= 0 && lengths[b] <= Tmax, "lengths[%d]=%d outside [0,%d]", b, lengths[b], Tmax);
      len[b] = lengths[b];
    }
  // Packed batch (tensor-core path, B > 1): the items lie back to back on ONE frame axis, G = max dilation rows of zero
  // padding between them (the conv's zero padding of both neighbours: a tap never reaches further than G), the axis
  // rounded up to whole 256-frame pair tiles.  No per-item tile rounding, no dead tile slots: 8 slices of 689 +- 25 %
  // frames are 48 frame tiles = one wave of 256-wide tiles, where the per-item layout needs 50-52 tiles = two waves
  // (measured 1716 -> see DESIGN.md 3.1e).  rowmap[row] = (item, frame); the caller-facing tensors (x, cond, noise,
  // eval output) keep their [B][..][Tmax] layout and are gathered / scattered through it.  DSVC_PACK=0 disables.
  const int user_B = B, user_T = Tmax;
  bool pack = false;
  {
    const int cyc = h->cfg.dilation_cycle_length < L ? h->cfg.dilation_cycle_length : L;
    const char* pe = getenv("DSVC_PACK");
    pack = tc && B > 1 && cyc <= 7 && !(pe && atoi(pe) == 0);
    if (pack) {
      const int G = 1 << (cyc - 1);
      std::vector<int2> rm;
      for (int b = 0; b < B; ++b) {
        for (int p = 0; p < len[b]; ++p) rm.push_back(make_int2(b, p));
        if (b + 1 < B) rm.insert(rm.end(), (size_t)G, make_int2(-1, 0));
      }
      const int Tp = 2 * TC_BM * ceil_div((int)rm.size(), 2 * TC_BM);
      rm.resize((size_t)Tp, make_int2(-1, 0));
      DSVC_TRY(h->rowmap.reserve(rm.size() * sizeof(int2)));
      DSVC_CUDA(cudaMemcpyAsync(h->rowmap.p, rm.data(), rm.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
      DSVC_CUDA(cudaStreamSynchronize(s));   // `rm` is a stack-owned staging buffer
      B = 1; Tmax = Tp;
      len.assign(1, Tp);
    }
  }
  const bool resized = (B != h->B || Tmax != h->Tmax || pack != h->packed);
  h->B = B; h->Tmax = Tmax; h->uB = user_B; h->uT = user_T; h->packed = pack;
  const size_t n = (size_t)B * Tmax;
  DSVC_TRY(h->X.reserve(n * C * 4));
  DSVC_TRY(h->S.reserve(n * C * 4));
  DSVC_TRY(h->XS.reserve(n * h->Mp * 4));
  DSVC_TRY(h->hist.reserve(4 * n * h->Mp * 4));
  DSVC_TRY(h->CP.reserve((size_t)L * n * 2 * C * 4));
  DSVC_TRY(h->cond_cl.reserve(n * H * 4));
  DSVC_TRY(h->lengths.reserve((size_t)B * 4));
  DSVC_TRY(h->state.reserve(sizeof(StepState)));
  if (tc && (2 * C) % SK_BN == 0 && (long long)ceil_div(Tmax, TC_BM) * ((2 * C) / SK_BN) * B * SK_SPLIT <= 4 * h->num_sms)
    DSVC_TRY(h->sk_slab.reserve(tc_splitk_slab_bytes(B, Tmax, 2 * C)));
  {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess) h->num_sms = sms;
  }
  DSVC_TRY(h->Y.reserve(n * C, tc));
  if (h->pingpong) {
    DSVC_TRY(h->Y2.reserve(n * C, tc));
    DSVC_TRY(tc_layer_probe((2 * C) / LY_BN, &h->fused_usable));
  }
  DSVC_TRY(h->Z.reserve(n * C, tc));
  DSVC_TRY(h->SP.reserve(n * C, tc));
  DSVC_TRY(h->R.reserve(n * C, tc));
  DSVC_TRY(h->XIN.reserve(n * h->Mp, tc));
  if (h->Mp != M) {
    // the input projection's TMA reads all Mp columns of XIN; only the first M are ever written (load_x, head epilogue).
    // The pad must be zero, not whatever the allocation held: an fp16 NaN times a zero weight is still NaN.
    DSVC_CUDA(cudaMemsetAsync(h->XIN.hi.p, 0, n * h->Mp * sizeof(__half), s));
    DSVC_CUDA(cudaMemsetAsync(h->XIN.lo.p, 0, n * h->Mp * sizeof(__half), s));
  }
  DSVC_CUDA(cudaMemcpyAsync(h->lengths.p, len.data(), (size_t)B * 4, cudaMemcpyHostToDevice, s));
  // Ragged batch on the tensor-core path: only the frame tiles that hold a valid frame do work.  The grid keeps the
  // dense size (a captured graph stays valid whatever the lengths are); dead slots exit at once.  Frames beyond an
  // item's length are then never written, so the conv-input planes -- whose rows just past the end ARE read, as the
  // zero padding of the item's last frames -- are cleared here once.
  std::vector<int2> tab;
  const int dense = B * ceil_div(Tmax, TC_BM);
  if (tc) {
    for (int b = 0; b < B; ++b)
      for (int m0 = 0; m0 < len[b]; m0 += TC_BM) tab.push_back(make_int2(b, m0));
  }
  const bool ragged = tc && (int)tab.size() < dense;
  const bool ragged_changed = ragged != (h->tile_slots > 0);
  if (ragged) {
    h->tile_live = (int)tab.size();
    h->tile_slots = 2 * ceil_div(dense, 2);
    tab.resize(h->tile_slots, make_int2(0, -1));
    DSVC_TRY(h->tile_tab.reserve(tab.size() * sizeof(int2)));
    DSVC_CUDA(cudaMemcpyAsync(h->tile_tab.p, tab.data(), tab.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
    DSVC_CUDA(cudaMemsetAsync(h->Y.hi.p, 0, n * C * sizeof(__half), s));
    DSVC_CUDA(cudaMemsetAsync(h->Y.lo.p, 0, n * C * sizeof(__half), s));
  } else {
    h->tile_slots = h->tile_live = 0;
  }
  DSVC_CUDA(cudaStreamSynchronize(s));   // `len` / `tab` are stack-owned staging buffers
  {
    const int bn = step_pick_bn(h);
    if (bn != h->step_bn) h->g_ddpm_valid = h->g_plms_valid = false;
    h->step_bn = bn;
    if (bn > 0) {
      const size_t fb = ((size_t)2 * ceil_div(Tmax, 2 * TC_BM) * 32 + 32) * sizeof(unsigned);
      DSVC_TRY(h->step_flags.reserve(fb));
      DSVC_CUDA(cudaMemsetAsync(h->step_flags.p, 0, fb, s));      // both counter sets and the sequence word start at 0
    }
  }
  const bool defer = skip_defer_pick(h);        // the Z planes the maps point at depend on it
  if (defer) DSVC_TRY(h->Z2.reserve(n * C, tc));
  if (resized || !h->prepared || ragged_changed || defer != h->skip_defer) {
    h->g_ddpm_valid = h->g_plms_valid = false;
    h->skip_defer = defer;
    if (tc) DSVC_TRY(tc_build_maps(h));
  }
  // cond [B][H][T] -> channels-last, then all L conditioner projections in one GEMM
  {
    Plane none{nullptr, nullptr, nullptr};
    dim3 grid(ceil_div(Tmax, 32), ceil_div(H, 32), B), block(32, 8);
    if (pack) pack_rows_kernel<<<grid, block, 0, s>>>(cond, h->cond_cl.as<float>(), none, h->rowmap.as<int2>(), Tmax, H, user_T, H);
    else
    transpose_kernel<<<grid, block, 0, s>>>(cond, h->cond_cl.as<float>(), none, H, Tmax, Tmax, H);
    DSVC_LAUNCH_CHECK();
    ConvGemmParams p = base_params(h->cond_cl.as<float>(), h->w_cond.as<float>(), B, Tmax, H, L * 2 * C, 1, 0);
    EpiCondProj::Params e{};
    e.bias = h->b_cond.as<float>(); e.CP = h->CP.as<float>(); e.B = B; e.Tmax = Tmax; e.C2 = 2 * C;
    DSVC_TRY((launch_conv_gemm_tile<128, 128, 8, 8, EpiCondProj>(p, e, s)));
  }
  h->prepared = true;
  return DSVC_OK;
}

int dsvc_diffnet_eval(dsvc_diffnet_t* h, const float* spec, int32_t t, float* out, void* stream) {
  DSVC_REQUIRE(h && spec && out, "dsvc_diffnet_eval: null argument");
  if (!h->prepared) { set_error("dsvc_diffnet_eval: call dsvc_diffnet_prepare first"); return DSVC_ESTATE; }
  DSVC_REQUIRE(t >= 0 && t < h->cfg.num_timesteps, "diffusion step %d outside [0,%d)", t, h->cfg.num_timesteps);
  cudaStream_t s = (cudaStream_t)stream;
  set_state_kernel<<<1, 1, 0, s>>>(h->state.as<StepState>(), t, 0, 0ull, nullptr);
  DSVC_LAUNCH_CHECK();
  DSVC_TRY(load_x(h, spec, s));
  HeadArgs ha; ha.mode = HEAD_EVAL; ha.out = out;
  return enqueue_eval(h, ha, s);
}

int dsvc_cond_encode(const float* hubert, const int64_t* mel2ph, const float* f0, const float* pitch_embed, int32_t B,
                     int32_t Th, int32_t T, int32_t H, int32_t f0_bin, float f0_min, float f0_max, float* decoder_inp,
                     float* f0_denorm, void* stream) {
  DSVC_REQUIRE(hubert && mel2ph && f0 && pitch_embed && decoder_inp && f0_denorm, "dsvc_cond_encode: null argument");
  DSVC_REQUIRE(B > 0 && Th > 0 && T > 0 && H > 0 && f0_bin > 2, "dsvc_cond_encode: bad dimensions");
  DSVC_TRY(require_device());
  const float mel_min = (float)(1127.0 * std::log(1.0 + (double)f0_min / 700.0));
  const float mel_max = (float)(1127.0 * std::log(1.0 + (double)f0_max / 700.0));
  cond_encode_kernel<<<dim3(T, B), 128, 0, (cudaStream_t)stream>>>(hubert, reinterpret_cast<const long long*>(mel2ph), f0,
                                                                 pitch_embed, Th, T, H, f0_bin, mel_min, mel_max,
                                                                 decoder_inp, f0_denorm);
  DSVC_LAUNCH_CHECK();
  return DSVC_OK;
}

int dsvc_diffnet_run_layer(dsvc_diffnet_t* h, int32_t layer, int32_t part, int32_t iters, void* stream) {
  DSVC_REQUIRE(h, "dsvc_diffnet_run_layer: null handle");
  if (!h->prepared) { set_error("dsvc_diffnet_run_layer: call dsvc_diffnet_prepare first"); return DSVC_ESTATE; }
  DSVC_REQUIRE(layer >= 0 && layer < h->cfg.residual_layers && part >= 0 && part <= 4 && iters >= 0, "bad layer/part/iters");
  if (part == 3) {
    // developer probe: `iters` whole evaluations through the step kernel; a -DDSVC_TIMELINE build prints its phase stamps
    if (h->step_bn == 0) { set_error("dsvc_diffnet_run_layer: part 3 needs the step kernel (tc_step.cuh) for this shape"); return DSVC_ESTATE; }
    cudaStream_t s3 = (cudaStream_t)stream;
    set_state_kernel<<<1, 1, 0, s3>>>(h->state.as<StepState>(), 500, 1, 1ull, nullptr);
    DSVC_LAUNCH_CHECK();
    HeadArgs ha3; ha3.mode = HEAD_DDPM;
    for (int i = 0; i < iters; ++i) DSVC_TRY(enqueue_eval(h, ha3, s3));
#ifdef DSVC_TIMELINE
    {
      static long long tl[160][2 * STEP_MAXL + 3][10];
      DSVC_CUDA(cudaStreamSynchronize(s3));
      DSVC_CUDA(cudaMemcpyFromSymbol(tl, g_step_tl, sizeof(tl)));
      const int np = 2 * h->cfg.residual_layers + 3;
      const int nct = 2 * h->step_pairs;
      printf("step kernel timeline (last launch), cycles.  per phase of CTA c: start->deps | deps->first operands | first->MMAs issued | "
             "issued->acc ready | acc->staged | staged->epi done | epi->signalled | phase total || start, ns after CTA 0's\n");
      const int show[6] = {0, 1, 2, nct / 2, nct - 2, nct - 1};
      for (int k = 0; k < 6; ++k) {
        const int c = show[k];
        if (c < 0 || c >= 160) continue;
        for (int ph = 9; ph < 15 && ph < np; ++ph) {
          const long long* t = tl[c][ph];
          const long long first = (c & 1) ? tl[c - 1][ph][2] : t[2], issued = (c & 1) ? tl[c - 1][ph][3] : t[3];
          printf("  cta %3d ph %2d: %6lld %6lld %6lld %6lld %6lld %6lld %6lld | %6lld || %7lld\n", c, ph, t[1] - t[0], (c & 1) ? -1 : first - t[1],
                 (c & 1) ? -1 : issued - first, (c & 1) ? -1 : t[4] - issued, t[5] - t[4], t[6] - t[5], t[7] - t[6],
                 tl[c][ph + 1][0] - t[0], t[8] - tl[0][ph][8]);
        }
      }
      // averages over the conv (odd) and out-projection (even >= 2) phases of the even CTAs
      for (int par = 0; par < 2; ++par) {
        double a[8] = {0, 0, 0, 0, 0, 0, 0, 0}; int n = 0;
        for (int c = 0; c < nct && c < 160; c += 2)
          for (int ph = 1 + par; ph < np - 2; ph += 2) {
            const long long* t = tl[c][ph];
            a[0] += t[1] - t[0]; a[1] += t[2] - t[1]; a[2] += t[3] - t[2]; a[3] += t[4] - t[3]; a[4] += t[5] - t[4]; a[5] += t[6] - t[5];
            a[6] += t[7] - t[6]; a[7] += tl[c][ph + 1][0] - t[0]; ++n;
          }
        printf("  mean %s: deps %.0f | first operands %.0f | MMA issue %.0f | acc ready %.0f | staged %.0f | epi %.0f | signal %.0f | total %.0f\n",
               par ? "out-proj" : "conv    ", a[0] / n, a[1] / n, a[2] / n, a[3] / n, a[4] / n, a[5] / n, a[6] / n, a[7] / n);
      }
      fflush(stdout);
    }
#endif
    return DSVC_OK;
  }
  if (part == 4) {
    // developer probe: layer `layer`'s two kernels in the alternation of a real evaluation.  Run 0 enqueues the evaluation
    // up to that layer's conv kernel, run 1 up to its out-projection; a -DDSVC_TIMELINE build prints the stamps of the
    // kernel each run ends with.
    if (!h->tc || h->step_bn > 0 || fused_layers(h)) {
      set_error("dsvc_diffnet_run_layer: part 4 needs the per-layer tensor-core kernels");
      return DSVC_ESTATE;
    }
    cudaStream_t s4 = (cudaStream_t)stream;
    for (int run = 0; run < 2; ++run) {
      set_state_kernel<<<1, 1, 0, s4>>>(h->state.as<StepState>(), 500, 1, 1ull, nullptr);
      DSVC_LAUNCH_CHECK();
      DSVC_TRY(enqueue_inproj(h, 0, s4));
      for (int l = 0; l <= layer; ++l) {
        DSVC_TRY(enqueue_layer_conv(h, l, 0, s4));
        if (l < layer || run == 1) DSVC_TRY(enqueue_layer_out(h, l, 0, s4));
      }
#ifdef DSVC_TIMELINE
      static long long tl4[1024][16];
      DSVC_CUDA(cudaStreamSynchronize(s4));
      DSVC_CUDA(cudaMemcpyFromSymbol(tl4, g_timeline, sizeof(tl4)));
      const int C = h->cfg.residual_channels, gx = tc_pair_frame_ctas(h->Tmax), bn = tc_pick_bn(h->B, h->Tmax, 2 * C);
      // block rows of the kernel and the role of each: 0 gate, 1 skip half, 2 out-projection (residual half when deferred)
      const int n_conv = 2 * C / bn, n_skip = (h->skip_defer && layer > 0) ? C / 64 : 0;
      const int rows = run == 0 ? n_conv + n_skip : (h->skip_defer ? C / 64 : 2 * C / bn);
      const int nct = gx * rows * h->B;
      if (nct > 1024) { printf("part 4: %d CTAs, more than the timeline holds\n", nct); continue; }
      auto role = [&](int c) { const int y = (c / gx) % rows; return run == 1 ? 2 : (y < n_conv ? 0 : 1); };
      long long e0 = tl4[0][15], rel = tl4[0][13];
      for (int c = 0; c < nct; ++c) { e0 = std::min(e0, tl4[c][15]); rel = std::min(rel, tl4[c][13]); }
      const char* names[3] = {"gate", "skip", "out"};
      printf("timeline part 4, layer %d, %s kernel (%s schedule), %d CTAs; ns after the first CTA entry; release = the earliest "
             "return from griddepcontrol.wait (%lld)\n", layer, run == 0 ? "conv" : "out-projection",
             h->skip_defer ? "deferred-skip" : "layer-by-layer", nct, rel - e0);
      // a CTA that was resident and waiting leaves griddepcontrol.wait at the release; one that entered as the previous
      // kernel drained reaches it only after its own set-up (barrier init, TMEM alloc, weight prefetch: ~1-2 us)
      for (int r = 0; r < 3; ++r) {
        int n = 0, waiting = 0;
        long long last_in = 0, first_done = LLONG_MAX, last_done = 0, last_ops = 0;
        for (int c = 0; c < nct; ++c) {
          if (role(c) != r) continue;
          ++n;
          waiting += tl4[c][13] - rel < 500;
          last_in = std::max(last_in, tl4[c][15] - e0);
          first_done = std::min(first_done, tl4[c][14] - e0);
          last_done = std::max(last_done, tl4[c][14] - e0);
          last_ops = std::max(last_ops, tl4[c][13] - e0);
        }
        if (n == 0) continue;
        printf("  %-4s %3d CTAs: %3d waiting at the release (past the wait < 0.5 us after it) | last entry %6lld | last past the wait "
               "%6lld | done %6lld .. %6lld\n", names[r], n, waiting, last_in, last_ops, first_done, last_done);
      }
      for (int c = 0; c < nct; c += 2)
        printf("  cta %3d %-4s: entry %6lld | past wait %6lld | first operands +%5lld cyc | done %6lld\n", c, names[role(c)],
               tl4[c][15] - e0, tl4[c][13] - e0, tl4[c][1], tl4[c][14] - e0);
      fflush(stdout);
#endif
    }
    return DSVC_OK;
  }
  if (part == 2 && !fused_layers(h)) {
    set_error("dsvc_diffnet_run_layer: part 2 (fused layer kernel) needs DSVC_FUSED_LAYER and a tensor-core handle whose "
              "2C/64 channel tiles form a schedulable cluster");
    return DSVC_ESTATE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  set_state_kernel<<<1, 1, 0, s>>>(h->state.as<StepState>(), 0, 1, 0ull, nullptr);   // a valid step-table row
  DSVC_LAUNCH_CHECK();
  for (int i = 0; i < iters; ++i) {
    if (part == 0) DSVC_TRY(enqueue_layer_conv(h, layer, 0, s));
    else if (part == 1) DSVC_TRY(enqueue_layer_out(h, layer, 0, s));
    else DSVC_TRY(enqueue_layer_fused(h, layer, 0, s));
  }
#ifdef DSVC_TIMELINE
  if (h->tc) {
    static long long host_tl[1024][16];
    DSVC_CUDA(cudaStreamSynchronize(s));
    DSVC_CUDA(cudaMemcpyFromSymbol(host_tl, g_timeline, sizeof(host_tl)));
    const int nct = 2 * ceil_div(ceil_div(h->Tmax, TC_BM), 2) * ceil_div(2 * h->cfg.residual_channels, 64) * h->B;
    if (part == 2) {
      printf("timeline fused layer (cycles since CTA entry): setup | A:first-operands | A:mma-issued | A:epi-prefetch | A:acc-ready | "
             "A:staged | A:epi-done | fences | cluster-barrier | B:first-operands | B:mma-issued | B:epi-prefetch | B:acc-ready | "
             "B:staged | B:epi-done\n");
      for (int c = 0; c < nct && c < 1024; c += (nct > 12 ? nct / 12 : 1))
        printf("  cta %3d: %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld\n", c,
               host_tl[c][0], host_tl[c][1], host_tl[c][2], host_tl[c][3], host_tl[c][4], host_tl[c][5], host_tl[c][6], host_tl[c][7],
               host_tl[c][8], host_tl[c][9], host_tl[c][10], host_tl[c][11], host_tl[c][12], host_tl[c][13], host_tl[c][14]);
    } else {
    long long e0 = host_tl[0][15];
    for (int c = 0; c < nct && c < 1024; ++c) e0 = host_tl[c][15] < e0 ? host_tl[c][15] : e0;
    printf("timeline part %d (cycles since CTA entry): setup | first-operands | mma-issued | epi-prefetch | acc-ready | staged | epi-done"
           " || CTA entry, ns after the first CTA of the last launch (globaltimer)\n", part);
    for (int c = 0; c < nct && c < 1024; c += (nct > 24 ? nct / 24 : 1))
      printf("  cta %3d: %6lld %6lld %6lld %6lld %6lld %6lld %6lld || %7lld\n", c, host_tl[c][0], host_tl[c][1], host_tl[c][2],
             host_tl[c][3], host_tl[c][4], host_tl[c][5], host_tl[c][6], host_tl[c][15] - e0);
    }
    fflush(stdout);
  }
#endif
  return DSVC_OK;
}

int dsvc_sample_ddpm(dsvc_diffnet_t* h, float* x, int32_t t_start, const float* noise, uint64_t seed, void* stream) {
  DSVC_REQUIRE(h && x, "dsvc_sample_ddpm: null argument");
  if (!h->prepared || !h->have_schedule) { set_error("dsvc_sample_ddpm: prepare + set_schedule first"); return DSVC_ESTATE; }
  DSVC_REQUIRE(t_start >= 0 && t_start <= h->cfg.num_timesteps, "t_start %d outside [0,%d]", t_start, h->cfg.num_timesteps);
  cudaStream_t s = (cudaStream_t)stream;
  DSVC_TRY(load_x(h, x, s));
  if (t_start > 0) {
    set_state_kernel<<<1, 1, 0, s>>>(h->state.as<StepState>(), t_start - 1, 1, seed, noise);
    DSVC_LAUNCH_CHECK();
    // the per-call arguments (seed, external noise pointer) live in the device-side StepState, so the captured step
    // graph is call-invariant: one capture per (B, Tmax)
    HeadArgs ha; ha.mode = HEAD_DDPM;
    if (!h->g_ddpm_valid) {
      DSVC_TRY(capture_graph(h, &h->g_ddpm, &h->g_ddpm_nodes, [&](cudaStream_t cs) -> int {
        DSVC_TRY(enqueue_eval(h, ha, cs));
        advance_state_kernel<<<1, 1, 0, cs>>>(h->state.as<StepState>(), 0);
        DSVC_LAUNCH_CHECK();
        return DSVC_OK;
      }));
      constexpr int DDPM_UNROLL = 10;
      DSVC_TRY(capture_graph(h, &h->g_ddpm_x, &h->g_ddpm_x_nodes, [&](cudaStream_t cs) -> int {
        for (int u = 0; u < DDPM_UNROLL; ++u) {
          DSVC_TRY(enqueue_eval(h, ha, cs));
          advance_state_kernel<<<1, 1, 0, cs>>>(h->state.as<StepState>(), 0);
          DSVC_LAUNCH_CHECK();
        }
        return DSVC_OK;
      }));
      h->g_ddpm_valid = true;
    }
    {
      constexpr int DDPM_UNROLL = 10;
      const int blocks = t_start / DDPM_UNROLL, rest = t_start - blocks * DDPM_UNROLL;
      for (int i = 0; i < blocks; ++i) DSVC_CUDA(cudaGraphLaunch(h->g_ddpm_x, s));
      for (int i = 0; i < rest; ++i) DSVC_CUDA(cudaGraphLaunch(h->g_ddpm, s));
      g_launches.fetch_add(h->g_ddpm_x_nodes * (uint64_t)blocks + h->g_ddpm_nodes * (uint64_t)rest, std::memory_order_relaxed);
    }
  }
  return store_x(h, x, s);
}

int dsvc_sample_plms(dsvc_diffnet_t* h, float* x, int32_t t_start, int32_t interval, void* stream) {
  DSVC_REQUIRE(h && x, "dsvc_sample_plms: null argument");
  if (!h->prepared || !h->have_schedule) { set_error("dsvc_sample_plms: prepare + set_schedule first"); return DSVC_ESTATE; }
  DSVC_REQUIRE(interval >= 1, "interval must be >= 1");
  DSVC_REQUIRE(t_start >= 0 && t_start <= h->cfg.num_timesteps, "t_start %d outside [0,%d]", t_start, h->cfg.num_timesteps);
  cudaStream_t s = (cudaStream_t)stream;
  DSVC_TRY(load_x(h, x, s));
  // reversed(range(0, t_start, interval)): first t is the largest multiple of interval below t_start
  const int n_iter = t_start > 0 ? (t_start - 1) / interval + 1 : 0;
  if (n_iter > 0) {
    set_state_kernel<<<1, 1, 0, s>>>(h->state.as<StepState>(), (n_iter - 1) * interval, interval, 0ull, nullptr);
    DSVC_LAUNCH_CHECK();
    // first iteration: two evaluations (diffusion.py:184-187)
    HeadArgs a; a.mode = HEAD_PLMS_FIRST; a.tsel = 0;
    DSVC_TRY(enqueue_eval(h, a, s));
    HeadArgs b2; b2.mode = HEAD_PLMS_SECOND; b2.tsel = 1;
    DSVC_TRY(enqueue_eval(h, b2, s));
    advance_state_kernel<<<1, 1, 0, s>>>(h->state.as<StepState>(), 1);
    DSVC_LAUNCH_CHECK();
    if (n_iter > 1) {
      HeadArgs c; c.mode = HEAD_PLMS_NEXT;
      if (!h->g_plms_valid) {
        DSVC_TRY(capture_graph(h, &h->g_plms, &h->g_plms_nodes, [&](cudaStream_t cs) -> int {
          DSVC_TRY(enqueue_eval(h, c, cs));
          advance_state_kernel<<<1, 1, 0, cs>>>(h->state.as<StepState>(), 1);
          DSVC_LAUNCH_CHECK();
          return DSVC_OK;
        }));
        h->g_plms_valid = true;
      }
      for (int i = 1; i < n_iter; ++i) DSVC_CUDA(cudaGraphLaunch(h->g_plms, s));
      g_launches.fetch_add(h->g_plms_nodes * (uint64_t)(n_iter - 1), std::memory_order_relaxed);
    }
  }
  return store_x(h, x, s);
}

}  // extern "C"
