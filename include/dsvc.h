/*
 * dsvc.h -- C-ABI of the B200-native diffusion-SVC inference hot path (libdsvc.so).
 *
 * The reference (prophesier/diff-svc) has no FFI: its plug-in surface for this path is a set of
 * Python classes.  Each entry point below names the reference call site it replaces
 * (file:line into the reference tree); the Python host mirror in diffsvc_b200/ binds them with
 * ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain C: opaque handles, raw pointers, ints.  No torch / C++ types cross this boundary.
 *   - every call returns 0 on success, a negative DSVC_E* code otherwise; dsvc_last_error()
 *     returns a thread-local human-readable message for the last failure.
 *   - "host" pointers are read during the call only.  "device" pointers are caller-owned device
 *     memory (e.g. PyTorch storage) valid on `stream`; the library never frees or reallocates
 *     them, allocates no caller-visible memory and never synchronises the device implicitly,
 *     except dsvc_*_create / dsvc_diffnet_prepare which (re)allocate private workspace.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - there is NO CPU fallback: every compute entry point fails with DSVC_ENODEVICE when no
 *     sm_100 device is present.
 *   - one in-flight call per handle (the reference is not re-entrant either:
 *     infer_tools/infer_tool.py, flask_api.py:54 threaded=False).
 */
#ifndef DSVC_H_
#define DSVC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSVC_OK          0
#define DSVC_EINVAL     -1   /* bad argument / unsupported shape */
#define DSVC_ECUDA      -2   /* CUDA runtime / driver error */
#define DSVC_ENODEVICE  -3   /* no sm_100 device: the product path has no CPU fallback */
#define DSVC_ESTATE     -4   /* call out of order (e.g. eval before prepare) */

/* arithmetic of the 20-layer WaveNet contractions */
#define DSVC_MATH_TC3F16   0  /* tcgen05 tensor cores, error-compensated fp16 hi/lo split, 3 MMAs per
                                 product, fp32 accumulate in TMEM: fp32-class results (default) */
#define DSVC_MATH_FP32     1  /* fp32 FFMA kernels (any channel count; validation + odd shapes) */
#define DSVC_MATH_TC1F16   2  /* tcgen05, single fp16 pass: "fast mode", NOT within the parity gate */

const char* dsvc_version(void);
/* CRC-32 of this header as the library was built against it.  Bindings that mirror the structs below by hand (ctypes)
 * compare it with the CRC-32 of the header they were written for and refuse a library built from another one. */
uint32_t dsvc_abi(void);
const char* dsvc_last_error(void);
/* number of sm_100 devices visible (0 on a CPU-only box); never fails */
int dsvc_device_count(void);
/* cumulative number of kernels this library launched in this process (bench.py "gpu_launches") */
uint64_t dsvc_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * DiffNet denoiser + Gaussian-diffusion samplers
 * replaces network/diff/net.py:86-135 (DiffNet), :58-84 (ResidualBlock) and the sampling loop
 * network/diff/diffusion.py:146-198, :269-278.
 * ---------------------------------------------------------------------------------------- */
typedef struct dsvc_diffnet dsvc_diffnet_t;

typedef struct {
  int32_t mel_bins;              /* M: in_dims (net.py:87)                       */
  int32_t residual_channels;     /* C: hparams['residual_channels'] (net.py:93)  */
  int32_t encoder_hidden;        /* H: hparams['hidden_size'] (net.py:91)        */
  int32_t residual_layers;       /* L: hparams['residual_layers'] (net.py:92)    */
  int32_t dilation_cycle_length; /* hparams['dilation_cycle_length'] (net.py:94) */
  int32_t num_timesteps;         /* rows of the schedule / step tables           */
  int32_t math;                  /* DSVC_MATH_*                                   */
} dsvc_diffnet_config;

/* All weights are HOST fp32 pointers in the reference's state_dict layouts (SURVEY.md 8b);
 * per-layer arrays are indexed [residual_layers]. */
typedef struct {
  const float* input_projection_w;        /* [C, M, 1]   */
  const float* input_projection_b;        /* [C]         */
  const float* mlp0_w;                    /* [4C, C]     */
  const float* mlp0_b;                    /* [4C]        */
  const float* mlp2_w;                    /* [C, 4C]     */
  const float* mlp2_b;                    /* [C]         */
  const float* const* dilated_conv_w;     /* L x [2C, C, 3] */
  const float* const* dilated_conv_b;     /* L x [2C]    */
  const float* const* diffusion_proj_w;   /* L x [C, C]  */
  const float* const* diffusion_proj_b;   /* L x [C]     */
  const float* const* conditioner_proj_w; /* L x [2C, H, 1] */
  const float* const* conditioner_proj_b; /* L x [2C]    */
  const float* const* output_proj_w;      /* L x [2C, C, 1] */
  const float* const* output_proj_b;      /* L x [2C]    */
  const float* skip_projection_w;         /* [C, C, 1]   */
  const float* skip_projection_b;         /* [C]         */
  const float* output_projection_w;       /* [M, C, 1]   */
  const float* output_projection_b;       /* [M]         */
  /* SinusoidalPosEmb(t) for t = 0..num_timesteps-1, [num_timesteps, C] (net.py:37-44).  The host
   * evaluates this weight-free basis with the reference's own float ops so that the table is
   * bit-identical; the MLP and the per-layer diffusion projections (net.py:99-103, :67) run on
   * the device at create time and are cached as a [num_timesteps, L, C] table. */
  const float* step_basis;
} dsvc_diffnet_weights;

/* DiffNet.__init__ + load_state_dict (net.py:87-110).  Uploads and repacks the weights. */
int dsvc_diffnet_create(dsvc_diffnet_t** out, const dsvc_diffnet_config* cfg,
                        const dsvc_diffnet_weights* w, void* stream);
void dsvc_diffnet_destroy(dsvc_diffnet_t* h);

/* The registered schedule buffers of GaussianDiffusion (diffusion.py:102-120), host fp32
 * [num_timesteps] each.  Taken from the module's buffers (i.e. the checkpoint), never recomputed. */
int dsvc_diffnet_set_schedule(dsvc_diffnet_t* h,
                              const float* sqrt_recip_alphas_cumprod,
                              const float* sqrt_recipm1_alphas_cumprod,
                              const float* posterior_mean_coef1,
                              const float* posterior_mean_coef2,
                              const float* posterior_log_variance_clipped,
                              const float* alphas_cumprod);

/* Per-utterance (batch) setup: sizes the private workspace for [B, Tmax] and computes the
 * step-invariant conditioner projections of all L layers once (net.py:68, hoisted out of the
 * T-step loop).  cond: device fp32 [B, H, Tmax] (= ret['decoder_inp'].transpose(1,2),
 * diffusion.py:232-234).  lengths: host int32 [B] valid frames per item (NULL = all Tmax); each
 * item is computed as if alone (its own length is the zero-padding boundary of every conv). */
int dsvc_diffnet_prepare(dsvc_diffnet_t* h, int32_t B, int32_t Tmax, const int32_t* lengths,
                         const float* cond, void* stream);

/* denoise_fn(x, t, cond=cond) (net.py:112-135; called at diffusion.py:147,182,186).
 * spec, out: device fp32 [B, 1, M, Tmax]; all items share the integer step t. */
int dsvc_diffnet_eval(dsvc_diffnet_t* h, const float* spec, int32_t t, float* out, void* stream);

/* for i in reversed(range(0, t_start)): x = p_sample(x, i, cond)   (diffusion.py:276-278,
 * p_sample :157-163, p_mean_variance :146-154).  x: device fp32 [B,1,M,Tmax], updated in place.
 * noise: device fp32 [t_start, B, 1, M, Tmax] in consumption order (one draw per step including
 * the masked t==0 draw, diffusion.py:160) or NULL to draw N(0,1) from the library's counter-based
 * Philox generator keyed by `seed`. */
int dsvc_sample_ddpm(dsvc_diffnet_t* h, float* x, int32_t t_start, const float* noise,
                     uint64_t seed, void* stream);

/* for i in reversed(range(0, t_start, interval)): x = p_sample_plms(x, i, interval, cond)
 * (diffusion.py:269-275, p_sample_plms :166-198).  The eps history (noise_list, :96,:270) is
 * reset at entry and lives in the handle. */
int dsvc_sample_plms(dsvc_diffnet_t* h, float* x, int32_t t_start, int32_t interval, void* stream);

/* Conditioning encoder, FastSpeech2.forward with no_fs2 (modules/fastspeech/fs2.py:94-154, add_pitch :185-238,
 * utils/pitch_utils.py:17-31,63-76): decoder_inp[b][t] = (pad(hubert)[mel2ph] + pitch_embed[f0_to_coarse(2^f0)])
 * * (mel2ph > 0).  SURVEY.md 8(f) row 1.  All pointers are device pointers:
 * hubert fp32 [B, Th, H]; mel2ph int64 [B, T] (0 = padding, else 1-based unit index); f0 fp32 [B, T] (log2 Hz);
 * pitch_embed fp32 [300, H]; outputs decoder_inp fp32 [B, T, H] and f0_denorm fp32 [B, T] (Hz, 0 on padding). */
int dsvc_cond_encode(const float* hubert, const int64_t* mel2ph, const float* f0, const float* pitch_embed,
                     int32_t B, int32_t Th, int32_t T, int32_t H, int32_t f0_bin, float f0_min, float f0_max,
                     float* decoder_inp, float* f0_denorm, void* stream);

/* Measurement hook (bench.py roofline): enqueue `iters` back-to-back launches of one kernel of the
 * WaveNet layer `layer` on the prepared workspace.  part 0 = dilated conv + conditioner + gate
 * (net.py:69-77), part 1 = output projection + residual + skip (net.py:79-84), part 2 = both as the
 * one fused layer kernel (opt-in DSVC_FUSED_LAYER; DSVC_ESTATE when that mode is not active).  Under the
 * deferred-skip schedule (the default for one clip, DESIGN.md 3.1d) part 0 is the conv kernel of `layer`
 * together with the skip half of layer `layer` - 1's output projection (the conv alone for layer 0), and
 * part 1 is the residual half of the output projection.  part 4 = developer probe: the evaluation up to
 * `layer`'s conv kernel, then up to its output projection (`iters` ignored; a -DDSVC_TIMELINE build
 * prints both kernels' in-kernel stamps).  The workspace contents afterwards are unspecified (call
 * prepare / a sampler again before trusting results). */
int dsvc_diffnet_run_layer(dsvc_diffnet_t* h, int32_t layer, int32_t part, int32_t iters, void* stream);

/* ------------------------------------------------------------------------------------------
 * NSF-HiFiGAN generator
 * replaces modules/nsf_hifigan/models.py:325-387 (Generator), :148-323 (SineGen,
 * SourceModuleHnNSF), :33-64 (ResBlock1), :73-94 (ResBlock2), called from network/vocoders/nsf_hifigan.py:36-45,:62-72.
 * ---------------------------------------------------------------------------------------- */
typedef struct dsvc_nsf dsvc_nsf_t;

#define DSVC_NSF_MAX_STAGES 8
#define DSVC_NSF_MAX_KERNELS 8
#define DSVC_NSF_MAX_DILATIONS 8

typedef struct {
  int32_t num_mels;
  int32_t sampling_rate;
  int32_t upsample_initial_channel;
  int32_t num_upsamples;                                   /* len(h.upsample_rates) */
  int32_t upsample_rates[DSVC_NSF_MAX_STAGES];
  int32_t upsample_kernel_sizes[DSVC_NSF_MAX_STAGES];
  int32_t num_kernels;                                     /* len(h.resblock_kernel_sizes) */
  int32_t resblock_kernel_sizes[DSVC_NSF_MAX_KERNELS];
  int32_t num_dilations;                                   /* dilations per ResBlock1 (3); 2 for ResBlock2 */
  int32_t resblock_dilation_sizes[DSVC_NSF_MAX_KERNELS][DSVC_NSF_MAX_DILATIONS];
  int32_t harmonic_num;                                    /* 8 (models.py:334) */
  int32_t has_source;                                      /* 1: m_source + noise_convs weights are given (NSF);
                                                              0: plain HiFi-GAN (modules/hifigan/hifigan.py with
                                                              use_pitch_embed = false) */
} dsvc_nsf_config;

/* HOST fp32 pointers, weight-norm already folded (remove_weight_norm, models.py:389-396),
 * PyTorch layouts. resblocks are indexed [stage * num_kernels + j][dilation m]. */
typedef struct {
  const float* source_linear_w;      /* m_source.l_linear.weight [1, harmonic_num+1] */
  const float* source_linear_b;      /* [1] */
  const float* conv_pre_w;           /* [C0, num_mels, 7] */
  const float* conv_pre_b;
  const float* const* ups_w;         /* stages x [Cin, Cout, K] (ConvTranspose1d layout) */
  const float* const* ups_b;
  const float* const* noise_convs_w; /* stages x [Cout, 1, Kn] */
  const float* const* noise_convs_b;
  const float* const* convs1_w;      /* (stages*num_kernels*num_dilations) x [ch, ch, k] */
  const float* const* convs1_b;
  const float* const* convs2_w;
  const float* const* convs2_b;
  const float* conv_post_w;          /* [1, ch_last, 7] */
  const float* conv_post_b;
} dsvc_nsf_weights;

/* Generator(h) with h.resblock == '1' + load_state_dict: dsvc_nsf_create_ex(out, cfg, 1, w, stream). */
int dsvc_nsf_create(dsvc_nsf_t** out, const dsvc_nsf_config* cfg, const dsvc_nsf_weights* w,
                    void* stream);
/* resblock: 1 = ResBlock1 (models.py:33-70), 2 = ResBlock2 (models.py:73-94; modules/hifigan/hifigan.py:70-91),
 * chosen as at models.py:337 / hifigan.py:119.  For 2: num_dilations must be 2 (ResBlock2 builds its two convs from
 * dilation[0] and dilation[1]), convs1_w / convs1_b carry resblocks.{n}.convs.{m} (indexed [stage*num_kernels + j][m]),
 * convs2_* must be NULL. */
int dsvc_nsf_create_ex(dsvc_nsf_t** out, const dsvc_nsf_config* cfg, int32_t resblock,
                       const dsvc_nsf_weights* w, void* stream);
void dsvc_nsf_destroy(dsvc_nsf_t* h);

/* Generator.forward(x, f0) (models.py:361-387); also HifiGanGenerator.forward(x, f0=None) of the 24 kHz
 * vocoder (modules/hifigan/hifigan.py:144-169): the same network, mel_scale = 1, and f0 == NULL skips the
 * harmonic source exactly like the reference's `if f0 is not None` branches.
 * mel: device fp32 [B, T, num_mels] log10-mel as produced by the diffusion side; it is scaled by
 *      `mel_scale` (2.30259: log10 -> ln, nsf_hifigan.py:39,65) on load;
 * f0:  device fp32 [B, T] in Hz, 0 = unvoiced; NULL = no source (needs no has_source weights);
 * rand_ini: device fp32 [B, harmonic_num+1] replacing torch.rand at models.py:192 (column 0 is
 *      forced to 0 as at :194), or NULL -> Philox(seed);
 * sine_noise: device fp32 [B, T*hop, harmonic_num+1] replacing randn_like at models.py:271, or
 *      NULL -> Philox(seed);
 * wav: device fp32 [B, T*hop] (= y.view(-1) per item, nsf_hifigan.py:43). */
int dsvc_nsf_forward(dsvc_nsf_t* h, const float* mel, const float* f0, const float* rand_ini,
                     const float* sine_noise, uint64_t seed, float mel_scale, float* wav,
                     int32_t B, int32_t T, void* stream);

/* ------------------------------------------------------------------------------------------
 * Data formats either side of the hot path (SURVEY.md section 8f rows 2-3)
 * ---------------------------------------------------------------------------------------- */

/* Mel analysis: replaces STFT.get_mel (modules/nsf_hifigan/nvSTFT.py:72-104: reflect pad by
 * (n_fft - hop)/2, torch.stft(center=False) with the window, sqrt(re^2 + im^2 + 1e-9), mel_basis @ spec,
 * log(clamp(., clip_val))) and the `0.434294 *` + transpose of NsfHifiGAN.wav2spec
 * (network/vocoders/nsf_hifigan.py:76-92). */
typedef struct {
  int32_t n_fft;       /* power of two in [64, 4096]; the window is given at this length */
  int32_t hop_size;
  int32_t n_mels;
  float clip_val;      /* 1e-5 (nvSTFT.py:59) */
  float out_scale;     /* 0.434294 for the log10 mel of wav2spec, 1 for get_mel's natural log */
} dsvc_mel_config;

/* frames produced for n_samples (>= 0), or -1 if the reflect padding is impossible */
int64_t dsvc_mel_frames(const dsvc_mel_config* cfg, int64_t n_samples);

/* wav: device fp32 [n_samples]; window: device fp32 [n_fft] (torch.hann_window(win_size), centre-padded
 * to n_fft by the caller when win_size < n_fft, as torch.stft does); mel_basis: device fp32
 * [n_mels, n_fft/2+1] (librosa.filters.mel layout); band_lo/band_hi: device int32 [n_mels], the half-open
 * range of non-zero columns of each basis row, or both NULL for dense rows;
 * mel_out: device fp32 [frames, n_mels]. */
int dsvc_mel_analysis(const dsvc_mel_config* cfg, const float* wav, int64_t n_samples,
                      const float* window, const float* mel_basis, const int32_t* band_lo,
                      const int32_t* band_hi, float* mel_out, void* stream);

/* The tensor half of Svc.after_infer (infer_tools/infer_tool.py:172-200) on the device: keep the frames
 * with abs(mel).sum(-1) > 0, clip them to [vmin, vmax] (hparams mel_vmin / mel_vmax), and keep f0 on the
 * same frames, so the vocoder can run on mel_out/f0_out without a host round trip.
 * mel: device fp32 [T, M]; f0 / f0_out: device fp32 [T] or both NULL; mel_out: device fp32 [T, M] (the
 * first *n_kept rows are written); n_kept: device int32 [1]. */
int dsvc_compact_frames(const float* mel, const float* f0, int32_t T, int32_t M, float vmin, float vmax,
                        float* mel_out, float* f0_out, int32_t* n_kept, void* stream);

/* ------------------------------------------------------------------------------------------
 * PitchExtractor (mel -> f0) of the 24 kHz models (SURVEY.md section 8f row 4)
 * replaces modules/fastspeech/pe.py:120-149 (PitchExtractor.forward: Prenet :8-44, ConvStacks :83-117),
 * modules/fastspeech/tts_modules.py:192-235 (PitchPredictor) and utils/pitch_utils.py:63-76 (denorm_f0),
 * called from Svc.infer (infer_tools/infer_tool.py:164-165).
 * ---------------------------------------------------------------------------------------- */
typedef struct dsvc_pe dsvc_pe_t;

#define DSVC_PE_MAX_LAYERS 8

typedef struct {
  int32_t n_mel_bins;        /* 80; multiple of 16 */
  int32_t hidden_size;       /* hparams['hidden_size'] (256); multiple of 64 */
  int32_t predictor_hidden;  /* hparams['predictor_hidden'] or hidden_size */
  int32_t prenet_layers;     /* 3 (pe.py:9) */
  int32_t prenet_kernel;     /* 5 */
  int32_t enc_layers;        /* conv_layers (2); 0 = no mel_encoder */
  int32_t enc_kernel;        /* 5 (pe.py:84) */
  int32_t gn_groups;         /* hidden_size / 16 (pe.py:56) */
  int32_t pred_layers;       /* 5 (pe.py:135) */
  int32_t pred_kernel;       /* hparams['predictor_kernel'] */
  int32_t pad_same;          /* hparams['ffn_padding'] == 'SAME' (else causal left padding) */
  int32_t odim;              /* 2 */
  int32_t pos_rows;          /* rows of the sinusoidal position table (>= T + 1) */
  int32_t pitch_norm;        /* 0 none, 1 'log' (2 ** f0), 2 'standard' (f0 * f0_std + f0_mean) */
  int32_t apply_uv;          /* pitch_type == 'frame' and hparams['use_uv'] */
  float f0_mean, f0_std;
  float bn_eps, gn_eps, ln_eps;   /* 1e-5, 1e-5, 1e-12 */
} dsvc_pe_config;

/* HOST fp32 pointers, PyTorch layouts (Conv1d [Cout, Cin, K], Linear [out, in]). */
typedef struct {
  const float* const* prenet_conv_w;   /* mel_prenet.layers.{l}.0.weight */
  const float* const* prenet_conv_b;
  const float* const* prenet_bn_w;     /* mel_prenet.layers.{l}.2.{weight,bias,running_mean,running_var} */
  const float* const* prenet_bn_b;
  const float* const* prenet_bn_mean;
  const float* const* prenet_bn_var;
  const float* prenet_out_w;           /* mel_prenet.out_proj */
  const float* prenet_out_b;
  const float* enc_in_w;               /* mel_encoder.in_proj */
  const float* enc_in_b;
  const float* const* enc_conv_w;      /* mel_encoder.conv.{l}.conv.conv */
  const float* const* enc_conv_b;
  const float* const* enc_gn_w;        /* mel_encoder.conv.{l}.norm */
  const float* const* enc_gn_b;
  const float* enc_out_w;              /* mel_encoder.out_proj */
  const float* enc_out_b;
  const float* const* pred_conv_w;     /* pitch_predictor.conv.{l}.1 */
  const float* const* pred_conv_b;
  const float* const* pred_ln_w;       /* pitch_predictor.conv.{l}.3 */
  const float* const* pred_ln_b;
  const float* pred_linear_w;          /* pitch_predictor.linear [odim, predictor_hidden] */
  const float* pred_linear_b;
  const float* pos_table;              /* SinusoidalPositionalEmbedding.weights [pos_rows, hidden_size], row 0 zero */
  const float* pos_embed_alpha;        /* [1] */
} dsvc_pe_weights;

int dsvc_pe_create(dsvc_pe_t** out, const dsvc_pe_config* cfg, const dsvc_pe_weights* w, void* stream);
void dsvc_pe_destroy(dsvc_pe_t* h);

/* mel: device fp32 [B, T, n_mel_bins] (log10 mel as produced by the sampler; all-zero frames are padding);
 * pitch_pred: device fp32 [B, T, odim] (ret['pitch_pred']); f0_denorm: device fp32 [B, T]
 * (ret['f0_denorm_pred'], 0 on padding frames). */
int dsvc_pe_forward(dsvc_pe_t* h, const float* mel, int32_t B, int32_t T, float* pitch_pred, float* f0_denorm,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DSVC_H_ */
