// Epilogue functors shared by the fp32 FFMA main loop (simt_gemm.cuh) and the tcgen05 main loop
// (tc_gemm.cuh).  An epilogue sees one output row (b, p) and a chunk of 4 consecutive output
// channels n..n+3 with their fp32 accumulators.  Its global inputs are split in three so that the
// main loops can batch loads ahead of use (the epilogues are latency-, not bandwidth-bound):
//   Col  : per-column constants (bias, diffusion-step shift)   -- loaded once per thread
//   Pre  : per-row inputs (residual stream, skip sum, conditioner projection, sampler state)
//   l2_prefetch(): the addresses Pre will read, for an early L2 prefetch while the MMAs run
//
// Everything the WaveNet layer does besides its two contractions is fused here
// (reference network/diff/net.py:66-84, :112-135 and network/diff/diffusion.py:146-198).
#pragma once
#include "common.cuh"

namespace dsvc {

// Device-resident sampler state, advanced by a 1-thread kernel at the end of each step so that one
// captured CUDA graph serves every step of the loop.
struct StepState {
  int t;        // current diffusion step
  int t_prev;   // PLMS: max(t - interval, 0)
  int interval; // t decrement per step (1 for DDPM)
  int step;     // number of completed steps (index of the noise slab to consume)
  int n_hist;   // PLMS: valid entries in the eps history (0..3)
  int head;     // PLMS: slot the current eps is written to (ring of 4)
  // per-call DDPM arguments (device-resident so that the captured step graph does not depend on them)
  unsigned long long seed;   // Philox key of the library's own N(0,1) stream
  const float* noise;        // caller-provided noise [steps][B][1][M][Tmax], or null
};

// An operand "plane": the activation tensor a later contraction reads.  fp32 for the FFMA path;
// an fp16 (hi, lo) pair, hi + lo == x to ~2^-22, for the 3-pass tcgen05 path.
struct Plane {
  float* f32;
  __half* hi;
  __half* lo;
};

struct EpiCol { float4 bias; float4 d; };
struct EpiPre { float4 a; float4 b; int2 row; };   // row: raw row_of() lookup (see row_live)

// Row validity of internal row (b, p), in two halves so that the LOAD can be batched with the other per-row inputs (one
// round of independent loads, issued while the MMAs run) and nothing waits on it before apply():
//   row_of()   the raw lookup: the row map entry (item, frame) of a packed batch, else (length of item b, p)
//   row_live() padding test on that raw value: item < 0 (packed) or p >= length
// A lookup inside apply() -- between the stores of consecutive rows -- serialises one L2 round trip per row; a lookup
// whose RESULT is consumed inside pre() serialises the pre-loads of the MMA issuer warp, which enters the epilogue last
// (measured: +1 us per out-projection kernel).
__device__ __forceinline__ int2 row_of(const int2* rowmap, const int* lengths, int b, int p) {
  if (rowmap) return __ldg(rowmap + p);
  return make_int2(__ldg(lengths + b), p);
}
__device__ __forceinline__ bool row_live(const int2* rowmap, const int2& row) {
  return rowmap ? row.x >= 0 : row.y < row.x;
}

__device__ __forceinline__ void l2_prefetch_line(const void* p) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

__device__ __forceinline__ void split_f16(float v, __half& hi, __half& lo) {
  hi = __float2half_rn(v);
  lo = __float2half_rn(v - __half2float(hi));
}

__device__ __forceinline__ void plane_store4(const Plane& pl, size_t idx, const float (&v)[4]) {
  if (pl.f32) *reinterpret_cast<float4*>(pl.f32 + idx) = make_float4(v[0], v[1], v[2], v[3]);
  if (pl.hi) {
    // packed conversions: hi = rn_f16(v), lo = rn_f16(v - hi), two elements per instruction
    const __half2 h01 = __floats2half2_rn(v[0], v[1]), h23 = __floats2half2_rn(v[2], v[3]);
    const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
    const __half2 l01 = __floats2half2_rn(v[0] - f01.x, v[1] - f01.y), l23 = __floats2half2_rn(v[2] - f23.x, v[3] - f23.y);
    uint2 hp, lp;
    hp.x = *reinterpret_cast<const uint32_t*>(&h01); hp.y = *reinterpret_cast<const uint32_t*>(&h23);
    lp.x = *reinterpret_cast<const uint32_t*>(&l01); lp.y = *reinterpret_cast<const uint32_t*>(&l23);
    *reinterpret_cast<uint2*>(pl.hi + idx) = hp;
    *reinterpret_cast<uint2*>(pl.lo + idx) = lp;
  }
}

// Packed ragged batches (diffnet.cu, dsvc_diffnet_prepare): the items of a batch lie back to back on ONE frame axis,
// separated by max-dilation rows of zero padding; rowmap[row] = (item, frame) of the caller's [B][Tmax] layout, or
// (-1, 0) for a padding row.  Null: the dense [B][Tmax] layout, padding = frames at or beyond the item's length.

// sigmoid(g) * tanh(f) from two ex2.approx and two rcp.approx:  1/(1+e^-g) * (1 - 2/(1+e^2f)).
// Absolute error ~1e-7 on a value in (-1, 1) -- what matters for an operand of the next contraction;
// used by the tensor-core path only (its own arithmetic error is ~1e-6), the FFMA path keeps expf/tanhf.
__device__ __forceinline__ float gate_fast(float g, float f) {
  const float eg = __expf(-g);
  const float ef = __expf(2.0f * f);
  const float sg = __fdividef(1.0f, 1.0f + eg);
  const float th = 1.0f - __fdividef(2.0f, 1.0f + ef);      // ef = inf -> 1, ef = 0 -> -1
  return sg * th;
}

// ---- input_projection + ReLU (net.py:121,123), and the conv-input plane of layer 0 ----------
struct EpiInProj {
  static constexpr bool kPair = false;
  struct Params {
    const float* bias;       // [C]
    const float* dtab;       // [Tn][L][C] diffusion-step shifts d_l(t)
    const StepState* st;
    const int* lengths;      // [B]
    const int2* rowmap;      // packed batch: row -> (item, frame), null otherwise
    float* X;                // [B][Tmax][C] residual stream
    Plane Y;                 // (x + d_0) masked to the item's own length: what the dilated conv reads
    int Tmax, C, L;
    int tsel;                // 0: step-table row st->t; 1: st->t_prev (2nd eval of the first PLMS iteration)
    float wscale;            // inverse power-of-two weight scale of the tcgen05 path (1 for FFMA)
  };
  __device__ static __forceinline__ EpiCol col(const Params& e, int n) {
    EpiCol c;
    c.bias = __ldg(reinterpret_cast<const float4*>(e.bias + n));
    const int tt = e.tsel ? e.st->t_prev : e.st->t;
    c.d = __ldg(reinterpret_cast<const float4*>(e.dtab + ((size_t)tt * e.L + 0) * e.C + n));
    return c;
  }
  __device__ static __forceinline__ void l2_prefetch(const Params&, int, int, int) {}
  __device__ static __forceinline__ EpiPre pre(const Params& e, int b, int p, int) {
    EpiPre r{};
    r.row = row_of(e.rowmap, e.lengths, b, p);
    return r;
  }
  __device__ static __forceinline__ void apply(const Params& e, int b, int p, int n, const float (&a)[4],
                                               const EpiCol& c, const EpiPre& r) {
    float x[4] = {fmaxf(a[0] * e.wscale + c.bias.x, 0.f), fmaxf(a[1] * e.wscale + c.bias.y, 0.f),
                  fmaxf(a[2] * e.wscale + c.bias.z, 0.f), fmaxf(a[3] * e.wscale + c.bias.w, 0.f)};
    const size_t idx = ((size_t)b * e.Tmax + p) * e.C + n;
    *reinterpret_cast<float4*>(e.X + idx) = make_float4(x[0], x[1], x[2], x[3]);
    const bool live = row_live(e.rowmap, r.row);
    float y[4] = {live ? x[0] + c.d.x : 0.f, live ? x[1] + c.d.y : 0.f, live ? x[2] + c.d.z : 0.f, live ? x[3] + c.d.w : 0.f};
    plane_store4(e.Y, idx, y);
  }
};

// ---- hoisted conditioner projections of all layers (net.py:68), + both conv biases ----------
struct EpiCondProj {
  static constexpr bool kPair = false;
  struct Params {
    const float* bias;   // [L*2C]: conditioner_projection.bias + dilated_conv.bias
    float* CP;           // [L][B][Tmax][2C]
    int B, Tmax, C2;
  };
  __device__ static __forceinline__ EpiCol col(const Params& e, int n) {
    EpiCol c;
    c.bias = __ldg(reinterpret_cast<const float4*>(e.bias + n));
    c.d = make_float4(0.f, 0.f, 0.f, 0.f);
    return c;
  }
  __device__ static __forceinline__ void l2_prefetch(const Params&, int, int, int) {}
  __device__ static __forceinline__ EpiPre pre(const Params&, int, int, int) { return EpiPre{}; }
  __device__ static __forceinline__ void apply(const Params& e, int b, int p, int n, const float (&a)[4],
                                               const EpiCol& c, const EpiPre&) {
    const int l = n / e.C2, nn = n - l * e.C2;
    const size_t idx = (((size_t)l * e.B + b) * e.Tmax + p) * e.C2 + nn;
    *reinterpret_cast<float4*>(e.CP + idx) = make_float4(a[0] + c.bias.x, a[1] + c.bias.y, a[2] + c.bias.z, a[3] + c.bias.w);
  }
};

// ---- gated activation: sigmoid(gate) * tanh(filter) (net.py:71-77) ---------------------------
struct EpiGate {
  static constexpr bool kPair = true;
  struct Params {
    const float* CP;     // this layer's slab [B][Tmax][2C] (biases folded in)
    Plane Z;             // [B][Tmax][C]
    int Tmax, C;
    float wscale;
    int fast;            // tensor-core path: gate_fast()
  };
  __device__ static __forceinline__ EpiCol col(const Params&, int) { return EpiCol{}; }
  __device__ static __forceinline__ void l2_prefetch(const Params& e, int b, int p, int c0) {
    const float* row = e.CP + ((size_t)b * e.Tmax + p) * (2 * e.C);
    l2_prefetch_line(row + c0);
    l2_prefetch_line(row + e.C + c0);
  }
  __device__ static __forceinline__ EpiPre pre(const Params& e, int b, int p, int c0) {
    const float* row = e.CP + ((size_t)b * e.Tmax + p) * (2 * e.C);
    EpiPre r;
    r.a = __ldg(reinterpret_cast<const float4*>(row + c0));
    r.b = __ldg(reinterpret_cast<const float4*>(row + e.C + c0));
    return r;
  }
  __device__ static __forceinline__ void apply_pair(const Params& e, int b, int p, int c0, const float (&g)[4],
                                                    const float (&f)[4], const EpiCol&, const EpiPre& r) {
    const float gg[4] = {g[0] * e.wscale + r.a.x, g[1] * e.wscale + r.a.y, g[2] * e.wscale + r.a.z, g[3] * e.wscale + r.a.w};
    const float ff[4] = {f[0] * e.wscale + r.b.x, f[1] * e.wscale + r.b.y, f[2] * e.wscale + r.b.z, f[3] * e.wscale + r.b.w};
    float z[4];
    if (e.fast) {
#pragma unroll
      for (int i = 0; i < 4; ++i) z[i] = gate_fast(gg[i], ff[i]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) z[i] = sigmoidf_(gg[i]) * tanhf(ff[i]);
    }
    plane_store4(e.Z, ((size_t)b * e.Tmax + p) * e.C + c0, z);
  }
};

// ---- output_projection: residual half -> x' = (x + r)/sqrt(2) (net.py:79-84); skip half -> running
//      skip sum (net.py:129-131, never materialising the [L,B,C,T] stack) ----------------------
struct EpiOutProj {
  static constexpr bool kPair = false;
  struct Params {
    const float* bias;       // [2C]
    const float* dtab;       // [Tn][L][C]
    const StepState* st;
    const int* lengths;
    const int2* rowmap;      // packed batch: row -> (item, frame), null otherwise
    float* X;                // [B][Tmax][C] in/out
    float* S;                // [B][Tmax][C] running skip sum
    Plane Y;                 // (x' + d_{l+1}) masked (not written by the last layer)
    Plane SP;                // last layer only: sum(skip)/sqrt(L), operand of skip_projection
    int Tmax, C, L, layer;
    int tsel;
    float wscale;
    int fast;                // tensor-core path: (x + r) * (1/sqrt 2) instead of the IEEE division
  };
  __device__ static __forceinline__ EpiCol col(const Params& e, int n) {
    EpiCol c;
    c.bias = __ldg(reinterpret_cast<const float4*>(e.bias + n));
    c.d = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n < e.C && e.layer + 1 < e.L) {
      const int tt = e.tsel ? e.st->t_prev : e.st->t;
      c.d = __ldg(reinterpret_cast<const float4*>(e.dtab + ((size_t)tt * e.L + e.layer + 1) * e.C + n));
    }
    return c;
  }
  __device__ static __forceinline__ const float* src(const Params& e, int b, int p, int n) {
    if (n < e.C) return e.X + ((size_t)b * e.Tmax + p) * e.C + n;
    return e.layer > 0 ? e.S + ((size_t)b * e.Tmax + p) * e.C + (n - e.C) : nullptr;
  }
  __device__ static __forceinline__ void l2_prefetch(const Params& e, int b, int p, int n) {
    const float* s = src(e, b, p, n);
    if (s) l2_prefetch_line(s);
  }
  __device__ static __forceinline__ EpiPre pre(const Params& e, int b, int p, int n) {
    EpiPre r{};
    const float* s = src(e, b, p, n);
    if (s) r.a = *reinterpret_cast<const float4*>(s);
    if (n < e.C && e.layer + 1 < e.L) r.row = row_of(e.rowmap, e.lengths, b, p);
    return r;
  }
  __device__ static __forceinline__ void apply(const Params& e, int b, int p, int n, const float (&a)[4],
                                               const EpiCol& c, const EpiPre& r) {
    const float v[4] = {a[0] * e.wscale + c.bias.x, a[1] * e.wscale + c.bias.y, a[2] * e.wscale + c.bias.z, a[3] * e.wscale + c.bias.w};
    if (n < e.C) {
      const size_t idx = ((size_t)b * e.Tmax + p) * e.C + n;
      const float s2 = 1.41421356237309504880f, is2 = 0.70710678118654752440f;
      float x[4];
      if (e.fast) {
        x[0] = (r.a.x + v[0]) * is2; x[1] = (r.a.y + v[1]) * is2; x[2] = (r.a.z + v[2]) * is2; x[3] = (r.a.w + v[3]) * is2;
      } else {
        x[0] = div_rn(add_rn(r.a.x, v[0]), s2); x[1] = div_rn(add_rn(r.a.y, v[1]), s2);
        x[2] = div_rn(add_rn(r.a.z, v[2]), s2); x[3] = div_rn(add_rn(r.a.w, v[3]), s2);
      }
      *reinterpret_cast<float4*>(e.X + idx) = make_float4(x[0], x[1], x[2], x[3]);
      if (e.layer + 1 < e.L) {
        const bool live = row_live(e.rowmap, r.row);
        float y[4] = {live ? x[0] + c.d.x : 0.f, live ? x[1] + c.d.y : 0.f, live ? x[2] + c.d.z : 0.f, live ? x[3] + c.d.w : 0.f};
        plane_store4(e.Y, idx, y);
      }
    } else {
      const size_t idx = ((size_t)b * e.Tmax + p) * e.C + (n - e.C);
      float s[4] = {v[0], v[1], v[2], v[3]};
      if (e.layer > 0) {
        s[0] = add_rn(r.a.x, v[0]); s[1] = add_rn(r.a.y, v[1]); s[2] = add_rn(r.a.z, v[2]); s[3] = add_rn(r.a.w, v[3]);
      }
      if (e.layer + 1 < e.L) {
        *reinterpret_cast<float4*>(e.S + idx) = make_float4(s[0], s[1], s[2], s[3]);
      } else {
        const float sl = sqrtf((float)e.L);
        float q[4] = {div_rn(s[0], sl), div_rn(s[1], sl), div_rn(s[2], sl), div_rn(s[3], sl)};
        plane_store4(e.SP, idx, q);
      }
    }
  }
};

// ---- skip_projection + ReLU (net.py:132-133) -------------------------------------------------
struct EpiSkipProj {
  static constexpr bool kPair = false;
  struct Params {
    const float* bias;   // [C]
    Plane R;             // [B][Tmax][C]
    int Tmax, C;
    float wscale;
  };
  __device__ static __forceinline__ EpiCol col(const Params& e, int n) {
    EpiCol c;
    c.bias = __ldg(reinterpret_cast<const float4*>(e.bias + n));
    c.d = make_float4(0.f, 0.f, 0.f, 0.f);
    return c;
  }
  __device__ static __forceinline__ void l2_prefetch(const Params&, int, int, int) {}
  __device__ static __forceinline__ EpiPre pre(const Params&, int, int, int) { return EpiPre{}; }
  __device__ static __forceinline__ void apply(const Params& e, int b, int p, int n, const float (&a)[4],
                                               const EpiCol& c, const EpiPre&) {
    float r[4] = {fmaxf(a[0] * e.wscale + c.bias.x, 0.f), fmaxf(a[1] * e.wscale + c.bias.y, 0.f),
                  fmaxf(a[2] * e.wscale + c.bias.z, 0.f), fmaxf(a[3] * e.wscale + c.bias.w, 0.f)};
    plane_store4(e.R, ((size_t)b * e.Tmax + p) * e.C + n, r);
  }
};

// ---- output_projection of DiffNet (net.py:134) fused with the sampler update ------------------
enum HeadMode : int {
  HEAD_EVAL = 0,        // write eps to `out` in the reference layout [B,1,M,T]
  HEAD_DDPM = 1,        // p_sample (diffusion.py:146-163)
  HEAD_PLMS_FIRST = 2,  // first eval of the first PLMS iteration: x_pred into the operand plane
  HEAD_PLMS_SECOND = 3, // second eval: eps' -> (eps+eps')/2 -> x
  HEAD_PLMS_NEXT = 4,   // Adams-Bashforth combination of the history (diffusion.py:188-196)
};

struct EpiHead {
  static constexpr bool kPair = false;
  struct Params {
    const float* bias;   // [Mp]
    const StepState* st;
    int mode;
    int B, Tmax, M;      // M: the model's mel bins -- what the caller's tensors, the noise index and the Philox counter use
    int Mp;              // row stride of xs / hist / XIN: M padded to whole tiles on the tensor-core path (columns past M:
                         // zero weights and bias, never stored)
    float wscale;
    float* out;          // HEAD_EVAL: [B,1,M,Tmax]
    float* xs;           // sampler state x, channels-last [B][Tmax][Mp]
    Plane XIN;           // operand plane of input_projection for the next eval
    const int2* rowmap;  // packed batch: row -> (item, frame) of the caller's layout (noise / Philox / HEAD_EVAL indexing)
    int uB, uT;          // the caller's batch size and Tmax (== B, Tmax when rowmap is null)
    // DDPM
    const float* c_recip; const float* c_recipm1; const float* c_coef1; const float* c_coef2; const float* c_logvar;
    // PLMS
    const float* alphas_cumprod;
    float* hist;         // [4][B][Tmax][Mp] eps ring
  };

  // get_x_pred coefficients (diffusion.py:171-177), evaluated in the reference's op order
  __device__ static __forceinline__ void plms_coefs(const Params& e, float& dA, float& cx, float& ce) {
    const float a_t = e.alphas_cumprod[e.st->t], a_prev = e.alphas_cumprod[e.st->t_prev];
    const float a_t_sq = sqrtf(a_t), a_prev_sq = sqrtf(a_prev);
    dA = sub_rn(a_prev, a_t);
    cx = div_rn(1.0f, mul_rn(a_t_sq, add_rn(a_t_sq, a_prev_sq)));
    const float s1 = sqrtf(mul_rn(sub_rn(1.0f, a_prev), a_t));
    const float s2 = sqrtf(mul_rn(sub_rn(1.0f, a_t), a_prev));
    ce = div_rn(1.0f, mul_rn(a_t_sq, add_rn(s1, s2)));
  }
  __device__ static __forceinline__ float x_pred(float x, float eps, float dA, float cx, float ce) {
    return add_rn(x, mul_rn(dA, sub_rn(mul_rn(cx, x), mul_rn(ce, eps))));
  }

  __device__ static __forceinline__ EpiCol col(const Params& e, int n) {
    EpiCol c;
    c.bias = __ldg(reinterpret_cast<const float4*>(e.bias + n));
    c.d = make_float4(0.f, 0.f, 0.f, 0.f);
    if (e.mode == HEAD_DDPM) {     // per-step scalars ride in the column context
      const int t = e.st->t;
      c.d = make_float4(e.c_recip[t], e.c_recipm1[t], e.c_coef1[t], e.c_coef2[t]);
    }
    return c;
  }
  __device__ static __forceinline__ void l2_prefetch(const Params& e, int b, int p, int n) {
    if (e.mode != HEAD_EVAL) l2_prefetch_line(e.xs + ((size_t)b * e.Tmax + p) * e.Mp + n);
  }
  __device__ static __forceinline__ EpiPre pre(const Params& e, int b, int p, int n) {
    EpiPre r{};
    if (e.mode != HEAD_EVAL) r.a = *reinterpret_cast<const float4*>(e.xs + ((size_t)b * e.Tmax + p) * e.Mp + n);
    r.row = e.rowmap ? __ldg(e.rowmap + p) : make_int2(b, p);
    return r;
  }

  __device__ static __forceinline__ void apply(const Params& e, int b, int p, int n, const float (&a)[4],
                                               const EpiCol& c, const EpiPre& r) {
    if (n >= e.M) return;                    // pad columns of the tensor-core path's Mp-wide head tile
    const float eps[4] = {a[0] * e.wscale + c.bias.x, a[1] * e.wscale + c.bias.y, a[2] * e.wscale + c.bias.z, a[3] * e.wscale + c.bias.w};
    const size_t idx = ((size_t)b * e.Tmax + p) * e.Mp + n;
    const int ub = r.row.x, up = r.row.y;    // (item, frame) in the caller's [uB][..][uT] tensors
    if (ub < 0) return;                      // padding row of a packed batch: nothing of the caller's lives here
    if (e.mode == HEAD_EVAL) {
#pragma unroll
      for (int i = 0; i < 4; ++i) e.out[((size_t)ub * e.M + n + i) * e.uT + up] = eps[i];
      return;
    }
    const float x[4] = {r.a.x, r.a.y, r.a.z, r.a.w};
    float xn[4];
    if (e.mode == HEAD_DDPM) {
      const int t = e.st->t;
      const float cr = c.d.x, crm1 = c.d.y, c1 = c.d.z, c2 = c.d.w;
      const float sd = (t == 0) ? 0.0f : expf(mul_rn(0.5f, e.c_logvar[t]));
      float nz[4];
      const float* noise = e.st->noise;
      if (noise) {
#pragma unroll
        for (int i = 0; i < 4; ++i) nz[i] = __ldg(noise + (((size_t)e.st->step * e.uB + ub) * e.M + (n + i)) * e.uT + up);
      } else {
        // library stream: one Philox4x32-10 call yields the 4 draws of this (step, item, frame, channel-quad)
        const float4 q = philox_normal4(e.st->seed, 0x6e6f6973u, (((size_t)e.st->step * e.uB + ub) * (e.M >> 2) + (n >> 2)) * e.uT + up);
        nz[0] = q.x; nz[1] = q.y; nz[2] = q.z; nz[3] = q.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float x0 = sub_rn(mul_rn(cr, x[i]), mul_rn(crm1, eps[i]));       // predict_start_from_noise
        x0 = fminf(fmaxf(x0, -1.0f), 1.0f);                               // clamp_ (clip_denoised)
        const float mean = add_rn(mul_rn(c1, x0), mul_rn(c2, x[i]));      // q_posterior
        xn[i] = add_rn(mean, mul_rn(sd, nz[i]));
      }
      *reinterpret_cast<float4*>(e.xs + idx) = make_float4(xn[0], xn[1], xn[2], xn[3]);
      plane_store4(e.XIN, idx, xn);
      return;
    }
    // ---- PLMS ----
    const size_t hs = (size_t)e.B * e.Tmax * e.Mp;
    float dA, cx, ce;
    plms_coefs(e, dA, cx, ce);
    const int head = e.st->head;
    if (e.mode == HEAD_PLMS_FIRST) {
      // keep eps in the ring (it becomes noise_list[-1]); x is NOT advanced, only the operand plane
      *reinterpret_cast<float4*>(e.hist + head * hs + idx) = make_float4(eps[0], eps[1], eps[2], eps[3]);
#pragma unroll
      for (int i = 0; i < 4; ++i) xn[i] = x_pred(x[i], eps[i], dA, cx, ce);
      plane_store4(e.XIN, idx, xn);
      return;
    }
    float ep[4];
    if (e.mode == HEAD_PLMS_SECOND) {
      const float4 e0 = *reinterpret_cast<const float4*>(e.hist + head * hs + idx);
      const float e0a[4] = {e0.x, e0.y, e0.z, e0.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) ep[i] = div_rn(add_rn(e0a[i], eps[i]), 2.0f);
    } else {
      const int nh = e.st->n_hist;
      *reinterpret_cast<float4*>(e.hist + head * hs + idx) = make_float4(eps[0], eps[1], eps[2], eps[3]);
      const float4 h1v = *reinterpret_cast<const float4*>(e.hist + ((head + 3) & 3) * hs + idx);
      const float h1[4] = {h1v.x, h1v.y, h1v.z, h1v.w};
      if (nh == 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) ep[i] = div_rn(sub_rn(mul_rn(3.0f, eps[i]), h1[i]), 2.0f);
      } else {
        const float4 h2v = *reinterpret_cast<const float4*>(e.hist + ((head + 2) & 3) * hs + idx);
        const float h2[4] = {h2v.x, h2v.y, h2v.z, h2v.w};
        if (nh == 2) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            ep[i] = div_rn(add_rn(sub_rn(mul_rn(23.0f, eps[i]), mul_rn(16.0f, h1[i])), mul_rn(5.0f, h2[i])), 12.0f);
        } else {
          const float4 h3v = *reinterpret_cast<const float4*>(e.hist + ((head + 1) & 3) * hs + idx);
          const float h3[4] = {h3v.x, h3v.y, h3v.z, h3v.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
            ep[i] = div_rn(sub_rn(add_rn(sub_rn(mul_rn(55.0f, eps[i]), mul_rn(59.0f, h1[i])), mul_rn(37.0f, h2[i])),
                                  mul_rn(9.0f, h3[i])), 24.0f);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) xn[i] = x_pred(x[i], ep[i], dA, cx, ce);
    *reinterpret_cast<float4*>(e.xs + idx) = make_float4(xn[0], xn[1], xn[2], xn[3]);
    plane_store4(e.XIN, idx, xn);
  }
};

// ---- generic affine epilogue for the vocoder and the one-off tables ---------------------------
//   v = acc + bias[n];  v = act(v);  v = v + res[idx];  v = out[idx] + v;  v = v / div;  out[idx] = v
struct EpiAffine {
  static constexpr bool kPair = false;
  enum Act : int { ACT_NONE = 0, ACT_MISH = 1 };
  struct Params {
    const float* bias;   // [Cout] or null
    const float* res;    // same indexing as out, or null
    float* out;          // [B][Lout][Cout]
    int Lout, Cout;
    int accumulate;      // out = out + v (read-modify-write)
    float div;           // 1.0f = none
    int act;
  };
  __device__ static __forceinline__ EpiCol col(const Params& e, int n) {
    EpiCol c;
    c.bias = e.bias ? __ldg(reinterpret_cast<const float4*>(e.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
    c.d = make_float4(0.f, 0.f, 0.f, 0.f);
    return c;
  }
  __device__ static __forceinline__ void l2_prefetch(const Params&, int, int, int) {}
  __device__ static __forceinline__ EpiPre pre(const Params& e, int b, int op, int n) {
    EpiPre r{};
    const size_t idx = ((size_t)b * e.Lout + op) * e.Cout + n;
    if (e.res) r.a = *reinterpret_cast<const float4*>(e.res + idx);
    if (e.accumulate) r.b = *reinterpret_cast<const float4*>(e.out + idx);
    return r;
  }
  __device__ static __forceinline__ void apply(const Params& e, int b, int op, int n, const float (&a)[4],
                                               const EpiCol& c, const EpiPre& r) {
    float v[4] = {a[0] + c.bias.x, a[1] + c.bias.y, a[2] + c.bias.z, a[3] + c.bias.w};
    if (e.act == ACT_MISH) {
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = mishf_(v[i]);
    }
    if (e.res) { v[0] = add_rn(v[0], r.a.x); v[1] = add_rn(v[1], r.a.y); v[2] = add_rn(v[2], r.a.z); v[3] = add_rn(v[3], r.a.w); }
    if (e.accumulate) { v[0] = add_rn(r.b.x, v[0]); v[1] = add_rn(r.b.y, v[1]); v[2] = add_rn(r.b.z, v[2]); v[3] = add_rn(r.b.w, v[3]); }
    if (e.div != 1.0f) {
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = div_rn(v[i], e.div);
    }
    *reinterpret_cast<float4*>(e.out + ((size_t)b * e.Lout + op) * e.Cout + n) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

// ---- vocoder ResBlock convs on the tcgen05 path (modules/nsf_hifigan/models.py:57-64, :376-382) ---------------
//   v = acc * wscale + bias;  v += res;  v = out_old + v (MRF sum);  v /= div;  out_f32 = v;
//   act = split_f16(leaky_relu(v, slope))   -- the operand plane of the NEXT conv (its F.leaky_relu fused here)
struct EpiVoc {
  static constexpr bool kPair = false;
  struct Params {
    const float* bias;   // [Cout]
    const float* res;    // [B][Lout][Cout] fp32 or null
    float* out;          // [B][Lout][Cout] fp32 or null
    Plane act;           // hi/lo planes [B][Lout][Cout] or {null}
    int Lout, Cout;      // Cout: the real channel count (a narrow conv's weight rows are zero-padded to the 64-wide tile)
    int accumulate;      // out = out + v
    float div, slope, wscale;
  };
  __device__ static __forceinline__ EpiCol col(const Params& e, int n) {
    EpiCol c;
    c.bias = n < e.Cout ? __ldg(reinterpret_cast<const float4*>(e.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
    c.d = make_float4(0.f, 0.f, 0.f, 0.f);
    return c;
  }
  __device__ static __forceinline__ void l2_prefetch(const Params& e, int b, int p, int n) {
    if (n >= e.Cout) return;
    const size_t idx = ((size_t)b * e.Lout + p) * e.Cout + n;
    if (e.res) l2_prefetch_line(e.res + idx);
    if (e.accumulate) l2_prefetch_line(e.out + idx);
  }
  __device__ static __forceinline__ EpiPre pre(const Params& e, int b, int p, int n) {
    EpiPre r{};
    if (n >= e.Cout) return r;
    const size_t idx = ((size_t)b * e.Lout + p) * e.Cout + n;
    if (e.res) r.a = *reinterpret_cast<const float4*>(e.res + idx);
    if (e.accumulate) r.b = *reinterpret_cast<const float4*>(e.out + idx);
    return r;
  }
  __device__ static __forceinline__ void apply(const Params& e, int b, int p, int n, const float (&a)[4], const EpiCol& c,
                                               const EpiPre& r) {
    if (n >= e.Cout) return;                 // padding columns of a narrow conv's 64-wide tile
    float v[4] = {a[0] * e.wscale + c.bias.x, a[1] * e.wscale + c.bias.y, a[2] * e.wscale + c.bias.z, a[3] * e.wscale + c.bias.w};
    if (e.res) { v[0] = add_rn(v[0], r.a.x); v[1] = add_rn(v[1], r.a.y); v[2] = add_rn(v[2], r.a.z); v[3] = add_rn(v[3], r.a.w); }
    if (e.accumulate) { v[0] = add_rn(r.b.x, v[0]); v[1] = add_rn(r.b.y, v[1]); v[2] = add_rn(r.b.z, v[2]); v[3] = add_rn(r.b.w, v[3]); }
    if (e.div != 1.0f) {
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = div_rn(v[i], e.div);
    }
    const size_t idx = ((size_t)b * e.Lout + p) * e.Cout + n;
    if (e.out) *reinterpret_cast<float4*>(e.out + idx) = make_float4(v[0], v[1], v[2], v[3]);
    if (e.act.hi) {
      const float y[4] = {lrelu_(v[0], e.slope), lrelu_(v[1], e.slope), lrelu_(v[2], e.slope), lrelu_(v[3], e.slope)};
      plane_store4(e.act, idx, y);
    }
  }
};

}  // namespace dsvc
