// Guidance tail: everything between the per-layer attention-map accumulators and the scalar guidance loss, plus its
// gradient back to the accumulators, plus the bit-exact box-mask rasteriser.
//
//   K5  rasterize_kernel      helpers.inside_box over a res x res grid          (reference utils/helpers.py:164-173)
//   K3  phase R of tail_fwd   mean over layers/heads + x100 softmax over tokens (utils/ptp_utils.py:287-288,
//                                                                                pipeline_guided_attention.py:217-219)
//   K4  phase S of tail_fwd   3x3 separable Gaussian, reflect padding           (pipeline :251-254, gaussian_smoothing.py)
//   K6  phase S of tail_fwd   max/argmax, normalise, centre of mass, box losses, loss assembly
//                                                                               (pipeline :255-296, :390-451; helpers.py:215-277)
//       tail_bwd_kernel       gradient of all of the above in ONE launch
//
// These are HBM/latency-bound integer-and-float streaming kernels (no contraction): the design rules are coalesced
// rows (one warp per pixel, lanes over the 77 text tokens = one 308-byte row per slice), warp-shuffle reductions, no
// atomics on data (summation order is fixed, results are run-to-run bit-stable), and ONE launch per direction: the
// forward's per-token stage runs in the last CTA to finish the per-pixel stage (ticket counter), the backward needs no
// second stage at all because every per-token scalar it needs was saved by the forward.
#include "ga_common.cuh"

namespace ga {
namespace tail {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kKPL = GA_MAX_CTX / 32;  // text tokens per lane

struct AccArgs {
  const float* ptr[GA_MAX_ACC_SLICES];
  int32_t slices[GA_MAX_ACC_SLICES];
  int32_t n;
};
struct TokArgs {
  ga_token_t t[GA_MAX_TOKENS];
};
struct BoxArgs {
  double x[GA_MAX_BOXES], y[GA_MAX_BOXES], w[GA_MAX_BOXES], h[GA_MAX_BOXES];
};

__device__ __forceinline__ int reflect(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// ------------------------------------------------------------------------------------------------ K5 rasteriser
// float64, round-to-nearest intrinsics (no FMA contraction), the reference's operation order:
//   ratio = float(res / 1);  x*ratio ...;  off = shrink * width;  x + off <= cx <= (x + width) - off   (inclusive)
__global__ void rasterize_kernel(BoxArgs a, int n, int res, double shrink, uint8_t* __restrict__ masks) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int npix = res * res;
  if (idx >= n * npix) return;
  const int i = idx / npix, pix = idx - i * npix, ii = pix / res, jj = pix - ii * res;
  const double ratio = (double)res;
  const double x = __dmul_rn(a.x[i], ratio), y = __dmul_rn(a.y[i], ratio);
  const double w = __dmul_rn(a.w[i], ratio), h = __dmul_rn(a.h[i], ratio);
  const double off_x = __dmul_rn(shrink, w), off_y = __dmul_rn(shrink, h);
  const double cx = __dadd_rn((double)jj, 0.5), cy = __dadd_rn((double)ii, 0.5);
  const bool in_x = cx >= __dadd_rn(x, off_x) && cx <= __dsub_rn(__dadd_rn(x, w), off_x);
  const bool in_y = cy >= __dadd_rn(y, off_y) && cy <= __dsub_rn(__dadd_rn(y, h), off_y);
  masks[idx] = (in_x && in_y) ? 1 : 0;
}

// ------------------------------------------------------------------------------------------- smoothing helpers
__device__ __forceinline__ float smooth_at(const float* img, int y, int x, int res, const float* w) {
  float acc = 0.f;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const int yy = reflect(y + a - 1, res);
    float rowacc = 0.f;
#pragma unroll
    for (int b = 0; b < 3; ++b) rowacc = fmaf(w[b], img[yy * res + reflect(x + b - 1, res)], rowacc);
    acc = fmaf(w[a], rowacc, acc);
  }
  return acc;
}

// adjoint tap of the 1-D reflect-padded filter: weight with which output position `src` reads input position `dst`
__device__ __forceinline__ float adjoint_tap(int dst, int src, int n, const float* w) {
  float m = 0.f;
#pragma unroll
  for (int a = 0; a < 3; ++a)
    if (reflect(src + a - 1, n) == dst) m += w[a];
  return m;
}

// ------------------------------------------------------------------------------------------ phase S (per token)
// One warp per tracked token.  `img` is a per-warp shared-memory staging buffer of res*res floats.
__device__ void token_stage(const ga_tail_params_t& p, const ga_token_t& tk, int t, const float* attn_text,
                            const uint8_t* masks, const float* weights, float* img, float* smoothed, float* stats,
                            int32_t* argmax) {
  const int lane = threadIdx.x & 31;
  const int res = p.res, npix = res * res, tp = p.last - p.first;
  for (int pix = lane; pix < npix; pix += 32) img[pix] = __ldcg(attn_text + (int64_t)pix * tp + tk.column);
  __syncwarp();
  const bool is_box = tk.kind == GA_TOKEN_BOX && tk.box >= 0;
  const uint8_t* mask = is_box ? masks + (int64_t)tk.box * npix : nullptr;
  const float* wts = (is_box && p.strict && weights != nullptr) ? weights + (int64_t)tk.box * npix : nullptr;
  float* sm = smoothed + (int64_t)t * npix;

  float vmax = -INFINITY, sum = 0.f, rsum = 0.f, rcol = 0.f, rrow = 0.f;
  int imax = 0x7fffffff, nin = 0;
  for (int pix = lane; pix < npix; pix += 32) {
    const int y = pix / res, x = pix - y * res;
    const float s = p.smooth ? smooth_at(img, y, x, res, p.w1d) : img[pix];
    const float a = img[pix];                         // un-smoothed map: custom-loss statistics
    rsum += a;
    rcol = fmaf((float)x + 0.5f, a, rcol);
    rrow = fmaf((float)y + 0.5f, a, rrow);
    sm[pix] = s;
    if (s > vmax) { vmax = s; imax = pix; }
    sum += s;
    if (is_box) nin += mask[pix];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, vmax, o);
    const int oi = __shfl_xor_sync(0xffffffffu, imax, o);
    if (ov > vmax || (ov == vmax && oi < imax)) { vmax = ov; imax = oi; }
    nin += __shfl_xor_sync(0xffffffffu, nin, o);
  }
  sum = warp_sum(sum);
  rsum = warp_sum(rsum); rcol = warp_sum(rcol); rrow = warp_sum(rrow);

  const float at_most = nin > 0 ? 1.f / (float)nin : 0.f;
  float col = 0.f, row = 0.f, sin_ = 0.f, sout = 0.f, hin = 0.f, hout = 0.f;
  for (int pix = lane; pix < npix; pix += 32) {
    const int y = pix / res, x = pix - y * res;
    const float pr = sm[pix] / sum;
    col = fmaf((float)x + 0.5f, pr, col);
    row = fmaf((float)y + 0.5f, pr, row);
    if (is_box) {
      const bool in = mask[pix] != 0;
      if (p.strict) {
        const float w = wts != nullptr ? wts[pix] : 1.f;
        if (in) {
          const float gap = at_most - pr;
          if (gap > 0.f) { sin_ = fmaf(w * 2.f, gap, sin_); hin = fmaf(w, pr, hin); }
        } else if (pr > 0.f) {
          sout = fmaf(w, pr, sout);
          hout = fmaf(w, pr, hout);
        }
      } else {
        if (in) sin_ += pr; else sout += pr;
      }
    }
  }
  col = warp_sum(col); row = warp_sum(row); sin_ = warp_sum(sin_); sout = warp_sum(sout);
  hin = warp_sum(hin); hout = warp_sum(hout);

  if (lane == 0) {
    const float inside = is_box ? (p.strict ? sin_ : 1.f - sin_) : 0.f;
    const float outside = is_box ? sout : 0.f;
    const float denom = (float)(res - 1);
    const float center = fabsf(col - tk.target_x) / denom + 4.f * fabsf(row - tk.target_y) / denom;
    float scaled = 0.f, unscaled = 0.f;
    if (tk.kind == GA_TOKEN_COOR) {
      scaled = unscaled = center;
    } else if (tk.kind == GA_TOKEN_BOX) {
      scaled = p.inside_scale * inside + p.outside_scale * outside;
      if (tk.center_weight > 0.f) scaled += tk.center_weight * center;
      unscaled = inside + outside;
    }
    float* st = stats + (int64_t)t * GA_STATS;
    st[GA_STAT_MAX] = vmax; st[GA_STAT_SUM] = sum; st[GA_STAT_COL] = col; st[GA_STAT_ROW] = row;
    st[GA_STAT_INSIDE] = inside; st[GA_STAT_OUTSIDE] = outside; st[GA_STAT_SCALED] = scaled;
    st[GA_STAT_UNSCALED] = unscaled; st[GA_STAT_HINGE_IN] = hin; st[GA_STAT_HINGE_OUT] = hout;
    st[GA_STAT_NINSIDE] = (float)nin; st[GA_STAT_CENTER] = center;
    st[GA_STAT_RAW_SUM] = rsum; st[GA_STAT_RAW_COL] = rcol / rsum; st[GA_STAT_RAW_ROW] = rrow / rsum;
    st[15] = 0.f;
    argmax[t] = imax;
  }
}

// --------------------------------------------------------------------------------------------------- forward
// Phase R (per pixel): mean over the accumulator slices, x100, softmax over the text tokens -> attn_text rows.
__device__ __forceinline__ void tail_phase_r(const AccArgs& acc, const ga_tail_params_t& p, float* attn_text, int smp,
                                             float (*srow)[4 * GA_MAX_CTX]) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int npix = p.res * p.res, T = p.n_ctx, tp = p.last - p.first;
  // Phase R.  A warp owns 4 consecutive pixels = 4*T contiguous floats of every slice = T aligned float4 chunks
  // (npix % 4 == 0 is guaranteed by the host wrapper): 128-bit coalesced loads, lanes over chunks, slices summed in a
  // fixed order; the sums are re-distributed through shared memory so that lanes become text tokens for the softmax.
  const int group = blockIdx.x * kWarps + warp;
  if (group * 4 < npix) {
    float4 v[kKPL];
#pragma unroll
    for (int kk = 0; kk < kKPL; ++kk) v[kk] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t slice4 = (int64_t)npix * T / 4;
    for (int a = 0; a < acc.n; ++a) {
      const float4* base = reinterpret_cast<const float4*>(acc.ptr[a]) + (int64_t)smp * acc.slices[a] * slice4 +
                           (int64_t)group * T;
#pragma unroll 2
      for (int s = 0; s < acc.slices[a]; ++s) {
#pragma unroll
        for (int kk = 0; kk < kKPL; ++kk) {
          const int c = lane + 32 * kk;
          if (c < T) {
            const float4 x = __ldg(base + (int64_t)s * slice4 + c);
            v[kk].x += x.x; v[kk].y += x.y; v[kk].z += x.z; v[kk].w += x.w;
          }
        }
      }
    }
#pragma unroll
    for (int kk = 0; kk < kKPL; ++kk) {
      const int c = lane + 32 * kk;
      if (c < T)
        reinterpret_cast<float4*>(srow[warp])[c] =
            make_float4((v[kk].x * p.inv_count) * p.temperature, (v[kk].y * p.inv_count) * p.temperature,
                        (v[kk].z * p.inv_count) * p.temperature, (v[kk].w * p.inv_count) * p.temperature);
    }
    __syncwarp();
    for (int q = 0; q < 4; ++q) {
      const int pix = group * 4 + q;
      const float* row = srow[warp] + q * T;
      float x[kKPL], m = -INFINITY;
#pragma unroll
      for (int kk = 0; kk < kKPL; ++kk) {
        const int j = lane + 32 * kk;
        x[kk] = (j < T) ? row[j] : 0.f;
        if (j >= p.first && j < p.last) m = fmaxf(m, x[kk]);
      }
      m = warp_max(m);
      float e[kKPL], sum = 0.f;
#pragma unroll
      for (int kk = 0; kk < kKPL; ++kk) {
        const int j = lane + 32 * kk;
        e[kk] = (j >= p.first && j < p.last) ? expf(x[kk] - m) : 0.f;
        sum += e[kk];
      }
      sum = warp_sum(sum);
#pragma unroll
      for (int kk = 0; kk < kKPL; ++kk) {
        const int j = lane + 32 * kk;
        if (j >= p.first && j < p.last) attn_text[(int64_t)pix * tp + (j - p.first)] = e[kk] / sum;
      }
    }
  }

}

// Phase S (per tracked token) + the total, for one sample; `simg` holds min(kWarps, n_tokens) maps of res*res floats.
__device__ __forceinline__ void tail_phase_s(const ga_tail_params_t& p, const TokArgs& toks, const uint8_t* masks,
                                             const float* weights, const float* attn_text, float* smoothed, float* stats,
                                             int32_t* argmax, float* total, unsigned int* ticket, float* simg) {
  const int warp = threadIdx.x >> 5;
  const int npix = p.res * p.res;
  for (int t0 = 0; t0 < p.n_tokens; t0 += kWarps) {
    const int t = t0 + warp;
    if (t < p.n_tokens)
      token_stage(p, toks.t[t], t, attn_text, masks, weights, simg + (size_t)warp * npix, smoothed, stats, argmax);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int t = 0; t < p.n_tokens; ++t) tot += toks.t[t].group_weight * stats[(int64_t)t * GA_STATS + GA_STAT_SCALED];
    total[0] = tot;
    *ticket = 0u;  // leave the workspace zero for the next launch
  }
}

// Small launches: ONE launch.  grid = (ceil(res^2 / 32), n_samples) CTAs x 256 threads; phase R in every CTA, the last
// CTA of a sample to finish (ticket counter) runs phase S.
__global__ void __launch_bounds__(kThreads)
tail_fwd_kernel(AccArgs acc, ga_tail_params_t p, TokArgs toks, const uint8_t* __restrict__ masks,
                const float* __restrict__ weights, float* attn_text, float* smoothed, float* stats, int32_t* argmax,
                float* total, unsigned int* ticket) {
  extern __shared__ float simg[];  // min(kWarps, n_tokens) * res*res floats (phase S only)
  __shared__ __align__(16) float srow[kWarps][4 * GA_MAX_CTX];   // phase R: 4 pixels x T tokens per warp
  __shared__ bool is_last;
  const int npix = p.res * p.res, tp = p.last - p.first;
  const int smp = blockIdx.y;                       // independent sample
  attn_text += (int64_t)smp * npix * tp;
  smoothed += (int64_t)smp * p.n_tokens * npix;
  stats += (int64_t)smp * p.n_tokens * GA_STATS;
  argmax += (int64_t)smp * p.n_tokens;
  total += smp;
  ticket += smp;
  tail_phase_r(acc, p, attn_text, smp, srow);
  // ---- hand-over to phase S: the last CTA to take a ticket sees every other CTA's attn_text
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int tkt = atomicAdd(ticket, 1u);
    is_last = (tkt == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  tail_phase_s(p, toks, masks, weights, attn_text, smoothed, stats, argmax, total, ticket, simg);
}

// Large launches (many samples): two launches.  Fused, the kernel needs 64 registers and the phase-S staging of every
// CTA although one CTA per sample uses it: 4 CTAs per SM, ncu warps-active 49 %, DRAM 48-58 %.  The per-pixel phase on
// its own is a lean streaming kernel (6 CTAs per SM), the per-token phase one CTA per sample.  Same device code, same
// bits as the fused kernel.
__global__ void __launch_bounds__(kThreads, 6)
tail_fwd_r_kernel(AccArgs acc, ga_tail_params_t p, float* attn_text) {
  __shared__ __align__(16) float srow[kWarps][4 * GA_MAX_CTX];
  const int smp = blockIdx.y;
  attn_text += (int64_t)smp * p.res * p.res * (p.last - p.first);
  tail_phase_r(acc, p, attn_text, smp, srow);
}

__global__ void __launch_bounds__(kThreads)
tail_fwd_s_kernel(ga_tail_params_t p, TokArgs toks, const uint8_t* __restrict__ masks, const float* __restrict__ weights,
                  const float* attn_text, float* smoothed, float* stats, int32_t* argmax, float* total) {
  extern __shared__ float simg[];
  const int npix = p.res * p.res, tp = p.last - p.first;
  const int smp = blockIdx.x;
  unsigned int dummy_ticket = 0u;
  tail_phase_s(p, toks, masks, weights, attn_text + (int64_t)smp * npix * tp, smoothed + (int64_t)smp * p.n_tokens * npix,
               stats + (int64_t)smp * p.n_tokens * GA_STATS, argmax + (int64_t)smp * p.n_tokens, total + smp,
               &dummy_ticket, simg);
}

// -------------------------------------------------------------------------------------------------- backward
// One launch, one warp per pixel.  Lane t (< n_tokens) owns tracked token t: it turns the upstream gradients and the
// forward's saved per-token scalars into d loss / d smoothed-map at the 3x3 neighbourhood of this pixel, pulls it
// through the adjoint of the reflect-padded filter, and hands the result to the lane that owns the token's column;
// then the warp does the x100-softmax backward over the tokens of this pixel.
struct TokenGrad {
  float g_col, g_row, g_in, g_out, g_max, g_sum, dp_mean, inv_sum, at_most;
  float r_gsum, r_gcol, r_grow, r_col, r_row, r_inv_sum;   // upstream gradients on / saved values of the raw statistics
  int argmax, box, strict_box, column;
};

__device__ __forceinline__ TokenGrad make_token_grad(const ga_tail_params_t& p, const ga_token_t& tk,
                                                     const float* st, int amax, float g_total, const float* gs) {
  TokenGrad g;
  const float denom = (float)(p.res - 1);
  const bool is_box = tk.kind == GA_TOKEN_BOX && tk.box >= 0;
  const float g_scaled = g_total * tk.group_weight + (gs ? gs[GA_STAT_SCALED] : 0.f);
  const float g_unscaled = gs ? gs[GA_STAT_UNSCALED] : 0.f;
  float g_center = gs ? gs[GA_STAT_CENTER] : 0.f;
  g.g_in = gs ? gs[GA_STAT_INSIDE] : 0.f;
  g.g_out = gs ? gs[GA_STAT_OUTSIDE] : 0.f;
  if (tk.kind == GA_TOKEN_COOR) {
    g_center += g_scaled + g_unscaled;
  } else if (tk.kind == GA_TOKEN_BOX) {
    g.g_in += g_scaled * p.inside_scale + g_unscaled;
    g.g_out += g_scaled * p.outside_scale + g_unscaled;
    if (tk.center_weight > 0.f) g_center += g_scaled * tk.center_weight;
  }
  if (!is_box) g.g_in = g.g_out = 0.f;
  const float dc = st[GA_STAT_COL] - tk.target_x, dr = st[GA_STAT_ROW] - tk.target_y;
  const float sgn_c = dc > 0.f ? 1.f : (dc < 0.f ? -1.f : 0.f);
  const float sgn_r = dr > 0.f ? 1.f : (dr < 0.f ? -1.f : 0.f);
  g.g_col = (gs ? gs[GA_STAT_COL] : 0.f) + g_center * sgn_c / denom;
  g.g_row = (gs ? gs[GA_STAT_ROW] : 0.f) + g_center * 4.f * sgn_r / denom;
  g.g_max = gs ? gs[GA_STAT_MAX] : 0.f;
  g.g_sum = gs ? gs[GA_STAT_SUM] : 0.f;
  g.r_gsum = gs ? gs[GA_STAT_RAW_SUM] : 0.f;
  g.r_gcol = gs ? gs[GA_STAT_RAW_COL] : 0.f;
  g.r_grow = gs ? gs[GA_STAT_RAW_ROW] : 0.f;
  g.r_col = st[GA_STAT_RAW_COL];
  g.r_row = st[GA_STAT_RAW_ROW];
  g.r_inv_sum = 1.f / st[GA_STAT_RAW_SUM];
  g.inv_sum = 1.f / st[GA_STAT_SUM];
  g.at_most = st[GA_STAT_NINSIDE] > 0.f ? 1.f / st[GA_STAT_NINSIDE] : 0.f;
  g.argmax = amax;
  g.column = tk.column;
  g.box = is_box ? tk.box : -1;
  g.strict_box = (is_box && p.strict) ? 1 : 0;
  // sum over pixels of dp * p, in closed form from the saved statistics
  g.dp_mean = g.g_col * st[GA_STAT_COL] + g.g_row * st[GA_STAT_ROW];
  if (is_box) {
    if (p.strict) g.dp_mean += -2.f * g.g_in * st[GA_STAT_HINGE_IN] + g.g_out * st[GA_STAT_HINGE_OUT];
    else g.dp_mean += -g.g_in * (1.f - st[GA_STAT_INSIDE]) + g.g_out * st[GA_STAT_OUTSIDE];
  }
  return g;
}

// d loss / d smoothed[pix] for one token
__device__ __forceinline__ float dsmoothed_at(const TokenGrad& g, int pix, int y, int x, int res, const uint8_t* masks,
                                              const float* weights, const float* sm) {
  const int npix = res * res;
  float dp = g.g_col * ((float)x + 0.5f) + g.g_row * ((float)y + 0.5f);
  if (g.box >= 0) {
    const bool in = masks[(int64_t)g.box * npix + pix] != 0;
    if (g.strict_box) {
      const float w = weights != nullptr ? weights[(int64_t)g.box * npix + pix] : 1.f;
      const float pr = sm[pix] * g.inv_sum;
      if (in) { if (g.at_most - pr > 0.f) dp -= 2.f * w * g.g_in; }
      else if (pr > 0.f) dp += w * g.g_out;
    } else {
      dp += in ? -g.g_in : g.g_out;
    }
  }
  float ds = (dp - g.dp_mean) * g.inv_sum + g.g_sum;
  if (pix == g.argmax) ds += g.g_max;
  return ds;
}

// One launch, one warp per group of 4 consecutive pixels (128-bit coalesced loads of the attn_text rows and stores of
// the d_abar rows, staged through shared memory); `groups_per_warp` groups per warp (1 when the launch is small).
__global__ void __launch_bounds__(kThreads)
tail_bwd_kernel(ga_tail_params_t p, TokArgs toks, const uint8_t* __restrict__ masks, const float* __restrict__ weights,
                const float* __restrict__ attn_text, const float* __restrict__ smoothed,
                const float* __restrict__ stats, const int32_t* __restrict__ argmax, const float* __restrict__ g_total,
                const float* __restrict__ g_stats, const float* __restrict__ g_attn_text, float* __restrict__ d_abar,
                int d_abar_rstride, int groups_per_warp) {
  extern __shared__ float sds[];            // d loss / d smoothed for [tile - halo, tile + halo), per token
  __shared__ TokenGrad tg[GA_MAX_TOKENS];
  __shared__ __align__(16) float s_in[kWarps][4 * GA_MAX_CTX];    // 4 attn_text rows
  __shared__ __align__(16) float s_out[kWarps][4 * GA_MAX_CTX];   // 4 d_abar rows
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int res = p.res, npix = res * res, tp = p.last - p.first;
  const int smp = blockIdx.y;
  attn_text += (int64_t)smp * npix * tp;
  smoothed += (int64_t)smp * p.n_tokens * npix;
  stats += (int64_t)smp * p.n_tokens * GA_STATS;
  argmax += (int64_t)smp * p.n_tokens;
  if (g_total != nullptr) g_total += smp;
  if (g_stats != nullptr) g_stats += (int64_t)smp * p.n_tokens * GA_STATS;
  if (g_attn_text != nullptr) g_attn_text += (int64_t)smp * npix * tp;
  d_abar += (int64_t)smp * npix * d_abar_rstride;

  // per-token scalars once per CTA: upstream gradients x the forward's saved statistics
  if ((int)threadIdx.x < p.n_tokens) {
    const int t = threadIdx.x;
    tg[t] = make_token_grad(p, toks.t[t], stats + (int64_t)t * GA_STATS, argmax[t],
                            g_total != nullptr ? g_total[0] : 0.f,
                            g_stats != nullptr ? g_stats + (int64_t)t * GA_STATS : nullptr);
  }
  __syncthreads();
  // d loss / d smoothed-map for the tile's pixels plus a halo of one row + one pixel on each side, every token:
  // computed once per CTA (each value is needed by up to 9 output pixels)
  const int ppc = 4 * kWarps * groups_per_warp;
  const int p0 = blockIdx.x * ppc;
  const int halo = p.smooth ? res + 1 : 0;
  const int lo = max(p0 - halo, 0), hi = min(p0 + ppc + halo, npix), span = ppc + 2 * halo;
  // (row / column of a pixel without an integer division: (pix + 0.5) / res in fp32 is exact for res <= 256)
  const float inv_res = 1.f / (float)res;
  const float inv_span = 1.f / (float)span;
  for (int i = threadIdx.x; i < p.n_tokens * span; i += blockDim.x) {
    const int t = (int)(((float)i + 0.5f) * inv_span), q = lo + (i - t * span);
    if (q < hi) {
      const int y = (int)(((float)q + 0.5f) * inv_res);
      sds[i] = dsmoothed_at(tg[t], q, y, q - y * res, res, masks, weights, smoothed + (int64_t)t * npix);
    }
  }
  __syncthreads();

  // d loss / d raw-map for the tile's own pixels, every token: the adjoint of the reflect-padded 3x3 filter applied to
  // the staged values, again once per CTA and spread over all threads (in the per-pixel loop below this used to run
  // on n_tokens lanes of every warp)
  float* sdi = sds + p.n_tokens * span;            // [token][pixel of the tile]
  for (int i = threadIdx.x; i < p.n_tokens * ppc; i += blockDim.x) {
    const int t = (int)(((float)i + 0.5f) / (float)ppc), pix = p0 + (i - t * ppc);
    float dimg = 0.f;
    if (pix < npix) {
      const float* ds = sds + t * span - lo;
      if (p.smooth) {
        const int y = (int)(((float)pix + 0.5f) * inv_res), x = pix - y * res;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy) {
          const int yy = y + dy;
          if (yy < 0 || yy >= res) continue;
          const float wy = p.w1d[1 - dy] + ((y == 1 && dy == -1) ? p.w1d[0] : 0.f) +
                           ((y == res - 2 && dy == 1) ? p.w1d[2] : 0.f);
#pragma unroll
          for (int dx = -1; dx <= 1; ++dx) {
            const int xx = x + dx;
            if (xx < 0 || xx >= res) continue;
            const float wx = p.w1d[1 - dx] + ((x == 1 && dx == -1) ? p.w1d[0] : 0.f) +
                             ((x == res - 2 && dx == 1) ? p.w1d[2] : 0.f);
            dimg = fmaf(wy * wx, ds[yy * res + xx], dimg);
          }
        }
      } else {
        dimg = ds[pix];
      }
      // raw-map statistics (custom losses) act on the un-smoothed map directly:
      // d rcol / d A[pix] = ((x + .5) - rcol) / rsum, d rsum / d A[pix] = 1
      const TokenGrad& g = tg[t];
      if (g.r_gcol != 0.f || g.r_grow != 0.f || g.r_gsum != 0.f) {
        const int y = (int)(((float)pix + 0.5f) * inv_res), x = pix - y * res;
        dimg += g.r_gsum + (g.r_gcol * (((float)x + 0.5f) - g.r_col) + g.r_grow * (((float)y + 0.5f) - g.r_row)) * g.r_inv_sum;
      }
    }
    sdi[i] = dimg;
  }
  __syncthreads();

  const float k = p.temperature * p.inv_count;
  const bool vec_out = (d_abar_rstride & 3) == 0;
  const bool sparse = g_attn_text == nullptr;      // the map gradient is non-zero only in the tracked tokens' columns
  for (int gi = 0; gi < groups_per_warp; ++gi) {
    const int g0 = p0 + (gi * kWarps + warp) * 4;     // first pixel of this warp's group
    if (g0 >= npix) break;
    // stage the 4 attn_text rows: tp float4 chunks, contiguous and 16-byte aligned (g0 % 4 == 0)
    const float4* src = reinterpret_cast<const float4*>(attn_text + (int64_t)g0 * tp);
#pragma unroll
    for (int kk = 0; kk < kKPL; ++kk) {
      const int c = lane + 32 * kk;
      if (c < tp) reinterpret_cast<float4*>(s_in[warp])[c] = __ldg(src + c);
    }
    __syncwarp();
    if (sparse && vec_out) {
      // Fast path (no upstream gradient on attn_text: the map gradient is non-zero only in the tracked tokens' columns,
      // so sum_j a_j da_j has n_tokens terms and everything else is elementwise).  Lanes 0..3 compute the dot product of
      // "their" pixel; then the warp writes the 4 rows as aligned float4 chunks straight to global memory with
      // da = 0, and 4 * n_tokens lanes patch the tracked columns.
      const int rs4 = d_abar_rstride >> 2;
      float dotq = 0.f;
      if (lane < 4 && g0 + lane < npix) {
        for (int t = 0; t < p.n_tokens; ++t)
          dotq = fmaf(s_in[warp][lane * tp + tg[t].column], sdi[t * ppc + (g0 + lane - p0)], dotq);
      }
      float dots[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) dots[q] = __shfl_sync(0xffffffffu, dotq, q);
      float* dst = d_abar + (int64_t)g0 * d_abar_rstride;
      for (int c = lane; c < 4 * rs4; c += 32) {
        const int q = (c >= rs4) + (c >= 2 * rs4) + (c >= 3 * rs4);      // c / rs4 without the runtime division
        const int jc = (c - q * rs4) << 2;
        if (g0 + q >= npix) break;
        const float* arow = s_in[warp] + q * tp - p.first;
        const float nk = -k * (q == 0 ? dots[0] : q == 1 ? dots[1] : q == 2 ? dots[2] : dots[3]);
        float4 o;
        o.x = (jc + 0 >= p.first && jc + 0 < p.last) ? nk * arow[jc + 0] : 0.f;
        o.y = (jc + 1 >= p.first && jc + 1 < p.last) ? nk * arow[jc + 1] : 0.f;
        o.z = (jc + 2 >= p.first && jc + 2 < p.last) ? nk * arow[jc + 2] : 0.f;
        o.w = (jc + 3 >= p.first && jc + 3 < p.last) ? nk * arow[jc + 3] : 0.f;
        *reinterpret_cast<float4*>(dst + q * d_abar_rstride + jc) = o;
      }
      __syncwarp();                                   // orders the patch stores below after the row stores above
      for (int i = lane; i < 4 * p.n_tokens; i += 32) {
        const int q = i & 3, t = i >> 2;
        if (g0 + q < npix) {
          const int col = tg[t].column;
          float da = 0.f;
          for (int t2 = 0; t2 < p.n_tokens; ++t2)     // tokens that share a column (never in practice) add up
            if (tg[t2].column == col) da += sdi[t2 * ppc + (g0 + q - p0)];
          const float dq = q == 0 ? dots[0] : q == 1 ? dots[1] : q == 2 ? dots[2] : dots[3];
          dst[q * d_abar_rstride + col + p.first] = k * s_in[warp][q * tp + col] * (da - dq);
        }
      }
      __syncwarp();
      continue;
    }
    for (int q = 0; q < 4; ++q) {
      const int pix = g0 + q;
      const float* arow = s_in[warp] + q * tp;
      // softmax backward over the text tokens of this pixel: lanes are tokens
      float a[kKPL], da[kKPL], dot = 0.f;
#pragma unroll
      for (int kk = 0; kk < kKPL; ++kk) {
        const int j = lane + 32 * kk;
        const bool live = j >= p.first && j < p.last;
        a[kk] = live ? arow[j - p.first] : 0.f;
        da[kk] = (live && !sparse) ? g_attn_text[(int64_t)pix * tp + (j - p.first)] : 0.f;
      }
      for (int t = 0; t < p.n_tokens; ++t) {         // smem broadcasts: every lane reads the same words
        const float gv = sdi[t * ppc + (pix - p0)];
        const int col = tg[t].column;
        if (sparse) dot = fmaf(arow[col], gv, dot);   // sum_j a_j da_j has n_tokens terms: no warp reduction
#pragma unroll
        for (int kk = 0; kk < kKPL; ++kk)
          if (col + p.first == lane + 32 * kk) da[kk] += gv;
      }
      if (!sparse) {
#pragma unroll
        for (int kk = 0; kk < kKPL; ++kk) dot = fmaf(a[kk], da[kk], dot);
        dot = warp_sum(dot);
      }
#pragma unroll
      for (int kk = 0; kk < kKPL; ++kk) {
        const int j = lane + 32 * kk;
        if (j < d_abar_rstride) {   // padding columns (>= n_ctx) are written as zeros too
          const float val = (j >= p.first && j < p.last) ? k * a[kk] * (da[kk] - dot) : 0.f;
          if (vec_out) s_out[warp][q * d_abar_rstride + j] = val;
          else d_abar[(int64_t)pix * d_abar_rstride + j] = val;
        }
      }
    }
    if (vec_out) {
      __syncwarp();
      float4* dst = reinterpret_cast<float4*>(d_abar + (int64_t)g0 * d_abar_rstride);
#pragma unroll
      for (int kk = 0; kk < kKPL; ++kk) {
        const int c = lane + 32 * kk;
        if (c < d_abar_rstride) dst[c] = reinterpret_cast<const float4*>(s_out[warp])[c];
      }
    }
    __syncwarp();
  }
}

// Rows of the sparse backward: out[px][j] = -k dot[px] a[px][j - first] for the text columns, 0 elsewhere.  One warp per
// pixel row, lanes over the padded output row (three slots: columns lane, lane + 32, lane + 64): every load and store
// instruction of a warp covers one contiguous 128-byte span; four pixels per iteration keep 12 loads per lane in flight.
// With compile-time row lengths (TP, RS, FIRST != 0: the Stable Diffusion shape) every access of an iteration is an
// immediate offset from two base pointers: 13 warp-instructions per pixel instead of the 68 of the first version
// (64-bit address arithmetic per access, per-slot token tests; ncu: 75 % of the kernel's instructions, issue slots 64 %).
template <int TP, int RS, int FIRST>
__device__ __forceinline__ void tail_bwd_rows(const float* a0, float* __restrict__ o0,
                                              const float* __restrict__ sdot, float k, int n_own, int tp_rt, int rs_rt,
                                              int first_rt) {
  const int tp = TP ? TP : tp_rt, rs = RS ? RS : rs_rt, first = TP ? FIRST : first_rt;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  bool rd[3], wr[3];
#pragma unroll
  for (int sl = 0; sl < 3; ++sl) {
    const int j = lane + 32 * sl;
    rd[sl] = j >= first && j < first + tp;
    wr[sl] = j < rs;
  }
  constexpr int kPix = 4;
  for (int px0 = warp * kPix; px0 < n_own; px0 += kWarps * kPix) {
    const float* ar = a0 + px0 * tp + (lane - first);
    float* orow = o0 + px0 * rs + lane;
    float x[kPix][3];
#pragma unroll
    for (int u = 0; u < kPix; ++u) {
      const bool live = TP ? true : (px0 + u < n_own);       // (the fixed-shape path is only taken with n_own % 4 == 0)
#pragma unroll
      for (int sl = 0; sl < 3; ++sl) x[u][sl] = (live && rd[sl]) ? ar[u * tp + 32 * sl] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < kPix; ++u) {
      if (!TP && px0 + u >= n_own) break;
      const float nk = -k * sdot[px0 + u];
#pragma unroll
      for (int sl = 0; sl < 3; ++sl)
        if (wr[sl]) orow[u * rs + 32 * sl] = nk * x[u][sl];
    }
  }
}

// Backward, fast path (no upstream gradient on attn_text -- every launch of the guided pipeline): the map gradient is
// non-zero only in the tracked tokens' columns, so a row of d_abar is the attn_text row of the same pixel scaled by one
// per-pixel scalar (-k * sum_t a[col_t] dA_t), with n_tokens entries patched.  The kernel is therefore a shifted,
// scaled row copy (75-float rows in, 80-float padded rows out) and is laid out for instruction count, which is what
// bounded the previous version (ncu: issue slots 81 %, DRAM 36 %): one CTA owns `tile` row-major pixels of one sample
// plus a halo of one row + one pixel on each side for the 3x3 filter adjoint; the per-token gradients dA_t are computed
// once per CTA, one thread per pixel; the streaming phase gives every thread whole float4 chunks of the output (4 scalar
// loads, 4 multiplies, one 128-bit store).
constexpr int kTailBwdMinCtas = 4;    // resident CTAs per SM the register allocation must allow
// (round 2, second pass) The tile's attn_text rows -- tile x 75 contiguous floats -- are fetched by ONE bulk copy
// (cp.async.bulk global -> shared, mbarrier complete_tx) issued before anything else, so the stream is in flight while
// phases 1-2 chase their small dependent loads; phase 2 and the row phase then read shared memory.  Before, a CTA's
// global row loads only started after two __syncthreads (ncu: 40 % of the stall samples sat in phases 1-2 with the
// memory pipe idle).
__global__ void __launch_bounds__(kThreads, kTailBwdMinCtas)
tail_bwd_sparse_kernel(ga_tail_params_t p, TokArgs toks, const uint8_t* __restrict__ masks,
                       const float* __restrict__ weights, const float* __restrict__ attn_text,
                       const float* __restrict__ smoothed, const float* __restrict__ stats,
                       const int32_t* __restrict__ argmax, const float* __restrict__ g_total,
                       const float* __restrict__ g_stats, float* __restrict__ d_abar, int d_abar_rstride, int tile) {
  extern __shared__ __align__(16) float srows[];   // [tile][tp] attn_text rows | sds (see below)
  __shared__ TokenGrad tg[GA_MAX_TOKENS];
  __shared__ __align__(8) uint64_t rows_bar;
  const int res = p.res, npix = res * res, tp = p.last - p.first, nt = p.n_tokens;
  const int smp = blockIdx.y;
  attn_text += (int64_t)smp * npix * tp;
  smoothed += (int64_t)smp * nt * npix;
  stats += (int64_t)smp * nt * GA_STATS;
  argmax += (int64_t)smp * nt;
  d_abar += (int64_t)smp * npix * d_abar_rstride;
  float* sds = srows + tile * tp;           // [token][tile + 2 halo] d loss / d smoothed | [token][tile] dA | [tile] dot
  {
    const int p0b = blockIdx.x * tile, n_ownb = min(tile, npix - p0b);
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&rows_bar);
    if (threadIdx.x == 0) {
      const uint32_t bytes = (uint32_t)n_ownb * tp * 4u;     // multiple of 16: npix % 4 == 0, tile % 4 == 0
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(srows)), "l"(attn_text + (int64_t)p0b * tp), "r"(bytes), "r"(bar)
                   : "memory");
    }
  }
  if ((int)threadIdx.x < nt) {
    const int t = threadIdx.x;
    tg[t] = make_token_grad(p, toks.t[t], stats + (int64_t)t * GA_STATS, argmax[t],
                            g_total != nullptr ? g_total[smp] : 0.f,
                            g_stats != nullptr ? g_stats + ((int64_t)smp * nt + t) * GA_STATS : nullptr);
  }
  __syncthreads();
  const int p0 = blockIdx.x * tile;
  const int halo = p.smooth ? res + 1 : 0;
  const int lo = max(p0 - halo, 0), hi = min(p0 + tile + halo, npix), span = tile + 2 * halo;
  const int n_own = min(tile, npix - p0);
  const float inv_res = 1.f / (float)res;
  float* sdi = sds + nt * span;
  float* sdot = sdi + nt * tile;
  bool has_dup = false;
  for (int t = 1; t < nt; ++t)
    for (int t2 = 0; t2 < t; ++t2) has_dup |= tg[t].column == tg[t2].column;
  float* sda = has_dup ? sdot + tile : sdi;       // per-column sums of dA; the launcher sizes the extra [token][tile]
  // phase 1: d loss / d smoothed over tile + halo, one thread per pixel, tokens in the inner loop
  for (int i = threadIdx.x; i < hi - lo; i += kThreads) {
    const int q = lo + i;
    const int y = (int)(((float)q + 0.5f) * inv_res), x = q - y * res;
    for (int t = 0; t < nt; ++t)
      sds[t * span + i] = dsmoothed_at(tg[t], q, y, x, res, masks, weights, smoothed + (int64_t)t * npix);
  }
  __syncthreads();
  // the tile's rows have landed? (init + copy were issued by thread 0 before the first __syncthreads)
  {
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&rows_bar);
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                   : "=r"(done) : "r"(bar) : "memory");
      if (spin > (1u << 24)) __trap();       // a lost copy must fail the launch, not hang the GPU
    }
  }
  // phase 2: adjoint of the reflect-padded 3x3 filter (+ raw-map statistics) -> dA_t for the tile's own pixels, and
  // the per-pixel dot product sum_t a[col_t] dA_t in token order (same fma chain as the general kernel)
  for (int px = threadIdx.x; px < n_own; px += kThreads) {
    const int pix = p0 + px;
    const int y = (int)(((float)pix + 0.5f) * inv_res), x = pix - y * res;
    float wy[3], wx[3];
#pragma unroll
    for (int dd = -1; dd <= 1; ++dd) {
      wy[dd + 1] = p.w1d[1 - dd] + ((y == 1 && dd == -1) ? p.w1d[0] : 0.f) + ((y == res - 2 && dd == 1) ? p.w1d[2] : 0.f);
      wx[dd + 1] = p.w1d[1 - dd] + ((x == 1 && dd == -1) ? p.w1d[0] : 0.f) + ((x == res - 2 && dd == 1) ? p.w1d[2] : 0.f);
    }
    float dot = 0.f;
    for (int t = 0; t < nt; ++t) {
      const float* ds = sds + t * span - lo;
      float dimg = 0.f;
      if (p.smooth) {
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy) {
          const int yy = y + dy;
          if (yy < 0 || yy >= res) continue;
#pragma unroll
          for (int dx = -1; dx <= 1; ++dx) {
            const int xx = x + dx;
            if (xx < 0 || xx >= res) continue;
            dimg = fmaf(wy[dy + 1] * wx[dx + 1], ds[yy * res + xx], dimg);
          }
        }
      } else {
        dimg = ds[pix];
      }
      const TokenGrad& g = tg[t];
      if (g.r_gcol != 0.f || g.r_grow != 0.f || g.r_gsum != 0.f)
        dimg += g.r_gsum + (g.r_gcol * (((float)x + 0.5f) - g.r_col) + g.r_grow * (((float)y + 0.5f) - g.r_row)) * g.r_inv_sum;
      sdi[t * tile + px] = dimg;
      dot = fmaf(srows[px * tp + g.column], dimg, dot);
    }
    sdot[px] = dot;
    if (has_dup) {          // tokens that share a column (never in practice): their gradients add up
      for (int t = 0; t < nt; ++t) {
        float da = 0.f;
        for (int t2 = 0; t2 < nt; ++t2)
          if (tg[t2].column == tg[t].column) da += sdi[t2 * tile + px];
        sda[t * tile + px] = da;
      }
    }
  }
  __syncthreads();
  // phase 3: the rows -- a shifted, scaled copy (see tail_bwd_rows) -- then the nt patched entries of every row
  const float k = p.temperature * p.inv_count;
  const float* a0 = srows;
  float* o0 = d_abar + (int64_t)p0 * d_abar_rstride;
  if (tp == 75 && d_abar_rstride == 80 && p.first == 1 && (n_own & 3) == 0)
    tail_bwd_rows<75, 80, 1>(a0, o0, sdot, k, n_own, tp, d_abar_rstride, p.first);      // SD: 77 tokens, text = [1, 76)
  else
    tail_bwd_rows<0, 0, 0>(a0, o0, sdot, k, n_own, tp, d_abar_rstride, p.first);
  __syncthreads();          // the copy wrote (a scaled value into) the tracked columns too: order the patch after it
  for (int px = threadIdx.x; px < n_own; px += kThreads) {
    const float dot = sdot[px];
    const float* arow = a0 + px * tp;
    float* orow = o0 + (int64_t)px * d_abar_rstride + p.first;
    for (int t = 0; t < nt; ++t) {
      const int col = tg[t].column;
      orow[col] = k * arow[col] * (sda[t * tile + px] - dot);                              // k a (dA - dot)
    }
  }
}

// --------------------------------------------------------------------------------------- stand-alone stages
__global__ void smooth_fwd_kernel(const float* __restrict__ maps, float* __restrict__ out, int n, int res, float w0,
                                  float w1, float w2) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x, npix = res * res;
  if (idx >= n * npix) return;
  const int i = idx / npix, pix = idx - i * npix, y = pix / res, x = pix - y * res;
  const float w[3] = {w0, w1, w2};
  out[idx] = smooth_at(maps + (int64_t)i * npix, y, x, res, w);
}

__global__ void smooth_bwd_kernel(const float* __restrict__ g_out, float* __restrict__ g_maps, int n, int res, float w0,
                                  float w1, float w2) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x, npix = res * res;
  if (idx >= n * npix) return;
  const int i = idx / npix, pix = idx - i * npix, y = pix / res, x = pix - y * res;
  const float w[3] = {w0, w1, w2};
  const float* g = g_out + (int64_t)i * npix;
  float acc = 0.f;
  for (int dy = -1; dy <= 1; ++dy) {
    const int yy = y + dy;
    if (yy < 0 || yy >= res) continue;
    const float my = adjoint_tap(y, yy, res, w);
    for (int dx = -1; dx <= 1; ++dx) {
      const int xx = x + dx;
      if (xx < 0 || xx >= res) continue;
      acc = fmaf(my * adjoint_tap(x, xx, res, w), g[yy * res + xx], acc);
    }
  }
  g_maps[idx] = acc;
}

// one CTA; out2 = (inside, outside)
__global__ void box_loss_fwd_kernel(const float* __restrict__ pmap, const uint8_t* __restrict__ mask,
                                    const float* __restrict__ weights, int res, int strict, float* out2) {
  __shared__ float red[3][kWarps];
  const int npix = res * res, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float nin = 0.f;
  for (int pix = threadIdx.x; pix < npix; pix += blockDim.x) nin += mask[pix];
  nin = warp_sum(nin);
  if (lane == 0) red[0][warp] = nin;
  __syncthreads();
  nin = 0.f;
  for (int w = 0; w < kWarps; ++w) nin += red[0][w];
  const float at_most = nin > 0.f ? 1.f / nin : 0.f;
  float sin_ = 0.f, sout = 0.f;
  for (int pix = threadIdx.x; pix < npix; pix += blockDim.x) {
    const float pr = pmap[pix];
    const bool in = mask[pix] != 0;
    if (strict) {
      const float w = weights != nullptr ? weights[pix] : 1.f;
      if (in) { const float gap = at_most - pr; if (gap > 0.f) sin_ = fmaf(2.f * w, gap, sin_); }
      else if (pr > 0.f) sout = fmaf(w, pr, sout);
    } else {
      if (in) sin_ += pr; else sout += pr;
    }
  }
  sin_ = warp_sum(sin_); sout = warp_sum(sout);
  if (lane == 0) { red[1][warp] = sin_; red[2][warp] = sout; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int w = 0; w < kWarps; ++w) { a += red[1][w]; b += red[2][w]; }
    out2[0] = strict ? a : 1.f - a;
    out2[1] = b;
  }
}

__global__ void box_loss_bwd_kernel(const float* __restrict__ pmap, const uint8_t* __restrict__ mask,
                                    const float* __restrict__ weights, int res, int strict,
                                    const float* __restrict__ g_out2, float* __restrict__ g_p) {
  __shared__ float red[kWarps];
  const int npix = res * res, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float nin = 0.f;
  for (int pix = threadIdx.x; pix < npix; pix += blockDim.x) nin += mask[pix];
  nin = warp_sum(nin);
  if (lane == 0) red[warp] = nin;
  __syncthreads();
  nin = 0.f;
  for (int w = 0; w < kWarps; ++w) nin += red[w];
  const float at_most = nin > 0.f ? 1.f / nin : 0.f;
  const float gi = g_out2[0], go = g_out2[1];
  for (int pix = threadIdx.x; pix < npix; pix += blockDim.x) {
    const bool in = mask[pix] != 0;
    float g = 0.f;
    if (strict) {
      const float w = weights != nullptr ? weights[pix] : 1.f;
      const float pr = pmap[pix];
      if (in) { if (at_most - pr > 0.f) g = -2.f * w * gi; }
      else if (pr > 0.f) g = w * go;
    } else {
      g = in ? -gi : go;
    }
    g_p[pix] = g;
  }
}

}  // namespace tail
}  // namespace ga

// =============================================================================================== C ABI wrappers
using namespace ga;

static int check_tail_params(const ga_tail_params_t* p, const ga_token_t* toks) {
  GA_CHECK_ARG(p != nullptr, "params_host is NULL");
  GA_CHECK_ARG(p->res >= 2 && p->res <= 256, "res %d out of range [2, 256]", p->res);
  GA_CHECK_ARG(p->n_ctx >= 1 && p->n_ctx <= GA_MAX_CTX, "n_ctx %d out of range [1, %d]", p->n_ctx, GA_MAX_CTX);
  GA_CHECK_ARG(p->first >= 0 && p->first < p->last && p->last <= p->n_ctx, "bad token window [%d, %d) for n_ctx %d",
               p->first, p->last, p->n_ctx);
  GA_CHECK_ARG(p->n_tokens >= 0 && p->n_tokens <= GA_MAX_TOKENS, "n_tokens %d out of range [0, %d]", p->n_tokens,
               GA_MAX_TOKENS);
  GA_CHECK_ARG(p->n_tokens == 0 || toks != nullptr, "tokens_host is NULL");
  GA_CHECK_ARG(p->n_samples >= 1 && p->n_samples <= 65535, "n_samples %d out of range [1, 65535]", p->n_samples);
  for (int t = 0; t < p->n_tokens; ++t) {
    GA_CHECK_ARG(toks[t].column >= 0 && toks[t].column < p->last - p->first,
                 "token %d: column %d outside the renormalised window of %d tokens", t, toks[t].column,
                 p->last - p->first);
    GA_CHECK_ARG(toks[t].kind >= GA_TOKEN_COOR && toks[t].kind <= GA_TOKEN_KEYWORD, "token %d: bad kind %d", t,
                 toks[t].kind);
  }
  return GA_OK;
}

extern "C" int ga_rasterize_boxes(const double* boxes_host, int n_boxes, int res, double shrink, uint8_t* masks,
                                  ga_stream_t stream) {
  GA_CHECK_ARG(n_boxes >= 0 && res >= 1 && res <= 4096, "bad n_boxes %d / res %d", n_boxes, res);
  if (n_boxes == 0) return GA_OK;
  GA_CHECK_ARG(boxes_host != nullptr && masks != nullptr, "NULL pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int b0 = 0; b0 < n_boxes; b0 += GA_MAX_BOXES) {
    const int n = n_boxes - b0 < GA_MAX_BOXES ? n_boxes - b0 : GA_MAX_BOXES;
    tail::BoxArgs a;
    for (int i = 0; i < n; ++i) {
      a.x[i] = boxes_host[4 * (b0 + i) + 0]; a.y[i] = boxes_host[4 * (b0 + i) + 1];
      a.w[i] = boxes_host[4 * (b0 + i) + 2]; a.h[i] = boxes_host[4 * (b0 + i) + 3];
    }
    const int total = n * res * res;
    tail::rasterize_kernel<<<(total + 255) / 256, 256, 0, st>>>(a, n, res, shrink, masks + (size_t)b0 * res * res);
    int rc = check_launch("rasterize_boxes");
    if (rc != GA_OK) return rc;
  }
  return GA_OK;
}

extern "C" int ga_guidance_tail_fwd(const float* const* acc_host, const int32_t* slices_host, int n_acc,
                                    const ga_tail_params_t* params_host, const ga_token_t* tokens_host,
                                    const uint8_t* masks, const float* weights, float* attn_text, float* smoothed,
                                    float* stats, int32_t* argmax, float* total, uint32_t* ticket,
                                    ga_stream_t stream) {
  int rc = check_tail_params(params_host, tokens_host);
  if (rc != GA_OK) return rc;
  GA_CHECK_ARG(n_acc >= 1 && n_acc <= GA_MAX_ACC_SLICES, "n_acc %d out of range [1, %d]", n_acc, GA_MAX_ACC_SLICES);
  GA_CHECK_ARG(acc_host != nullptr && slices_host != nullptr && attn_text != nullptr && total != nullptr,
               "NULL pointer");
  const ga_tail_params_t& p = *params_host;
  GA_CHECK_ARG(p.n_tokens == 0 || (smoothed != nullptr && stats != nullptr && argmax != nullptr), "NULL output");
  tail::AccArgs acc;
  acc.n = n_acc;
  for (int i = 0; i < n_acc; ++i) {
    GA_CHECK_ARG(acc_host[i] != nullptr && slices_host[i] >= 1, "accumulator %d is NULL or empty", i);
    acc.ptr[i] = acc_host[i];
    acc.slices[i] = slices_host[i];
  }
  tail::TokArgs toks;
  for (int t = 0; t < p.n_tokens; ++t) {
    toks.t[t] = tokens_host[t];
    GA_CHECK_ARG(toks.t[t].kind != GA_TOKEN_BOX || toks.t[t].box < 0 || masks != nullptr, "BOX token without masks");
  }
  GA_CHECK_ARG(ticket != nullptr, "ticket workspace is NULL");
  const int npix = p.res * p.res;
  const int n_maps = p.n_tokens < tail::kWarps ? (p.n_tokens > 0 ? p.n_tokens : 1) : tail::kWarps;
  const size_t smem = (size_t)n_maps * npix * sizeof(float);     // phase S: one staged map per concurrently processed token
  if (smem > 200 * 1024) return fail(GA_ERR_UNSUPPORTED, "res %d too large for the fused tail", p.res);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (smem > 24 * 1024) {   // static (phase R rows) + dynamic (phase S maps) can pass the 48 KB default from res 32 up
    static bool raised[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !raised[dev]) {
      cudaError_t e = cudaFuncSetAttribute(tail::tail_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      raised[dev] = true;
    }
  }
  GA_CHECK_ARG(npix % 4 == 0, "res*res must be a multiple of 4 (res %d)", p.res);
  for (int i = 0; i < n_acc; ++i) GA_CHECK_ALIGN(acc_host[i], 16, "accumulator");
  const dim3 grid((npix / 4 + tail::kWarps - 1) / tail::kWarps, p.n_samples);
  if ((int64_t)p.n_samples * npix >= 96 * 1024 && smem <= 48 * 1024) {
    // many samples: lean per-pixel kernel + one CTA per sample for the per-token phase (see the kernels' comment)
    tail::tail_fwd_r_kernel<<<grid, tail::kThreads, 0, st>>>(acc, p, attn_text);
    int rc2 = check_launch("guidance_tail_fwd_r");
    if (rc2 != GA_OK) return rc2;
    // one warp per tracked token: a block of n_maps warps (3 for the usual prompts) keeps ~3x more samples resident
    // per SM than 8-warp blocks with 5 idle warps (the per-token phase is latency-bound: strided column gathers)
    tail::tail_fwd_s_kernel<<<p.n_samples, 32 * n_maps, smem, st>>>(p, toks, masks, weights, attn_text, smoothed,
                                                                   stats, argmax, total);
    return check_launch("guidance_tail_fwd_s");
  }
  tail::tail_fwd_kernel<<<grid, tail::kThreads, smem, st>>>(acc, p, toks, masks, weights, attn_text, smoothed, stats,
                                                            argmax, total, reinterpret_cast<unsigned int*>(ticket));
  return check_launch("guidance_tail_fwd");
}

extern "C" int ga_guidance_tail_bwd(const ga_tail_params_t* params_host, const ga_token_t* tokens_host,
                                    const uint8_t* masks, const float* weights, const float* attn_text,
                                    const float* smoothed, const float* stats, const int32_t* argmax,
                                    const float* g_total, const float* g_stats, const float* g_attn_text,
                                    float* d_abar, int d_abar_row_stride, ga_stream_t stream) {
  int rc = check_tail_params(params_host, tokens_host);
  if (rc != GA_OK) return rc;
  const ga_tail_params_t& p = *params_host;
  GA_CHECK_ARG(attn_text != nullptr && d_abar != nullptr, "NULL pointer");
  GA_CHECK_ARG(d_abar_row_stride >= p.n_ctx && d_abar_row_stride <= GA_MAX_CTX, "d_abar_row_stride %d out of range",
               d_abar_row_stride);
  GA_CHECK_ARG(p.n_tokens == 0 || (smoothed != nullptr && stats != nullptr && argmax != nullptr), "NULL saved tensor");
  tail::TokArgs toks;
  for (int t = 0; t < p.n_tokens; ++t) toks.t[t] = tokens_host[t];
  const int npix = p.res * p.res;
  GA_CHECK_ARG(npix % 4 == 0, "res*res must be a multiple of 4 (res %d)", p.res);
  GA_CHECK_ALIGN(attn_text, 16, "attn_text");
  if ((d_abar_row_stride & 3) == 0) GA_CHECK_ALIGN(d_abar, 16, "d_abar");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (g_attn_text == nullptr && (d_abar_row_stride & 3) == 0) {
    // the pipeline's case: sparse map gradient.  A CTA owns 128 pixels (half of a 16x16 map) and their halo.
    const int tile = 128;
    const int nt = p.n_tokens > 0 ? p.n_tokens : 1;
    const int tp = p.last - p.first;
    const size_t smem = ((size_t)tile * tp + (size_t)nt * (3 * tile + 2 * (p.res + 1)) + tile) * sizeof(float);
    // (small launches -- the pipeline's own single evaluation, small seed batches -- are latency-bound and stay on the
    // general kernel below, which spreads its 4-pixel groups over more CTAs: 4.4 vs 10 us at 1 sample, 6.2 vs 13.5 us
    // at 64; the crossover measured on B200 is ~400 samples at res 16: profiles/r02_microbench_tail_bwd.jsonl)
    if (smem <= 100 * 1024 && (int64_t)p.n_samples * npix >= 96 * 1024) {
      static bool attr_set = false;
      if (!attr_set) {
        cudaFuncSetAttribute(tail::tail_bwd_sparse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        cudaFuncSetAttribute(tail::tail_bwd_sparse_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        attr_set = true;
      }
      const dim3 grid((npix + tile - 1) / tile, p.n_samples);
      tail::tail_bwd_sparse_kernel<<<grid, tail::kThreads, smem, st>>>(p, toks, masks, weights, attn_text, smoothed,
                                                                      stats, argmax, g_total, g_stats, d_abar,
                                                                      d_abar_row_stride, tile);
      return check_launch("guidance_tail_bwd_sparse");
    }
  }
  // general path (upstream gradient on attn_text: Python custom-loss plug-ins)
  int groups_per_warp = ((int64_t)p.n_samples * npix >= 128 * 1024) ? 4 : 1;
  auto halo_bytes = [&](int gpw) {
    // staged d loss / d smoothed (tile + halo) and d loss / d raw map (tile), per token
    return (size_t)(p.n_tokens > 0 ? p.n_tokens : 1) * (2 * 4 * tail::kWarps * gpw + 2 * (p.res + 1)) * sizeof(float);
  };
  if (halo_bytes(groups_per_warp) > 14 * 1024) groups_per_warp = 1;
  const int ppc = 4 * tail::kWarps * groups_per_warp;
  const dim3 grid((npix + ppc - 1) / ppc, p.n_samples);
  const size_t smem = halo_bytes(groups_per_warp);
  if (smem > 14 * 1024) return fail(GA_ERR_UNSUPPORTED, "res %d x %d tokens too large for the tail backward", p.res, p.n_tokens);
  tail::tail_bwd_kernel<<<grid, tail::kThreads, smem, st>>>(
      p, toks, masks, weights, attn_text, smoothed, stats, argmax, g_total, g_stats, g_attn_text, d_abar,
      d_abar_row_stride, groups_per_warp);
  return check_launch("guidance_tail_bwd");
}

extern "C" int ga_smooth_fwd(const float* maps, float* out, int n_maps, int res, const float* w1d_host,
                             ga_stream_t stream) {
  GA_CHECK_ARG(maps && out && w1d_host && n_maps >= 0 && res >= 2, "bad argument");
  const int total = n_maps * res * res;
  if (total == 0) return GA_OK;
  tail::smooth_fwd_kernel<<<(total + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      maps, out, n_maps, res, w1d_host[0], w1d_host[1], w1d_host[2]);
  return check_launch("smooth_fwd");
}

extern "C" int ga_smooth_bwd(const float* g_out, float* g_maps, int n_maps, int res, const float* w1d_host,
                             ga_stream_t stream) {
  GA_CHECK_ARG(g_out && g_maps && w1d_host && n_maps >= 0 && res >= 2, "bad argument");
  const int total = n_maps * res * res;
  if (total == 0) return GA_OK;
  tail::smooth_bwd_kernel<<<(total + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      g_out, g_maps, n_maps, res, w1d_host[0], w1d_host[1], w1d_host[2]);
  return check_launch("smooth_bwd");
}

extern "C" int ga_box_loss_fwd(const float* p, const uint8_t* mask, const float* weights, int res, int strict,
                               float* out2, ga_stream_t stream) {
  GA_CHECK_ARG(p && mask && out2 && res >= 1, "bad argument");
  tail::box_loss_fwd_kernel<<<1, tail::kThreads, 0, static_cast<cudaStream_t>(stream)>>>(p, mask, weights, res, strict,
                                                                                        out2);
  return check_launch("box_loss_fwd");
}

extern "C" int ga_box_loss_bwd(const float* p, const uint8_t* mask, const float* weights, int res, int strict,
                               const float* g_out2, float* g_p, ga_stream_t stream) {
  GA_CHECK_ARG(p && mask && g_out2 && g_p && res >= 1, "bad argument");
  tail::box_loss_bwd_kernel<<<1, tail::kThreads, 0, static_cast<cudaStream_t>(stream)>>>(p, mask, weights, res, strict,
                                                                                        g_out2, g_p);
  return check_launch("box_loss_bwd");
}
