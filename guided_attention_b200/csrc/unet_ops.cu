// UNet-side kernels of the guidance path (sm_100a): GroupNorm (+ SiLU, + shift) forward / backward, conv bias + residual,
// the GEGLU gate forward / backward and the LayerNorm forward, all on channels-last / token-major 16-bit activations with
// 128-bit accesses.  GroupNorm is described here; the three smaller kernels have their own headers further down.
//
// Why it is here: the guidance path differentiates the loss with respect to the LATENTS, so every guided step runs the
// UNet forward AND backward (reference pipeline_guided_attention.py:455-470 `_update_latent`, :583-743 the UNet forward
// the pipeline drives).  In the launch list of a guided image (profiles/r02b_ncu_launches_summary.txt) the GroupNorm
// of the ResNet / transformer blocks is the largest non-GEMM item: PyTorch runs it as RowwiseMoments (one CTA per
// (sample, group): 32 CTAs on 148 SMs at batch 1, 26 us) + ComputeFusedParams + an elementwise kernel + a separate
// SiLU, and five more kernels in the backward -- 27 % of the device time of an image.  Here one GroupNorm(+SiLU) is two
// launches per direction, each spread over the whole GPU, HBM/L2-bound byte work:
//
//   stats kernel   grid (pixel chunks, channel slices, samples).  A thread owns one 8-channel vector (128-bit loads,
//                  coalesced along the channel axis of the NHWC tensor) and walks the pixels of its chunk, per-channel
//                  sums in registers; per-group partials are combined in a FIXED order through shared memory and written
//                  as (mean, M2) of the chunk.
//   apply kernel   same decomposition.  Prologue: every CTA merges the <= 128 chunk partials of the groups of ITS slice
//                  with Chan's parallel-variance update, 8-32 threads per group, all loads issued before the first merge,
//                  fixed order: bit-stable run to run (the repo's multi-GPU sweep is an equality test), no atomics, no
//                  grid-wide hand-off (a first version let the last CTA of the stats kernel merge everything: its
//                  serial tail grew with the batch, 85 us at 8 samples).  Then y = silu(x * a + b) with
//                  a = rstd * gamma, b = beta - mean * a per channel.
//   backward       the same two-launch shape: partial sums of  dxh = dz * gamma  and  dxh * xhat  per (sample, group)
//                  (dz = dy * silu'(z), z recomputed from x), then
//                  dx = rstd * (dxh - mean(dxh) - xhat * mean(dxh * xhat)).
// The second launch of each direction re-reads x (and dy) from L2 (the largest activation of an SD UNet is 7.9 MB).
// Statistics are fp32; the affine parameters are read in the activation dtype.  d gamma / d beta are not produced (the
// UNet is frozen on the guidance path: ptp_utils.register_attention_control).  The optional `shift[n, c]` (the bias of
// the convolution that produced x + the block's time-embedding projection) is added on load.  The second kernel of a
// pair is launched with programmatic stream serialisation and starts with griddepcontrol.wait: its CTAs are scheduled
// while the first kernel drains.
#include "ga_common.cuh"
#include <stdlib.h>

namespace ga {
namespace gn {

constexpr int kThreads = 256;

struct Params {
  const void* x;
  const void* dy;
  const void* gamma;
  const void* beta;
  const void* shift;      // optional (n, c): the kernels normalise x + shift[n, c] (a conv bias + time embedding folded in)
  int64_t shift_stride;   // elements between the shift rows of consecutive samples (>= c: a column slice of a wider matrix)
  void* out;              // y (forward) or dx (backward)
  float* stats;           // [n][groups][2] = mean, rstd
  float* ws;              // chunk partials [n][P][groups][2]: (mean, M2) forward, (sum dxh, sum dxh * xhat) backward
  int n, hw, c, groups, cpg;
  int cs;                 // channel slices per pixel (grid.y); a slice holds whole groups
  int vs;                 // 8-channel vectors per slice (<= kThreads)
  int pl;                 // pixel lanes = kThreads / vs
  int chunk;              // pixels per CTA
  int P;                  // chunks (grid.x)
  float eps;
};

template <typename T> __device__ __forceinline__ void unpack8(const uint4& w, float* f) {
  const float2 a = Word<T>::unpack(w.x), b = Word<T>::unpack(w.y), c = Word<T>::unpack(w.z), d = Word<T>::unpack(w.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
template <typename T> __device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(Word<T>::pack(f[0], f[1]), Word<T>::pack(f[2], f[3]), Word<T>::pack(f[4], f[5]),
                    Word<T>::pack(f[6], f[7]));
}
__device__ __forceinline__ float sigmoidf_fast(float z) { return __fdividef(1.f, 1.f + __expf(-z)); }
// Programmatic dependent launch: the second kernel of a pair is launched while the first still runs (its CTAs are
// scheduled as the first one's retire) and waits here until the first has completed and its writes are visible.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// A thread's coordinates: which 8-channel vector of which slice, which pixel lane.
struct Coord {
  int n, c0, pl, p0, p1;
  bool active;
  __device__ __forceinline__ void init(const Params& p) {
    const int tid = threadIdx.x;
    pl = tid / p.vs;
    const int v = tid - pl * p.vs;
    active = pl < p.pl;
    n = blockIdx.z;
    c0 = ((int)blockIdx.y * p.vs + v) * 8;
    p0 = (int)blockIdx.x * p.chunk;
    p1 = min(p0 + p.chunk, p.hw);
  }
};

template <typename T> __device__ __forceinline__ void load_shift(const Params& p, const Coord& t, float* sh) {
  if (p.shift != nullptr) {
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.shift) + (int64_t)t.n * p.shift_stride + t.c0)), sh);
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) sh[e] = 0.f;
  }
}

// Per-channel sums of a thread -> per-group sums of the CTA's slice, fixed order.  A vector touches at most two groups
// (checked on the host): the first `k` elements belong to group c0 / cpg, the rest to the next one.
__device__ __forceinline__ void group_partials(const Params& p, const Coord& t, const float* s, const float* q,
                                               float4* part, float& S, float& Q, int& g_out, bool& owner) {
  const int g0 = t.c0 / p.cpg;
  const int k = min(8, (g0 + 1) * p.cpg - t.c0);
  float sA = 0.f, qA = 0.f, sB = 0.f, qB = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    if (e < k) { sA += s[e]; qA += q[e]; } else { sB += s[e]; qB += q[e]; }
  }
  part[threadIdx.x] = t.active ? make_float4(sA, qA, sB, qB) : make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  // `sub` threads per group (a power of two inside one warp): sub-lane j sums the pixel lanes j, j + sub, ... of the
  // vectors that overlap its group, then a shuffle tree in a fixed order
  const int gps = p.groups / p.cs;
  const int sub = gps * 8 <= kThreads ? 8 : 1;
  const int gl = (int)threadIdx.x / sub, j = (int)threadIdx.x - gl * sub;
  const bool live = gl < gps;
  const int slice_c0 = (int)blockIdx.y * p.vs * 8;
  const int g = (int)blockIdx.y * gps + gl;
  S = 0.f; Q = 0.f;
  if (live) {
    const int v_lo = (g * p.cpg - slice_c0) >> 3, v_hi = ((g + 1) * p.cpg - 1 - slice_c0) >> 3;
    for (int l = j; l < p.pl; l += sub)
      for (int v = v_lo; v <= v_hi; ++v) {
        const float4 w = part[l * p.vs + v];
        // a vector that starts inside the group contributes its first part, one that starts before it its second part
        if (slice_c0 + v * 8 >= g * p.cpg) { S += w.x; Q += w.y; } else { S += w.z; Q += w.w; }
      }
  }
  if (sub == 8) {
#pragma unroll
    for (int off = 4; off > 0; off >>= 1) {
      S += __shfl_down_sync(0xffffffffu, S, off, 8);
      Q += __shfl_down_sync(0xffffffffu, Q, off, 8);
    }
  }
  owner = live && j == 0;
  g_out = g;
}

constexpr int kMaxChunks = 128;       // chunk partials per (sample, group)
constexpr int kMaxSliceGroups = 32;   // groups one CTA's slice may hold (SD: 32 groups, one or two slices)
constexpr int kMergeLoads = 16;       // partials one thread of the merging prologue holds: kMaxChunks / 8

// Layout of the merging prologues: `tpg` = 8, 16 or 32 threads per group (all inside one warp), so that the whole CTA
// merges all groups of its slice at once and every thread has ALL its partials in flight before the first merge (one
// L2 round trip instead of one per group).
__device__ __forceinline__ int merge_tpg(int gps) {
  int tpg = 8;
  while (tpg < 32 && tpg * 2 * gps <= kThreads) tpg *= 2;
  return tpg;
}

// Prologue of the apply kernels: (mean, rstd) of every group of this CTA's slice from the chunk partials (mean, M2),
// Chan's parallel update in a fixed order (thread-sequential over its chunks, then a shuffle tree).
__device__ __forceinline__ void merge_stats(const Params& p, float2* sst) {
  pdl_wait();
  const int gps = p.groups / p.cs, n = blockIdx.z;
  const int tpg = merge_tpg(gps);
  const int gl = (int)threadIdx.x / tpg, j = (int)threadIdx.x - gl * tpg;
  const bool live = gl < gps;
  const int g = (int)blockIdx.y * gps + gl;
  float2 w[kMergeLoads];
#pragma unroll
  for (int i = 0; i < kMergeLoads; ++i) {
    const int ch = j + tpg * i;
    w[i] = (live && ch < p.P) ? __ldg(reinterpret_cast<const float2*>(p.ws) + ((int64_t)n * p.P + ch) * p.groups + g)
                              : make_float2(0.f, 0.f);
  }
  float cnt = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll
  for (int i = 0; i < kMergeLoads; ++i) {
    const int ch = j + tpg * i;
    if (live && ch < p.P) {
      const float cb = (float)((min((ch + 1) * p.chunk, p.hw) - ch * p.chunk) * p.cpg);
      const float tot = cnt + cb, delta = w[i].x - mean, f = __fdividef(cb, tot);
      mean = fmaf(delta, f, mean);
      m2 += w[i].y + delta * delta * cnt * f;
      cnt = tot;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    if (off < tpg) {
      const float cb = __shfl_down_sync(0xffffffffu, cnt, off, 32);
      const float mb = __shfl_down_sync(0xffffffffu, mean, off, 32);
      const float qb = __shfl_down_sync(0xffffffffu, m2, off, 32);
      if (cb > 0.f && j + off < tpg) {
        const float tot = cnt + cb, delta = mb - mean, f = __fdividef(cb, tot);
        mean = fmaf(delta, f, mean);
        m2 += qb + delta * delta * cnt * f;
        cnt = tot;
      }
    }
  }
  if (live && j == 0) {
    const float2 st = make_float2(mean, rsqrtf(m2 / cnt + p.eps));
    sst[gl] = st;
    if (blockIdx.x == 0) reinterpret_cast<float2*>(p.stats)[n * p.groups + g] = st;   // kept for the backward
  }
  __syncthreads();
}

// Prologue of the backward apply kernel: mean(dxh), mean(dxh * xhat) of every group of the slice (plain sums).
__device__ __forceinline__ void merge_sums(const Params& p, float2* scf) {
  pdl_wait();
  const int gps = p.groups / p.cs, n = blockIdx.z;
  const int tpg = merge_tpg(gps);
  const int gl = (int)threadIdx.x / tpg, j = (int)threadIdx.x - gl * tpg;
  const bool live = gl < gps;
  const int g = (int)blockIdx.y * gps + gl;
  float2 w[kMergeLoads];
#pragma unroll
  for (int i = 0; i < kMergeLoads; ++i) {
    const int ch = j + tpg * i;
    w[i] = (live && ch < p.P) ? __ldg(reinterpret_cast<const float2*>(p.ws) + ((int64_t)n * p.P + ch) * p.groups + g)
                              : make_float2(0.f, 0.f);
  }
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < kMergeLoads; ++i) { s1 += w[i].x; s2 += w[i].y; }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    if (off < tpg) {
      const float a1 = __shfl_down_sync(0xffffffffu, s1, off, 32), a2 = __shfl_down_sync(0xffffffffu, s2, off, 32);
      if (j + off < tpg) { s1 += a1; s2 += a2; }
    }
  }
  if (live && j == 0) {
    const float inv_m = 1.f / ((float)p.hw * (float)p.cpg);
    scf[gl] = make_float2(s1 * inv_m, s2 * inv_m);
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------- forward: stats
template <typename T>
__global__ void __launch_bounds__(kThreads) gn_stats_kernel(const Params p) {
  __shared__ float4 part[kThreads];
  pdl_launch_dependents();
  Coord t;
  t.init(p);
  float s[8], q[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { s[e] = 0.f; q[e] = 0.f; }
  if (t.active) {
    const uint4* xp = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.x) + ((int64_t)t.n * p.hw) * p.c + t.c0);
    const int64_t stride = (int64_t)p.c / 8;
    float sh[8];
    load_shift<T>(p, t, sh);
#pragma unroll 4
    for (int px = t.p0 + t.pl; px < t.p1; px += p.pl) {
      float f[8];
      unpack8<T>(__ldg(xp + px * stride), f);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float v = f[e] + sh[e];
        s[e] += v;
        q[e] = fmaf(v, v, q[e]);
      }
    }
  }
  float S, Q;
  int g;
  bool owner;
  group_partials(p, t, s, q, part, S, Q, g, owner);
  if (owner) {
    const float cnt = (float)((t.p1 - t.p0) * p.cpg);
    const float mean = cnt > 0.f ? S / cnt : 0.f;
    const float m2 = fmaxf(Q - S * mean, 0.f);
    float* w = p.ws + (((int64_t)t.n * p.P + blockIdx.x) * p.groups + g) * 2;
    w[0] = mean;
    w[1] = m2;
  }
}

// ------------------------------------------------------------------------------------------------- forward: apply
template <typename T, bool kSilu>
__global__ void __launch_bounds__(kThreads) gn_apply_kernel(const Params p) {
  __shared__ float2 sst[kMaxSliceGroups];
  Coord t;
  t.init(p);
  merge_stats(p, sst);
  if (!t.active) return;
  float a[8], b[8];
  {
    float gm[8], bt[8];
    const int g_first = (int)blockIdx.y * (p.groups / p.cs);
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.gamma) + t.c0)), gm);
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.beta) + t.c0)), bt);
    float sh[8];
    load_shift<T>(p, t, sh);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float2 st = sst[(t.c0 + e) / p.cpg - g_first];
      a[e] = st.y * gm[e];
      b[e] = fmaf(sh[e] - st.x, a[e], bt[e]);        // (x + shift - mean) * rstd * gamma + beta
    }
  }
  const int64_t base = ((int64_t)t.n * p.hw) * p.c + t.c0;
  const uint4* xp = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.x) + base);
  uint4* yp = reinterpret_cast<uint4*>(reinterpret_cast<T*>(p.out) + base);
  const int64_t stride = (int64_t)p.c / 8;
#pragma unroll 4
  for (int px = t.p0 + t.pl; px < t.p1; px += p.pl) {
    float f[8];
    unpack8<T>(__ldg(xp + px * stride), f);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float z = fmaf(f[e], a[e], b[e]);
      f[e] = kSilu ? z * sigmoidf_fast(z) : z;
    }
    yp[px * stride] = pack8<T>(f);
  }
}

// ------------------------------------------------------------------------------------------------ backward: sums
template <typename T, bool kSilu>
__global__ void __launch_bounds__(kThreads) gn_bwd_sums_kernel(const Params p) {
  __shared__ float4 part[kThreads];
  pdl_launch_dependents();
  Coord t;
  t.init(p);
  float s[8], q[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { s[e] = 0.f; q[e] = 0.f; }
  if (t.active) {
    float a[8], b[8], gm[8], r[8], mr[8];
    {
      float bt[8];
      unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.gamma) + t.c0)), gm);
      unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.beta) + t.c0)), bt);
      float sh[8];
      load_shift<T>(p, t, sh);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int g = (t.c0 + e) / p.cpg;
        const float2 st = __ldg(reinterpret_cast<const float2*>(p.stats) + t.n * p.groups + g);
        const float mu = st.x - sh[e];               // everything below is a function of x + shift
        r[e] = st.y;
        mr[e] = mu * st.y;
        a[e] = st.y * gm[e];
        b[e] = fmaf(-mu, a[e], bt[e]);
      }
    }
    const int64_t base = ((int64_t)t.n * p.hw) * p.c + t.c0;
    const uint4* xp = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.x) + base);
    const uint4* gp = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.dy) + base);
    const int64_t stride = (int64_t)p.c / 8;
#pragma unroll 2
    for (int px = t.p0 + t.pl; px < t.p1; px += p.pl) {
      float f[8], d[8];
      unpack8<T>(__ldg(xp + px * stride), f);
      unpack8<T>(__ldg(gp + px * stride), d);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float dz = d[e];
        if (kSilu) {
          const float z = fmaf(f[e], a[e], b[e]);
          const float sg = sigmoidf_fast(z);
          dz *= sg * fmaf(z, 1.f - sg, 1.f);
        }
        const float dxh = dz * gm[e];
        const float xh = fmaf(f[e], r[e], -mr[e]);
        s[e] += dxh;
        q[e] = fmaf(dxh, xh, q[e]);
      }
    }
  }
  float S, Q;
  int g;
  bool owner;
  group_partials(p, t, s, q, part, S, Q, g, owner);
  if (owner) {
    float* w = p.ws + (((int64_t)t.n * p.P + blockIdx.x) * p.groups + g) * 2;
    w[0] = S;
    w[1] = Q;
  }
}

// ----------------------------------------------------------------------------------------------- backward: apply
template <typename T, bool kSilu>
__global__ void __launch_bounds__(kThreads) gn_bwd_apply_kernel(const Params p) {
  __shared__ float2 scf[kMaxSliceGroups];
  Coord t;
  t.init(p);
  merge_sums(p, scf);
  if (!t.active) return;
  float a[8], b[8], gr[8], r[8], mr[8], k1[8], k2[8];
  {
    float gm[8], bt[8];
    const int g_first = (int)blockIdx.y * (p.groups / p.cs);
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.gamma) + t.c0)), gm);
    unpack8<T>(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.beta) + t.c0)), bt);
    float sh[8];
    load_shift<T>(p, t, sh);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int g = (t.c0 + e) / p.cpg;
      const float2 st = __ldg(reinterpret_cast<const float2*>(p.stats) + t.n * p.groups + g);
      const float2 cf = scf[g - g_first];
      const float mu = st.x - sh[e];
      r[e] = st.y;
      mr[e] = mu * st.y;
      a[e] = st.y * gm[e];
      b[e] = fmaf(-mu, a[e], bt[e]);
      gr[e] = gm[e] * st.y;
      k1[e] = cf.x * st.y;
      k2[e] = cf.y * st.y;
    }
  }
  const int64_t base = ((int64_t)t.n * p.hw) * p.c + t.c0;
  const uint4* xp = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.x) + base);
  const uint4* gp = reinterpret_cast<const uint4*>(reinterpret_cast<const T*>(p.dy) + base);
  uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<T*>(p.out) + base);
  const int64_t stride = (int64_t)p.c / 8;
#pragma unroll 2
  for (int px = t.p0 + t.pl; px < t.p1; px += p.pl) {
    float f[8], d[8];
    unpack8<T>(__ldg(xp + px * stride), f);
    unpack8<T>(__ldg(gp + px * stride), d);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float dz = d[e];
      if (kSilu) {
        const float z = fmaf(f[e], a[e], b[e]);
        const float sg = sigmoidf_fast(z);
        dz *= sg * fmaf(z, 1.f - sg, 1.f);
      }
      const float xh = fmaf(f[e], r[e], -mr[e]);
      f[e] = fmaf(dz, gr[e], -k1[e]) - xh * k2[e];
    }
    op[px * stride] = pack8<T>(f);
  }
}

// ----------------------------------------------------------------------------------------------------------- host
// Decomposition of one (n, hw, c) tensor with `groups` groups; false when the shape is outside what the kernels assume.
static bool plan(Params& p, int n, int hw, int c, int groups) {
  if (n < 1 || hw < 1 || c < 8 || groups < 1 || c % groups != 0 || c % 8 != 0) return false;
  if ((int64_t)n * groups > (1 << 20)) return false;
  p.n = n; p.hw = hw; p.c = c; p.groups = groups; p.cpg = c / groups;
  const int V = c / 8;
  int cs = (V + kThreads - 1) / kThreads;
  while (cs <= groups && (groups % cs != 0 || V % cs != 0 || ((V / cs) * 8) % p.cpg != 0 || V / cs > kThreads)) ++cs;
  if (cs > groups) return false;
  p.cs = cs;
  p.vs = V / cs;
  p.pl = kThreads / p.vs;
  for (int v = 0; v < V; ++v)                      // a vector may touch at most two groups
    if ((v * 8 + 7) / p.cpg - (v * 8) / p.cpg > 1) return false;
  int chunk = (hw + 127) / 128;
  if (chunk < p.pl) chunk = p.pl;
  if (chunk > hw) chunk = hw;
  p.chunk = chunk;
  p.P = (hw + chunk - 1) / chunk;
  if (p.P > kMaxChunks || groups / cs > kMaxSliceGroups || n > 65535 || cs > 65535) return false;
  return true;
}

int64_t ws_bytes(int n, int hw, int c, int groups) {
  Params p;
  if (!plan(p, n, hw, c, groups)) return -1;
  return (int64_t)n * p.P * groups * 2 * (int64_t)sizeof(float);
}

template <typename K>
static void launch_second(K kernel, const dim3& grid, const Params& p, cudaStream_t st) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, p);
}

template <typename T>
static void launch_fwd(const Params& p, bool silu, cudaStream_t st) {
  const dim3 grid(p.P, p.cs, p.n);
  gn_stats_kernel<T><<<grid, kThreads, 0, st>>>(p);
  if (silu) launch_second(gn_apply_kernel<T, true>, grid, p, st);
  else launch_second(gn_apply_kernel<T, false>, grid, p, st);
}
template <typename T>
static void launch_bwd(const Params& p, bool silu, cudaStream_t st) {
  const dim3 grid(p.P, p.cs, p.n);
  if (silu) {
    gn_bwd_sums_kernel<T, true><<<grid, kThreads, 0, st>>>(p);
    launch_second(gn_bwd_apply_kernel<T, true>, grid, p, st);
  } else {
    gn_bwd_sums_kernel<T, false><<<grid, kThreads, 0, st>>>(p);
    launch_second(gn_bwd_apply_kernel<T, false>, grid, p, st);
  }
}

int fwd(const void* x, const void* shift, int64_t shift_stride, const void* gamma, const void* beta, void* y, float* stats, float* ws, int n,
        int hw, int c, int groups, float eps, int silu, int dtype, cudaStream_t st) {
  Params p;
  if (!plan(p, n, hw, c, groups))
    return fail(GA_ERR_UNSUPPORTED, "group norm: shape n=%d hw=%d c=%d groups=%d is not supported", n, hw, c, groups);
  p.x = x; p.shift = shift; p.shift_stride = shift_stride; p.dy = nullptr; p.gamma = gamma; p.beta = beta; p.out = y; p.stats = stats; p.ws = ws;
  p.eps = eps;
  if (dtype == GA_F16) launch_fwd<__half>(p, silu != 0, st);
  else launch_fwd<__nv_bfloat16>(p, silu != 0, st);
  return check_launch("group_norm_fwd");
}

int bwd(const void* x, const void* shift, int64_t shift_stride, const void* dy, const void* gamma, const void* beta, const float* stats,
        void* dx, float* ws, int n, int hw, int c, int groups, int silu, int dtype, cudaStream_t st) {
  Params p;
  if (!plan(p, n, hw, c, groups))
    return fail(GA_ERR_UNSUPPORTED, "group norm: shape n=%d hw=%d c=%d groups=%d is not supported", n, hw, c, groups);
  p.x = x; p.shift = shift; p.shift_stride = shift_stride; p.dy = dy; p.gamma = gamma; p.beta = beta; p.out = dx; p.stats = const_cast<float*>(stats); p.ws = ws;
  p.eps = 0.f;
  if (dtype == GA_F16) launch_bwd<__half>(p, silu != 0, st);
  else launch_bwd<__nv_bfloat16>(p, silu != 0, st);
  return check_launch("group_norm_bwd");
}

// ---------------------------------------------------------------------------- bias (+ residual) epilogue of a conv
// out = a + bias[c] (+ b): PyTorch adds a convolution's bias with a broadcast `add_` (a non-vectorised elementwise
// kernel, ~5 us per convolution) and the block's residual with another launch; on the channels-last tensor the bias
// index is the fastest dimension, so both fit one 128-bit-vectorised pass.
template <typename T>
__global__ void __launch_bounds__(kThreads) add_bias_residual_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b,
                                                                     const uint4* __restrict__ bias, uint4* __restrict__ out,
                                                                     int64_t n_vec, int vec_per_pixel) {
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * kThreads) {
    float fa[8], fb[8], fc[8];
    unpack8<T>(__ldg(a + i), fa);
    unpack8<T>(__ldg(bias + (int)(i % vec_per_pixel)), fc);
    if (b != nullptr) {
      unpack8<T>(__ldg(b + i), fb);
#pragma unroll
      for (int e = 0; e < 8; ++e) fa[e] += fb[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) fa[e] += fc[e];
    out[i] = pack8<T>(fa);
  }
}

int add_bias_residual(const void* a, const void* b, const void* bias, void* out, int64_t n_pixels, int c, int dtype,
                      cudaStream_t st) {
  const int64_t n_vec = n_pixels * (c / 8);
  if (n_vec == 0) return GA_OK;
  int64_t blocks = (n_vec + kThreads - 1) / kThreads;
  if (blocks > 148 * 8) blocks = 148 * 8;
  const uint4 *pa = static_cast<const uint4*>(a), *pb = static_cast<const uint4*>(b), *pc = static_cast<const uint4*>(bias);
  if (dtype == GA_F16)
    add_bias_residual_kernel<__half><<<(int)blocks, kThreads, 0, st>>>(pa, pb, pc, static_cast<uint4*>(out), n_vec, c / 8);
  else
    add_bias_residual_kernel<__nv_bfloat16><<<(int)blocks, kThreads, 0, st>>>(pa, pb, pc, static_cast<uint4*>(out), n_vec,
                                                                             c / 8);
  return check_launch("add_bias_residual");
}

// ------------------------------------------------------------------------------------------------------- GEGLU
// The transformer blocks' feed-forward gate (diffusers `GEGLU.forward`: `h, gate = proj(x).chunk(2, -1); h * gelu(gate)`)
// on the projection output p (rows, 2 * inner): PyTorch runs gelu and the product as two NON-vectorised elementwise
// kernels (the chunks are strided views) and the backward as gelu_backward + two products + a concatenating copy.
//   forward   out[r, j] = p[r, j] * gelu(p[r, inner + j])                         (exact erf GELU)
//   backward  d_p[r, j] = d_out * gelu(g),  d_p[r, inner + j] = d_out * h * gelu'(g)
__device__ __forceinline__ float gelu_f(float g) { return 0.5f * g * (1.f + erff(g * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad_f(float g) {
  return 0.5f * (1.f + erff(g * 0.70710678118654752f)) + g * 0.3989422804014327f * __expf(-0.5f * g * g);
}

template <typename T>
__global__ void __launch_bounds__(kThreads) geglu_fwd_kernel(const uint4* __restrict__ p, uint4* __restrict__ out,
                                                             int64_t n_vec, int vec_per_row) {
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * kThreads) {
    const int64_t r = i / vec_per_row;
    const int v = (int)(i - r * vec_per_row);
    float h[8], g[8];
    unpack8<T>(__ldg(p + r * 2 * vec_per_row + v), h);
    unpack8<T>(__ldg(p + r * 2 * vec_per_row + vec_per_row + v), g);
#pragma unroll
    for (int e = 0; e < 8; ++e) h[e] *= gelu_f(g[e]);
    out[i] = pack8<T>(h);
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) geglu_bwd_kernel(const uint4* __restrict__ p, const uint4* __restrict__ d_out,
                                                             uint4* __restrict__ d_p, int64_t n_vec, int vec_per_row) {
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * kThreads) {
    const int64_t r = i / vec_per_row;
    const int v = (int)(i - r * vec_per_row);
    float h[8], g[8], d[8], dh[8], dg[8];
    unpack8<T>(__ldg(p + r * 2 * vec_per_row + v), h);
    unpack8<T>(__ldg(p + r * 2 * vec_per_row + vec_per_row + v), g);
    unpack8<T>(__ldg(d_out + i), d);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      dh[e] = d[e] * gelu_f(g[e]);
      dg[e] = d[e] * h[e] * gelu_grad_f(g[e]);
    }
    d_p[r * 2 * vec_per_row + v] = pack8<T>(dh);
    d_p[r * 2 * vec_per_row + vec_per_row + v] = pack8<T>(dg);
  }
}

int geglu(const void* p, const void* d_out, void* out, int64_t rows, int inner, int dtype, bool backward, cudaStream_t st) {
  const int64_t n_vec = rows * (inner / 8);
  if (n_vec == 0) return GA_OK;
  int64_t blocks = (n_vec + kThreads - 1) / kThreads;
  if (blocks > 148 * 16) blocks = 148 * 16;
  const uint4* pp = static_cast<const uint4*>(p);
  if (!backward) {
    if (dtype == GA_F16) geglu_fwd_kernel<__half><<<(int)blocks, kThreads, 0, st>>>(pp, static_cast<uint4*>(out), n_vec, inner / 8);
    else geglu_fwd_kernel<__nv_bfloat16><<<(int)blocks, kThreads, 0, st>>>(pp, static_cast<uint4*>(out), n_vec, inner / 8);
  } else {
    const uint4* pd = static_cast<const uint4*>(d_out);
    if (dtype == GA_F16) geglu_bwd_kernel<__half><<<(int)blocks, kThreads, 0, st>>>(pp, pd, static_cast<uint4*>(out), n_vec, inner / 8);
    else geglu_bwd_kernel<__nv_bfloat16><<<(int)blocks, kThreads, 0, st>>>(pp, pd, static_cast<uint4*>(out), n_vec, inner / 8);
  }
  return check_launch(backward ? "geglu_bwd" : "geglu_fwd");
}

// --------------------------------------------------------------------------------------------------- LayerNorm
// The three LayerNorms of every transformer block (diffusers `BasicTransformerBlock.norm1/2/3`) on (rows, C) tokens,
// C = 320 / 640 / 1280: one WARP per row, the row held in registers (<= 8 vectors of 8 channels per lane), exact two-pass
// mean / variance with warp shuffles, 128-bit loads and stores.  mean / rstd are saved for the backward.
constexpr int kLnMaxVec = 8;   // vectors per lane: C <= 32 * 8 * 8 = 2048

template <typename T>
__global__ void __launch_bounds__(kThreads) layer_norm_fwd_kernel(const uint4* __restrict__ x, const uint4* __restrict__ gamma,
                                                                  const uint4* __restrict__ beta, uint4* __restrict__ y,
                                                                  float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                                  int64_t rows, int V, float eps) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const uint4* xr = x + row * V;
  float f[kLnMaxVec][8];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i) {
    const int v = lane + 32 * i;
    if (v < V) {
      unpack8<T>(__ldg(xr + v), f[i]);
#pragma unroll
      for (int e = 0; e < 8; ++e) sum += f[i][e];
    }
  }
  const float inv_c = 1.f / (float)(V * 8);
  const float mean = warp_sum(sum) * inv_c;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i) {
    if (lane + 32 * i < V) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float d = f[i][e] - mean;
        sq = fmaf(d, d, sq);
      }
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) * inv_c + eps);
  if (lane == 0) {
    mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
  uint4* yr = y + row * V;
#pragma unroll
  for (int i = 0; i < kLnMaxVec; ++i) {
    const int v = lane + 32 * i;
    if (v < V) {
      float g[8], b[8];
      unpack8<T>(__ldg(gamma + v), g);
      unpack8<T>(__ldg(beta + v), b);
#pragma unroll
      for (int e = 0; e < 8; ++e) f[i][e] = fmaf((f[i][e] - mean) * rstd, g[e], b[e]);
      yr[v] = pack8<T>(f[i]);
    }
  }
}

int layer_norm_fwd(const void* x, const void* gamma, const void* beta, void* y, float* mean, float* rstd, int64_t rows,
                   int c, float eps, int dtype, cudaStream_t st) {
  if (rows == 0) return GA_OK;
  const int V = c / 8;
  const int64_t blocks = (rows + kThreads / 32 - 1) / (kThreads / 32);
  const uint4 *px = static_cast<const uint4*>(x), *pg = static_cast<const uint4*>(gamma), *pb = static_cast<const uint4*>(beta);
  if (dtype == GA_F16)
    layer_norm_fwd_kernel<__half><<<(unsigned)blocks, kThreads, 0, st>>>(px, pg, pb, static_cast<uint4*>(y), mean, rstd, rows, V, eps);
  else
    layer_norm_fwd_kernel<__nv_bfloat16><<<(unsigned)blocks, kThreads, 0, st>>>(px, pg, pb, static_cast<uint4*>(y), mean, rstd, rows,
                                                                                V, eps);
  return check_launch("layer_norm_fwd");
}

}  // namespace gn
}  // namespace ga

using namespace ga;

extern "C" int ga_layer_norm_fwd(const void* x, const void* gamma, const void* beta, void* y, float* mean, float* rstd,
                                 int64_t rows, int channels, float eps, int dtype, ga_stream_t stream) {
  GA_CHECK_ARG(x && gamma && beta && y && mean && rstd, "NULL operand");
  GA_CHECK_ARG(dtype == GA_F16 || dtype == GA_BF16, "layer norm: 16-bit activations only (dtype %d)", dtype);
  GA_CHECK_ARG(rows >= 0 && rows < ((int64_t)1 << 34) && channels >= 8 && channels % 8 == 0 &&
                   channels <= 32 * 8 * gn::kLnMaxVec,
               "layer norm: channels %d must be a multiple of 8 in [8, %d]", channels, 32 * 8 * gn::kLnMaxVec);
  GA_CHECK_ALIGN(x, 16, "x");
  GA_CHECK_ALIGN(y, 16, "y");
  GA_CHECK_ALIGN(gamma, 16, "gamma");
  GA_CHECK_ALIGN(beta, 16, "beta");
  return gn::layer_norm_fwd(x, gamma, beta, y, mean, rstd, rows, channels, eps, dtype, static_cast<cudaStream_t>(stream));
}

static int check_geglu_args(const void* p, const void* out, int64_t rows, int inner, int dtype) {
  GA_CHECK_ARG(p && out, "NULL operand");
  GA_CHECK_ARG(dtype == GA_F16 || dtype == GA_BF16, "geglu: 16-bit activations only (dtype %d)", dtype);
  GA_CHECK_ARG(rows >= 0 && inner >= 8 && inner % 8 == 0, "geglu: inner width %d must be a multiple of 8", inner);
  GA_CHECK_ALIGN(p, 16, "proj");
  GA_CHECK_ALIGN(out, 16, "output");
  return GA_OK;
}

extern "C" int ga_geglu_fwd(const void* proj, void* out, int64_t rows, int inner, int dtype, ga_stream_t stream) {
  int rc = check_geglu_args(proj, out, rows, inner, dtype);
  if (rc != GA_OK) return rc;
  return gn::geglu(proj, nullptr, out, rows, inner, dtype, false, static_cast<cudaStream_t>(stream));
}

extern "C" int ga_geglu_bwd(const void* proj, const void* d_out, void* d_proj, int64_t rows, int inner, int dtype,
                            ga_stream_t stream) {
  int rc = check_geglu_args(proj, d_proj, rows, inner, dtype);
  if (rc != GA_OK) return rc;
  GA_CHECK_ARG(d_out != nullptr, "NULL operand");
  GA_CHECK_ALIGN(d_out, 16, "d_out");
  return gn::geglu(proj, d_out, d_proj, rows, inner, dtype, true, static_cast<cudaStream_t>(stream));
}

extern "C" int ga_add_bias_residual(const void* a, const void* b, const void* bias, void* out, int64_t n_pixels,
                                    int channels, int dtype, ga_stream_t stream) {
  GA_CHECK_ARG(a && bias && out, "NULL operand");
  GA_CHECK_ARG(dtype == GA_F16 || dtype == GA_BF16, "add_bias_residual: 16-bit activations only (dtype %d)", dtype);
  GA_CHECK_ARG(n_pixels >= 0 && channels >= 8 && channels % 8 == 0, "add_bias_residual: channels %d must be a multiple of 8",
               channels);
  GA_CHECK_ALIGN(a, 16, "a");
  GA_CHECK_ALIGN(out, 16, "out");
  GA_CHECK_ALIGN(bias, 16, "bias");
  if (b != nullptr) GA_CHECK_ALIGN(b, 16, "b");
  return gn::add_bias_residual(a, b, bias, out, n_pixels, channels, dtype, static_cast<cudaStream_t>(stream));
}

extern "C" int64_t ga_group_norm_ws_bytes(int n, int hw, int channels, int groups) {
  return gn::ws_bytes(n, hw, channels, groups);
}

static int check_gn_args(const void* x, const void* gamma, const void* beta, const void* out, const void* stats,
                         const void* ws, int dtype) {
  GA_CHECK_ARG(x && gamma && beta && out && stats && ws, "NULL operand");
  GA_CHECK_ARG(dtype == GA_F16 || dtype == GA_BF16, "group norm: 16-bit activations only (dtype %d)", dtype);
  GA_CHECK_ALIGN(x, 16, "x");
  GA_CHECK_ALIGN(out, 16, "output");
  GA_CHECK_ALIGN(gamma, 16, "gamma");
  GA_CHECK_ALIGN(beta, 16, "beta");
  GA_CHECK_ALIGN(stats, 8, "stats");
  GA_CHECK_ALIGN(ws, 8, "ws");
  return GA_OK;
}

extern "C" int ga_group_norm_fwd(const void* x, const void* shift, int64_t shift_stride, const void* gamma, const void* beta, void* y,
                                 float* stats, float* ws, int n, int hw, int channels, int groups, float eps, int silu,
                                 int dtype, ga_stream_t stream) {
  int rc = check_gn_args(x, gamma, beta, y, stats, ws, dtype);
  if (rc != GA_OK) return rc;
  if (shift != nullptr) {
    GA_CHECK_ALIGN(shift, 16, "shift");
    GA_CHECK_ARG(shift_stride >= channels && shift_stride % 8 == 0, "shift_stride %lld must be a multiple of 8 >= channels",
                 (long long)shift_stride);
  }
  return gn::fwd(x, shift, shift_stride, gamma, beta, y, stats, ws, n, hw, channels, groups, eps, silu, dtype,
                 static_cast<cudaStream_t>(stream));
}

extern "C" int ga_group_norm_bwd(const void* x, const void* shift, int64_t shift_stride, const void* d_y, const void* gamma, const void* beta,
                                 const float* stats, void* d_x, float* ws, int n, int hw, int channels, int groups,
                                 int silu, int dtype, ga_stream_t stream) {
  int rc = check_gn_args(x, gamma, beta, d_x, stats, ws, dtype);
  if (rc != GA_OK) return rc;
  GA_CHECK_ARG(d_y != nullptr, "NULL operand");
  GA_CHECK_ALIGN(d_y, 16, "d_y");
  if (shift != nullptr) {
    GA_CHECK_ALIGN(shift, 16, "shift");
    GA_CHECK_ARG(shift_stride >= channels && shift_stride % 8 == 0, "shift_stride %lld must be a multiple of 8 >= channels",
                 (long long)shift_stride);
  }
  return gn::bwd(x, shift, shift_stride, d_y, gamma, beta, stats, d_x, ws, n, hw, channels, groups, silu, dtype,
                 static_cast<cudaStream_t>(stream));
}
