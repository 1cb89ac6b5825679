// Exact self-attention (queries and keys are the same N image tokens) on the tcgen05 tensor cores, without ever
// materialising the (B*H, N, N) probability tensor that the reference builds, keeps for autograd and streams through
// four ATen kernels per layer (utils/ptp_utils.py:77-85, 97-146 on the attn1 layers: 268 MB per tensor at 64x64).
// SURVEY.md section 8 row f4.  These layers are off the guidance path (their maps are never read) but on the autograd
// path, so the backward is provided too.
//
// Forward, one CTA = 128 query rows of one (batch, head), ONE pass over the keys in blocks of BK (128 or 64) with an
// online softmax: per block S_j = Q K_j^T, P_j = exp(scale (S_j - running max)) (un-normalised, 16-bit, back into
// TMEM), O += P_j V_j.  The two compute groups own alternate key blocks, each with its own output accumulator and
// running max / sum; the epilogue merges the two partial results and divides by the row sum once.
//
//   warp 0      TMA producer   Q tile once, then a ring of K+V blocks
//   warp 1      MMA issuer 1   S(j) = Q K_j^T into score buffer j % 3
//   warp 2      MMA issuer 2   O_(j & 1) += P(j) V_j; its commit frees the K/V stage and the score buffer
//   warps 4-7   compute group 0 (even key blocks), warps 8-11 compute group 1 (odd key blocks): thread = query row =
//               TMEM lane.
// Three score buffers for two groups: the scores of a group's next block are computed while it works on the current
// one, and the two issuers are ordered by completion (P_FREE), not by sharing one instruction stream -- with a single
// issuer warp and two buffers every group waited a full issue -> tensor pipe -> commit round trip per block.
#include "tc_common.cuh"

namespace ga {
namespace sa {

using namespace ga::tc;

constexpr int kM = 128;
constexpr int kThreads = 384;
constexpr int kGroupThreads = 128;
constexpr int kQBlockBytes = kM * 128;
constexpr int kMaxStages = 4;
constexpr int kSBuf = 3;       // score buffers in TMEM (P overwrites the head of its S buffer); O follows them

struct FwdParams {
  void* o;
  float* lse;
  int B, H, N, d;
  int nblk, npv, bf16;
  int bk;        // keys per block: 128 (d <= 64) or 64
  int nb;        // key blocks
  int stages;    // K/V ring depth (>= 2)
  float scale;
};

// position in a ring of `n` buffers + parity of the current use of that buffer
struct RingPos {
  int idx;
  uint32_t par;
  __device__ __forceinline__ void advance(int n) {
    if (++idx == n) { idx = 0; par ^= 1u; }
  }
};

// ============================================================================================ forward
// QK^T is issued once per key block and the scores cross TMEM -> registers once.  Each compute group keeps its OWN
// output accumulator in TMEM (O_0 for the even key blocks, O_1 for the odd ones) together with its own running row
// maximum and row sum, so the groups never have to agree on a maximum while the blocks stream; the epilogue merges the
// two partial results
//     m = max(m_0, m_1),  l = l_0 2^(m_0 - m) + l_1 2^(m_1 - m),  O = (O_0 2^(m_0 - m) + O_1 2^(m_1 - m)) / l.
// The running maximum is LAZY: a group keeps exponentiating against a stale maximum as long as the block maximum
// exceeds it by less than 2^kLazyBits (P <= 256: harmless for the 16-bit P operand and the fp32 sums), and only when a
// row jumps further does its warp rescale its O accumulator in TMEM (tcgen05.ld -> multiply -> tcgen05.st, after the
// group's previous PV GEMM has completed).  After the first block of a group that is rare, so the common path of a
// block is: tcgen05.ld S -> max -> exp2 -> sum -> pack -> tcgen05.st P -> arrive.  Every exponential runs on the SFU:
// handing some of them to the FMA pipe as a polynomial measured slower (profiles/r02_microbench_self_attn_poly_ab.txt).
//
//   TMEM:  3 score buffers of `bk` columns | O_0 (npv) | O_1 (npv)      (d = 160: 192 + 320 = 512 columns)
constexpr float kLazyBits = 8.f;

template <int BK>
__global__ void __launch_bounds__(kThreads, 1)
self_attn_fwd1_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                      const __grid_constant__ CUtensorMap map_v, const FwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  // q_full, o_ready, kv_full[4], kv_free[4], s_ready[3], p_ready[3], p_free[3]
  __shared__ __align__(8) uint64_t bars[19];
  __shared__ uint32_t tmem_base_slot;
  __shared__ float xm[2][kM], xl[2][kM];   // running maxima / sums of the two compute groups

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int tile = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int row0 = tile * kM;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  constexpr uint32_t kv_block_bytes = (uint32_t)BK * 128u;
  const uint32_t k_bytes = (uint32_t)p.nblk * kv_block_bytes;
  const uint32_t stage_bytes = 2u * k_bytes;
  const uint32_t sQ = base;
  const uint32_t sKV = sQ + (uint32_t)p.nblk * kQBlockBytes;
  auto Q_FULL = [&]() { return smem_u32(&bars[0]); };
  auto O_READY = [&]() { return smem_u32(&bars[1]); };
  auto KV_FULL = [&](int s) { return smem_u32(&bars[2 + s]); };
  auto KV_FREE = [&](int s) { return smem_u32(&bars[6 + s]); };
  auto S_READY = [&](int i) { return smem_u32(&bars[10 + i]); };
  auto P_READY = [&](int i) { return smem_u32(&bars[13 + i]); };
  auto P_FREE = [&](int i) { return smem_u32(&bars[16 + i]); };
  constexpr uint32_t colO = (uint32_t)(kSBuf * BK);

  if (tid == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_k); prefetch_tmap(&map_v);
    mbar_init(Q_FULL(), 1);
    mbar_init(O_READY(), 1);
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(KV_FULL(s), 1); mbar_init(KV_FREE(s), 1); }
    for (int i = 0; i < kSBuf; ++i) {
      mbar_init(S_READY(i), 1);
      mbar_init(P_READY(i), kGroupThreads);
      mbar_init(P_FREE(i), 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const int nb = p.nb, NS = p.stages;
  const int ksteps = (p.d + 15) >> 4;
  const int fmt = p.bf16 ? 1 : 0;

  if (warp < 4) {
    reg_dealloc<40>();
    if (warp == 0) {
      // ------------------------------------------------------------------------------------------- producer
      if (elect_one()) {
        mbar_expect_tx(Q_FULL(), (uint32_t)p.nblk * kQBlockBytes);
        for (int blk = 0; blk < p.nblk; ++blk)
          tma_load_4d(sQ + blk * kQBlockBytes, &map_q, Q_FULL(), blk * kBlockCols, h, row0, b);
      }
      RingPos st = {0, 0};
      for (int it = 0; it < nb; ++it) {
        if (it >= NS) mbar_wait(KV_FREE(st.idx), st.par ^ 1u);
        if (elect_one()) {
          const uint32_t sK = sKV + st.idx * stage_bytes, sV = sK + k_bytes;
          mbar_expect_tx(KV_FULL(st.idx), stage_bytes);
          for (int blk = 0; blk < p.nblk; ++blk) {
            tma_load_4d(sK + blk * kv_block_bytes, &map_k, KV_FULL(st.idx), blk * kBlockCols, h, it * BK, b);
            tma_load_4d(sV + blk * kv_block_bytes, &map_v, KV_FULL(st.idx), blk * kBlockCols, h, it * BK, b);
          }
        }
        __syncwarp();
        st.advance(NS);
      }
    } else if (warp == 1) {
      // ----------------------------------------------------------------------------- MMA issuer 1: S = Q K^T
      const uint32_t idesc_qk = make_idesc(fmt, 0, BK, kM);
      const uint64_t dQ0 = smem_desc_sw128(sQ, 16, 1024);
      const uint64_t dK0 = smem_desc_sw128(sKV, 16, 1024);                          // stage 0, K-major
      mbar_wait(Q_FULL(), 0);
      RingPos st = {0, 0}, sb = {0, 0};
      for (int it = 0; it < nb; ++it) {
        // the buffer's previous item (it - 3): its P has been consumed by its PV GEMM
        if (it >= kSBuf) mbar_wait(P_FREE(sb.idx), sb.par ^ 1u);
        mbar_wait(KV_FULL(st.idx), st.par);
        tc_fence_after();
        if (elect_one()) {
          issue_kmajor_gemm(tmem + (uint32_t)(sb.idx * BK), dQ0, kQBlockBytes, desc_advance(dK0, st.idx * stage_bytes),
                            kv_block_bytes, ksteps, idesc_qk);
          tc_commit(S_READY(sb.idx));
        }
        __syncwarp();
        st.advance(NS);
        sb.advance(kSBuf);
      }
    } else if (warp == 2) {
      // ------------------------------------------------------------------- MMA issuer 2: O_(it & 1) += P V
      const uint32_t idesc_pv = make_idesc(fmt, 1, p.npv, kM);
      const uint64_t dV0 = smem_desc_sw128(sKV + k_bytes, kv_block_bytes, 1024);    // stage 0, MN-major
      RingPos st = {0, 0}, sb = {0, 0};
      for (int it = 0; it < nb; ++it) {
        mbar_wait(P_READY(sb.idx), sb.par);
        tc_fence_after();
        if (elect_one()) {
          issue_tmem_gemm(tmem + colO + (uint32_t)((it & 1) * p.npv), tmem + (uint32_t)(sb.idx * BK),
                          desc_advance(dV0, st.idx * stage_bytes), BK / 16, idesc_pv, it >= 2);
          tc_commit(KV_FREE(st.idx));
          tc_commit(P_FREE(sb.idx));
        }
        __syncwarp();
        st.advance(NS);
        sb.advance(kSBuf);
      }
      if (elect_one()) tc_commit(O_READY());
      __syncwarp();
    }
  } else {
    reg_alloc<232>();
    // --------------------------------------------------------------------------------------- compute groups
    const int g = (warp - 4) >> 2;
    const int r = ((warp & 3) << 5) + lane;
    const int row = row0 + r;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t colOg = colO + (uint32_t)(g * p.npv);
    const float sc = p.scale * 1.4426950408889634f;
    const bool bf16 = p.bf16 != 0;
    const float lazy = kLazyBits / sc;               // the lazy-maximum slack in raw score units

    float m_used = -INFINITY;                        // the maximum this row's exponentials are taken against (raw units)
    float l4[4] = {0.f, 0.f, 0.f, 0.f};
    for (int it = g; it < nb; it += 2) {
      const int buf = it % kSBuf;
      const uint32_t colS = (uint32_t)(buf * BK);
      mbar_wait(S_READY(buf), (uint32_t)(it / kSBuf) & 1u);
      tc_fence_after();
      float s[BK];
#pragma unroll
      for (int c = 0; c < BK / 16; ++c) tmem_ld16(lane_base + colS + c * 16, s + c * 16);
      tmem_ld_wait();
      const int key0 = it * BK;
      if (key0 + BK > p.N) {
#pragma unroll
        for (int j = 0; j < BK; ++j)
          if (key0 + j >= p.N) s[j] = -INFINITY;
      }
      float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int j = 0; j < BK; ++j) m4[j & 3] = fmaxf(m4[j & 3], s[j]);
      const float bm = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
      const bool jump = bm > m_used + lazy;          // first block: m_used = -inf
      if (__any_sync(0xffffffffu, jump)) {
        if (it >= 2) {
          // rescale this group's accumulator: its previous PV GEMM (item it - 2) must have completed
          const int pit = it - 2;
          mbar_wait(P_FREE(pit % kSBuf), (uint32_t)(pit / kSBuf) & 1u);
          tc_fence_after();
          const float f = jump ? ex2_approx((m_used - bm) * sc) : 1.f;
          for (int cc = 0; cc < p.npv / 16; ++cc) {
            float ov[16];
            tmem_ld16(lane_base + colOg + cc * 16, ov);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) ov[i] *= f;
            tmem_st16(lane_base + colOg + cc * 16, ov);
          }
          tmem_st_wait();
#pragma unroll
          for (int i = 0; i < 4; ++i) l4[i] *= f;
        }
        if (jump) m_used = bm;
      }
      const float mo = m_used * sc;
#pragma unroll
      for (int j = 0; j < BK; ++j) {
        s[j] = ex2_approx(fmaf(s[j], sc, -mo));
        l4[j & 3] += s[j];
      }
      // P (packed 16-bit, BK / 2 columns) over the head of the score buffer: every score is in registers by now
#pragma unroll
      for (int c = 0; c < BK / 16; ++c) {
        uint32_t packed[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) packed[i] = pack16(s[c * 16 + 2 * i], s[c * 16 + 2 * i + 1], bf16);
        tmem_st8(lane_base + colS + c * 8, packed);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(P_READY(buf));
    }
    // ---- merge the two groups' partial softmax states
    xm[g][r] = m_used;
    xl[g][r] = (l4[0] + l4[1]) + (l4[2] + l4[3]);
    named_bar_sync(1, 2 * kGroupThreads);
    const bool has1 = nb >= 2;                       // group 1 saw no key block otherwise: O_1 is unwritten TMEM
    const float m0 = xm[0][r], m1 = has1 ? xm[1][r] : -INFINITY;
    const float m = fmaxf(m0, m1);
    const float f0 = ex2_approx((m0 - m) * sc), f1 = has1 ? ex2_approx((m1 - m) * sc) : 0.f;
    const float l = xl[0][r] * f0 + (has1 ? xl[1][r] * f1 : 0.f);
    const float inv = 1.f / l;
    if (g == 0 && row < p.N) p.lse[((int64_t)b * p.H + h) * p.N + row] = m * p.scale + logf(l);
    const float w0 = f0 * inv, w1 = f1 * inv;

    // ---- epilogue: the two groups take alternate 16-column chunks of O = w0 O_0 + w1 O_1
    mbar_wait(O_READY(), 0);
    tc_fence_after();
    uint8_t* orow = reinterpret_cast<uint8_t*>(p.o) + (((int64_t)b * p.N + row) * p.H + h) * (int64_t)p.d * 2;
    for (int cc = g; cc < p.npv / 16; cc += 2) {
      float oa[16], ob[16];
      tmem_ld16(lane_base + colO + cc * 16, oa);
      if (has1) tmem_ld16(lane_base + colO + (uint32_t)p.npv + cc * 16, ob);
      tmem_ld_wait();
      if (row < p.N) {
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float a0 = has1 ? fmaf(ob[2 * i], w1, oa[2 * i] * w0) : oa[2 * i] * w0;
          const float a1 = has1 ? fmaf(ob[2 * i + 1], w1, oa[2 * i + 1] * w0) : oa[2 * i + 1] * w0;
          w[i] = pack16(a0, a1, bf16);
        }
        const int col = cc * 16;
        if (col < p.d) *reinterpret_cast<uint4*>(orow + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
        if (col + 8 < p.d) *reinterpret_cast<uint4*>(orow + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512u);
}

// ------------------------------------------------------------------------------------------------------ host
bool supports(int dtype, int head_dim) {
  return (dtype == GA_F16 || dtype == GA_BF16) && head_dim % 8 == 0 && head_dim >= 8 && head_dim <= 160;
}

int fwd(const void* q, const void* k, const void* v, void* o, float* lse, int B, int H, int N, int d, float scale,
        int dtype, cudaStream_t st) {
  FwdParams p;
  p.o = o; p.lse = lse; p.B = B; p.H = H; p.N = N; p.d = d;
  p.nblk = (d + kBlockCols - 1) / kBlockCols;
  p.npv = (d + 15) & ~15;
  p.bf16 = dtype == GA_BF16;
  p.bk = p.nblk == 1 ? 128 : 64;
  p.nb = (N + p.bk - 1) / p.bk;
  p.scale = scale;
  const size_t q_bytes = (size_t)p.nblk * kQBlockBytes, stage = (size_t)2 * p.nblk * p.bk * 128;
  p.stages = 0;
  for (int n = kMaxStages; n >= 2; --n)
    if (1024 + q_bytes + n * stage <= 226 * 1024) { p.stages = n; break; }
  if (p.stages == 0) return fail(GA_ERR_UNSUPPORTED, "self-attention: head_dim %d does not fit shared memory", d);
  // two output accumulators behind the three score buffers: 3 bk + 2 npv <= 512 TMEM columns (every head_dim <= 160)
  if (kSBuf * p.bk + 2 * p.npv > 512)
    return fail(GA_ERR_UNSUPPORTED, "self-attention: head_dim %d does not fit tensor memory", d);
  const size_t smem = 1024 + q_bytes + p.stages * stage;
  CUtensorMap mq, mk, mv;
  int rc;
  if ((rc = make_map(&mq, q, dtype, B, N, H, d, kM)) != GA_OK) return rc;
  if ((rc = make_map(&mk, k, dtype, B, N, H, d, p.bk)) != GA_OK) return rc;
  if ((rc = make_map(&mv, v, dtype, B, N, H, d, p.bk)) != GA_OK) return rc;
  dim3 grid((N + kM - 1) / kM, H, B);
  const void* kern = p.bk == 128 ? reinterpret_cast<const void*>(self_attn_fwd1_kernel<128>)
                                 : reinterpret_cast<const void*>(self_attn_fwd1_kernel<64>);
  cudaError_t e = ensure_smem(kern, p.bk == 128 ? 4 : 5, smem);
  if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  if (p.bk == 128) self_attn_fwd1_kernel<128><<<grid, kThreads, smem, st>>>(mq, mk, mv, p);
  else self_attn_fwd1_kernel<64><<<grid, kThreads, smem, st>>>(mq, mk, mv, p);
  return check_launch("self_attn_fwd1");
}


// ===================================================================================================== backward
// Autograd of the forward above (reference: torch autograd through utils/ptp_utils.py:77-85 on the attn1 layers, which
// keeps the (B*H, N, N) probabilities and streams them through softmax-backward and four batched GEMMs).  Here P is
// recomputed from the saved row log-sum-exp; two launches, no atomics (results are bit-stable run to run):
//
//   dQ kernel   one CTA = 128 query rows of one (batch, head); streams the keys in blocks of 64:
//                 S = Q K_j^T, dP = dO V_j^T (two K-major GEMMs into TMEM) -> P = exp(scale S - lse),
//                 dS = P o (dP - D) * scale -> 16-bit into TMEM -> dQ += dS K_j (K_j as the MN-major B operand).
//               It also produces D[row] = sum_c dO[row, c] O[row, c] for the second kernel.
//   dK/dV kernel one CTA = 128 keys of one (batch, head) (TMEM lane = key); streams the queries in blocks of BQ:
//                 S^T = K Q_i^T, dP^T = V dO_i^T -> P^T, dS^T (lse and D are per COLUMN here: staged in shared memory)
//                 -> dV += P^T dO_i, dK += dS^T Q_i (Q_i / dO_i tiles as MN-major B operands).
// Both kernels use the forward's warp roles: warp 0 TMA producer, warp 1 MMA issuer, warps 4-7 / 8-11 compute groups
// that own alternate blocks (TMEM stage = block & 1).
constexpr int kBK = 64;        // keys per block in the dQ kernel

struct BwdParams {
  const void* o;
  const void* d_o;
  const float* lse;
  float* dvec;                 // (B, H, N) fp32: D, written by the dQ kernel, read by the dK/dV kernel
  void* d_q;
  void* d_k;
  void* d_v;
  int B, H, N, d;
  int nblk, npv, bf16;
  int nb;                      // streamed blocks (keys for dQ, queries for dK/dV)
  int bq;                      // queries per block in the dK/dV kernel (64 or 32)
  int tstages;                 // TMEM stages of the streamed GEMM outputs: 3 when the accumulators fit behind them
  int stages;
  float scale;
};

__device__ __forceinline__ float dot8(const uint4& a, const uint4& b, bool bf16) {
  const uint32_t* pa = reinterpret_cast<const uint32_t*>(&a);
  const uint32_t* pb = reinterpret_cast<const uint32_t*>(&b);
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 fa, fb;
    if (bf16) {
      fa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pa[i]));
      fb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pb[i]));
    } else {
      fa = __half22float2(*reinterpret_cast<const __half2*>(&pa[i]));
      fb = __half22float2(*reinterpret_cast<const __half2*>(&pb[i]));
    }
    acc = fmaf(fa.x, fb.x, acc);
    acc = fmaf(fa.y, fb.y, acc);
  }
  return acc;
}

// ------------------------------------------------------------------------------------------------------ dQ
__global__ void __launch_bounds__(kThreads, 1)
self_attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                        const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                        const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  // qg_full, dq_ready, kv_full[4], kv_free[4], sd_ready[3], ds_ready[3], ds_free[3]
  __shared__ __align__(8) uint64_t bars[19];
  __shared__ uint32_t tmem_base_slot;

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int tile = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int row0 = tile * kM;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t kv_block_bytes = (uint32_t)kBK * 128u;
  const uint32_t k_bytes = (uint32_t)p.nblk * kv_block_bytes;
  const uint32_t stage_bytes = 2u * k_bytes;
  const uint32_t sQ = base;
  const uint32_t sG = sQ + (uint32_t)p.nblk * kQBlockBytes;
  const uint32_t sKV = sG + (uint32_t)p.nblk * kQBlockBytes;
  auto QG_FULL = [&]() { return smem_u32(&bars[0]); };
  auto DQ_READY = [&]() { return smem_u32(&bars[1]); };
  auto KV_FULL = [&](int s) { return smem_u32(&bars[2 + s]); };
  auto KV_FREE = [&](int s) { return smem_u32(&bars[6 + s]); };
  auto SD_READY = [&](int i) { return smem_u32(&bars[10 + i]); };
  auto DS_READY = [&](int i) { return smem_u32(&bars[13 + i]); };
  auto DS_FREE = [&](int i) { return smem_u32(&bars[16 + i]); };
  // TMEM: nT stages of 128 columns (S at +0 -- dS is written over it -- and dP at +64), dQ after them.  Three stages
  // when dQ fits behind them (d <= 128): see the forward kernel for why two groups want three buffers.
  const int nT = p.tstages;
  const uint32_t kColDQ = (uint32_t)(nT * 128);
  auto colS = [](int i) { return (uint32_t)(i * 128); };

  if (tid == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_do); prefetch_tmap(&map_k); prefetch_tmap(&map_v);
    mbar_init(QG_FULL(), 1);
    mbar_init(DQ_READY(), 1);
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(KV_FULL(s), 1); mbar_init(KV_FREE(s), 1); }
    for (int i = 0; i < 3; ++i) {
      mbar_init(SD_READY(i), 1);
      mbar_init(DS_READY(i), kGroupThreads);
      mbar_init(DS_FREE(i), 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const int nb = p.nb, NS = p.stages;
  const int ksteps = (p.d + 15) >> 4;
  const int fmt = p.bf16 ? 1 : 0;

  if (warp < 4) {
    reg_dealloc<40>();
    if (warp == 0) {
      // ------------------------------------------------------------------------------------------- producer
      if (elect_one()) {
        mbar_expect_tx(QG_FULL(), 2u * (uint32_t)p.nblk * kQBlockBytes);
        for (int blk = 0; blk < p.nblk; ++blk) {
          tma_load_4d(sQ + blk * kQBlockBytes, &map_q, QG_FULL(), blk * kBlockCols, h, row0, b);
          tma_load_4d(sG + blk * kQBlockBytes, &map_do, QG_FULL(), blk * kBlockCols, h, row0, b);
        }
      }
      int ss = 0;
      uint32_t par = 0;
      for (int it = 0; it < nb; ++it) {
        if (it >= NS) mbar_wait(KV_FREE(ss), par ^ 1u);
        if (elect_one()) {
          const uint32_t sK = sKV + ss * stage_bytes, sV = sK + k_bytes;
          mbar_expect_tx(KV_FULL(ss), stage_bytes);
          for (int blk = 0; blk < p.nblk; ++blk) {
            tma_load_4d(sK + blk * kv_block_bytes, &map_k, KV_FULL(ss), blk * kBlockCols, h, it * kBK, b);
            tma_load_4d(sV + blk * kv_block_bytes, &map_v, KV_FULL(ss), blk * kBlockCols, h, it * kBK, b);
          }
        }
        __syncwarp();
        if (++ss == NS) { ss = 0; par ^= 1u; }
      }
    } else if (warp == 1) {
      // ------------------------------------------------------------------ MMA issuer 1: S = Q K^T, dP = dO V^T
      const uint32_t idesc_s = make_idesc(fmt, 0, kBK, kM);
      const uint64_t dQ0 = smem_desc_sw128(sQ, 16, 1024), dG0 = smem_desc_sw128(sG, 16, 1024);
      const uint64_t dK0 = smem_desc_sw128(sKV, 16, 1024), dV0 = smem_desc_sw128(sKV + k_bytes, 16, 1024);   // K-major
      mbar_wait(QG_FULL(), 0);
      RingPos st = {0, 0}, tb = {0, 0};
      for (int it = 0; it < nb; ++it) {
        if (it >= nT) mbar_wait(DS_FREE(tb.idx), tb.par ^ 1u);   // dS of the stage's previous block consumed by its GEMM
        mbar_wait(KV_FULL(st.idx), st.par);
        tc_fence_after();
        if (elect_one()) {
          issue_kmajor_gemm(tmem + colS(tb.idx), dQ0, kQBlockBytes, desc_advance(dK0, st.idx * stage_bytes), kv_block_bytes,
                            ksteps, idesc_s);
          issue_kmajor_gemm(tmem + colS(tb.idx) + kBK, dG0, kQBlockBytes, desc_advance(dV0, st.idx * stage_bytes),
                            kv_block_bytes, ksteps, idesc_s);
          tc_commit(SD_READY(tb.idx));
        }
        __syncwarp();
        st.advance(NS);
        tb.advance(nT);
      }
    } else if (warp == 2) {
      // ------------------------------------------------------------------ MMA issuer 2: dQ += dS K
      const uint32_t idesc_dq = make_idesc(fmt, 1, p.npv, kM);
      const uint64_t dKmn0 = smem_desc_sw128(sKV, kv_block_bytes, 1024);                                   // MN-major
      RingPos st = {0, 0}, tb = {0, 0};
      for (int it = 0; it < nb; ++it) {
        mbar_wait(DS_READY(tb.idx), tb.par);
        tc_fence_after();
        if (elect_one()) {
          issue_tmem_gemm(tmem + kColDQ, tmem + colS(tb.idx), desc_advance(dKmn0, st.idx * stage_bytes), kBK / 16, idesc_dq,
                          it > 0);
          tc_commit(KV_FREE(st.idx));
          tc_commit(DS_FREE(tb.idx));
        }
        __syncwarp();
        st.advance(NS);
        tb.advance(nT);
      }
      if (elect_one()) tc_commit(DQ_READY());
      __syncwarp();
    }
  } else {
    reg_alloc<232>();
    // --------------------------------------------------------------------------------------- compute groups
    const int g = (warp - 4) >> 2;
    const int r = ((warp & 3) << 5) + lane;
    const int row = row0 + r;
    const bool live = row < p.N;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float sc = p.scale * 1.4426950408889634f;
    const bool bf16 = p.bf16 != 0;

    // D = rowsum(dO o O) for this thread's row (both groups compute it; group 0 publishes it for the dK/dV kernel)
    float Drow = 0.f, l2 = 0.f;
    if (live) {
      const int64_t off = (((int64_t)b * p.N + row) * p.H + h) * (int64_t)p.d;
      const uint4* po = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(p.o) + off * 2);
      const uint4* pg = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(p.d_o) + off * 2);
      for (int c = 0; c < p.d / 8; ++c) Drow += dot8(__ldg(po + c), __ldg(pg + c), bf16);
      const int64_t vi = ((int64_t)b * p.H + h) * p.N + row;
      l2 = __ldg(p.lse + vi) * 1.4426950408889634f;
      if (g == 0) p.dvec[vi] = Drow;
    }

    for (int it = g; it < nb; it += 2) {
      const int ti = nT == 3 ? it % 3 : (it & 1);     // constant divisors: no runtime division per block
      mbar_wait(SD_READY(ti), (uint32_t)(nT == 3 ? it / 3 : it >> 1) & 1u);
      tc_fence_after();
      float s[kBK], dp[kBK];
#pragma unroll
      for (int c = 0; c < kBK / 16; ++c) {
        tmem_ld16(lane_base + colS(ti) + c * 16, s + c * 16);
        tmem_ld16(lane_base + colS(ti) + kBK + c * 16, dp + c * 16);
      }
      tmem_ld_wait();
      const int key0 = it * kBK;
      const bool ragged = key0 + kBK > p.N;
      uint32_t packed[kBK / 2];
#pragma unroll
      for (int j = 0; j < kBK; ++j) {
        float pr = ex2_approx(fmaf(s[j], sc, -l2));
        if (ragged && key0 + j >= p.N) pr = 0.f;
        s[j] = pr * (dp[j] - Drow) * p.scale;
      }
#pragma unroll
      for (int j = 0; j < kBK; j += 2) packed[j >> 1] = pack16(s[j], s[j + 1], bf16);
#pragma unroll
      for (int c = 0; c < kBK / 16; ++c) tmem_st8(lane_base + colS(ti) + c * 8, packed + c * 8);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(DS_READY(ti));
    }

    // ---- epilogue: the two groups take alternate 16-column chunks of dQ
    mbar_wait(DQ_READY(), 0);
    tc_fence_after();
    uint8_t* grow = reinterpret_cast<uint8_t*>(p.d_q) + (((int64_t)b * p.N + row) * p.H + h) * (int64_t)p.d * 2;
    for (int cc = g; cc < p.npv / 16; cc += 2) {
      float ov[16];
      tmem_ld16(lane_base + kColDQ + cc * 16, ov);
      tmem_ld_wait();
      if (live) {
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = pack16(ov[2 * i], ov[2 * i + 1], bf16);
        const int col = cc * 16;
        if (col < p.d) *reinterpret_cast<uint4*>(grow + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
        if (col + 8 < p.d) *reinterpret_cast<uint4*>(grow + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512u);
}

// --------------------------------------------------------------------------------------------------- dK, dV
template <int BQ>
__global__ void __launch_bounds__(kThreads, 1)
self_attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                         const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                         const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  // kv_full, acc_ready, qg_full[4], qg_free[4], sd_ready[3], pds_ready[3], pds_free[3]
  __shared__ __align__(8) uint64_t bars[19];
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float xl[2][2][BQ];       // [group][block parity][query]: lse * log2(e)
  __shared__ __align__(16) float xd[2][2][BQ];       //                                D

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int tile = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int key0 = tile * kM;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t q_block_bytes = (uint32_t)BQ * 128u;
  const uint32_t q_bytes = (uint32_t)p.nblk * q_block_bytes;
  const uint32_t stage_bytes = 2u * q_bytes;
  const uint32_t sK = base;
  const uint32_t sV = sK + (uint32_t)p.nblk * kQBlockBytes;
  const uint32_t sQG = sV + (uint32_t)p.nblk * kQBlockBytes;
  auto KV_FULL = [&]() { return smem_u32(&bars[0]); };
  auto ACC_READY = [&]() { return smem_u32(&bars[1]); };
  auto QG_FULL = [&](int s) { return smem_u32(&bars[2 + s]); };
  auto QG_FREE = [&](int s) { return smem_u32(&bars[6 + s]); };
  auto SD_READY = [&](int i) { return smem_u32(&bars[10 + i]); };
  auto PDS_READY = [&](int i) { return smem_u32(&bars[13 + i]); };
  auto PDS_FREE = [&](int i) { return smem_u32(&bars[16 + i]); };
  // TMEM: stage g at g*2*BQ: S^T at +0 (P^T written over it), dP^T at +BQ (dS^T written over it); accumulators after
  const int nT = p.tstages;                          // 3 when the two accumulators fit behind three stages
  auto colST = [](int i) { return (uint32_t)(i * 2 * BQ); };
  const uint32_t kColDV = (uint32_t)(nT * 2 * BQ);
  const uint32_t colDK = kColDV + (uint32_t)p.npv;

  if (tid == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_do); prefetch_tmap(&map_k); prefetch_tmap(&map_v);
    mbar_init(KV_FULL(), 1);
    mbar_init(ACC_READY(), 1);
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(QG_FULL(s), 1); mbar_init(QG_FREE(s), 1); }
    for (int i = 0; i < 3; ++i) {
      mbar_init(SD_READY(i), 1);
      mbar_init(PDS_READY(i), kGroupThreads);
      mbar_init(PDS_FREE(i), 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const int nb = p.nb, NS = p.stages;
  const int ksteps = (p.d + 15) >> 4;
  const int fmt = p.bf16 ? 1 : 0;

  if (warp < 4) {
    reg_dealloc<40>();
    if (warp == 0) {
      // ------------------------------------------------------------------------------------------- producer
      if (elect_one()) {
        mbar_expect_tx(KV_FULL(), 2u * (uint32_t)p.nblk * kQBlockBytes);
        for (int blk = 0; blk < p.nblk; ++blk) {
          tma_load_4d(sK + blk * kQBlockBytes, &map_k, KV_FULL(), blk * kBlockCols, h, key0, b);
          tma_load_4d(sV + blk * kQBlockBytes, &map_v, KV_FULL(), blk * kBlockCols, h, key0, b);
        }
      }
      int ss = 0;
      uint32_t par = 0;
      for (int it = 0; it < nb; ++it) {
        if (it >= NS) mbar_wait(QG_FREE(ss), par ^ 1u);
        if (elect_one()) {
          const uint32_t sQi = sQG + ss * stage_bytes, sGi = sQi + q_bytes;
          mbar_expect_tx(QG_FULL(ss), stage_bytes);
          for (int blk = 0; blk < p.nblk; ++blk) {
            tma_load_4d(sQi + blk * q_block_bytes, &map_q, QG_FULL(ss), blk * kBlockCols, h, it * BQ, b);
            tma_load_4d(sGi + blk * q_block_bytes, &map_do, QG_FULL(ss), blk * kBlockCols, h, it * BQ, b);
          }
        }
        __syncwarp();
        if (++ss == NS) { ss = 0; par ^= 1u; }
      }
    } else if (warp == 1) {
      // ------------------------------------------------------------ MMA issuer 1: S^T = K Q_i^T, dP^T = V dO_i^T
      const uint32_t idesc_s = make_idesc(fmt, 0, BQ, kM);
      const uint64_t dK0 = smem_desc_sw128(sK, 16, 1024), dV0 = smem_desc_sw128(sV, 16, 1024);
      const uint64_t dQ0 = smem_desc_sw128(sQG, 16, 1024), dG0 = smem_desc_sw128(sQG + q_bytes, 16, 1024);       // K-major
      mbar_wait(KV_FULL(), 0);
      RingPos st = {0, 0}, tb = {0, 0};
      for (int it = 0; it < nb; ++it) {
        if (it >= nT) mbar_wait(PDS_FREE(tb.idx), tb.par ^ 1u);
        mbar_wait(QG_FULL(st.idx), st.par);
        tc_fence_after();
        if (elect_one()) {
          issue_kmajor_gemm(tmem + colST(tb.idx), dK0, kQBlockBytes, desc_advance(dQ0, st.idx * stage_bytes), q_block_bytes,
                            ksteps, idesc_s);
          issue_kmajor_gemm(tmem + colST(tb.idx) + BQ, dV0, kQBlockBytes, desc_advance(dG0, st.idx * stage_bytes),
                            q_block_bytes, ksteps, idesc_s);
          tc_commit(SD_READY(tb.idx));
        }
        __syncwarp();
        st.advance(NS);
        tb.advance(nT);
      }
    } else if (warp == 2) {
      // ------------------------------------------------------------ MMA issuer 2: dV += P^T dO_i, dK += dS^T Q_i
      const uint32_t idesc_acc = make_idesc(fmt, 1, p.npv, kM);
      const uint64_t dQmn0 = smem_desc_sw128(sQG, q_block_bytes, 1024);                                       // MN-major
      const uint64_t dGmn0 = smem_desc_sw128(sQG + q_bytes, q_block_bytes, 1024);
      RingPos st = {0, 0}, tb = {0, 0};
      for (int it = 0; it < nb; ++it) {
        mbar_wait(PDS_READY(tb.idx), tb.par);
        tc_fence_after();
        if (elect_one()) {
          issue_tmem_gemm(tmem + kColDV, tmem + colST(tb.idx), desc_advance(dGmn0, st.idx * stage_bytes), BQ / 16,
                          idesc_acc, it > 0);
          issue_tmem_gemm(tmem + colDK, tmem + colST(tb.idx) + BQ, desc_advance(dQmn0, st.idx * stage_bytes), BQ / 16,
                          idesc_acc, it > 0);
          tc_commit(QG_FREE(st.idx));
          tc_commit(PDS_FREE(tb.idx));
        }
        __syncwarp();
        st.advance(NS);
        tb.advance(nT);
      }
      if (elect_one()) tc_commit(ACC_READY());
      __syncwarp();
    }
  } else {
    reg_alloc<232>();
    // --------------------------------------------------------------------------------------- compute groups
    const int g = (warp - 4) >> 2;
    const int gt = tid - 128 - g * kGroupThreads;    // thread index inside the group
    const int r = ((warp & 3) << 5) + lane;          // key row of the tile = TMEM lane
    const int key = key0 + r;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float sc = p.scale * 1.4426950408889634f;
    const bool bf16 = p.bf16 != 0;
    const int64_t vbase = ((int64_t)b * p.H + h) * p.N;

    int n = 0;
    for (int it = g; it < nb; it += 2, ++n) {
      // stage the per-query log-sum-exp and D of this block (columns of S^T) in shared memory
      const int buf = n & 1;
      if (gt < BQ) {
        const int q = it * BQ + gt;
        xl[g][buf][gt] = q < p.N ? __ldg(p.lse + vbase + q) * 1.4426950408889634f : INFINITY;
        xd[g][buf][gt] = q < p.N ? __ldg(p.dvec + vbase + q) : 0.f;
      }
      named_bar_sync(1 + g, kGroupThreads);
      const int ti = nT == 3 ? it % 3 : (it & 1);     // constant divisors: no runtime division per block
      mbar_wait(SD_READY(ti), (uint32_t)(nT == 3 ? it / 3 : it >> 1) & 1u);
      tc_fence_after();
      float s[BQ], dp[BQ];
#pragma unroll
      for (int c = 0; c < BQ / 16; ++c) {
        tmem_ld16(lane_base + colST(ti) + c * 16, s + c * 16);
        tmem_ld16(lane_base + colST(ti) + BQ + c * 16, dp + c * 16);
      }
      tmem_ld_wait();
      uint32_t pk[BQ / 2], dk[BQ / 2];
#pragma unroll
      for (int j = 0; j < BQ; j += 4) {
        const float4 l4 = *reinterpret_cast<const float4*>(&xl[g][buf][j]);
        const float4 d4 = *reinterpret_cast<const float4*>(&xd[g][buf][j]);
        const float lj[4] = {l4.x, l4.y, l4.z, l4.w}, dj[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float pr = ex2_approx(fmaf(s[j + u], sc, -lj[u]));
          s[j + u] = pr;
          dp[j + u] = pr * (dp[j + u] - dj[u]) * p.scale;
        }
      }
#pragma unroll
      for (int j = 0; j < BQ; j += 2) {
        pk[j >> 1] = pack16(s[j], s[j + 1], bf16);
        dk[j >> 1] = pack16(dp[j], dp[j + 1], bf16);
      }
#pragma unroll
      for (int c = 0; c < BQ / 16; ++c) {
        tmem_st8(lane_base + colST(ti) + c * 8, pk + c * 8);
        tmem_st8(lane_base + colST(ti) + BQ + c * 8, dk + c * 8);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(PDS_READY(ti));
    }

    // ---- epilogue: group 0 stores dV, group 1 stores dK
    mbar_wait(ACC_READY(), 0);
    tc_fence_after();
    const uint32_t col0 = g == 0 ? kColDV : colDK;
    uint8_t* out = reinterpret_cast<uint8_t*>(g == 0 ? p.d_v : p.d_k) +
                   (((int64_t)b * p.N + key) * p.H + h) * (int64_t)p.d * 2;
    for (int cc = 0; cc < p.npv / 16; ++cc) {
      float ov[16];
      tmem_ld16(lane_base + col0 + cc * 16, ov);
      tmem_ld_wait();
      if (key < p.N) {
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = pack16(ov[2 * i], ov[2 * i + 1], bf16);
        const int col = cc * 16;
        if (col < p.d) *reinterpret_cast<uint4*>(out + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
        if (col + 8 < p.d) *reinterpret_cast<uint4*>(out + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512u);
}

template <int BQ>
static int launch_dkv(const CUtensorMap& mk, const CUtensorMap& mv, const CUtensorMap& mq, const CUtensorMap& mg,
                      BwdParams p, int slot, cudaStream_t st) {
  const size_t kv_bytes = (size_t)2 * p.nblk * kQBlockBytes, stage = (size_t)2 * p.nblk * BQ * 128;
  p.bq = BQ;
  p.nb = (p.N + BQ - 1) / BQ;
  p.tstages = (3 * 2 * BQ + 2 * p.npv <= 512) ? 3 : 2;
  p.stages = 0;
  for (int n = kMaxStages; n >= 2; --n)
    if (1024 + kv_bytes + n * stage <= 226 * 1024) { p.stages = n; break; }
  if (p.stages == 0) return fail(GA_ERR_UNSUPPORTED, "self-attention dK/dV: head_dim %d does not fit shared memory", p.d);
  const size_t smem = 1024 + kv_bytes + p.stages * stage;
  cudaError_t e = ensure_smem(reinterpret_cast<const void*>(self_attn_bwd_dkv_kernel<BQ>), slot, smem);
  if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  dim3 grid((p.N + kM - 1) / kM, p.H, p.B);
  self_attn_bwd_dkv_kernel<BQ><<<grid, kThreads, smem, st>>>(mk, mv, mq, mg, p);
  return check_launch("self_attn_bwd_dkv");
}

int bwd(const void* q, const void* k, const void* v, const void* o, const float* lse, const void* d_o, void* d_q,
        void* d_k, void* d_v, float* dvec, int B, int H, int N, int d, float scale, int dtype, cudaStream_t st) {
  BwdParams p;
  p.o = o; p.d_o = d_o; p.lse = lse; p.dvec = dvec; p.d_q = d_q; p.d_k = d_k; p.d_v = d_v;
  p.B = B; p.H = H; p.N = N; p.d = d;
  p.nblk = (d + kBlockCols - 1) / kBlockCols;
  p.npv = (d + 15) & ~15;
  p.bf16 = dtype == GA_BF16;
  p.scale = scale;
  p.bq = 0;
  int rc;
  // ---- dQ (+ D)
  {
    p.nb = (N + kBK - 1) / kBK;
    p.tstages = (3 * 128 + p.npv <= 512) ? 3 : 2;
    const size_t qg_bytes = (size_t)2 * p.nblk * kQBlockBytes, stage = (size_t)2 * p.nblk * kBK * 128;
    p.stages = 0;
    for (int n = kMaxStages; n >= 2; --n)
      if (1024 + qg_bytes + n * stage <= 226 * 1024) { p.stages = n; break; }
    if (p.stages == 0) return fail(GA_ERR_UNSUPPORTED, "self-attention dQ: head_dim %d does not fit shared memory", d);
    const size_t smem = 1024 + qg_bytes + p.stages * stage;
    CUtensorMap mq, mg, mk, mv;
    if ((rc = make_map(&mq, q, dtype, B, N, H, d, kM)) != GA_OK) return rc;
    if ((rc = make_map(&mg, d_o, dtype, B, N, H, d, kM)) != GA_OK) return rc;
    if ((rc = make_map(&mk, k, dtype, B, N, H, d, kBK)) != GA_OK) return rc;
    if ((rc = make_map(&mv, v, dtype, B, N, H, d, kBK)) != GA_OK) return rc;
    cudaError_t e = ensure_smem(reinterpret_cast<const void*>(self_attn_bwd_dq_kernel), 1, smem);
    if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    dim3 grid((N + kM - 1) / kM, H, B);
    self_attn_bwd_dq_kernel<<<grid, kThreads, smem, st>>>(mq, mg, mk, mv, p);
    if ((rc = check_launch("self_attn_bwd_dq")) != GA_OK) return rc;
  }
  // ---- dK, dV
  {
    const int bq = (4 * 64 + 2 * p.npv <= 512) ? 64 : 32;
    CUtensorMap mk, mv, mq, mg;
    if ((rc = make_map(&mk, k, dtype, B, N, H, d, kM)) != GA_OK) return rc;
    if ((rc = make_map(&mv, v, dtype, B, N, H, d, kM)) != GA_OK) return rc;
    if ((rc = make_map(&mq, q, dtype, B, N, H, d, bq)) != GA_OK) return rc;
    if ((rc = make_map(&mg, d_o, dtype, B, N, H, d, bq)) != GA_OK) return rc;
    return bq == 64 ? launch_dkv<64>(mk, mv, mq, mg, p, 2, st) : launch_dkv<32>(mk, mv, mq, mg, p, 3, st);
  }
}

}  // namespace sa
}  // namespace ga
