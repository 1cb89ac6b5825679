// K1, tcgen05 variant: fused cross-attention forward against the short text context on the 5th-gen tensor cores.
//
//   one CTA  = 128 query rows x (heads_per_cta heads, looped)            one cluster = all heads of a row tile
//   TMA      : Q tile, K, V of the head -> shared memory, 128-byte swizzle (cp.async.bulk.tensor.4d + mbarrier)
//   MMA 1    : S[128 x 80]  = Q[128 x d] . K^T          tcgen05.mma kind::f16, A/B K-major from smem, D in TMEM
//   softmax  : one thread per row (TMEM lane), tcgen05.ld, exp2, fp32; P normalised before the second GEMM
//   MMA 2    : O[128 x d]   = P[128 x 80] . V[80 x d]    A = P written back to TMEM as packed 16-bit, B = V MN-major
//   epilogue : tcgen05.ld O -> 16-bit -> global;  row log-sum-exp -> global
//   maps     : every thread keeps its row of head-summed probabilities in registers; the heads of one row tile form a
//              thread-block cluster and the per-head tiles are reduced over distributed shared memory in a fixed order
//              -> the AttentionStore accumulator `acc[b]` is written once, coalesced, without atomics (deterministic).
//
// Replaces reference utils/ptp_utils.py:77-85, 97-146, 226-230 (+ the per-layer part of :273-289) for 16-bit operands.
// The probability tensor never reaches HBM.  This kernel is HBM/latency-bound (77 keys: 60-76 FLOP/B, DESIGN.md): the
// tensor cores are used because the contraction is dense, not because it is the bottleneck.
#include <cuda.h>
#include <cooperative_groups.h>
#include <stdlib.h>

#include "ga_common.cuh"
#include "tc_common.cuh"

namespace cg = cooperative_groups;

namespace ga {
namespace tc {

constexpr int kM = 128;         // query rows per tile = UMMA M
constexpr int kThreads = 128;
constexpr int kQBlockBytes = kM * 128;      // one 64-column block of the Q tile
constexpr int kKVBlockBytes = kTpad * 128;  // one 64-column block of K or V
constexpr int kAccStride = kTpad + 1;       // padded row stride (floats) of the cluster-reduction staging tile

// TMEM column map (fp32 columns).  P (packed 16-bit, 40 columns) overwrites the head of S once every thread has read
// its row of S; O follows.  Everything fits 256 columns up to d = 160, so two CTAs share an SM's 512 columns.
constexpr int kColS = 0;
constexpr int kColP = 0;
constexpr int kColO = 96;

struct FwdParams {
  void* o;
  float* lse;
  float* acc;
  int B, H, N, T, d;
  int nblk;           // 64-column blocks of the head dimension
  int npv;            // UMMA N of the second GEMM: d rounded up to 16
  int heads_per_cta;
  int tmem_cols;
  int bf16;
  float scale;
};

// ------------------------------------------------------------------------------------------------------ kernel
__global__ void __launch_bounds__(kThreads)
cross_attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                         const __grid_constant__ CUtensorMap map_v, const FwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2];
  __shared__ uint32_t tmem_base_slot;

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int tile = blockIdx.y, b = blockIdx.z;
  const int head0 = blockIdx.x * p.heads_per_cta;
  const int row0 = tile * kM;

  // 1024-byte aligned carve-up (the 128-byte swizzle pattern repeats every 8 rows = 1024 bytes)
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sQ = base;
  const uint32_t sK = sQ + p.nblk * kQBlockBytes;
  const uint32_t sV = sK + p.nblk * kKVBlockBytes;
  float* sAcc = reinterpret_cast<float*>(base_ptr + p.nblk * (kQBlockBytes + 2 * kKVBlockBytes));
  const uint32_t bar_load = smem_u32(&bars[0]), bar_mma = smem_u32(&bars[1]);

  if (tid == 0) {
    prefetch_tmap(&map_q);
    prefetch_tmap(&map_k);
    prefetch_tmap(&map_v);
    mbar_init(bar_load, 1);
    mbar_init(bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);   // this warp's quarter of the 128 TMEM lanes

  const int fmt = p.bf16 ? 1 : 0;
  const uint32_t idesc_qk = make_idesc(fmt, 0, kTpad, kM);
  const uint32_t idesc_pv = make_idesc(fmt, 1, p.npv, kM);
  const uint32_t tx_bytes = (uint32_t)p.nblk * (kQBlockBytes + 2 * kKVBlockBytes);
  const float sc = p.scale * 1.4426950408889634f;
  const int ksteps = (p.d + 15) >> 4;

  float pacc[kTpad];
#pragma unroll
  for (int j = 0; j < kTpad; ++j) pacc[j] = 0.f;

  uint32_t ph_load = 0, ph_mma = 0;   // mbarrier phase parities: bar_load flips once per head, bar_mma twice
  for (int hh = 0; hh < p.heads_per_cta; ++hh) {
    const int h = head0 + hh;
    // ---- TMA: Q tile + K + V of this head; MMA 1 (warp 0, warp-uniform; one elected lane issues) ---------------
    if (warp == 0) {
      if (elect_one()) {
        mbar_expect_tx(bar_load, tx_bytes);
        for (int blk = 0; blk < p.nblk; ++blk) {
          tma_load_4d(sQ + blk * kQBlockBytes, &map_q, bar_load, blk * kBlockCols, h, row0, b);
          tma_load_4d(sK + blk * kKVBlockBytes, &map_k, bar_load, blk * kBlockCols, h, 0, b);
          tma_load_4d(sV + blk * kKVBlockBytes, &map_v, bar_load, blk * kBlockCols, h, 0, b);
        }
      }
      mbar_wait(bar_load, ph_load);
      tc_fence_after();
      if (elect_one()) {
        // S = Q K^T: K-major operands; a k-step of 16 elements is 32 bytes inside the 128-byte swizzled row
        issue_kmajor_gemm(tmem + kColS, smem_desc_sw128(sQ, 16, 1024), kQBlockBytes, smem_desc_sw128(sK, 16, 1024),
                          kKVBlockBytes, ksteps, idesc_qk);
        tc_commit(bar_mma);
      }
      __syncwarp();
    }
    mbar_wait(bar_mma, ph_mma);
    ph_mma ^= 1;
    tc_fence_after();

    // ---- softmax over the keys of this thread's row ----------------------------------------------------------
    float s[kTpad];
#pragma unroll
    for (int c = 0; c < kTpad / 16; ++c) tmem_ld16(lane_addr + kColS + c * 16, s + c * 16);
    tmem_ld_wait();
    float m, sum;
    row_softmax_ilp(s, p.T, sc, m, sum);
    // P (un-normalised, 16-bit) -> TMEM (A operand of the second GEMM), over the columns S occupied
#pragma unroll
    for (int c = 0; c < kTpad / 16; ++c) {
      uint32_t packed[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) packed[i] = pack16(s[c * 16 + 2 * i], s[c * 16 + 2 * i + 1], p.bf16 != 0);
      tmem_st8(lane_addr + kColP + c * 8, packed);
    }
    const float inv = __fdividef(1.f, sum);
    if (p.acc != nullptr) {
#pragma unroll
      for (int j = 0; j < kTpad; ++j) pacc[j] = fmaf(s[j], inv, pacc[j]);
    }
    const int row = row0 + tid;
    if (row < p.N) p.lse[((int64_t)b * p.H + h) * p.N + row] = (m * sc + lg2_approx(sum)) * 0.6931471805599453f;
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();

    // ---- MMA 2: O = P V  (V is MN-major: rows = keys, 128-byte rows of 64 channels) -------------------------
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        // 16 keys = two 8-row swizzle atoms (SBO = 1024 B apart); channel blocks are LBO = one K/V block apart
        issue_tmem_gemm(tmem + kColO, tmem + kColP, smem_desc_sw128(sV, kKVBlockBytes, 1024), kTpad / 16, idesc_pv, false);
        tc_commit(bar_mma);
      }
      __syncwarp();
    }
    mbar_wait(bar_mma, ph_mma);
    ph_mma ^= 1;
    tc_fence_after();

    // ---- epilogue: O row -> 16-bit -> global -----------------------------------------------------------------
    {
      uint8_t* orow = reinterpret_cast<uint8_t*>(p.o) + (((int64_t)b * p.N + row) * p.H + h) * (int64_t)p.d * 2;
      for (int c = 0; c < p.npv / 16; ++c) {
        float ov[16];
        tmem_ld16(lane_addr + kColO + c * 16, ov);
        tmem_ld_wait();
        if (row < p.N) {
          uint32_t w[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) w[i] = pack16(ov[2 * i] * inv, ov[2 * i + 1] * inv, p.bf16 != 0);
          const int col = c * 16;
          if (col < p.d) *reinterpret_cast<uint4*>(orow + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
          if (col + 8 < p.d) *reinterpret_cast<uint4*>(orow + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
        }
      }
    }
    // all TMEM reads of this head are done before the next head's MMA overwrites S / O, and before smem is reloaded
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    ph_load ^= 1;
  }

  if (warp == 0) tmem_dealloc(tmem, (uint32_t)p.tmem_cols);

  // ---- head reduction of the probability rows across the cluster (DSMEM), fixed order -----------------------
  if (p.acc != nullptr) {
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned csize = cluster.num_blocks(), crank = cluster.block_rank();
#pragma unroll
    for (int j = 0; j < kTpad; ++j) sAcc[tid * kAccStride + j] = pacc[j];
    cluster.sync();
    // every remote load of a row is issued before the first add (one DSMEM round trip per row instead of one per
    // peer); the sum itself runs in rank order, so the result does not depend on timing
    const float* peer[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) peer[c] = cluster.map_shared_rank(sAcc, c < (int)csize ? c : 0);
    for (int i = (int)crank + (int)csize * warp; i < kM; i += (int)csize * (kThreads / 32)) {
      const int r = row0 + i;
      if (r >= p.N) continue;
      float part[8][3];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) {
          const int j = lane + 32 * kk;
          part[c][kk] = (c < (int)csize && j < p.T) ? peer[c][i * kAccStride + j] : 0.f;
        }
      }
      float v[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < 8; ++c) {
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) v[kk] += part[c][kk];
      }
#pragma unroll
      for (int kk = 0; kk < 3; ++kk) {
        const int j = lane + 32 * kk;
        if (j < p.T) p.acc[((int64_t)b * p.N + r) * p.T + j] = v[kk];
      }
    }
    cluster.sync();   // nobody leaves while a peer may still read its staging tile
  }
}


// ============================================================================= K1, persistent pipelined variant
// The single-shot kernel above is latency-bound per CTA (TMA -> MMA -> softmax -> MMA -> epilogue in sequence).  For
// launches with enough work per SM this variant keeps ONE persistent CTA per SM (512 threads, four warpgroups) and
// overlaps the stages of consecutive work items:
//
//   WG0  warps  0-3   epilogue        O (TMEM) * 1/rowsum -> 16-bit -> shared memory (the item's dead Q tile, TMA swizzle)
//                                     -> TMA store; hands the TMEM O columns and the shared-memory stage back
//   WG1  warps  4-7   softmax group 0 items 0, 2, 4, ...   TMEM stage 0 (columns   0-255: S/P at +0, O at +96)
//   WG2  warps  8-11  softmax group 1 items 1, 3, 5, ...   TMEM stage 1 (columns 256-511)
//   WG3  warp  12     TMA producer    runs up to `smem_stages` items ahead (full / smem_free mbarriers)
//        warp  13     MMA issuer      MMA1(k) is issued before MMA2(k-1)
//
// A softmax group never waits for the second GEMM or for global stores: its per-item critical path is
// tcgen05.ld -> max / exp2 / sum -> tcgen05.st.  The O rows leave through the TMA (no per-thread 16-byte stores with
// a row stride between lanes, which is what saturated the LSU in the first pipelined version: profiles/).
//
// Work items: flat (b, tile, h) with h fastest (the heads of one row tile run on neighbouring SMs at the same time, so
// the 32-byte sectors two heads share are fetched / written once); with maps a CTA takes whole (b, tile) groups and
// streams the H heads through the pipeline, so the head-sum of P stays in the two groups' registers and is combined
// once per group through one shared staging tile, in a fixed order, then written coalesced: deterministic, no atomics.
constexpr int kPipeThreads = 512;
constexpr int kMaxStages = 6;   // shared-memory ring depth of the grouped forward and of the streaming K1 / K2
constexpr int kFwdStages = 12;  // flat forward: Q-only stages
constexpr int kStageCols = 256;
constexpr int kGroupThreads = 128;

struct PipeParams {
  void* o;
  float* lse;
  float* acc;
  int B, H, N, T, d;
  int nblk, npv, bf16;
  int tiles;        // row tiles per (b, h)
  int units;        // row tiles B*tiles: the work units of the grouped mode, the ranges the flat mode splits
  int grouped;      // 1: a unit is a (b, tile) group of H items
  int smem_stages;  // 1 .. kMaxStages
  int n_sbuf;       // S/P buffers in TMEM: 4 when 4*80 + 2*npv <= 512, else 2
  int n_obuf;       // O buffers in TMEM: as many as fit behind the S buffers (2 .. 4)
  int direct_store; // 1: epilogue stores from registers (short rings), 0: staged in the dead Q tile + TMA store
  float scale;
};

// Coordinates of the work items of one CTA, advanced incrementally.
//   grouped (maps kept): units (b, tile) dealt round-robin over the grid, H items (heads) per unit.
//   flat: the grid is `gridDim.x / H` teams of H CTAs; a team owns a contiguous range of the B * tiles row tiles and CTA
//         `blockIdx.x % H` of the team streams head h of that range in (b, tile) order.  Consecutive items of a CTA then
//         share (b, h) -- K and V stay in the shared-memory stage and are not re-loaded -- while the H CTAs of a team
//         sweep the same rows at the same time, so the 32-byte sectors neighbouring heads share are fetched once.
struct ItemIter {
  int unit, b, tile, h;
  __device__ __forceinline__ void init(const PipeParams& p) {
    if (p.grouped) {
      unit = blockIdx.x;
      h = 0;
      b = unit / p.tiles;
      tile = unit - b * p.tiles;
    } else {
      h = blockIdx.x % p.H;
      unit = flat_begin(p);                       // row tile index b * tiles + tile
      b = unit / p.tiles;
      tile = unit - b * p.tiles;
    }
  }
  __device__ __forceinline__ void next(const PipeParams& p) {
    if (p.grouped) {
      if (++h < p.H) return;
      h = 0;
      unit += gridDim.x;
      b = unit / p.tiles;
      tile = unit - b * p.tiles;
    } else {
      ++unit;
      if (++tile == p.tiles) { tile = 0; ++b; }
    }
  }
  static __device__ __forceinline__ int flat_begin(const PipeParams& p) {
    const int teams = gridDim.x / p.H, team = blockIdx.x / p.H;
    return (int)(((int64_t)p.units * team) / teams);
  }
  static __device__ __forceinline__ int flat_count(const PipeParams& p) {
    const int teams = gridDim.x / p.H, team = blockIdx.x / p.H;
    return (int)(((int64_t)p.units * (team + 1)) / teams) - (int)(((int64_t)p.units * team) / teams);
  }
};

// Two softmax groups (16 warps): with maps kept the head-sum lives in the groups' registers, 184 per softmax thread.
__global__ void __launch_bounds__(kPipeThreads, 1)
cross_attn_fwd_tc_pipe_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                              const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_o,
                              const PipeParams p) {
  extern __shared__ uint8_t smem_raw[];
  // full[12], smem_free[12] (per shared-memory stage); s_ready[4], p_ready[4], p_free[4] (per S/P buffer); o_ready[4],
  // tmem_free[4] (per O buffer); kv_full[2], kv_free[2] (flat mode: K/V slots outside the ring)
  __shared__ __align__(8) uint64_t bars[2 * kFwdStages + 24];
  __shared__ uint32_t tmem_base_slot;
  __shared__ float s_inv[8][kM];         // [item & 7][row]: 1 / rowsum, softmax group -> epilogue

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  // Flat mode (no maps): consecutive items of a CTA share (b, h), so K and V live in two slots OUTSIDE the ring and a ring
  // stage holds the Q tile only (16 KB per 64 channels instead of 36): up to 12 Q tiles in flight.  The ablation runs
  // showed the flat kernel bound by ring latency (load + store-read + seven barrier hand-offs ~ 5 us per item) times ring
  // depth, not by any unit.  Grouped mode (maps kept): every item has its own head -> K/V stay inside the stage.
  const bool kvres = !p.grouped;
  const uint32_t q_bytes = (uint32_t)p.nblk * kQBlockBytes, kv_bytes = 2u * (uint32_t)p.nblk * kKVBlockBytes;
  const uint32_t stage_bytes = kvres ? q_bytes : q_bytes + kv_bytes;
  const uint32_t kv_base = base + (uint32_t)p.smem_stages * stage_bytes;        // flat mode: two (K, V) slots
  float* sAcc = reinterpret_cast<float*>(base_ptr + (size_t)p.smem_stages * stage_bytes);
  auto KV_FULL = [&](int s) { return smem_u32(&bars[2 * kFwdStages + 20 + s]); };
  auto KV_FREE = [&](int s) { return smem_u32(&bars[2 * kFwdStages + 22 + s]); };
  auto FULL = [&](int s) { return smem_u32(&bars[s]); };
  auto SMEM_FREE = [&](int s) { return smem_u32(&bars[kFwdStages + s]); };
  auto S_READY = [&](int s) { return smem_u32(&bars[2 * kFwdStages + s]); };
  auto P_READY = [&](int s) { return smem_u32(&bars[2 * kFwdStages + 4 + s]); };
  auto O_READY = [&](int s) { return smem_u32(&bars[2 * kFwdStages + 8 + s]); };
  auto TMEM_FREE = [&](int s) { return smem_u32(&bars[2 * kFwdStages + 12 + s]); };
  auto P_FREE = [&](int s) { return smem_u32(&bars[2 * kFwdStages + 16 + s]); };
  // TMEM: nS score buffers of 80 columns (P, packed 16-bit, overwrites the head of its S buffer), then two O buffers.
  // With four S buffers (d <= 96) a softmax group finds the scores of its NEXT item already computed when it finishes
  // one: MMA1(k + 2) no longer has to wait for MMA2(k) to consume P(k) out of the same columns -- that round trip
  // (arrive -> issue -> tensor pipe -> commit -> wake-up, ~1.4 us) used to sit on every group's critical path.
  // (buffer counts are powers of two: index = k & mask, use parity = (k >> shift) & 1 -- no divisions on the issue path)
  const int nS = p.n_sbuf, nO = p.n_obuf;
  const int sMask = nS - 1, oMask = nO - 1, sShift = nS == 4 ? 2 : 1, oShift = nO == 4 ? 2 : 1;
  auto sIdx = [&](int k) { return k & sMask; };
  auto oIdx = [&](int k) { return k & oMask; };
  auto colS = [&](int k) { return (uint32_t)((k & sMask) * kTpad); };
  auto colO = [&](int k) { return (uint32_t)(nS * kTpad + (k & oMask) * p.npv); };
  auto sPar = [&](int k) { return (uint32_t)(k >> sShift) & 1u; };
  auto oPar = [&](int k) { return (uint32_t)(k >> oShift) & 1u; };

  // number of work units / items this CTA owns (units are dealt round-robin over the grid)
  const int my_units = (p.units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int n_items = p.grouped ? my_units * p.H : ItemIter::flat_count(p);

  if (tid == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_k); prefetch_tmap(&map_v); prefetch_tmap(&map_o);
    for (int s = 0; s < kFwdStages; ++s) { mbar_init(FULL(s), 1); mbar_init(SMEM_FREE(s), p.direct_store ? 1 : 4); }
    for (int s = 0; s < 4; ++s) {
      mbar_init(S_READY(s), 1);
      mbar_init(P_READY(s), kGroupThreads);
      mbar_init(O_READY(s), 1);
      mbar_init(TMEM_FREE(s), kGroupThreads);
      mbar_init(P_FREE(s), 1);
    }
    for (int s = 0; s < 2; ++s) { mbar_init(KV_FULL(s), 1); mbar_init(KV_FREE(s), 1); }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const int fmt = p.bf16 ? 1 : 0;
  const int ksteps = (p.d + 15) >> 4;
  const int S = p.smem_stages;
  const bool bf16 = p.bf16 != 0;
  // Short rings (big tiles: d > 64) cannot afford to hold a stage until the epilogue's TMA store has read it: there the
  // epilogue stores its rows straight from registers and the stage is released by the second GEMM's commit.
  const bool direct = p.direct_store != 0;

  constexpr int kCtlWarp = 12;                       // control warpgroup: producer, MMA issuer 1, MMA issuer 2, idle
  if (warp >= kCtlWarp) {
    reg_dealloc<56>();
    if (warp == kCtlWarp) {
      // ------------------------------------------------------------------------------------- TMA producer
      // Flat mode: K and V are loaded once per batch element of the CTA's range (the TMA handles one box row of <= 128
      // bytes per few cycles; at d = 40 the 2 x 80 K/V rows of an item would cost more TMA slots than its 128 Q rows).
      ItemIter it;
      it.init(p);
      int ss = 0, cur_b = -1, unit = -1;
      uint32_t par = 0;                                 // parity of the use of stage ss that is about to start
      for (int k = 0; k < n_items; ++k) {
        if (kvres && it.b != cur_b) {                   // flat mode: a new batch element -> its K, V into the next slot
          cur_b = it.b;
          ++unit;
          const int slot = unit & 1;
          if (unit >= 2) mbar_wait(KV_FREE(slot), (((uint32_t)(unit >> 1)) & 1u) ^ 1u);
          if (elect_one()) {
            const uint32_t sK = kv_base + slot * kv_bytes, sV = sK + p.nblk * kKVBlockBytes;
            mbar_expect_tx(KV_FULL(slot), kv_bytes);
            for (int blk = 0; blk < p.nblk; ++blk) {
              tma_load_4d(sK + blk * kKVBlockBytes, &map_k, KV_FULL(slot), blk * kBlockCols, it.h, 0, it.b);
              tma_load_4d(sV + blk * kKVBlockBytes, &map_v, KV_FULL(slot), blk * kBlockCols, it.h, 0, it.b);
            }
          }
          __syncwarp();
        }
        if (k >= S) mbar_wait(SMEM_FREE(ss), par ^ 1u);
        if (elect_one()) {
          const uint32_t sQ = base + ss * stage_bytes, sK = sQ + p.nblk * kQBlockBytes, sV = sK + p.nblk * kKVBlockBytes;
          mbar_expect_tx(FULL(ss), stage_bytes);
          for (int blk = 0; blk < p.nblk; ++blk) {
            tma_load_4d(sQ + blk * kQBlockBytes, &map_q, FULL(ss), blk * kBlockCols, it.h, it.tile * kM, it.b);
            if (!kvres) {
              tma_load_4d(sK + blk * kKVBlockBytes, &map_k, FULL(ss), blk * kBlockCols, it.h, 0, it.b);
              tma_load_4d(sV + blk * kKVBlockBytes, &map_v, FULL(ss), blk * kBlockCols, it.h, 0, it.b);
            }
          }
        }
        __syncwarp();
        it.next(p);
        if (++ss == S) { ss = 0; par ^= 1u; }
      }
    } else if (warp == kCtlWarp + 1) {
      // ------------------------------------------------------------------------------ MMA issuer 1: S = Q K^T
      // Two issuer warps, one per GEMM: a single thread issuing both was the critical path of the CTA once everything
      // else overlapped (its ~150 instructions per item take longer than the item's data movement).  Cross-warp
      // ordering is by completion: MMA1(k) overwrites the columns P(k - nS) lived in, so it waits for P_FREE of that
      // buffer, which MMA2's commit signals.
      const uint32_t idesc_qk = make_idesc(fmt, 0, kTpad, kM);
      const uint64_t dQ0 = smem_desc_sw128(base, 16, 1024);
      const uint64_t dK0 = smem_desc_sw128(kvres ? kv_base : base + p.nblk * kQBlockBytes, 16, 1024);
      ItemIter it;
      it.init(p);
      int ss = 0, cur_b = -1, unit = -1;
      uint32_t par = 0;
      for (int k = 0; k < n_items; ++k) {
        if (kvres && it.b != cur_b) {                   // first item of a batch element: its K, V must have landed
          cur_b = it.b;
          ++unit;
          mbar_wait(KV_FULL(unit & 1), ((uint32_t)(unit >> 1)) & 1u);
        }
        if (k >= nS) mbar_wait(P_FREE(sIdx(k)), sPar(k) ^ 1u);
        mbar_wait(FULL(ss), par);
        tc_fence_after();
        if (elect_one()) {
          issue_kmajor_gemm(tmem + colS(k), desc_advance(dQ0, ss * stage_bytes), kQBlockBytes,
                            desc_advance(dK0, kvres ? (unit & 1) * kv_bytes : ss * stage_bytes), kKVBlockBytes, ksteps,
                            idesc_qk);
          tc_commit(S_READY(sIdx(k)));
        }
        __syncwarp();
        it.next(p);
        if (++ss == S) { ss = 0; par ^= 1u; }
      }
    } else if (warp == kCtlWarp + 2) {
      // ------------------------------------------------------------------------------ MMA issuer 2: O = P V
      const uint32_t idesc_pv = make_idesc(fmt, 1, p.npv, kM);
      const uint64_t dV0 = smem_desc_sw128((kvres ? kv_base : base + p.nblk * kQBlockBytes) + p.nblk * kKVBlockBytes,
                                           kKVBlockBytes, 1024);
      ItemIter it;
      it.init(p);
      int ss = 0, cur_b = it.b, unit = 0;
      for (int k = 0; k < n_items; ++k) {
        mbar_wait(P_READY(sIdx(k)), sPar(k));
        if (k >= nO) mbar_wait(TMEM_FREE(oIdx(k)), oPar(k) ^ 1u);  // the epilogue of item k-nO has drained this O buffer
        tc_fence_after();
        const int slot = unit & 1;
        it.next(p);
        const bool last_of_unit = kvres && (k == n_items - 1 || it.b != cur_b);
        if (elect_one()) {
          issue_tmem_gemm(tmem + colO(k), tmem + colS(k), desc_advance(dV0, kvres ? slot * kv_bytes : ss * stage_bytes),
                          kTpad / 16, idesc_pv, false);
          tc_commit(O_READY(oIdx(k)));
          tc_commit(P_FREE(sIdx(k)));
          if (direct) tc_commit(SMEM_FREE(ss));          // nothing is staged in the stage: free it as soon as V is read
          if (last_of_unit) tc_commit(KV_FREE(slot));    // every GEMM that reads this slot has been issued (and S(k) done)
        }
        __syncwarp();
        if (last_of_unit) { cur_b = it.b; ++unit; }
        if (++ss == S) ss = 0;
      }
    }
  } else if (warp < 4) {
    reg_dealloc<88>();
    // ---------------------------------------------------------------------------------------- epilogue
    // The four warps run independently (no warpgroup barrier): each converts its 32 TMEM lanes, stages them in its
    // quarter of the tile and issues its own TMA store (box of 32 rows); the stage is handed back to the producer when
    // all four stores have read it (SMEM_FREE counts 4 arrivals).
    const int r = (warp << 5) + lane;                 // row of the tile = TMEM lane
    const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
    ItemIter it;
    it.init(p);
    int ss = 0;
    if (direct) {
      // short rings: rows go from registers to global memory (the stage was handed back by MMA2's commit)
      for (int k = 0; k < n_items; ++k) {
        const int ob = oIdx(k);
        mbar_wait(O_READY(ob), oPar(k));
        tc_fence_after();
        const float inv = s_inv[k & 7][r];
        const int row = it.tile * kM + r;
        uint8_t* orow = reinterpret_cast<uint8_t*>(p.o) + (((int64_t)it.b * p.N + row) * p.H + it.h) * (int64_t)p.d * 2;
        for (int cc = 0; cc < p.npv / 16; ++cc) {
          float ov[16];
          tmem_ld16(lane_base + colO(k) + cc * 16, ov);
          tmem_ld_wait();
          if (row < p.N) {
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = pack16(ov[2 * i] * inv, ov[2 * i + 1] * inv, bf16);
            const int col = cc * 16;
            if (col < p.d) *reinterpret_cast<uint4*>(orow + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
            if (col + 8 < p.d) *reinterpret_cast<uint4*>(orow + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
          }
        }
        tc_fence_before();
        mbar_arrive(TMEM_FREE(ob));
        it.next(p);
      }
    }
    for (int k = 0; k < n_items && !direct; ++k) {
      const int ob = oIdx(k);
      mbar_wait(O_READY(ob), oPar(k));
      tc_fence_after();
      const float inv = s_inv[k & 7][r];
      const uint32_t sO = base + ss * stage_bytes;    // the Q tile of this stage is dead once MMA1 has retired
      for (int c0 = 0; c0 < p.npv / 16; c0 += 4) {    // up to 64 columns per TMEM round trip
        float ov[64];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (c0 + u < p.npv / 16) tmem_ld16(lane_base + colO(k) + (c0 + u) * 16, ov + u * 16);
        tmem_ld_wait();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (c0 + u < p.npv / 16) {
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = pack16(ov[u * 16 + 2 * i] * inv, ov[u * 16 + 2 * i + 1] * inv, bf16);
            st_swizzled_32B(sO + (uint32_t)((c0 + u) >> 2) * kQBlockBytes, r, ((c0 + u) & 3) * 2, w);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(TMEM_FREE(ob));
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        for (int blk = 0; blk < p.nblk; ++blk)
          tma_store_4d(&map_o, sO + blk * kQBlockBytes + (uint32_t)warp * 4096u, blk * kBlockCols, it.h,
                       it.tile * kM + warp * 32, it.b);
        bulk_commit_group();
        // a stage may be refilled once its stores have read it.  Long rings wait for the PREVIOUS item's store only, so
        // the read of this one overlaps the next item's TMEM loads; short rings cannot afford the one-item delay.
        if (S < 5) {
          bulk_wait_read0();
          mbar_arrive(SMEM_FREE(ss));
        } else if (k >= 1) {
          bulk_wait_read1();
          mbar_arrive(SMEM_FREE(ss == 0 ? S - 1 : ss - 1));
        }
      }
      __syncwarp();
      it.next(p);
      if (++ss == S) ss = 0;
    }
    if (!direct && elect_one()) {
      bulk_wait_read0();
      if (n_items >= 1 && S >= 5) mbar_arrive(SMEM_FREE(ss == 0 ? S - 1 : ss - 1));
      bulk_wait_all0();
    }
    __syncwarp();
  } else {
    // setmaxnreg moves registers inside the CTA's OWN launch allocation (threads x registers at launch), not the SM's
    // file: 512 x 128 = 64 K (56 + 88 + 2 x 184 per 128 threads); asking for more spins forever in
    // USETMAXREG.TRY_ALLOC.
    reg_alloc<184>();
    // ------------------------------------------------------------------------------------ softmax groups
    const int g = (warp - 4) >> 2;                    // handles items k with k % 2 == g
    const int r = ((warp & 3) << 5) + lane;           // row of the tile = TMEM lane
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float sc = p.scale * 1.4426950408889634f;
    float pacc[kTpad];                                // head-sum of P (maps kept)
    if (p.grouped) {
#pragma unroll
      for (int j = 0; j < kTpad; ++j) pacc[j] = 0.f;
    }

    auto process = [&](int k, int b, int h, int tile) {
      const int row = tile * kM + r;
      const uint32_t lane_addr = lane_base + colS(k);
      mbar_wait(S_READY(sIdx(k)), sPar(k));
      tc_fence_after();
      float s[kTpad];
#pragma unroll
      for (int cc = 0; cc < kTpad / 16; ++cc) tmem_ld16(lane_addr + cc * 16, s + cc * 16);
      tmem_ld_wait();
      float m, sum;
      row_softmax_ilp(s, p.T, sc, m, sum);
#pragma unroll
      for (int cc = 0; cc < kTpad / 16; ++cc) {
        uint32_t packed[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) packed[i] = pack16(s[cc * 16 + 2 * i], s[cc * 16 + 2 * i + 1], bf16);
        tmem_st8(lane_addr + cc * 8, packed);
      }
      const float inv = __fdividef(1.f, sum);
      s_inv[k & 7][r] = inv;
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(P_READY(sIdx(k)));
      if (p.grouped) {
#pragma unroll
        for (int j = 0; j < kTpad; ++j) pacc[j] = fmaf(s[j], inv, pacc[j]);
      }
      if (row < p.N)
        p.lse[((int64_t)b * p.H + h) * p.N + row] = (m * sc + lg2_approx(sum)) * 0.6931471805599453f;
    };

    ItemIter it;
    it.init(p);
    if (!p.grouped) {
      for (int i = 0; i < g; ++i) it.next(p);
      for (int k = g; k < n_items; k += 2) {
        process(k, it.b, it.h, it.tile);
#pragma unroll
        for (int i = 0; i < 2; ++i) it.next(p);
      }
    } else {
      int k = 0;
      for (int u = 0; u < my_units; ++u) {
        const int unit = blockIdx.x + u * gridDim.x;
        const int b = unit / p.tiles, tile = unit - b * p.tiles;
        for (int h = 0; h < p.H; ++h, ++k)
          if ((k & 1) == g) process(k, b, h, tile);
        // ---- end of the (b, tile) group: combine the two groups' head sums, write the accumulator rows coalesced
        if (g == 1) {
#pragma unroll
          for (int j = 0; j < kTpad; ++j) sAcc[r * kAccStride + j] = pacc[j];
        }
        named_bar_sync(1, 2 * kGroupThreads);
        if (g == 0) {
#pragma unroll
          for (int j = 0; j < kTpad; ++j) sAcc[r * kAccStride + j] += pacc[j];
        }
        named_bar_sync(2, 2 * kGroupThreads);
        for (int i = warp - 4; i < kM; i += 8) {
          const int gr = tile * kM + i;
          if (gr >= p.N) break;
#pragma unroll
          for (int kk = 0; kk < 3; ++kk) {
            const int j = lane + 32 * kk;
            if (j < p.T) p.acc[((int64_t)b * p.N + gr) * p.T + j] = sAcc[i * kAccStride + j];
          }
        }
        named_bar_sync(3, 2 * kGroupThreads);
#pragma unroll
        for (int j = 0; j < kTpad; ++j) pacc[j] = 0.f;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512u);
}

// ================================================================ K1, persistent STREAMING variant (maps kept, d > 64)
// With maps a CTA streams the H heads of one (b, tile) unit, every item with its own K and V, so the pipelined kernel
// above must keep K/V inside the ring stage: 72 KB per stage at d = 80 and 108 KB at d = 160 next to the 41 KB
// head-sum staging tile, i.e. TWO stages / ONE stage -- the kernel is ring-latency bound (18 / 32 us per unit whatever
// the unit count, profiles/r02_crossover_sweep_before.jsonl).  Like the streaming K2 below, this variant rings
// 64-channel BLOCKS: a stage is (Q block, K block) = 26 KB, S is accumulated over the blocks as they land and a stage
// is released by the commit that follows its own k-steps; the item's V (needed only by the second GEMM) waits in a
// small ring of V slots; O rows leave from registers.  Softmax groups, head-sum accumulation and TMEM layout are
// those of the pipelined kernel.
struct FwdStreamParams {
  PipeParams b;
  int ring_stages;   // (Q block, K block) stages, 2 .. kMaxStages
  int v_slots;       // 2 .. 4
  int stage_out;     // leading 64-channel blocks of O that leave through per-warp TMA-store staging tiles (0, 1 or 2)
};
constexpr uint32_t kOutStageBytes = 4u * 4096u;   // one staged block: 4 epilogue warps x (32 rows x 128 bytes)

__global__ void __launch_bounds__(kPipeThreads, 1)
cross_attn_fwd_tc_stream_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                                const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_o,
                                const FwdStreamParams sp) {
  const PipeParams& p = sp.b;
  extern __shared__ uint8_t smem_raw[];
  // ring_full[6], ring_free[6], v_full[4], v_free[4], s_ready[4], p_ready[4], p_free[4], o_ready[4], tmem_free[4]
  __shared__ __align__(8) uint64_t bars[2 * kMaxStages + 28];
  __shared__ uint32_t tmem_base_slot;
  __shared__ float s_inv[8][kM];

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
  constexpr uint32_t ring_stage_bytes = kQBlockBytes + kKVBlockBytes;
  const int R = sp.ring_stages, NV = sp.v_slots;
  const uint32_t v_slot_bytes = (uint32_t)p.nblk * kKVBlockBytes;
  const uint32_t v_base = base + (uint32_t)R * ring_stage_bytes;
  const uint32_t out_stage = v_base + (uint32_t)NV * v_slot_bytes;                     // 1024-byte aligned
  const uint32_t out_stage_bytes = (uint32_t)sp.stage_out * kOutStageBytes;
  float* sAcc = reinterpret_cast<float*>(base_ptr + (size_t)R * ring_stage_bytes + (size_t)NV * v_slot_bytes +
                                         out_stage_bytes);
  auto RING_FULL = [&](int s) { return smem_u32(&bars[s]); };
  auto RING_FREE = [&](int s) { return smem_u32(&bars[kMaxStages + s]); };
  auto V_FULL = [&](int s) { return smem_u32(&bars[2 * kMaxStages + s]); };
  auto V_FREE = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 4 + s]); };
  auto S_READY = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 8 + s]); };
  auto P_READY = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 12 + s]); };
  auto P_FREE = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 16 + s]); };
  auto O_READY = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 20 + s]); };
  auto TMEM_FREE = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 24 + s]); };
  const int nS = p.n_sbuf, nO = p.n_obuf;
  const int sMask = nS - 1, oMask = nO - 1, sShift = nS == 4 ? 2 : 1, oShift = nO == 4 ? 2 : 1;
  auto sIdx = [&](int k) { return k & sMask; };
  auto oIdx = [&](int k) { return k & oMask; };
  auto colS = [&](int k) { return (uint32_t)((k & sMask) * kTpad); };
  auto colO = [&](int k) { return (uint32_t)(nS * kTpad + (k & oMask) * p.npv); };
  auto sPar = [&](int k) { return (uint32_t)(k >> sShift) & 1u; };
  auto oPar = [&](int k) { return (uint32_t)(k >> oShift) & 1u; };
  const int my_units = (p.units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int n_items = my_units * p.H;

  if (tid == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_k); prefetch_tmap(&map_v);
    if (sp.stage_out) prefetch_tmap(&map_o);
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(RING_FULL(s), 1); mbar_init(RING_FREE(s), 1); }
    for (int s = 0; s < 4; ++s) {
      mbar_init(V_FULL(s), 1);
      mbar_init(V_FREE(s), 1);
      mbar_init(S_READY(s), 1);
      mbar_init(P_READY(s), kGroupThreads);
      mbar_init(P_FREE(s), 1);
      mbar_init(O_READY(s), 1);
      mbar_init(TMEM_FREE(s), kGroupThreads);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const int fmt = p.bf16 ? 1 : 0;
  const int ksteps = (p.d + 15) >> 4;
  const bool bf16 = p.bf16 != 0;

  if (warp >= 12) {
    reg_dealloc<56>();
    if (warp == 12) {
      // ------------------------------------------------------------------------------------- TMA producer
      ItemIter it;
      it.init(p);
      int rs = 0, ring_fills = 0, vs = 0;
      uint32_t rpar = 0, vpar = 0;
      for (int k = 0; k < n_items; ++k) {
        for (int blk = 0; blk < p.nblk; ++blk) {
          if (ring_fills >= R) mbar_wait(RING_FREE(rs), rpar ^ 1u);
          if (elect_one()) {
            const uint32_t sQ = base + rs * ring_stage_bytes, sK = sQ + kQBlockBytes;
            mbar_expect_tx(RING_FULL(rs), ring_stage_bytes);
            tma_load_4d(sQ, &map_q, RING_FULL(rs), blk * kBlockCols, it.h, it.tile * kM, it.b);
            tma_load_4d(sK, &map_k, RING_FULL(rs), blk * kBlockCols, it.h, 0, it.b);
          }
          __syncwarp();
          ++ring_fills;
          if (++rs == R) { rs = 0; rpar ^= 1u; }
        }
        if (k >= NV) mbar_wait(V_FREE(vs), vpar ^ 1u);
        if (elect_one()) {
          const uint32_t sV = v_base + vs * v_slot_bytes;
          mbar_expect_tx(V_FULL(vs), v_slot_bytes);
          for (int blk = 0; blk < p.nblk; ++blk)
            tma_load_4d(sV + blk * kKVBlockBytes, &map_v, V_FULL(vs), blk * kBlockCols, it.h, 0, it.b);
        }
        __syncwarp();
        if (++vs == NV) { vs = 0; vpar ^= 1u; }
        it.next(p);
      }
    } else if (warp == 13) {
      // ------------------------------------------------------------- MMA issuer 1: S += Q_blk K_blk^T per block
      const uint32_t idesc_qk = make_idesc(fmt, 0, kTpad, kM);
      const uint64_t dQ0 = smem_desc_sw128(base, 16, 1024), dK0 = smem_desc_sw128(base + kQBlockBytes, 16, 1024);
      int rs = 0;
      uint32_t rpar = 0;
      for (int k = 0; k < n_items; ++k) {
        if (k >= nS) mbar_wait(P_FREE(sIdx(k)), sPar(k) ^ 1u);
        for (int blk = 0; blk < p.nblk; ++blk) {
          mbar_wait(RING_FULL(rs), rpar);
          tc_fence_after();
          if (elect_one()) {
            const int nks = min(4, ksteps - 4 * blk);
            const uint32_t roff = (uint32_t)rs * ring_stage_bytes;
            for (int ks = 0; ks < nks; ++ks)
              mma_ss(tmem + colS(k), desc_advance(dQ0, roff + ks * 32u), desc_advance(dK0, roff + ks * 32u), idesc_qk,
                     (blk > 0 || ks > 0) ? 1u : 0u);
            tc_commit(RING_FREE(rs));
            if (blk == p.nblk - 1) tc_commit(S_READY(sIdx(k)));
          }
          __syncwarp();
          if (++rs == R) { rs = 0; rpar ^= 1u; }
        }
      }
    } else if (warp == 14) {
      // ------------------------------------------------------------------------------ MMA issuer 2: O = P V
      const uint32_t idesc_pv = make_idesc(fmt, 1, p.npv, kM);
      const uint64_t dV0 = smem_desc_sw128(v_base, kKVBlockBytes, 1024);
      int vs = 0;
      uint32_t vpar = 0;
      for (int k = 0; k < n_items; ++k) {
        mbar_wait(P_READY(sIdx(k)), sPar(k));
        if (k >= nO) mbar_wait(TMEM_FREE(oIdx(k)), oPar(k) ^ 1u);
        mbar_wait(V_FULL(vs), vpar);
        tc_fence_after();
        if (elect_one()) {
          issue_tmem_gemm(tmem + colO(k), tmem + colS(k), desc_advance(dV0, (uint32_t)vs * v_slot_bytes), kTpad / 16,
                          idesc_pv, false);
          tc_commit(O_READY(oIdx(k)));
          tc_commit(P_FREE(sIdx(k)));
          tc_commit(V_FREE(vs));
        }
        __syncwarp();
        if (++vs == NV) { vs = 0; vpar ^= 1u; }
      }
    }
  } else if (warp < 4) {
    reg_dealloc<88>();
    // ---------------------------------------------------------------------------------------- epilogue
    const int r = (warp << 5) + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
    ItemIter it;
    it.init(p);
    for (int k = 0; k < n_items; ++k) {
      const int ob = oIdx(k);
      mbar_wait(O_READY(ob), oPar(k));
      tc_fence_after();
      const float inv = s_inv[k & 7][r];
      const int row = it.tile * kM + r;
      uint8_t* orow = reinterpret_cast<uint8_t*>(p.o) + (((int64_t)it.b * p.N + row) * p.H + it.h) * (int64_t)p.d * 2;
      int c_first = 0;
      if (sp.stage_out) {
        // The leading 64-channel blocks leave through the TMA: registers -> this warp's 4 KB staging tile per block (the
        // TMA's 128-byte swizzle, conflict-free) -> one cp.async.bulk.tensor store of 32 rows per block.  The per-thread
        // 16-byte stores they replace have their lanes a row apart: 32 LSU wavefronts per instruction, and the epilogue
        // warpgroup was the busiest role of this kernel (profiles/: 79 % of its samples outside the O_READY wait, the
        // second MMA issuer waiting 35 % of its time for it to free an O buffer).  Lane 0 issues every store of its warp
        // and is the one that waits for the previous item's stores to have READ the tiles before they are overwritten
        // (bulk groups are per thread).  Columns past head_dim in a block's tile are never written and never stored (the
        // TMA clips the box at the tensor's extent).
        const int chunks = p.npv / 16;
        for (int blk = 0; blk < sp.stage_out; ++blk) {
#pragma unroll
          for (int half = 0; half < 2; ++half) {        // 32 columns per TMEM round trip (88 registers per thread here)
            const int cb = blk * 4 + half * 2;
            if (cb >= chunks) break;
            float ov[32];
            tmem_ld16(lane_base + colO(k) + cb * 16, ov);
            if (cb + 1 < chunks) tmem_ld16(lane_base + colO(k) + (cb + 1) * 16, ov + 16);
            tmem_ld_wait();
            if (blk == 0 && half == 0 && k > 0) {
              if (lane == 0) bulk_wait_read0();
              __syncwarp();
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              if (cb + u >= chunks) break;
              uint32_t w[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) w[i] = pack16(ov[u * 16 + 2 * i] * inv, ov[u * 16 + 2 * i + 1] * inv, bf16);
              st_swizzled_32B(out_stage + (uint32_t)blk * kOutStageBytes, r, (half * 2 + u) * 2, w);
            }
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          for (int blk = 0; blk < sp.stage_out && blk * 4 < chunks; ++blk)
            tma_store_4d(&map_o, out_stage + (uint32_t)blk * kOutStageBytes + (uint32_t)warp * 4096u, blk * kBlockCols, it.h,
                         it.tile * kM + warp * 32, it.b);
          bulk_commit_group();
        }
        c_first = 4 * sp.stage_out;
      }
      for (int c0 = c_first; c0 < p.npv / 16; c0 += 2) {
        float ov[32];
        tmem_ld16(lane_base + colO(k) + c0 * 16, ov);
        if (c0 + 1 < p.npv / 16) tmem_ld16(lane_base + colO(k) + (c0 + 1) * 16, ov + 16);
        tmem_ld_wait();
        if (row < p.N) {
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            if (c0 + u >= p.npv / 16) break;
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = pack16(ov[u * 16 + 2 * i] * inv, ov[u * 16 + 2 * i + 1] * inv, bf16);
            const int col = (c0 + u) * 16;
            if (col < p.d) *reinterpret_cast<uint4*>(orow + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
            if (col + 8 < p.d) *reinterpret_cast<uint4*>(orow + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(TMEM_FREE(ob));
      it.next(p);
    }
    if (sp.stage_out && lane == 0) bulk_wait_all0();      // the last stores have left before the CTA exits
    __syncwarp();
  } else {
    reg_alloc<184>();
    // ------------------------------------------------------------------------------------ softmax groups
    const int g = (warp - 4) >> 2;
    const int r = ((warp & 3) << 5) + lane;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float sc = p.scale * 1.4426950408889634f;
    float pacc[kTpad];
#pragma unroll
    for (int j = 0; j < kTpad; ++j) pacc[j] = 0.f;
    int k = 0;
    for (int u = 0; u < my_units; ++u) {
      const int unit = blockIdx.x + u * gridDim.x;
      const int b = unit / p.tiles, tile = unit - b * p.tiles;
      const int row = tile * kM + r;
      for (int h = 0; h < p.H; ++h, ++k) {
        if ((k & 1) != g) continue;
        const uint32_t lane_addr = lane_base + colS(k);
        mbar_wait(S_READY(sIdx(k)), sPar(k));
        tc_fence_after();
        float s[kTpad];
#pragma unroll
        for (int cc = 0; cc < kTpad / 16; ++cc) tmem_ld16(lane_addr + cc * 16, s + cc * 16);
        tmem_ld_wait();
        float m, sum;
        row_softmax_ilp(s, p.T, sc, m, sum);
#pragma unroll
        for (int cc = 0; cc < kTpad / 16; ++cc) {
          uint32_t packed[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) packed[i] = pack16(s[cc * 16 + 2 * i], s[cc * 16 + 2 * i + 1], bf16);
          tmem_st8(lane_addr + cc * 8, packed);
        }
        const float inv = __fdividef(1.f, sum);
        s_inv[k & 7][r] = inv;
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(P_READY(sIdx(k)));
#pragma unroll
        for (int j = 0; j < kTpad; ++j) pacc[j] = fmaf(s[j], inv, pacc[j]);
        if (row < p.N)
          p.lse[((int64_t)b * p.H + h) * p.N + row] = (m * sc + lg2_approx(sum)) * 0.6931471805599453f;
      }
      // ---- end of the (b, tile) unit: combine the two groups' head sums and write the accumulator rows
      if (g == 1) {
#pragma unroll
        for (int j = 0; j < kTpad; ++j) sAcc[r * kAccStride + j] = pacc[j];
      }
      named_bar_sync(1, 2 * kGroupThreads);
      if (g == 0) {
#pragma unroll
        for (int j = 0; j < kTpad; ++j) sAcc[r * kAccStride + j] += pacc[j];
      }
      named_bar_sync(2, 2 * kGroupThreads);
      for (int i = warp - 4; i < kM; i += 8) {
        const int gr = tile * kM + i;
        if (gr >= p.N) break;
#pragma unroll
        for (int kk = 0; kk < 3; ++kk) {
          const int j = lane + 32 * kk;
          if (j < p.T) p.acc[((int64_t)b * p.N + gr) * p.T + j] = sAcc[i * kAccStride + j];
        }
      }
      named_bar_sync(3, 2 * kGroupThreads);
#pragma unroll
      for (int j = 0; j < kTpad; ++j) pacc[j] = 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512u);
}

// ============================================================================================== K2 (backward)
//   S  = Q K^T, dP = dO V^T                two K-major GEMMs into two TMEM regions
//   P  = exp(scale S - lse);  dP += d_acc[row]  (the attention-map gradient injected by the guidance tail)
//   dS = P o (dP - rowsum(P o dP)) * scale   -> packed 16-bit back into TMEM (A operand)
//   dQ = dS K                               K is the MN-major B operand (same tile the first GEMM read K-major)
// autograd of reference utils/ptp_utils.py:77-85 restricted to the latent path (dK / dV: SIMT variant).
constexpr int kColDP = 80;   // dP, later overwritten by dQ (dP is dead once it is in registers)

struct BwdParams {
  void* d_q;
  const float* lse;
  const float* d_acc;
  int64_t d_acc_bstride;
  int d_acc_rstride;   // elements between consecutive rows of the map gradient (>= T; 80 = 16-byte aligned rows)
  int B, H, N, T, d;
  int nblk, npv, tmem_cols, bf16;
  float scale;
};

__global__ void __launch_bounds__(kThreads)
cross_attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                         const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                         const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2];
  __shared__ uint32_t tmem_base_slot;

  const int tid = threadIdx.x, warp = uniform_warp_idx();
  const int h = blockIdx.x, tile = blockIdx.y, b = blockIdx.z;
  const int row0 = tile * kM, row = row0 + tid;

  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sQ = base;
  const uint32_t sG = sQ + p.nblk * kQBlockBytes;          // dO tile
  const uint32_t sK = sG + p.nblk * kQBlockBytes;
  const uint32_t sV = sK + p.nblk * kKVBlockBytes;
  const uint32_t bar_load = smem_u32(&bars[0]), bar_mma = smem_u32(&bars[1]);

  if (tid == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_do); prefetch_tmap(&map_k); prefetch_tmap(&map_v);
    mbar_init(bar_load, 1);
    mbar_init(bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);

  const int fmt = p.bf16 ? 1 : 0;
  const uint32_t idesc_nt = make_idesc(fmt, 0, kTpad, kM);
  const uint32_t idesc_dq = make_idesc(fmt, 1, p.npv, kM);
  const int ksteps = (p.d + 15) >> 4;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(bar_load, (uint32_t)p.nblk * 2u * (kQBlockBytes + kKVBlockBytes));
      for (int blk = 0; blk < p.nblk; ++blk) {
        tma_load_4d(sQ + blk * kQBlockBytes, &map_q, bar_load, blk * kBlockCols, h, row0, b);
        tma_load_4d(sK + blk * kKVBlockBytes, &map_k, bar_load, blk * kBlockCols, h, 0, b);
        tma_load_4d(sG + blk * kQBlockBytes, &map_do, bar_load, blk * kBlockCols, h, row0, b);
        tma_load_4d(sV + blk * kKVBlockBytes, &map_v, bar_load, blk * kBlockCols, h, 0, b);
      }
    }
    mbar_wait(bar_load, 0);
    tc_fence_after();
    if (elect_one()) {
      issue_kmajor_gemm(tmem + kColS, smem_desc_sw128(sQ, 16, 1024), kQBlockBytes, smem_desc_sw128(sK, 16, 1024),
                        kKVBlockBytes, ksteps, idesc_nt);
      issue_kmajor_gemm(tmem + kColDP, smem_desc_sw128(sG, 16, 1024), kQBlockBytes, smem_desc_sw128(sV, 16, 1024),
                        kKVBlockBytes, ksteps, idesc_nt);
      tc_commit(bar_mma);
    }
    __syncwarp();
  }
  mbar_wait(bar_mma, 0);
  tc_fence_after();

  float s[kTpad], dp[kTpad];
#pragma unroll
  for (int c = 0; c < kTpad / 16; ++c) {
    tmem_ld16(lane_addr + kColS + c * 16, s + c * 16);
    tmem_ld16(lane_addr + kColDP + c * 16, dp + c * 16);
  }
  tmem_ld_wait();
  const bool live = row < p.N;
  const float sc = p.scale * 1.4426950408889634f;
  const float l2 = live ? p.lse[((int64_t)b * p.H + h) * p.N + row] * 1.4426950408889634f : 0.f;
  const float* dacc = (p.d_acc != nullptr && live)
                          ? p.d_acc + (int64_t)b * p.d_acc_bstride + (int64_t)row * p.d_acc_rstride : nullptr;
  if (dacc != nullptr) {
    if ((p.d_acc_rstride & 3) == 0) {            // 16-byte aligned rows (the tail kernel pads them to 80 floats)
#pragma unroll
      for (int j = 0; j < kTpad; j += 4) {
        if (j + 3 < p.d_acc_rstride) {
          const float4 v4 = __ldg(reinterpret_cast<const float4*>(dacc + j));
          dp[j] += v4.x; dp[j + 1] += v4.y; dp[j + 2] += v4.z; dp[j + 3] += v4.w;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < kTpad; ++j)
        if (j < p.T) dp[j] += __ldg(dacc + j);
    }
  }
  float dsum = 0.f;
#pragma unroll
  for (int j = 0; j < kTpad; ++j) {
    const bool ok = live && j < p.T;
    const float pr = ok ? ex2_approx(fmaf(s[j], sc, -l2)) : 0.f;
    const float g = ok ? dp[j] : 0.f;
    s[j] = pr;
    dp[j] = g;
    dsum = fmaf(pr, g, dsum);
  }
  uint32_t packed[kTpad / 2];
#pragma unroll
  for (int j = 0; j < kTpad; j += 2)
    packed[j >> 1] = pack16(s[j] * (dp[j] - dsum) * p.scale, s[j + 1] * (dp[j + 1] - dsum) * p.scale, p.bf16 != 0);
#pragma unroll
  for (int c = 0; c < kTpad / 16; ++c) tmem_st8(lane_addr + kColP + c * 8, packed + c * 8);
  tmem_st_wait();
  tc_fence_before();
  __syncthreads();

  if (warp == 0) {
    tc_fence_after();
    if (elect_one()) {
      issue_tmem_gemm(tmem + kColDP, tmem + kColP, smem_desc_sw128(sK, kKVBlockBytes, 1024), kTpad / 16, idesc_dq, false);
      tc_commit(bar_mma);
    }
    __syncwarp();
  }
  mbar_wait(bar_mma, 1);
  tc_fence_after();

  uint8_t* grow = reinterpret_cast<uint8_t*>(p.d_q) + (((int64_t)b * p.N + row) * p.H + h) * (int64_t)p.d * 2;
  for (int c = 0; c < p.npv / 16; ++c) {
    float ov[16];
    tmem_ld16(lane_addr + kColDP + c * 16, ov);
    tmem_ld_wait();
    if (live) {
      uint32_t w[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) w[i] = pack16(ov[2 * i], ov[2 * i + 1], p.bf16 != 0);
      const int col = c * 16;
      if (col < p.d) *reinterpret_cast<uint4*>(grow + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
      if (col + 8 < p.d) *reinterpret_cast<uint4*>(grow + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, (uint32_t)p.tmem_cols);
}

// =================================================================================== K2, persistent STREAMING kernel
// One persistent CTA per SM with the warpgroup roles of the pipelined forward; the work items are the B * tiles row
// tiles of one head, split into contiguous ranges over teams of H CTAs (the forward's flat split).  Per item the first
// MMA warp issues S = Q K^T and dP = dO V^T into two TMEM regions, a compute group turns them into dS (16-bit, written
// over S), the second MMA warp issues dQ = dS K (K as the MN-major B operand) and the epilogue warpgroup converts dQ.
// What the shared memory holds is chosen so that the producer never waits for an epilogue (a ring of whole items --
// Q, dO, K, V of one 128-row tile: 104 KB per stage at d = 80, 156 KB at d = 160 -- left the SM with too few bytes in
// flight: DRAM 25-34 %, issue slots 12-19 %, tensor pipe 8-9 %, profiles/r02_ncu_summary.json):
//   * K and V of the current (batch element, head) live in two dedicated slots (the next element's K/V are fetched
//     into the other slot while the current one is in use); a CTA's items are consecutive row tiles of one head, so
//     they change rarely;
//   * the ring holds 64-channel BLOCKS of Q and dO (32 KB per stage: 4 stages at d = 80, 3 at d = 160).  S and dP
//     are accumulated over the blocks as they arrive, and a stage is released by the tcgen05.commit that follows
//     ITS OWN k-steps -- the producer streams Q / dO at HBM rate instead of waiting for epilogues;
//   * dQ rows leave from registers.
// TMEM: three stages of 160 columns (S | dP, dQ over dP) when npv <= 80, else two stages of 256 columns, so a compute
// group finds the GEMM outputs of its next item ready when it finishes one.  S and dP of item k overwrite the columns
// of dS(k - nT), and of dQ(k - nT) when dQ lies over dP: the first MMA warp waits for that item's dQ GEMM (DQ_READY)
// and, in the aliased case, for its epilogue (TMEM_FREE).
struct BwdPipeParams {
  void* d_q;
  const float* lse;
  const float* d_acc;
  int64_t d_acc_bstride;
  int d_acc_rstride;
  int B, H, N, T, d;
  int nblk, npv, bf16;
  int tiles, units;
  float scale;
  // col_dq and tstages are read together: at an 8-byte aligned offset they come in with one 64-bit constant load
  int col_dq;          // TMEM column of dQ inside a stage: 160 (own columns) or 80 (over dP)
  int tstages;         // TMEM stages: 3 (160 columns each, dQ over dP) when npv <= 80, else 2 (256 columns each)
};
struct BwdStreamParams {
  BwdPipeParams b;
  int ring_stages;   // 2 .. kMaxStages
  int g_slots;       // 0: the map-gradient rows are read with per-thread loads; 1: TMA-staged 128-row tiles (see below)
  int g_batched;     // 1: the map gradient has a batch stride (coordinate b), 0: one (N, rstride) matrix for every b
};

// The injected map gradient (round 2, second pass).  A compute thread needs ITS row of d_abar (80 floats): read with
// per-thread 128-bit loads, every load instruction of a warp touches 32 different 128-byte lines (rows are 320 bytes
// apart), i.e. 32 L1 tag cycles per instruction, 20 instructions per thread, 8 warps: ~1.2 us of LSU time per item --
// measured: d = 80, B = 256: 351 us with the map gradient, 214 us without.  With `g_slots` the otherwise idle fourth
// warp of the producer warpgroup streams the item's 128 x 80 fp32 tile into shared memory with three TMA boxes
// (32 + 32 + 16 columns x 128 rows, 128- / 64-byte swizzle: a thread reading its own row chunk by chunk is
// bank-conflict free), and the compute threads pick their row up with 20 shared-memory loads.
constexpr uint32_t kGPieceBytes = kM * 128;                  // 32 fp32 columns x 128 rows
constexpr uint32_t kGSlotBytes = 2 * kGPieceBytes + kM * 64; // columns 0..31 | 32..63 | 64..79 (64-byte rows)

template <bool kGStaged>
__global__ void __launch_bounds__(kPipeThreads, 1)
cross_attn_bwd_tc_stream_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                                const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                                const __grid_constant__ CUtensorMap map_g, const __grid_constant__ CUtensorMap map_g16,
                                const BwdStreamParams sp) {
  const BwdPipeParams& p = sp.b;
  extern __shared__ uint8_t smem_raw[];
  // ring_full[6], ring_free[6], kv_full[2], kv_free[2], then sd_ready / ds_ready / dq_ready / tmem_free x 3,
  // g_full[2] (one per compute group: a waiter must see every phase of its barrier), g_free
  __shared__ __align__(8) uint64_t bars[31];
  __shared__ uint32_t tmem_base_slot;

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t kv_half = (uint32_t)p.nblk * kKVBlockBytes;       // K (or V) of one head: nblk blocks
  const uint32_t kv_slot_bytes = 2u * kv_half;
  const uint32_t ring_base = base + 2u * kv_slot_bytes;
  constexpr uint32_t ring_stage_bytes = 2u * kQBlockBytes;         // one block of Q + one block of dO
  const int R = sp.ring_stages;
  auto RING_FULL = [&](int s) { return smem_u32(&bars[s]); };
  auto RING_FREE = [&](int s) { return smem_u32(&bars[kMaxStages + s]); };
  auto KV_FULL = [&](int s) { return smem_u32(&bars[2 * kMaxStages + s]); };
  auto KV_FREE = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 2 + s]); };
  auto SD_READY = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 4 + s]); };
  auto DS_READY = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 7 + s]); };
  auto DQ_READY = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 10 + s]); };
  auto TMEM_FREE = [&](int s) { return smem_u32(&bars[2 * kMaxStages + 13 + s]); };
  auto G_FULL = [&](int g) { return smem_u32(&bars[2 * kMaxStages + 16 + g]); };
  const uint32_t G_FREE = smem_u32(&bars[2 * kMaxStages + 18]);
  constexpr bool g_staged = kGStaged;       // (the host instantiates the staged kernel only with a map gradient)
  const uint32_t g_base = ring_base + (uint32_t)R * ring_stage_bytes;
  const int nT = p.tstages;
  const uint32_t stage_cols = nT == 3 ? 160u : (uint32_t)kStageCols;
  auto tIdx = [&](int k) { return nT == 3 ? k % 3 : (k & 1); };
  auto tPar = [&](int k) { return (uint32_t)(nT == 3 ? k / 3 : k >> 1) & 1u; };
  const int teams = gridDim.x / p.H, team = blockIdx.x / p.H, my_h = blockIdx.x % p.H;
  const int rt0 = (int)(((int64_t)p.units * team) / teams);
  const int n_items = (int)(((int64_t)p.units * (team + 1)) / teams) - rt0;
  const bool dq_aliased = p.col_dq == kColDP;

  if (tid == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_do); prefetch_tmap(&map_k); prefetch_tmap(&map_v);
    if (g_staged) { prefetch_tmap(&map_g); prefetch_tmap(&map_g16); }
    mbar_init(G_FULL(0), 1);
    mbar_init(G_FULL(1), 1);
    mbar_init(G_FREE, kGroupThreads);
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(RING_FULL(s), 1); mbar_init(RING_FREE(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(KV_FULL(s), 1); mbar_init(KV_FREE(s), 1); }
    for (int s = 0; s < 3; ++s) {
      mbar_init(SD_READY(s), 1);
      mbar_init(DS_READY(s), kGroupThreads);
      mbar_init(DQ_READY(s), 1);
      mbar_init(TMEM_FREE(s), kGroupThreads);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 512u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(tmem_base_slot);
  const int fmt = p.bf16 ? 1 : 0;
  const int ksteps = (p.d + 15) >> 4;
  const bool bf16 = p.bf16 != 0;

  auto batch_of = [&](int k) { return (rt0 + k) / p.tiles; };
  auto coords = [&](int k, int& b, int& h, int& tile) {
    const int rt = rt0 + k;
    h = my_h;
    b = rt / p.tiles;
    tile = rt - b * p.tiles;
  };

  if (warp >= 12) {
    reg_dealloc<56>();
    if (warp == 12) {
      // ------------------------------------------------------------------------------------------ TMA producer
      int cur_b = -1, kv_fills = 0, ring_fills = 0, rs = 0;
      uint32_t rpar = 0;
      for (int k = 0; k < n_items; ++k) {
        int b, h, tile;
        coords(k, b, h, tile);
        if (b != cur_b) {
          const int slot = kv_fills & 1;
          if (kv_fills >= 2) mbar_wait(KV_FREE(slot), (uint32_t)((kv_fills >> 1) - 1) & 1u);
          if (elect_one()) {
            const uint32_t sK = base + slot * kv_slot_bytes, sV = sK + kv_half;
            mbar_expect_tx(KV_FULL(slot), kv_slot_bytes);
            for (int blk = 0; blk < p.nblk; ++blk) {
              tma_load_4d(sK + blk * kKVBlockBytes, &map_k, KV_FULL(slot), blk * kBlockCols, h, 0, b);
              tma_load_4d(sV + blk * kKVBlockBytes, &map_v, KV_FULL(slot), blk * kBlockCols, h, 0, b);
            }
          }
          __syncwarp();
          ++kv_fills;
          cur_b = b;
        }
        for (int blk = 0; blk < p.nblk; ++blk) {
          if (ring_fills >= R) mbar_wait(RING_FREE(rs), rpar ^ 1u);
          if (elect_one()) {
            const uint32_t sQ = ring_base + rs * ring_stage_bytes, sG = sQ + kQBlockBytes;
            mbar_expect_tx(RING_FULL(rs), ring_stage_bytes);
            tma_load_4d(sQ, &map_q, RING_FULL(rs), blk * kBlockCols, h, tile * kM, b);
            tma_load_4d(sG, &map_do, RING_FULL(rs), blk * kBlockCols, h, tile * kM, b);
          }
          __syncwarp();
          ++ring_fills;
          if (++rs == R) { rs = 0; rpar ^= 1u; }
        }
      }
    } else if (warp == 13) {
      // --------------------------------------------- MMA issuer 1: S += Q_blk K_blk^T, dP += dO_blk V_blk^T per block
      const uint32_t idesc_nt = make_idesc(fmt, 0, kTpad, kM);
      const uint64_t dQ0 = smem_desc_sw128(ring_base, 16, 1024), dG0 = smem_desc_sw128(ring_base + kQBlockBytes, 16, 1024);
      const uint64_t dK0 = smem_desc_sw128(base, 16, 1024), dV0 = smem_desc_sw128(base + kv_half, 16, 1024);
      int cur_b = -1, kv_uses = 0, rs = 0;
      uint32_t rpar = 0;
      for (int k = 0; k < n_items; ++k) {
        const int ts = tIdx(k);
        const uint32_t ph = tPar(k);
        if (k >= nT) {
          mbar_wait(DQ_READY(ts), ph ^ 1u);
          if (dq_aliased) mbar_wait(TMEM_FREE(ts), ph ^ 1u);
        }
        const int b = batch_of(k);
        if (b != cur_b) {
          ++kv_uses;
          cur_b = b;
          mbar_wait(KV_FULL((kv_uses - 1) & 1), (uint32_t)((kv_uses - 1) >> 1) & 1u);
        }
        const uint32_t kv_off = (uint32_t)((kv_uses - 1) & 1) * kv_slot_bytes;
        for (int blk = 0; blk < p.nblk; ++blk) {
          mbar_wait(RING_FULL(rs), rpar);
          tc_fence_after();
          if (elect_one()) {
            const int nks = min(4, ksteps - 4 * blk);
            const uint32_t roff = (uint32_t)rs * ring_stage_bytes, koff = kv_off + (uint32_t)blk * kKVBlockBytes;
            for (int ks = 0; ks < nks; ++ks)
              mma_ss(tmem + ts * stage_cols + kColS, desc_advance(dQ0, roff + ks * 32u), desc_advance(dK0, koff + ks * 32u),
                     idesc_nt, (blk > 0 || ks > 0) ? 1u : 0u);
            for (int ks = 0; ks < nks; ++ks)
              mma_ss(tmem + ts * stage_cols + kColDP, desc_advance(dG0, roff + ks * 32u), desc_advance(dV0, koff + ks * 32u),
                     idesc_nt, (blk > 0 || ks > 0) ? 1u : 0u);
            tc_commit(RING_FREE(rs));            // this block's Q / dO are dead once these k-steps have retired
            if (blk == p.nblk - 1) tc_commit(SD_READY(ts));
          }
          __syncwarp();
          if (++rs == R) { rs = 0; rpar ^= 1u; }
        }
      }
    } else if (warp == 14) {
      // ------------------------------------------------------------------------------ MMA issuer 2: dQ = dS K
      const uint32_t idesc_dq = make_idesc(fmt, 1, p.npv, kM);
      const uint64_t dKmn0 = smem_desc_sw128(base, kKVBlockBytes, 1024);
      int cur_b = -1, kv_uses = 0;
      for (int k = 0; k < n_items; ++k) {
        const int ts = tIdx(k);
        const uint32_t ph = tPar(k);
        const int b = batch_of(k);
        if (b != cur_b) { ++kv_uses; cur_b = b; }
        const int slot = (kv_uses - 1) & 1;
        mbar_wait(DS_READY(ts), ph);
        if (!dq_aliased && k >= nT) mbar_wait(TMEM_FREE(ts), ph ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          issue_tmem_gemm(tmem + ts * stage_cols + p.col_dq, tmem + ts * stage_cols + kColP,
                          desc_advance(dKmn0, (uint32_t)slot * kv_slot_bytes), kTpad / 16, idesc_dq, false);
          tc_commit(DQ_READY(ts));
          // last item of this batch element on this CTA: its K/V slot may be refilled once this GEMM has retired
          if (k == n_items - 1 || batch_of(k + 1) != b) tc_commit(KV_FREE(slot));
        }
        __syncwarp();
      }
    } else if (g_staged && warp == 15) {
      // ------------------------------------------------- map-gradient producer: one 128 x 80 fp32 tile per item
      for (int k = 0; k < n_items; ++k) {
        int b, h, tile;
        coords(k, b, h, tile);
        if (k >= 1) mbar_wait(G_FREE, (uint32_t)(k - 1) & 1u);
        if (elect_one()) {
          mbar_expect_tx(G_FULL(k & 1), kGSlotBytes);
          const int gb = sp.g_batched ? b : 0;
          tma_load_3d(g_base, &map_g, G_FULL(k & 1), 0, tile * kM, gb);
          tma_load_3d(g_base + kGPieceBytes, &map_g, G_FULL(k & 1), 32, tile * kM, gb);
          tma_load_3d(g_base + 2 * kGPieceBytes, &map_g16, G_FULL(k & 1), 64, tile * kM, gb);
        }
        __syncwarp();
      }
    }
  } else if (warp < 4) {
    reg_dealloc<88>();
    // ---------------------------------------------------------------------------------------- epilogue (dQ)
    const int r = (warp << 5) + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
    for (int k = 0; k < n_items; ++k) {
      const int ts = tIdx(k);
      mbar_wait(DQ_READY(ts), tPar(k));
      tc_fence_after();
      int b, h, tile;
      coords(k, b, h, tile);
      const int row = tile * kM + r;
      uint8_t* grow = reinterpret_cast<uint8_t*>(p.d_q) + (((int64_t)b * p.N + row) * p.H + h) * (int64_t)p.d * 2;
      for (int c0 = 0; c0 < p.npv / 16; c0 += 2) {
        float ov[32];
        tmem_ld16(lane_base + ts * stage_cols + p.col_dq + c0 * 16, ov);
        if (c0 + 1 < p.npv / 16) tmem_ld16(lane_base + ts * stage_cols + p.col_dq + (c0 + 1) * 16, ov + 16);
        tmem_ld_wait();
        if (row < p.N) {
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            if (c0 + u >= p.npv / 16) break;
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = pack16(ov[u * 16 + 2 * i], ov[u * 16 + 2 * i + 1], bf16);
            const int col = (c0 + u) * 16;
            if (col < p.d) *reinterpret_cast<uint4*>(grow + col * 2) = make_uint4(w[0], w[1], w[2], w[3]);
            if (col + 8 < p.d) *reinterpret_cast<uint4*>(grow + col * 2 + 16) = make_uint4(w[4], w[5], w[6], w[7]);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(TMEM_FREE(ts));
    }
  } else {
    reg_alloc<184>();
    const int g = (warp - 4) >> 2;
    const int r = ((warp & 3) << 5) + lane;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float sc = p.scale * 1.4426950408889634f;
    for (int k = g; k < n_items; k += 2) {
      int b, h, tile;
      coords(k, b, h, tile);
      const int row = tile * kM + r;
      const bool live = row < p.N;
      const int ts = tIdx(k);
      const uint32_t ph = tPar(k);
      const uint32_t lane_addr = lane_base + ts * stage_cols;
      const float l2 = live ? __ldg(p.lse + ((int64_t)b * p.H + h) * p.N + row) * 1.4426950408889634f : 0.f;
      const float* dacc = (p.d_acc != nullptr && live)
                              ? p.d_acc + (int64_t)b * p.d_acc_bstride + (int64_t)row * p.d_acc_rstride : nullptr;
      // the row of the injected map gradient is fetched BEFORE waiting for the GEMMs (it is an L2 hit, shared by all
      // heads and batch elements, but 20 row-strided 16-byte loads per thread are ~0.5 us of exposed latency otherwise);
      // its registers are dead again before the scores are loaded
      float dp[kTpad];
      const bool vec_acc = (p.d_acc_rstride & 3) == 0;
      if constexpr (g_staged) {
        // this thread's row of the TMA-staged tile.  32-column pieces (128-byte rows, 128-byte swizzle): chunk c of
        // row r sits at chunk c ^ (r & 7); 16-column piece (64-byte rows, 64-byte swizzle): at chunk c ^ ((r >> 1) & 3).
        mbar_wait(G_FULL(g), (uint32_t)(k >> 1) & 1u);
        const uint32_t grow = g_base + (uint32_t)r * 128u;
#pragma unroll
        for (int j = 0; j < 64; j += 4) {
          const uint32_t a = grow + (uint32_t)(j >> 5) * kGPieceBytes + ((uint32_t)(((j >> 2) & 7) ^ (r & 7)) << 4);
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                       : "=f"(dp[j]), "=f"(dp[j + 1]), "=f"(dp[j + 2]), "=f"(dp[j + 3]) : "r"(a) : "memory");
        }
#pragma unroll
        for (int j = 64; j < kTpad; j += 4) {
          const uint32_t a = g_base + 2 * kGPieceBytes + (uint32_t)r * 64u +
                             ((uint32_t)(((j - 64) >> 2) ^ ((r >> 1) & 3)) << 4);
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                       : "=f"(dp[j]), "=f"(dp[j + 1]), "=f"(dp[j + 2]), "=f"(dp[j + 3]) : "r"(a) : "memory");
        }
        mbar_arrive(G_FREE);                  // (release: the loads above are performed before the arrival)
      } else if (dacc != nullptr) {
        if (vec_acc) {
#pragma unroll
          for (int j = 0; j < kTpad; j += 4) {
            float4 v4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j + 3 < p.d_acc_rstride) v4 = __ldg(reinterpret_cast<const float4*>(dacc + j));
            dp[j] = v4.x; dp[j + 1] = v4.y; dp[j + 2] = v4.z; dp[j + 3] = v4.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < kTpad; ++j) dp[j] = j < p.T ? __ldg(dacc + j) : 0.f;
        }
      } else {
#pragma unroll
        for (int j = 0; j < kTpad; ++j) dp[j] = 0.f;
      }
      mbar_wait(SD_READY(ts), ph);
      tc_fence_after();
      float s[kTpad];
#pragma unroll
      for (int cc = 0; cc < kTpad / 16; ++cc) {
        tmem_ld16(lane_addr + kColDP + cc * 16, s + cc * 16);      // dP through the registers the scores will use
      }
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < kTpad; ++j) dp[j] += s[j];
#pragma unroll
      for (int cc = 0; cc < kTpad / 16; ++cc) tmem_ld16(lane_addr + kColS + cc * 16, s + cc * 16);
      tmem_ld_wait();
      float d4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < kTpad; ++j) {
        const bool ok = live && (j < kTpad - 16 || j < p.T);
        const float pr = ok ? ex2_approx(fmaf(s[j], sc, -l2)) : 0.f;
        s[j] = pr;
        d4[j & 3] = fmaf(pr, dp[j], d4[j & 3]);
      }
      const float dsum = (d4[0] + d4[1]) + (d4[2] + d4[3]);
#pragma unroll
      for (int cc = 0; cc < kTpad / 16; ++cc) {
        uint32_t packed[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int j = cc * 16 + 2 * i;
          packed[i] = pack16(s[j] * (dp[j] - dsum) * p.scale, s[j + 1] * (dp[j + 1] - dsum) * p.scale, bf16);
        }
        tmem_st8(lane_addr + kColP + cc * 8, packed);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(DS_READY(ts));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512u);
}

// --------------------------------------------------------------------------------------------------- host side
static int heads_per_cta_for(int H) {
  for (int hpc = 1; hpc <= H; ++hpc)
    if (H % hpc == 0 && H / hpc <= 8) return hpc;
  return H;
}

static int fwd_pipe(const CUtensorMap& mq, const CUtensorMap& mk, const CUtensorMap& mv, const FwdParams& f, int dtype,
                    cudaStream_t st) {
  PipeParams p;
  p.o = f.o; p.lse = f.lse; p.acc = f.acc;
  p.B = f.B; p.H = f.H; p.N = f.N; p.T = f.T; p.d = f.d;
  p.nblk = f.nblk; p.npv = f.npv; p.bf16 = f.bf16; p.scale = f.scale;
  p.tiles = (f.N + kM - 1) / kM;
  p.grouped = f.acc != nullptr ? 1 : 0;
  p.units = f.B * p.tiles;
  p.n_sbuf = (4 * kTpad + 2 * p.npv <= 512) ? 4 : 2;
  p.n_obuf = (512 - p.n_sbuf * kTpad) / p.npv >= 4 ? 4 : 2;
  // maps kept and more than one 64-channel block: the streaming variant
  if (p.grouped && p.nblk >= 2) {
    FwdStreamParams sp;
    sp.b = p;
    const size_t acc_bytes = (size_t)kM * kAccStride * sizeof(float), ring = (size_t)kQBlockBytes + kKVBlockBytes;
    const size_t vslot = (size_t)p.nblk * kKVBlockBytes;
    // O staging tiles (TMA stores instead of row-strided 16-byte stores, see the epilogue) are paid for with the third
    // V slot where needed, never with a ring stage.  Measured on B200 (profiles/r02d_k1_stage_ab.txt): d = 80
    // 210 -> 167-171 us with one staged block, d = 160 191 -> 170 us with one staged block and two V slots, 158 us with two.
    // dynamic + static shared memory (barriers, s_inv: 4.4 KB) must stay within the 227 KB a CTA can opt in to
    auto stages_for = [&](int blocks, int v_slots) {
      for (int n = kMaxStages; n >= 2; --n)
        if (1024 + acc_bytes + (size_t)blocks * kOutStageBytes + v_slots * vslot + n * ring <= 222 * 1024) return n;
      return 0;
    };
    const int without = stages_for(0, 3);
    sp.stage_out = 0;
    sp.v_slots = 3;
    // first fit that keeps the ring depth: two staged blocks only when two FULL 64-channel blocks exist (staging the
    // 16-channel tail of d = 80 at the price of a V slot measured slower: 176 vs 171 us)
    const int full_blocks = p.d / kBlockCols;
    const int cand[4][2] = {{2, 3}, {2, 2}, {1, 3}, {1, 2}};
    for (int i = 0; i < 4; ++i) {
      if (cand[i][0] == 2 && full_blocks < 2) continue;
      if (stages_for(cand[i][0], cand[i][1]) == without) {
        sp.stage_out = cand[i][0];
        sp.v_slots = cand[i][1];
        break;
      }
    }
    sp.ring_stages = stages_for(sp.stage_out, sp.v_slots);
    if (sp.ring_stages >= p.nblk) {
      const size_t smem_s = 1024 + acc_bytes + (size_t)sp.stage_out * kOutStageBytes + sp.v_slots * vslot + sp.ring_stages * ring;
      cudaError_t es2 = ensure_smem(reinterpret_cast<const void*>(cross_attn_fwd_tc_stream_kernel), 6, smem_s);
      if (es2 != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(es2));
      CUtensorMap mo_s;
      int rc_s;
      if ((rc_s = make_map(&mo_s, f.o, dtype, f.B, f.N, f.H, f.d, 32)) != GA_OK) return rc_s;   // one store per epilogue warp
      const int grid_s = p.units < sm_count() ? p.units : sm_count();
      cross_attn_fwd_tc_stream_kernel<<<grid_s, kPipeThreads, smem_s, st>>>(mq, mk, mv, mo_s, sp);
      return check_launch("cross_attn_fwd_tc_stream");
    }
  }
  CUtensorMap mo;
  int rc;
  if ((rc = make_map(&mo, f.o, dtype, f.B, f.N, f.H, f.d, 32)) != GA_OK) return rc;   // one store per epilogue warp
  const size_t kv = (size_t)2 * p.nblk * kKVBlockBytes;
  const size_t stage = (size_t)p.nblk * kQBlockBytes + (p.grouped ? kv : 0);            // flat: Q-only stages
  const size_t extra = 1024 + (p.grouped ? (size_t)kM * kAccStride * sizeof(float) : 2 * kv);   // flat: two K/V slots
  p.smem_stages = 1;
  for (int n = (p.grouped ? kMaxStages : kFwdStages); n >= 2; --n)
    if (n * stage + extra <= 224 * 1024) { p.smem_stages = n; break; }
  const size_t smem = p.smem_stages * stage + extra;
  if (smem > 224 * 1024) return fail(GA_ERR_UNSUPPORTED, "tcgen05 pipelined cross-attention: %zu B of shared memory", smem);
  p.direct_store = p.smem_stages < 4 ? 1 : 0;
  cudaError_t e = ensure_smem(reinterpret_cast<const void*>(cross_attn_fwd_tc_pipe_kernel), 2, smem);
  if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  int grid;
  if (p.grouped) {
    grid = p.units < sm_count() ? p.units : sm_count();
  } else {                                   // teams of H CTAs, each team a contiguous range of row tiles
    if (f.H > sm_count()) return fail(GA_ERR_UNSUPPORTED, "pipelined cross-attention: %d heads", f.H);
    int teams = sm_count() / f.H;
    if (teams > p.units) teams = p.units;
    grid = teams * f.H;
  }
  cross_attn_fwd_tc_pipe_kernel<<<grid, kPipeThreads, smem, st>>>(mq, mk, mv, mo, p);
  return check_launch("cross_attn_fwd_tc_pipe");
}

bool supports_fwd(int dtype, int n_ctx, int head_dim, int heads, bool with_acc) {
  (void)heads; (void)with_acc;
  // the row softmax predicates only the last 16 of the 80 key columns on n_ctx: 65..80 keys (SD: 77)
  return (dtype == GA_F16 || dtype == GA_BF16) && n_ctx > kTpad - 16 && n_ctx <= kTpad &&
         head_dim % 8 == 0 && head_dim >= 8 && head_dim <= 256;
}
bool supports_bwd(int dtype, int n_ctx, int head_dim, int heads, bool with_dkv) {
  return !with_dkv && supports_fwd(dtype, n_ctx, head_dim, heads, false);
}

int fwd(const void* q, const void* k, const void* v, void* o, float* lse, float* acc, int B, int H, int N, int T, int d,
        float scale, int dtype, int force_variant, cudaStream_t st) {
  CUtensorMap mq, mk, mv;
  int rc;
  if ((rc = make_map(&mq, q, dtype, B, N, H, d, kM)) != GA_OK) return rc;
  if ((rc = make_map(&mk, k, dtype, B, T, H, d, kTpad)) != GA_OK) return rc;
  if ((rc = make_map(&mv, v, dtype, B, T, H, d, kTpad)) != GA_OK) return rc;

  FwdParams p;
  p.o = o; p.lse = lse; p.acc = acc;
  p.B = B; p.H = H; p.N = N; p.T = T; p.d = d;
  p.nblk = (d + kBlockCols - 1) / kBlockCols;
  p.npv = (d + 15) & ~15;
  p.heads_per_cta = acc != nullptr ? heads_per_cta_for(H) : 1;
  const int need_cols = kColO + p.npv;
  p.tmem_cols = need_cols <= 128 ? 128 : (need_cols <= 256 ? 256 : 512);
  p.bf16 = dtype == GA_BF16;
  p.scale = scale;

  // Variant choice: the persistent pipelined kernel needs enough work units to occupy the SMs (a unit is a (b, tile)
  // group of H heads when maps are kept, a single (b, h, tile) otherwise) and d <= 160 (two 256-column TMEM stages).
  {
    const int tiles = (N + kM - 1) / kM;
    const int units = acc != nullptr ? B * tiles : B * H * tiles;
    // Crossovers measured on B200 (profiles/r02_crossover_sweep_before.jsonl, r02_crossover_sweep.jsonl).  With maps a
    // persistent CTA streams the H heads of one (b, tile) unit back to back: ~17 us per unit at d = 80 and ~19-26 us
    // at d = 160 (streaming variant) however few units there are, while the single-shot cluster kernel costs ~9 us per
    // wave of ~8 units: the persistent kernel wins from ~24 units on (B = 3 at 32x32, B = 12 at 16x16) -- not from
    // sm_count / 2 = 74 as in round 1, which left the seed-batched launches (B = 8, 16) on the slow side.
    // (third pass, with the staged epilogue: 16 units already win when a batch element has more than one row tile --
    // B = 2 at 32x32, the CFG pass: 14.6 vs 17.4 us -- profiles/r02d_crossover_sweep.jsonl)
    const int min_units = acc != nullptr ? (tiles >= 2 ? 16 : 24) : 2 * sm_count();
    bool use_pipe = d <= 160 && units >= min_units;
    if (force_variant == 0) use_pipe = false;
    if (force_variant == 1) {
      if (d > 160) return fail(GA_ERR_UNSUPPORTED, "pipelined tcgen05 cross-attention needs head_dim <= 160");
      use_pipe = true;
    }
    if (use_pipe) return fwd_pipe(mq, mk, mv, p, dtype, st);
  }
  size_t smem = 1024 + (size_t)p.nblk * (kQBlockBytes + 2 * kKVBlockBytes);
  if (acc != nullptr) smem += (size_t)kM * kAccStride * sizeof(float);
  if (smem > 226 * 1024) return fail(GA_ERR_UNSUPPORTED, "tcgen05 cross-attention: %zu B of shared memory", smem);
  cudaError_t e = ensure_smem(reinterpret_cast<const void*>(cross_attn_fwd_tc_kernel), 0, smem);
  if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));

  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(H / p.heads_per_cta, (N + kM - 1) / kM, B);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = acc != nullptr ? H / p.heads_per_cta : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, cross_attn_fwd_tc_kernel, mq, mk, mv, p);
  if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cross_attn_fwd_tc launch: %s", cudaGetErrorString(e));
  return check_launch("cross_attn_fwd_tc");
}

int bwd(const void* q, const void* k, const void* v, const float* lse, const void* d_o, const float* d_acc,
        int64_t d_acc_bstride, int d_acc_rstride, void* d_q, int B, int H, int N, int T, int d, float scale, int dtype,
        int force_variant, cudaStream_t st) {
  CUtensorMap mq, mg, mk, mv;
  int rc;
  if ((rc = make_map(&mq, q, dtype, B, N, H, d, kM)) != GA_OK) return rc;
  if ((rc = make_map(&mg, d_o, dtype, B, N, H, d, kM)) != GA_OK) return rc;
  if ((rc = make_map(&mk, k, dtype, B, T, H, d, kTpad)) != GA_OK) return rc;
  if ((rc = make_map(&mv, v, dtype, B, T, H, d, kTpad)) != GA_OK) return rc;
  const int nblk = (d + kBlockCols - 1) / kBlockCols, npv = (d + 15) & ~15;
  const int tiles = (N + kM - 1) / kM, units = B * H * tiles;
  // crossover measured on B200 (profiles/r02b_crossover_sweep.jsonl): without a map gradient the persistent kernel wins
  // from ~2 items per SM; with one (TMA-staged tile vs per-thread row loads in the single-shot kernel) already at 256
  // items (N = 1024 d = 80: 10.9 vs 12.3 us, N = 256 d = 160: 15.0 vs 21.3 us), a tie at 128
  const int min_items = d_acc != nullptr ? (5 * sm_count()) / 4 : 2 * sm_count();
  bool use_pipe = d <= 160 && units >= min_items && H <= sm_count();
  if (force_variant == 0) use_pipe = false;
  if (force_variant == 1) {
    if (d > 160) return fail(GA_ERR_UNSUPPORTED, "pipelined tcgen05 cross-attention needs head_dim <= 160");
    use_pipe = true;
  }
  if (use_pipe) {
    // the streaming kernel -- K/V slots + a ring of Q/dO blocks -- measured faster than a ring of whole items at every
    // head dim (B200, profiles/r02_microbench_k2_stream.jsonl: d = 80: 386 vs 490 us, d = 160: 347 vs 419 us,
    // d = 40: 304 vs 320 us)
    BwdStreamParams sp;
    BwdPipeParams& p = sp.b;
    p.d_q = d_q; p.lse = lse; p.d_acc = d_acc; p.d_acc_bstride = d_acc_bstride; p.d_acc_rstride = d_acc_rstride;
    p.B = B; p.H = H; p.N = N; p.T = T; p.d = d;
    p.nblk = nblk; p.npv = npv; p.bf16 = dtype == GA_BF16; p.scale = scale;
    p.tiles = tiles; p.units = B * tiles;      // row tiles, split over teams of H CTAs
    p.tstages = npv <= kTpad ? 3 : 2;
    p.col_dq = p.tstages == 3 ? kColDP : ((2 * kTpad + npv <= kStageCols) ? 2 * kTpad : kColDP);
    const size_t kv = (size_t)2 * 2 * nblk * kKVBlockBytes, ring = (size_t)2 * kQBlockBytes;
    auto stages_for = [&](size_t extra) {
      for (int n = kMaxStages; n >= 2; --n)
        if (1024 + kv + extra + n * ring <= 226 * 1024) return n;
      return 0;
    };
    // TMA-staged map-gradient tile (40 KB) whenever the rows can be described to the TMA (16-byte aligned base and
    // strides, at most 80 columns) and two ring stages remain: d = 160 runs 242 us with two stages + the staged tile
    // vs 278 us with three stages + per-thread loads (B = 512, N = 256)
    sp.g_slots = 0;
    sp.g_batched = d_acc_bstride != 0 ? 1 : 0;
    CUtensorMap mgr = mq, mgr16 = mq;      // placeholders when the staged path is off (never dereferenced)
    const bool g_ok = d_acc != nullptr && (d_acc_rstride & 3) == 0 && d_acc_rstride <= kTpad && (d_acc_bstride & 3) == 0 &&
                      (reinterpret_cast<uintptr_t>(d_acc) & 15) == 0;
    if (g_ok && stages_for(kGSlotBytes) >= 2) {
      const int nb = sp.g_batched ? B : 1;
      const int64_t bs = sp.g_batched ? d_acc_bstride : (int64_t)N * d_acc_rstride;
      if ((rc = make_map_rows_f32(&mgr, d_acc, d_acc_rstride, N, nb, bs, 32, kM, CU_TENSOR_MAP_SWIZZLE_128B)) != GA_OK) return rc;
      if ((rc = make_map_rows_f32(&mgr16, d_acc, d_acc_rstride, N, nb, bs, 16, kM, CU_TENSOR_MAP_SWIZZLE_64B)) != GA_OK) return rc;
      sp.g_slots = 1;
    }
    const size_t g_bytes = sp.g_slots ? (size_t)kGSlotBytes : 0;
    sp.ring_stages = stages_for(g_bytes);
    // two stages fit for every head_dim <= 160: 1024 + 4 x 3 x 10240 + 2 x 32768 = 189 440 B
    if (sp.ring_stages < 2) return fail(GA_ERR_UNSUPPORTED, "streaming tcgen05 cross-attention backward: head_dim %d", d);
    const size_t smem_s = 1024 + kv + sp.ring_stages * ring + g_bytes;
    auto kern = sp.g_slots ? cross_attn_bwd_tc_stream_kernel<true> : cross_attn_bwd_tc_stream_kernel<false>;
    cudaError_t es2 = ensure_smem(reinterpret_cast<const void*>(kern), sp.g_slots ? 7 : 5, smem_s);
    if (es2 != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(es2));
    if (H > sm_count()) return fail(GA_ERR_UNSUPPORTED, "pipelined cross-attention backward: %d heads", H);
    int teams_s = sm_count() / H;
    if (teams_s > p.units) teams_s = p.units;
    kern<<<teams_s * H, kPipeThreads, smem_s, st>>>(mq, mg, mk, mv, mgr, mgr16, sp);
    return check_launch("cross_attn_bwd_tc_stream");
  }
  BwdParams p;
  p.d_q = d_q; p.lse = lse; p.d_acc = d_acc; p.d_acc_bstride = d_acc_bstride; p.d_acc_rstride = d_acc_rstride;
  p.B = B; p.H = H; p.N = N; p.T = T; p.d = d;
  p.nblk = nblk;
  p.npv = npv;
  p.tmem_cols = (kColDP + p.npv) <= 256 ? 256 : 512;
  p.bf16 = dtype == GA_BF16;
  p.scale = scale;
  const size_t smem = 1024 + (size_t)p.nblk * 2 * (kQBlockBytes + kKVBlockBytes);
  if (smem > 226 * 1024) return fail(GA_ERR_UNSUPPORTED, "tcgen05 cross-attention bwd: %zu B of shared memory", smem);
  cudaError_t e = ensure_smem(reinterpret_cast<const void*>(cross_attn_bwd_tc_kernel), 1, smem);
  if (e != cudaSuccess) return fail(GA_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  dim3 grid(H, (N + kM - 1) / kM, B);
  cross_attn_bwd_tc_kernel<<<grid, kThreads, smem, st>>>(mq, mg, mk, mv, p);
  return check_launch("cross_attn_bwd_tc");
}

}  // namespace tc
}  // namespace ga
