// tcgen05 / TMEM / TMA / mbarrier PTX wrappers and UMMA descriptor helpers shared by the tensor-core kernels
// (cross_attn_tc.cu, self_attn_tc.cu).  sm_100a only.
#pragma once
#include <cuda.h>
#include <stdint.h>

#include "ga_common.cuh"

namespace ga {
namespace tc {

constexpr uint32_t kSpinLimit = 1u << 24;
constexpr int kTpad = 80;       // cross-attention: keys padded to a multiple of 16 (UMMA N granularity at M = 128)

// ----------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (launch failure reported to the host) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  // not unrolled: nvcc otherwise expands every wait into 64 try_wait/branch pairs, and the five roles of the pipelined
  // kernels then thrash the instruction cache (stall_no_inst was 9 % of all samples)
#pragma unroll 1
  for (uint32_t i = 0; i < kSpinLimit; ++i)
    if (mbar_try_wait(bar, parity)) return;
  __trap();
}

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// Pull a tile into L2 without touching shared memory: lets a producer keep far more HBM requests in flight than its
// shared-memory ring has stages (the later cp.async.bulk.tensor of the same tile then hits L2).
__device__ __forceinline__ void tma_prefetch_l2_4d(const CUtensorMap* map, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
               ::"l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] . B[smem desc]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem desc]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors (cute/arch/mma_sm100_desc.hpp bit layout) -------------------------------------------------
// shared-memory matrix descriptor, 128-byte swizzle: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1
// [46,48) | layout_type=2 (SWIZZLE_128B) [61,64)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D fp32 [4,6)=1 | A fmt [7,10) | B fmt [10,13) | A major bit15 | B major bit16 | N>>3 [17,23)
// | M>>4 [24,29)      (fmt: 0 = f16, 1 = bf16; major: 0 = K, 1 = MN)
__host__ __device__ constexpr uint32_t make_idesc(int fmt, int b_mn_major, int n, int m) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ uint32_t pack16(float a, float b, bool bf16) {
  if (bf16) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- warp-uniform role helpers ----------------------------------------------------------------------------------
// The TMA-producer and MMA-issuer roles run as WHOLE warps in warp-uniform control flow and pick one lane with
// elect.sync for the asynchronous instructions.  A role entered through a divergent `lane == 0` branch makes the
// compiler wrap every UTCHMMA / UTMALDG in an ELECT / BRA.U.ANY loop and keep descriptors in vector registers
// (~13 SASS instructions per MMA): the single issuing thread then becomes the critical path of the whole CTA.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// warp-uniform non-blocking test (a completed phase stays completed, so "any lane saw it" is the right vote)
// (test_wait returns at once; try_wait may suspend the thread for an implementation-defined time when the phase is
// still pending, which would turn a poll over several barriers back into a blocking wait on the first one)
__device__ __forceinline__ bool mbar_test_uniform(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return __any_sync(0xffffffffu, (int)ok) != 0;
}
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
__device__ __forceinline__ uint32_t uniform_u32(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }

// start-address field of a shared-memory descriptor advanced by `bytes` (stays inside the 14-bit field: < 256 KB)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }

// D[tmem] = A . B^T with A and B K-major in 64-column blocks of 128-byte swizzled rows; one k-step = 16 columns =
// 32 bytes inside the row, four k-steps per block.
__device__ __forceinline__ void issue_kmajor_gemm(uint32_t d_tmem, uint64_t a_desc, uint32_t a_block_bytes, uint64_t b_desc,
                                                  uint32_t b_block_bytes, int ksteps, uint32_t idesc) {
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint32_t blk = (uint32_t)ks >> 2, in = ((uint32_t)ks & 3u) * 32u;
    mma_ss(d_tmem, desc_advance(a_desc, blk * a_block_bytes + in), desc_advance(b_desc, blk * b_block_bytes + in), idesc,
           ks > 0 ? 1u : 0u);
  }
}
// D[tmem] (+)= A[tmem, packed 16-bit: 8 columns per k-step] . B with B MN-major (k-step = 16 rows of 128 bytes)
__device__ __forceinline__ void issue_tmem_gemm(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, int ksteps, uint32_t idesc,
                                                bool accumulate) {
  for (int ks = 0; ks < ksteps; ++ks)
    mma_ts(d_tmem, a_tmem + (uint32_t)ks * 8u, desc_advance(b_desc, (uint32_t)ks * 2048u), idesc,
           (accumulate || ks > 0) ? 1u : 0u);
}

// ---- TMA stores (shared -> global, bulk async group) ---------------------------------------------------------------
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the bulk stores issued by this thread have finished READING shared memory (the buffer may be overwritten)
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the most recent bulk store of this thread have finished reading shared memory
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
// ... have completed (globally visible)
__device__ __forceinline__ void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy writes to shared memory made visible to the async proxy (TMA) before the store is issued
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// One thread's 16 consecutive 16-bit values (32 bytes: two 16-byte chunks) of row `r` written into a [rows x 64-column]
// block laid out with the 128-byte swizzle the TMA expects: chunk index XOR (row & 7).  `col16` = first column / 8.
__device__ __forceinline__ void st_swizzled_32B(uint32_t block_base, int r, int chunk, const uint32_t* w) {
  const uint32_t row_base = block_base + (uint32_t)r * 128u;
  const uint32_t a0 = row_base + (uint32_t)(((chunk) ^ (r & 7)) << 4);
  const uint32_t a1 = row_base + (uint32_t)(((chunk + 1) ^ (r & 7)) << 4);
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a0), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a1), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
}

// Row softmax with four independent max / sum chains (the serial 80-long chains of `row_softmax` leave a warp stalled on
// its own dependencies).  On return s[j] = exp2(sc * (s[j] - max)) for j < T and 0 beyond; `sum` is their sum.
__device__ __forceinline__ void row_softmax_ilp(float* s, int T, float sc, float& m, float& sum) {
  float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int j = 0; j < kTpad - 16; ++j) m4[j & 3] = fmaxf(m4[j & 3], s[j]);
#pragma unroll
  for (int j = kTpad - 16; j < kTpad; ++j)
    if (j < T) m4[j & 3] = fmaxf(m4[j & 3], s[j]);
  m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
  const float mo = m * sc;
  float a4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < kTpad - 16; ++j) {
    s[j] = ex2_approx(fmaf(s[j], sc, -mo));
    a4[j & 3] += s[j];
  }
#pragma unroll
  for (int j = kTpad - 16; j < kTpad; ++j) {
    s[j] = (j < T) ? ex2_approx(fmaf(s[j], sc, -mo)) : 0.f;
    a4[j & 3] += s[j];
  }
  sum = (a4[0] + a4[1]) + (a4[2] + a4[3]);
}

__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
template <int kRegs> __device__ __forceinline__ void reg_dealloc() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs));
}
template <int kRegs> __device__ __forceinline__ void reg_alloc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs));
}


// ---- host side --------------------------------------------------------------------------------------------------
constexpr int kBlockCols = 64;  // 16-bit elements per 128-byte swizzle row
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// (d, H, rows, B) view of a (B, rows, H*d) tensor; box = 64 channels x 1 head x box_rows rows; 128-byte swizzle;
// out-of-range channels / rows are filled with zeros.
static inline int make_map(CUtensorMap* map, const void* ptr, int dtype, int B, int rows, int H, int d, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) return fail(GA_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[4] = {(cuuint64_t)d, (cuuint64_t)H, (cuuint64_t)rows, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)d * 2, (cuuint64_t)H * d * 2, (cuuint64_t)rows * H * d * 2};
  cuuint32_t box[4] = {(cuuint32_t)kBlockCols, 1u, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  CUresult r = fn(map, dtype == GA_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4,
                  const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_ERROR_INVALID_CONTEXT) {
    // first call on a thread that has no current context yet (e.g. a fresh autograd worker): let the runtime bind the
    // primary context of the current device, then retry
    cudaFree(nullptr);
    r = fn(map, dtype == GA_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4,
           const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) return fail(GA_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return GA_OK;
}

// (cols, rows, batches) view of fp32 rows with a row pitch of `cols` floats and a batch stride of `bstride` floats;
// box = box_cols columns (box_cols * 4 bytes = the swizzle span) x box_rows rows; out-of-range columns / rows are
// filled with zeros.
static inline int make_map_rows_f32(CUtensorMap* map, const void* ptr, int cols, int rows, int batches, int64_t bstride,
                                    int box_cols, int box_rows, CUtensorMapSwizzle swizzle) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) return fail(GA_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batches};
  cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)bstride * 4};
  cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = CUDA_ERROR_INVALID_CONTEXT;
  for (int attempt = 0; attempt < 2 && r == CUDA_ERROR_INVALID_CONTEXT; ++attempt) {
    if (attempt == 1) cudaFree(nullptr);      // bind the primary context (see make_map)
    r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
           CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) return fail(GA_ERR_CUDA, "cuTensorMapEncodeTiled (fp32 rows) failed (%d)", (int)r);
  return GA_OK;
}

// The opt-in dynamic shared-memory limit is raised once per (device, kernel) to the largest size the kernel can ask
// for, so steady-state launches (and CUDA-graph captures) make no attribute call at all.
static inline cudaError_t ensure_smem(const void* kernel, int slot, size_t) {
  static bool done[64][8] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  if (done[dev][slot]) return cudaSuccess;
  int optin = 0;
  cudaFuncAttributes fa;
  if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
  if ((e = cudaFuncGetAttributes(&fa, kernel)) != cudaSuccess) return e;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
  if (e == cudaSuccess) done[dev][slot] = true;
  return e;
}

static inline int sm_count() {
  static int n[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (n[dev] == 0) cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
  return n[dev] > 0 ? n[dev] : 148;
}


}  // namespace tc
}  // namespace ga
