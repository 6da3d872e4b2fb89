// sm_100a building blocks written as inline PTX: mbarrier, TMA (cp.async.bulk.tensor), TMEM alloc/ld, tcgen05.mma
// with shared-memory matrix descriptors.  No CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace udh {
namespace tc {

// ------------------------------------------------------------------------------------------------ host: tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled through the runtime's driver entry point (libudh does not link libcuda, so the library
// still loads on a box without a driver — needed by the CPU-side ABI tests).
inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// `rank` dims (innermost first), 128-byte swizzle, zero fill out of bounds.  The inner box extent must span 128 bytes.
inline int make_tmap(CUtensorMap* map, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled is unavailable (no CUDA driver?)"); return UDH_ECUDA; }
  cuuint64_t gdim[5], gstr[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i + 1];   // stride of dim i+1 (dim 0 is contiguous)
  CUresult r = fn(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return UDH_ECUDA; }
  return UDH_OK;
}

inline int make_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                          const uint32_t* box) {
  return make_tmap(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rank, dims, strides_bytes, box);
}

// ------------------------------------------------------------------------------------------------ device: PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Bounded wait: a protocol bug traps after ~2 s (launch error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  while (!mbar_try_wait(bar, parity)) {
    if (globaltimer_ns() - t0 > 2000000000ull) {
      printf("libudh: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", (int)blockIdx.x, (int)threadIdx.x,
             smem_u32(bar), parity);
      asm volatile("trap;");
    }
  }
}

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, int c0, int c1, int c2, int c3, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}

// TMA store smem -> global (bulk async group), 2D tile
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives row (lane base + t), v[j] = column j.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, "
               "%24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
                 "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                 "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 16-byte vector reduction into global memory (REDG.E.ADD.F32x4): one L2 atomic transaction for four floats.
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ---- descriptors -------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, 128-byte swizzle.  start: smem byte address; lbo/sbo in bytes;
// base_offset = (start >> 7) & 7 when the start is not on a 1024-byte swizzle-pattern boundary.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t start, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t base_offset) {
  uint64_t d = 0;
  d |= (uint64_t)((start & 0x3FFFFu) >> 4);             // [0,14)  start address >> 4
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;    // [16,30) leading byte offset >> 4
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;    // [32,46) stride byte offset >> 4
  d |= (uint64_t)1 << 46;                               // [46,48) descriptor version = 1 (Blackwell)
  d |= (uint64_t)(base_offset & 7u) << 49;              // [49,52) matrix base offset
  d |= (uint64_t)2 << 61;                               // [61,64) layout type: SWIZZLE_128B
  return d;
}

// Fast path for issue loops: the upper word is constant (SBO = 1024 B, version 1, SWIZZLE_128B, base_offset 0); the lower
// word is (start >> 4) | (LBO >> 4) << 16, so stepping the start address is one 32-bit add.
constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo(uint32_t start, uint32_t lbo_bytes) { return ((start & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16); }
__device__ __forceinline__ uint64_t desc_from_lo(uint32_t lo) { return ((uint64_t)kDescHiSw128 << 32) | lo; }

// Instruction descriptor, kind::f16, bf16 x bf16 -> fp32, dense.  a_mn / b_mn: 1 = MN-major operand.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// ---- two-limb split of fp32 values (UDH_NUMERIC_BF16X3) ------------------------------------------------------------
// x = hi + lo with hi = bf16(x), lo = bf16(x - hi) (x - hi is exact in fp32).  The product of two split values is
// evaluated on the tensor pipe as hi*hi + hi*lo + lo*hi with fp32 accumulation; the dropped lo*lo term and the residual
// of the split are both <= 2^-16 |x y|.  Two values are packed per 32-bit word.
// Why bf16 and not fp16 limbs (22 bits instead of 16): kind::f16 MMAs with fp16 on one side and bf16 on the other raise
// an illegal-instruction error on B200, so both operands of every MMA share a format, and the weight gradient multiplies
// activations with gradients (1e-8 .. 1e-2), which do not fit fp16's range without per-tensor loss scaling.
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - __low2float(h), b - __high2float(h));
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// value of a packed pair of limbs: (hi.x + lo.x, hi.y + lo.y)
__device__ __forceinline__ float2 join2(uint32_t hi, uint32_t lo) {
  const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&hi), l = *reinterpret_cast<const __nv_bfloat162*>(&lo);
  return make_float2(__low2float(h) + __low2float(l), __high2float(h) + __high2float(l));
}

// D[tmem] (+)= A[smem] . B[smem]   (issued by ONE thread)
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

}  // namespace tc
}  // namespace udh
