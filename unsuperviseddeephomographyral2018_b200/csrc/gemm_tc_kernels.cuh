// tcgen05 GEMM for the fully connected head (fc1: 32768 -> 1024), bf16 operands, fp32 TMEM accumulation.
//   D[M][N] (+)= A . B over K, tiles of 128 x 256, k-blocks of 64, 4-stage TMA ring, two TMEM accumulator sets.
// Each operand is either K-major (contraction index contiguous in memory: tile = [rows][64 k], box (64, rows)) or
// MN-major (row/column index contiguous: tile = 64-wide column blocks of [64 k][64 mn]), which covers
//   forward   y  = x . W        A = x [B][F] K-major,      B = W [F][N] MN-major,   split-K, atomic accumulation
//   dgrad     dx = dy . W^T     A = dy [B][N] K-major,     B = W [F][N] as [n=f][k] K-major
//   wgrad     dW = x^T . dy     A = x [B][F] MN-major,     B = dy [B][N] MN-major   (K = batch)
// with no transposed copies.  warp 0: TMA | warp 1: MMA | warp 2: TMEM alloc | warps 4-7: epilogue.
#pragma once
#include "tc_common.cuh"

namespace udh {
namespace tc {

// The contraction may run over up to three SEGMENTS: segment s reads A at (k + a_koff[s], m + a_moff[s]) and B at
// (k + b_koff[s], n + b_noff[s]).  The two-limb mode (UDH_NUMERIC_BF16X3) uses this to evaluate
// lo.hi + hi.hi + hi.lo over operands stored as [hi | lo] without duplicating anything in memory; one segment with zero
// offsets is the plain GEMM.
struct GemmGeom {
  int M, N;            // logical output size (rows beyond M / cols beyond N are not stored)
  int m_tiles, n_tiles, k_splits;
  int kb_per_split;    // k-blocks (of 64) per split, counted over all segments
  int kb_per_seg;      // k-blocks of one segment
  int a_koff[3], a_moff[3], b_koff[3], b_noff[3];
  int64_t ldc;
};

constexpr int kGemmStages = 4;
constexpr int kGemmStageBytes = 16384 + 32768;   // A 128 x 64, B 256 x 64 (bf16)

constexpr int kGemmEpiBytes = 2 * 4 * 32 * 128;  // TMA-store staging of the non-atomic epilogue: 2 x (32 rows x 32 floats) per warp

// ATOMIC: split-K partial tiles are added with 16-byte vector reductions.  Otherwise the tile is stored through a swizzled
// shared-memory staging block and TMA (full 128-byte lines; rows / columns beyond M / N are clipped by the tensor map).
template <bool A_MN, bool B_MN, bool ATOMIC>
__global__ void __launch_bounds__(256, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
               const GemmGeom g, float* __restrict__ C) {
  extern __shared__ uint8_t raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sEpi = base + (size_t)kGemmStages * kGemmStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sEpi + (ATOMIC ? 0 : kGemmEpiBytes));
  uint64_t* full = bars;                       // [stages]
  uint64_t* empty = bars + kGemmStages;        // [stages]
  uint64_t* t_full = bars + 2 * kGemmStages;   // [2]
  uint64_t* t_empty = t_full + 2;              // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kGemmStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 128); }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { prefetch_tmap(&tmA); prefetch_tmap(&tmB); }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_tiles = g.m_tiles * g.n_tiles * g.k_splits;
  pdl_wait();                  // predecessor grid complete: global memory may be touched from here on
  pdl_trigger();
  const int my_tiles = (num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  auto decode = [&](int tile, int& mt, int& nt, int& ks) {
    ks = tile % g.k_splits; tile /= g.k_splits;
    nt = tile % g.n_tiles;
    mt = tile / g.n_tiles;
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t cnt = 0;
      for (int i = 0; i < my_tiles; ++i) {
        int mt, nt, ks;
        decode((int)blockIdx.x + i * (int)gridDim.x, mt, nt, ks);
        for (int kb = 0; kb < g.kb_per_split; ++kb, ++cnt) {
          const int s = cnt % kGemmStages;
          const int kg = ks * g.kb_per_split + kb;
          const int seg = kg / g.kb_per_seg;
          const int k0 = (kg - seg * g.kb_per_seg) * 64;
          const int ak = k0 + g.a_koff[seg], am = mt * 128 + g.a_moff[seg], bk = k0 + g.b_koff[seg], bn = nt * 256 + g.b_noff[seg];
          mbar_wait(&empty[s], ((cnt / kGemmStages) & 1) ^ 1);
          mbar_arrive_expect_tx(&full[s], kGemmStageBytes);
          uint8_t* sa = base + (size_t)s * kGemmStageBytes;
          uint8_t* sb = sa + 16384;
          if (A_MN) {
            for (int j = 0; j < 2; ++j) tma_load_2d(sa + j * 8192, &tmA, am + j * 64, ak, &full[s]);
          } else {
            tma_load_2d(sa, &tmA, ak, am, &full[s]);
          }
          if (B_MN) {
            for (int j = 0; j < 4; ++j) tma_load_2d(sb + j * 8192, &tmB, bn + j * 64, bk, &full[s]);
          } else {
            tma_load_2d(sb, &tmB, bk, bn, &full[s]);
          }
        }
      }
    }
  } else if (warp == 1) {
    // whole warp converged; one elected lane issues
    constexpr uint32_t idesc = make_idesc_bf16(128, 256, A_MN ? 1 : 0, B_MN ? 1 : 0);
    uint32_t cnt = 0;
    for (int i = 0; i < my_tiles; ++i) {
      const int b = i & 1;
      mbar_wait(&t_empty[b], ((i >> 1) & 1) ^ 1);
      tc_fence_after();
      for (int kb = 0; kb < g.kb_per_split; ++kb, ++cnt) {
        const int s = cnt % kGemmStages;
        mbar_wait(&full[s], (cnt / kGemmStages) & 1);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(base + (size_t)s * kGemmStageBytes), b_addr = a_addr + 16384;
        const uint32_t a_lo = desc_lo(a_addr, A_MN ? 8192 : 16), b_lo = desc_lo(b_addr, B_MN ? 8192 : 16);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_base + (uint32_t)(b * 256), desc_from_lo(a_lo + k * (A_MN ? 128 : 2)), desc_from_lo(b_lo + k * (B_MN ? 128 : 2)),
                      idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty[s]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&t_full[b]);
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int ew = warp - 4;
    uint8_t* stg0 = sEpi + ew * 8192;            // two staging blocks per warp: chunk c fills one while the TMA store
    const int sw = lane & 7;                      // of chunk c-1 still reads the other
    int stores_in_flight = 0;
    for (int i = 0; i < my_tiles; ++i) {
      const int b = i & 1;
      int mt, nt, ks;
      decode((int)blockIdx.x + i * (int)gridDim.x, mt, nt, ks);
      mbar_wait(&t_full[b], (i >> 1) & 1);
      tc_fence_after();
      const int m = mt * 128 + ew * 32 + lane;
      float* crow = C + (int64_t)m * g.ldc + nt * 256;
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(b * 256 + c * 32), v);
        const int n0 = nt * 256 + c * 32;
        if (ATOMIC) {
          if (m < g.M) {
            if (n0 + 32 <= g.N) {
#pragma unroll
              for (int j = 0; j < 8; ++j) red_add_v4(crow + c * 32 + 4 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (n0 + j < g.N) atomicAdd(crow + c * 32 + j, v[j]);
            }
          }
        } else {
          uint8_t* stg = stg0 + (c & 1) * 4096;
          const uint32_t my_row = smem_u32(stg) + lane * 128;
          if (stores_in_flight >= 2) { if (lane == 0) bulk_wait_read1(); __syncwarp(); stores_in_flight = 1; }
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4)
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(my_row + (uint32_t)((j4 ^ sw) << 4)), "f"(v[4 * j4]), "f"(v[4 * j4 + 1]),
                         "f"(v[4 * j4 + 2]), "f"(v[4 * j4 + 3]) : "memory");
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {                          // (always commit, possibly an empty group, so the group count stays uniform)
            if (n0 < g.N && mt * 128 + ew * 32 < g.M) tma_store_2d(&tmC, stg, n0, mt * 128 + ew * 32);
            bulk_commit();
          }
          ++stores_in_flight;
        }
      }
      tc_fence_before();
      mbar_arrive(&t_empty[b]);
    }
    if (!ATOMIC) { if (lane == 0) bulk_wait0(); __syncwarp(); }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// Host launcher.  C[M][N] (+)= A . B on tensor cores.  a_inner/a_outer: dims of A's tensor (innermost first); same for B.
// seg (nullable): offsets of the contraction segments (see GemmGeom), K is the length of ONE segment.
struct GemmSegments { int n; int a_koff[3], a_moff[3], b_koff[3], b_noff[3]; };

template <bool A_MN, bool B_MN, bool ATOMIC>
inline int launch_gemm(const void* A, uint64_t a_inner, uint64_t a_outer, const void* Bm, uint64_t b_inner, uint64_t b_outer,
                       float* C, int64_t ldc, int M, int N, int K, int k_splits, const GemmSegments* seg, cudaStream_t st) {
  GemmGeom g;
  g.M = M; g.N = N; g.ldc = ldc;
  g.m_tiles = (M + 127) / 128; g.n_tiles = (N + 255) / 256;
  const int nseg = seg ? seg->n : 1;
  g.kb_per_seg = (K + 63) / 64;
  const int kb = g.kb_per_seg * nseg;
  g.k_splits = k_splits;
  g.kb_per_split = (kb + k_splits - 1) / k_splits;
  UDH_REQUIRE(g.kb_per_split * k_splits == kb, "tc gemm: k-blocks (%d) must divide evenly into %d splits", kb, k_splits);
  for (int i = 0; i < 3; ++i) {
    g.a_koff[i] = seg && i < nseg ? seg->a_koff[i] : 0; g.a_moff[i] = seg && i < nseg ? seg->a_moff[i] : 0;
    g.b_koff[i] = seg && i < nseg ? seg->b_koff[i] : 0; g.b_noff[i] = seg && i < nseg ? seg->b_noff[i] : 0;
  }
  CUtensorMap tmA, tmB;
  uint64_t dA[2] = {a_inner, a_outer}, sA[2] = {2, a_inner * 2};
  uint32_t boxA[2] = {64, A_MN ? 64u : 128u};
  int rc = make_tmap_bf16(&tmA, A, 2, dA, sA, boxA);
  if (rc != UDH_OK) return rc;
  uint64_t dB[2] = {b_inner, b_outer}, sB[2] = {2, b_inner * 2};
  uint32_t boxB[2] = {64, B_MN ? 64u : 256u};
  rc = make_tmap_bf16(&tmB, Bm, 2, dB, sB, boxB);
  if (rc != UDH_OK) return rc;
  // output map for the TMA-store epilogue: fp32 [M][ldc], box = 32 floats (128 B) x 32 rows
  CUtensorMap tmC;
  uint64_t dC[2] = {(uint64_t)N, (uint64_t)M}, sC[2] = {4, (uint64_t)ldc * 4};
  uint32_t boxC[2] = {32, 32};
  rc = make_tmap(&tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, C, 2, dC, sC, boxC);
  if (rc != UDH_OK) return rc;
  const size_t smem = 1024 + (size_t)kGemmStages * kGemmStageBytes + (ATOMIC ? 0 : kGemmEpiBytes) + 256;
  auto kern = tc_gemm_kernel<A_MN, B_MN, ATOMIC>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = persistent_ctas();
  const int tiles = g.m_tiles * g.n_tiles * g.k_splits;
  launch_chain(kern, dim3(tiles < sms ? tiles : sms), dim3(256), smem, st, tmA, tmB, tmC, g, C);
  return check_launch("tc_gemm_kernel");
}

}  // namespace tc
}  // namespace udh
