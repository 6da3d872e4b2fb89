// Error-compensated tcgen05 weight-gradient kernels (UDH_NUMERIC_BF16X3) on two-limb padded streams.
//
//   dW[tap][ci][co] = sum_q X[q + off_tap][ci] * G[q][co]   with   X = X_hi + X_lo,  G = G_hi + G_lo
// evaluated as three passes  X_lo.G_hi + X_hi.G_hi + X_hi.G_lo  into the SAME fp32 TMEM accumulators, which stay resident
// for the CTA's whole run (split-K over CTAs, one epilogue of vector reductions) — see wgrad_tc_kernels.cuh for the
// operand formulation (MN-major operands, tap pairs through the leading-dimension offset, N = 192 for the 64 -> 64 layers).
//
// Shared memory holds ONE buffer per (operand, limb) — X_hi, X_lo, G_hi, G_lo — each with its own full/empty mbarrier
// pair.  The pass order (X_lo,G_hi) -> (X_hi,G_hi) -> (X_hi,G_lo) staggers their lifetimes: X_lo is free after the first
// third of an item, G_hi after the second, X_hi / G_lo at its end, and each is needed again one third later than it was
// released at the earliest, so every refill runs under the MMAs of another pass although nothing is double-buffered.
//
// Bias gradient: db = sum_q G[q] = ones.(G_hi + G_lo).  The constant-one rows ride along as an extra M block of the X_hi
// passes; in the X_lo pass that M block reads a block of zeros.  Both constant blocks are 16 rows (one k-step) long: the
// descriptor's leading-dimension offset is recomputed per k-step so that it always lands on the same 2 KB.
#pragma once
#include "wgrad_tc_kernels.cuh"

namespace udh {
namespace tc {

constexpr int kConstBlockBytes = 2048;     // 16 positions x 64 channels x 2 bytes

constexpr uint32_t kOnePair = 0x3F803F80u;   // two bf16 1.0 packed in one word

__device__ __forceinline__ void fill_const_blocks(uint8_t* sOnes, uint8_t* sZeros) {
  uint32_t* o = reinterpret_cast<uint32_t*>(sOnes);
  uint32_t* z = reinterpret_cast<uint32_t*>(sZeros);
  for (int i = threadIdx.x; i < kConstBlockBytes / 4; i += blockDim.x) { o[i] = kOnePair; z[i] = 0u; }
  fence_proxy_async();                                          // generic-proxy writes -> visible to the tensor (async) proxy
}

// buffer indices
constexpr int kXH = 0, kXL = 1, kGH = 2, kGL = 3;

// ---------------------------------------------------------------------------------------------------------------------
// generic kernel: N_OUT = 128; CBX = 1 (64 -> 128: two taps per MMA) or 2 (128 -> 128: one tap per MMA + ones group)
template <int N_OUT, int CBX, int T>
__global__ void __launch_bounds__(256, 1)
tc_wgrad_x3_kernel(const __grid_constant__ CUtensorMap tmX128, const __grid_constant__ CUtensorMap tmXhh,
                   const __grid_constant__ CUtensorMap tmG, const WgradGeom g, float* __restrict__ dW, float* __restrict__ db) {
  constexpr int CBO = N_OUT / 64;
  constexpr int CIN = CBX * 64;
  extern __shared__ uint8_t raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  const int xblk_bytes = g.xrows * 128;                         // one 64-channel block of one limb of X
  constexpr int gblk_bytes = T * 128 * 128;                     // one 64-channel block of one limb of G
  const int xl_bytes = CBX * xblk_bytes, gl_bytes = CBO * gblk_bytes;
  uint8_t* sX[2] = {base, base + xl_bytes};                     // [limb][CBX blocks]
  uint8_t* sG[2] = {base + 2 * (size_t)xl_bytes, base + 2 * (size_t)xl_bytes + gl_bytes};
  uint8_t* sOnes = sG[1] + gl_bytes;
  uint8_t* sZeros = sOnes + kConstBlockBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sZeros + kConstBlockBytes);
  uint64_t* full = bars;        // [4]
  uint64_t* empty = bars + 4;   // [4]
  uint64_t* acc_full = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int sl = 0;
  while (sl + 1 < g.num_slices && (int)blockIdx.x >= g.slice_cta[sl + 1]) ++sl;
  const int bx = (int)blockIdx.x - g.slice_cta[sl], gxs = g.slice_cta[sl + 1] - g.slice_cta[sl];
  const int g_begin = g.slice_group[sl];
  const int g_count = g.slice_group[sl + 1] - g_begin;
  constexpr int kTmemCols = 512;

  fill_const_blocks(sOnes, sZeros);
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { prefetch_tmap(&tmX128); prefetch_tmap(&tmXhh); prefetch_tmap(&tmG); }
  if (warp == 2) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                  // predecessor grid complete: global memory may be touched from here on
  pdl_trigger();
  const int my_items = (g.num_items - bx + gxs - 1) / gxs;

  if (warp == 0) {
    if (lane == 0) {
      auto load_x = [&](int l, int q0, uint32_t par) {
        mbar_wait(&empty[l], par);
        mbar_arrive_expect_tx(&full[l], (uint32_t)xl_bytes);
        for (int cb = 0; cb < CBX; ++cb) {
          uint8_t* dst = sX[l] + (size_t)cb * xblk_bytes;
          const int c0 = (l * CBX + cb) * 64;
          tma_load_2d(dst, &tmXhh, c0, q0 - g.hh, &full[l]);
          for (int t = 0; t < T; ++t) tma_load_2d(dst + (size_t)(g.hh + t * 128) * 128, &tmX128, c0, q0 + t * 128, &full[l]);
          tma_load_2d(dst + (size_t)(g.hh + T * 128) * 128, &tmXhh, c0, q0 + T * 128, &full[l]);
        }
      };
      auto load_g = [&](int l, int q0, uint32_t par) {
        mbar_wait(&empty[2 + l], par);
        mbar_arrive_expect_tx(&full[2 + l], (uint32_t)gl_bytes);
        for (int cb = 0; cb < CBO; ++cb)
          for (int t = 0; t < T; ++t)
            tma_load_2d(sG[l] + (size_t)cb * gblk_bytes + (size_t)t * 16384, &tmG, (l * CBO + cb) * 64, q0 + t * 128, &full[2 + l]);
      };
      for (int it = 0; it < my_items; ++it) {
        const int q0 = (bx + it * gxs) * T * 128;
        const uint32_t par = (it & 1) ^ 1;
        load_x(1, q0, par);      // in the order the MMA passes release the buffers
        load_g(0, q0, par);
        load_x(0, q0, par);
        load_g(1, q0, par);
      }
    }
  } else if (warp == 1) {
    // One elected lane runs the whole MMA role (waits included); the per-group operand geometry (row shift of the first M
    // block, leading-dimension offset to the second one, constant-block mode) does not depend on the item and is tabulated once.
    constexpr uint32_t idesc = make_idesc_bf16(128, N_OUT, 1, 1);
    constexpr uint32_t idesc_ones = make_idesc_bf16(64, N_OUT, 1, 1);
    const uint32_t ones_addr = smem_u32(sOnes), zeros_addr = smem_u32(sZeros);
    if (elect_one()) {
      int goff[4]; uint32_t glbo[4]; int gmode[4];               // mode 0: fixed lbo; 1: second M block = constant rows; 2: ones group (M = 64)
#pragma unroll
      for (int gi_l = 0; gi_l < 4; ++gi_l) {
        const int gi = g_begin + gi_l;
        goff[gi_l] = 0; glbo[gi_l] = 0; gmode[gi_l] = 0;
        if (gi_l >= g_count) continue;
        if (CBX == 1) {
          const int tap0 = 2 * gi;
          const int off0 = (tap0 / 3 - 1) * g.Wp + (tap0 % 3 - 1);
          goff[gi_l] = off0;
          if (gi < 4) {
            const int tap1 = tap0 + 1;
            glbo[gi_l] = (uint32_t)(((tap1 / 3 - 1) * g.Wp + (tap1 % 3 - 1)) - off0) * 128;
          } else {
            gmode[gi_l] = 1;
          }
        } else if (gi < 9) {
          goff[gi_l] = (gi / 3 - 1) * g.Wp + (gi % 3 - 1);
          glbo[gi_l] = (uint32_t)xblk_bytes;                      // second M block = channels 64..127
        } else {
          gmode[gi_l] = 2;
        }
      }
      for (int it = 0; it < my_items; ++it) {
        const uint32_t par = it & 1;
#pragma unroll 1
        for (int pass = 0; pass < 3; ++pass) {
          const int xl = pass == 0 ? 1 : 0;                       // X limb of this pass
          const int gl_ = pass == 2 ? 1 : 0;                      // G limb of this pass
          if (pass == 0) { mbar_wait(&full[kXL], par); mbar_wait(&full[kGH], par); }
          else if (pass == 1) mbar_wait(&full[kXH], par);
          else mbar_wait(&full[kGL], par);
          tc_fence_after();
          const uint32_t x_addr = smem_u32(sX[xl]);
          const uint32_t g_addr = smem_u32(sG[gl_]);
          const uint32_t const_addr = xl ? zeros_addr : ones_addr; // the constant-one channel has no lo limb
#pragma unroll 1
          for (int t = 0; t < T; ++t) {
            const uint32_t b_lo = desc_lo(g_addr + (uint32_t)t * 16384, (uint32_t)gblk_bytes);
#pragma unroll
            for (int gi_l = 0; gi_l < 4; ++gi_l) {
              if (gi_l >= g_count) continue;
              const int mode = gmode[gi_l];
              if (mode == 2 && xl) continue;                      // ones group: X_hi passes only
              const uint32_t a_start = mode == 2 ? ones_addr : x_addr + (uint32_t)(g.hh + t * 128 + goff[gi_l]) * 128;
              const uint32_t id = mode == 2 ? idesc_ones : idesc;
              const uint32_t d_tmem = tmem_base + (uint32_t)(gi_l * N_OUT);
              // the first MMA into an accumulator overwrites it: pass 0 (or pass 1 for the ones group, which skips pass 0)
              const bool fresh = it == 0 && t == 0 && (pass == 0 || (mode == 2 && pass == 1));
#pragma unroll
              for (int kk = 0; kk < 8; ++kk) {                     // 16 positions = 2048 bytes per k-step
                uint32_t a_lo;
                if (mode == 0) a_lo = desc_lo(a_start + kk * 2048, glbo[gi_l]);
                else if (mode == 1) a_lo = desc_lo(a_start + kk * 2048, const_addr - (a_start + kk * 2048));
                else a_lo = desc_lo(a_start, 0);
                umma_bf16(d_tmem, desc_from_lo(a_lo), desc_from_lo(b_lo + kk * 128), id, (fresh && kk == 0) ? 0u : 1u);
              }
            }
          }
          if (pass == 0) umma_commit(&empty[kXL]);
          else if (pass == 1) umma_commit(&empty[kGH]);
          else { umma_commit(&empty[kXH]); umma_commit(&empty[kGL]); }
        }
      }
      umma_commit(acc_full);
    }
    __syncwarp();
  } else if (warp >= 4 && my_items > 0) {
    const int ew = warp - 4;
    const int m = ew * 32 + lane;                               // accumulator row == TMEM lane
    mbar_wait(acc_full, 0);
    tc_fence_after();
#pragma unroll 1
    for (int gl = 0; gl < g_count; ++gl) {
      const int gi = g_begin + gl;
      int tap, ci;
      bool is_ones = false;
      if (CBX == 1) {
        ci = m & 63;
        tap = 2 * gi + (m >> 6);
        if (tap == 9) is_ones = true;
      } else {
        ci = m; tap = gi;
        if (gi == 9) is_ones = true;
      }
      float* dst = is_ones ? db : dW + ((size_t)tap * CIN + ci) * N_OUT;
      const bool active = is_ones ? (m == (CBX == 1 ? 64 : 0) && db != nullptr) : true;
#pragma unroll 1
      for (int c = 0; c < N_OUT / 32; ++c) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(gl * N_OUT + c * 32), v);
        if (active) {
#pragma unroll
          for (int j = 0; j < 8; ++j)                                  // 16-byte vector reductions: 4x fewer L2 atomics
            red_add_v4(dst + c * 32 + 4 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
}

// ---------------------------------------------------------------------------------------------------------------------
// 64 -> 64 channel layers: the N = 192 formulation of tc_wgrad64_kernel (B = three row shifts of G, A = two row shifts of X;
// two MMAs per 16 positions and pass), with the limb passes above.
template <int T>
__global__ void __launch_bounds__(256, 1)
tc_wgrad64_x3_kernel(const __grid_constant__ CUtensorMap tmX128, const __grid_constant__ CUtensorMap tmXhh,
                     const __grid_constant__ CUtensorMap tmG136, const Wgrad64Geom g, float* __restrict__ dW, float* __restrict__ db) {
  static_assert(T == 2, "G is staged as two 136-row boxes");
  extern __shared__ uint8_t raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  const int xblk_bytes = g.xrows * 128;
  constexpr int kGRows = T * 128 + 16;                          // 8 halo rows on each side
  constexpr int gblk_bytes = kGRows * 128;
  uint8_t* sX[2] = {base, base + xblk_bytes};
  uint8_t* sG[2] = {base + 2 * (size_t)xblk_bytes, base + 2 * (size_t)xblk_bytes + gblk_bytes};
  uint8_t* sOnes = sG[1] + gblk_bytes;
  uint8_t* sZeros = sOnes + kConstBlockBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sZeros + kConstBlockBytes);
  uint64_t* full = bars;        // [4]
  uint64_t* empty = bars + 4;   // [4]
  uint64_t* acc_full = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kTmemCols = 512;                                // 2 groups x 192 columns

  fill_const_blocks(sOnes, sZeros);
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { prefetch_tmap(&tmX128); prefetch_tmap(&tmXhh); prefetch_tmap(&tmG136); }
  if (warp == 2) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                  // predecessor grid complete: global memory may be touched from here on
  pdl_trigger();
  const int my_items = (g.num_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 0) {
    if (lane == 0) {
      auto load_x = [&](int l, int q0, uint32_t par) {
        mbar_wait(&empty[l], par);
        mbar_arrive_expect_tx(&full[l], (uint32_t)xblk_bytes);
        uint8_t* dst = sX[l];
        tma_load_2d(dst, &tmXhh, l * 64, q0 - g.hh, &full[l]);
        for (int t = 0; t < T; ++t) tma_load_2d(dst + (size_t)(g.hh + t * 128) * 128, &tmX128, l * 64, q0 + t * 128, &full[l]);
        tma_load_2d(dst + (size_t)(g.hh + T * 128) * 128, &tmXhh, l * 64, q0 + T * 128, &full[l]);
      };
      auto load_g = [&](int l, int q0, uint32_t par) {
        mbar_wait(&empty[2 + l], par);
        mbar_arrive_expect_tx(&full[2 + l], (uint32_t)gblk_bytes);
        tma_load_2d(sG[l], &tmG136, l * 64, q0 - 8, &full[2 + l]);
        tma_load_2d(sG[l] + 136 * 128, &tmG136, l * 64, q0 + 128, &full[2 + l]);
      };
      for (int it = 0; it < my_items; ++it) {
        const int q0 = ((int)blockIdx.x + it * (int)gridDim.x) * T * 128;
        const uint32_t par = (it & 1) ^ 1;
        load_x(1, q0, par);
        load_g(0, q0, par);
        load_x(0, q0, par);
        load_g(1, q0, par);
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(128, 192, 1, 1);
    const uint32_t ones_addr = smem_u32(sOnes), zeros_addr = smem_u32(sZeros);
    for (int it = 0; it < my_items; ++it) {
      const uint32_t par = it & 1;
#pragma unroll 1
      for (int pass = 0; pass < 3; ++pass) {
        const int xl = pass == 0 ? 1 : 0;
        const int gl_ = pass == 2 ? 1 : 0;
        if (pass == 0) { mbar_wait(&full[kXL], par); mbar_wait(&full[kGH], par); }
        else if (pass == 1) mbar_wait(&full[kXH], par);
        else mbar_wait(&full[kGL], par);
        tc_fence_after();
        const uint32_t x_addr = smem_u32(sX[xl]);
        const uint32_t g_addr = smem_u32(sG[gl_]);
        const uint32_t const_addr = xl ? zeros_addr : ones_addr;
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
          const uint32_t b_lo = desc_lo(g_addr + (uint32_t)(8 + t * 128 - 1) * 128, 128);     // G[q-1] | G[q] | G[q+1]
#pragma unroll
          for (int gl = 0; gl < 2; ++gl) {
            const uint32_t a_start = x_addr + (uint32_t)(g.hh + t * 128 + (gl == 0 ? -g.Wp : g.Wp)) * 128;
            const uint32_t d_tmem = tmem_base + (uint32_t)(gl * 192);
            const bool fresh = it == 0 && t == 0 && pass == 0;
            if (elect_one()) {
#pragma unroll
              for (int kk = 0; kk < 8; ++kk) {
                const uint32_t as = a_start + kk * 2048;
                const uint32_t a_lo = desc_lo(as, gl == 0 ? (uint32_t)g.Wp * 128 : const_addr - as);
                umma_bf16(d_tmem, desc_from_lo(a_lo), desc_from_lo(b_lo + kk * 128), idesc, (fresh && kk == 0) ? 0u : 1u);
              }
            }
            __syncwarp();
          }
        }
        if (elect_one()) {
          if (pass == 0) umma_commit(&empty[kXL]);
          else if (pass == 1) umma_commit(&empty[kGH]);
          else { umma_commit(&empty[kXH]); umma_commit(&empty[kGL]); }
        }
        __syncwarp();
      }
    }
    if (elect_one()) umma_commit(acc_full);
    __syncwarp();
  } else if (warp >= 4 && my_items > 0) {
    const int ew = warp - 4;
    const int m = ew * 32 + lane;
    const int ci = m & 63;
    mbar_wait(acc_full, 0);
    tc_fence_after();
#pragma unroll 1
    for (int gl = 0; gl < 2; ++gl) {
      const int ky = gl == 0 ? (m >> 6) - 1 : 1;                  // rows 64.. of group 1 are the ones rows
      const bool is_ones = gl == 1 && m >= 64;
#pragma unroll 1
      for (int c = 0; c < 6; ++c) {
        const int j = c >> 1;                                     // N block: G shift c = j - 1  ->  kx = 1 - j
        const int tap = (ky + 1) * 3 + (2 - j);
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(gl * 192 + c * 32), v);
        float* dst = is_ones ? db : dW + ((size_t)tap * 64 + ci) * 64;
        const bool active = is_ones ? (m == 64 && j == 1 && db != nullptr) : true;
        if (active) {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj)
            red_add_v4(dst + (c & 1) * 32 + 4 * jj, v[4 * jj], v[4 * jj + 1], v[4 * jj + 2], v[4 * jj + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
}

}  // namespace tc
}  // namespace udh
