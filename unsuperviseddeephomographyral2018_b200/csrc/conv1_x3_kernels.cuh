// conv1_1 (2 -> 64 channels, K = 18) in the two-limb mode (UDH_NUMERIC_BF16X3); see conv1_tc_kernels.cuh for the design.
// The explicit im2col row of a pixel holds BOTH limbs of its 18 taps:  k = tap*2+plane  -> hi limb,  k + 32 -> lo limb
// (k = 18: the constant 1 of the wgrad's bias row; it has no lo limb).
// forward : D = A . W1^T + A[:, 0:32] . W2^T  with W1[co] = [w_hi (k < 18) | w_hi (k - 32 < 18)] and W2[co] = [w_lo | 0]
//           = x_hi.w_hi + x_lo.w_hi + x_hi.w_lo; column 18 carries the constant 1 and the bias limbs as its weight, so the
//           accumulator already holds conv + bias; the epilogue splits its ReLU into limbs again.
// wgrad   : D[k][co] += A^T . G_hi + A^T . G_lo ; rows k and k + 32 are added into the same dW row by the epilogue
//           (x_hi.g + x_lo.g; the extra x_lo.g_lo term is harmless), row 18 is the bias gradient.
#pragma once
#include "conv1_tc_kernels.cuh"

namespace udh {
namespace tc {

__device__ __forceinline__ void build_im2col_row_x3(uint8_t* tile, int r, const float* __restrict__ I1, const float* __restrict__ I2,
                                                    int n, int y, int x, int H, int W, bool ones_col) {
  float v[24];
#pragma unroll
  for (int i = 0; i < 24; ++i) v[i] = 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int gy = y + ky - 1;
    const bool rowok = gy >= 0 && gy < H;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int gx = x + kx - 1;
      if (rowok && gx >= 0 && gx < W) {
        const size_t o = ((size_t)n * H + gy) * W + gx;
        v[(ky * 3 + kx) * 2] = __ldg(I1 + o);
        v[(ky * 3 + kx) * 2 + 1] = __ldg(I2 + o);
      }
    }
  }
  if (ones_col) v[18] = 1.0f;
  const uint32_t rowaddr = smem_u32(tile) + r * 128;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int h = 0; h < 4; ++h) split2(v[c * 8 + 2 * h], v[c * 8 + 2 * h + 1], hi[h], lo[h]);
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(rowaddr + (uint32_t)((c ^ (r & 7)) << 4)), "r"(hi[0]), "r"(hi[1]),
                 "r"(hi[2]), "r"(hi[3]) : "memory");
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(rowaddr + (uint32_t)(((4 + c) ^ (r & 7)) << 4)), "r"(lo[0]), "r"(lo[1]),
                 "r"(lo[2]), "r"(lo[3]) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------------------- forward
constexpr int kConv1X3CtasPerSm = 3;
static __global__ void __launch_bounds__(160, kConv1X3CtasPerSm)
conv1_x3_fwd_kernel(const __grid_constant__ CUtensorMap tmOut, const Conv1Geom g, const float* __restrict__ I1,
                    const float* __restrict__ I2, const float* __restrict__ w, const float* __restrict__ bias,
                    uint32_t* __restrict__ mask_out) {
  extern __shared__ uint8_t raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = base;                       // [2][128][128 B]
  uint8_t* sW = base + 2 * 16384;           // W1, W2: [64 co][128 B] each
  uint8_t* sEpi = sW + 16384;               // [4 warps][32][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sEpi + 16384);
  uint64_t* a_full = bars;                  // [2] count 128 (workers)
  uint64_t* a_empty = bars + 2;             // [2] count 1 (MMA commit)
  uint64_t* t_full = bars + 4;              // [2] count 1 (MMA commit)
  uint64_t* t_empty = bars + 6;             // [2] count 128 (workers)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // zero both A tiles (the unused columns stay zero for ever) and build the two weight tiles
  for (int i = threadIdx.x; i < 2 * 16384 / 16; i += blockDim.x) reinterpret_cast<uint4*>(sA)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 64 * 8; i += blockDim.x) {
    const int co = i >> 3, c = i & 7;       // chunk c holds k = 8c .. 8c+7
    uint32_t p1[4], p2[4];
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const int k0 = c * 8 + 2 * h;
      const int kk = c < 4 ? k0 : k0 - 32;  // tap index this column multiplies (hi columns 0.., lo columns 32..)
      // tap 18 is the constant-1 column of the im2col row: its "weight" is the bias, added by the MMA (hi.b_hi + hi.b_lo)
      const float f0 = kk < 18 ? __ldg(w + kk * 64 + co) : (kk == 18 ? __ldg(bias + co) : 0.f);
      const float f1 = kk + 1 < 18 ? __ldg(w + (kk + 1) * 64 + co) : (kk + 1 == 18 ? __ldg(bias + co) : 0.f);
      uint32_t hi, lo;
      split2(f0, f1, hi, lo);
      p1[h] = hi;
      p2[h] = c < 4 ? lo : 0u;
    }
    *reinterpret_cast<uint4*>(sW + co * 128 + ((c ^ (co & 7)) << 4)) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
    *reinterpret_cast<uint4*>(sW + 8192 + co * 128 + ((c ^ (co & 7)) << 4)) = make_uint4(p2[0], p2[1], p2[2], p2[3]);
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&a_full[i], 128); mbar_init(&a_empty[i], 1); mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 128); }
    fence_barrier_init();
    prefetch_tmap(&tmOut);
  }
  if (warp == 4) tmem_alloc(tmem_slot, 128);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                  // predecessor grid complete (the prologue above touched only parameters, written long before)
  pdl_trigger();
  const int my_tiles = (g.tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int segs = g.W / 128;

  if (warp < 4) {
    const int px = threadIdx.x;              // pixel within the segment == TMEM lane
    uint8_t* stg = sEpi + warp * 4096;
    const uint32_t my_row = smem_u32(stg) + lane * 128;
    const int sw = lane & 7;
    bool store_pending = false;
    for (int i = 0; i <= my_tiles; ++i) {
      if (i < my_tiles) {
        // ---- build the im2col tile of item i
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        const int seg = tile % segs, row = tile / segs;
        const int n = row / g.H, y = row - n * g.H;
        const int b = i & 1;
        mbar_wait(&a_empty[b], ((i >> 1) & 1) ^ 1);
        build_im2col_row_x3(sA + b * 16384, px, I1, I2, n, y, seg * 128 + px, g.H, g.W, true);
        fence_proxy_async();
        mbar_arrive(&a_full[b]);
      }
      if (i > 0) {
        // ---- drain the accumulator of item i-1
        const int j = i - 1, b = j & 1;
        const int tile = (int)blockIdx.x + j * (int)gridDim.x;
        const int seg = tile % segs, row = tile / segs;
        const int n = row / g.H, y = row - n * g.H;
        const int q0w = (n * (g.H + 2) + y + 1) * (g.W + 2) + 1 + seg * 128 + warp * 32;    // padded position of this warp's first pixel
        mbar_wait(&t_full[b], (j >> 1) & 1);
        tc_fence_after();
        uint32_t mo[2];
        uint32_t hi[2][16], lo[2][16];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          float v[32];
          tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(b * 64 + c * 32), v);
          // the bias arrived through the constant-1 column; ReLU, then the mask bit of channel k = [v > 0] = the sign of
          // (0 - bits(v)) for v >= +0, shifted in from the top (one negate + one funnel shift per channel)
          uint32_t mw = 0;
#pragma unroll
          for (int k = 31; k >= 0; --k) {
            v[k] = fmaxf(v[k], 0.f);
            mw = __funnelshift_l((uint32_t)(-__float_as_int(v[k])), mw, 1);
          }
          mo[c] = mw;
#pragma unroll
          for (int k = 0; k < 16; ++k) split2(v[2 * k], v[2 * k + 1], hi[c][k], lo[c][k]);
        }
        tc_fence_before();
        mbar_arrive(&t_empty[b]);
        if (mask_out) *reinterpret_cast<uint2*>(mask_out + (size_t)(q0w + lane) * 2) = make_uint2(mo[0], mo[1]);
#pragma unroll
        for (int limb = 0; limb < 2; ++limb) {
          if (store_pending) { if (lane == 0) bulk_wait_read0(); __syncwarp(); }
#pragma unroll
          for (int c = 0; c < 2; ++c) {
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const uint32_t* s = limb ? lo[c] : hi[c];
              asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(my_row + (uint32_t)(((c * 4 + j4) ^ sw) << 4)),
                           "r"(s[j4 * 4]), "r"(s[j4 * 4 + 1]), "r"(s[j4 * 4 + 2]), "r"(s[j4 * 4 + 3]) : "memory");
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) { tma_store_2d(&tmOut, stg, limb * 64, q0w); bulk_commit(); }
          store_pending = true;
        }
      }
    }
    if (lane == 0) bulk_wait0();
    __syncwarp();
  } else {
    // ---- MMA issuer (whole warp converged)
    constexpr uint32_t idesc = make_idesc_bf16(128, 64, 0, 0);
    const uint32_t w1_lo = desc_lo(smem_u32(sW), 16), w2_lo = desc_lo(smem_u32(sW + 8192), 16);
    for (int i = 0; i < my_tiles; ++i) {
      const int b = i & 1;
      const uint32_t ph = (i >> 1) & 1;
      mbar_wait(&a_full[b], ph);
      mbar_wait(&t_empty[b], ph ^ 1);
      tc_fence_after();
      const uint32_t a_lo = desc_lo(smem_u32(sA + b * 16384), 16);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k)            // all 64 columns against W1: hi.w_hi (k-steps 0,1) + lo.w_hi (k-steps 2,3)
          umma_bf16(tmem_base + (uint32_t)(b * 64), desc_from_lo(a_lo + k * 2), desc_from_lo(w1_lo + k * 2), idesc, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < 2; ++k)            // hi columns against W2: hi.w_lo
          umma_bf16(tmem_base + (uint32_t)(b * 64), desc_from_lo(a_lo + k * 2), desc_from_lo(w2_lo + k * 2), idesc, 1u);
        umma_commit(&a_empty[b]);
        umma_commit(&t_full[b]);
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 128);
}

// ------------------------------------------------------------------------------------------------------------- wgrad
constexpr int kConv1X3WgradCtasPerSm = 2;
static __global__ void __launch_bounds__(160, kConv1X3WgradCtasPerSm)
conv1_x3_wgrad_kernel(const __grid_constant__ CUtensorMap tmG, const Conv1Geom g, const float* __restrict__ I1,
                      const float* __restrict__ I2, float* __restrict__ dW, float* __restrict__ db) {
  extern __shared__ uint8_t raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = base;                       // [2][128][128 B]
  uint8_t* sG = base + 2 * 16384;           // [2 stages][2 limbs][128][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sG + 4 * 16384);
  uint64_t* a_full = bars;                  // [2] count 128
  uint64_t* g_full = bars + 2;              // [2] TMA
  uint64_t* empty = bars + 4;               // [2] MMA commit
  uint64_t* acc_full = bars + 6;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  for (int i = threadIdx.x; i < 2 * 16384 / 16; i += blockDim.x) reinterpret_cast<uint4*>(sA)[i] = make_uint4(0, 0, 0, 0);
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&a_full[i], 128); mbar_init(&g_full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(acc_full, 1);
    fence_barrier_init();
    prefetch_tmap(&tmG);
  }
  if (warp == 4) tmem_alloc(tmem_slot, 64);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_trigger();
  const int my_tiles = (g.tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int segs = g.W / 128;

  if (warp < 4) {
    const int px = threadIdx.x;
    for (int i = 0; i < my_tiles; ++i) {
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      const int seg = tile % segs, row = tile / segs;
      const int n = row / g.H, y = row - n * g.H;
      const int b = i & 1;
      mbar_wait(&empty[b], ((i >> 1) & 1) ^ 1);
      build_im2col_row_x3(sA + b * 16384, px, I1, I2, n, y, seg * 128 + px, g.H, g.W, true);
      fence_proxy_async();
      mbar_arrive(&a_full[b]);
    }
    if (my_tiles > 0) {
      // epilogue: M = 64 accumulator rows live in lanes 32*(r/16) + r%16; rows 0..17 (x_hi) and 32..49 (x_lo) = dW[k][co],
      // row 18 = db[co]
      mbar_wait(acc_full, 0);
      tc_fence_after();
      const int r = warp * 16 + lane;        // valid for lane < 16
      const int rr = r & 31;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c * 32), v);
        if (lane < 16 && (rr < 18 || r == 18)) {
          float* dst = rr < 18 ? dW + rr * 64 + c * 32 : db + c * 32;
#pragma unroll
          for (int j = 0; j < 8; ++j) red_add_v4(dst + 4 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
      }
    }
  } else {
    constexpr uint32_t idesc = make_idesc_bf16(64, 64, 1, 1);
    for (int i = 0; i < my_tiles; ++i) {
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      const int seg = tile % segs, row = tile / segs;
      const int n = row / g.H, y = row - n * g.H;
      const int q0 = (n * (g.H + 2) + y + 1) * (g.W + 2) + 1 + seg * 128;
      const int b = i & 1;
      const uint32_t ph = (i >> 1) & 1;
      mbar_wait(&empty[b], ph ^ 1);                                  // both tiles of the stage are free again
      if (elect_one()) {
        mbar_arrive_expect_tx(&g_full[b], 2 * 16384);
        tma_load_2d(sG + b * 32768, &tmG, 0, q0, &g_full[b]);
        tma_load_2d(sG + b * 32768 + 16384, &tmG, 64, q0, &g_full[b]);
      }
      __syncwarp();
      mbar_wait(&a_full[b], ph);
      mbar_wait(&g_full[b], ph);
      tc_fence_after();
      const uint32_t a_lo = desc_lo(smem_u32(sA + b * 16384), 16384);
      const uint32_t gh_lo = desc_lo(smem_u32(sG + b * 32768), 16384), gl_lo = desc_lo(smem_u32(sG + b * 32768 + 16384), 16384);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          umma_bf16(tmem_base, desc_from_lo(a_lo + kk * 128), desc_from_lo(gh_lo + kk * 128), idesc, (i > 0 || kk > 0) ? 1u : 0u);
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          umma_bf16(tmem_base, desc_from_lo(a_lo + kk * 128), desc_from_lo(gl_lo + kk * 128), idesc, 1u);
        umma_commit(&empty[b]);
      }
      __syncwarp();
    }
    if (elect_one()) umma_commit(acc_full);
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 64);
}

}  // namespace tc
}  // namespace udh
