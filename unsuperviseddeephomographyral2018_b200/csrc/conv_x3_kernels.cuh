// Error-compensated tcgen05 implicit-GEMM 3x3 convolution (UDH_NUMERIC_BF16X3): fp32-grade results from 16-bit tensor-core
// operands.  Same padded-stream formulation as conv_tc_kernels.cuh (every tap is a row shift of the flattened activation
// matrix), but every fp32 value travels as TWO 16-bit limbs, x = hi + lo:
//   * activation / gradient streams are [Q positions][hi(C) | lo(C)], packed weights hold [tap][cb][hi | lo][N][64];
//   * a product is evaluated as  lo_x.hi_w + hi_x.hi_w + hi_x.lo_w  — three tcgen05.mma passes into ONE fp32 TMEM
//     accumulator (the dropped lo.lo term and the residual of the split are 2^-16 relative for bf16 limbs);
//   * the epilogue applies bias / ReLU / ReLU-backward mask on the fp32 accumulator, splits the result into limbs again and
//     TMA-stores both (so rounding to 16 bits never enters the data path: the only approximation is the 2^-16 split).
// Shared memory cannot hold double-buffered operands of twice the size, so the two limbs of the A rows live in two SINGLE
// buffers that are consumed in staggered phases: phase LO (A_lo x W_hi, 1/3 of the MMAs) then phase HI (A_hi x W_hi,
// A_hi x W_lo).  A_lo is free again after a third of the item and is refilled under phase HI; A_hi is refilled under the
// next item's phase LO — each limb buffer has its own full/empty mbarrier pair, and a dedicated producer warp so that the
// weight ring (a second producer warp) never waits behind an activation buffer.  Weights always stream through a TMA ring
// (hi + lo of all 9 taps do not fit next to the activations); each ring block is reused by the T tiles of the item.
//   warp 0: weight-ring producer | warp 1: MMA issuer | warp 2: TMEM allocator | warp 3: activation producer |
//   warps 4-11: epilogue (two per TMEM lane quarter, as in the bf16 kernel).
// Phase order: HI first (its first MMA initialises the accumulators), then LO.
// WIDE (64 -> 64 channels): an (M128,N64,K16) MMA is capped at ~50 clk by the A-operand fetch (64 % of the tensor peak), so
// phase HI issues ONE N = 128 MMA per k-step against the ring stage [W_hi | W_lo] (64 clk, full rate) into a MAIN and an AUX
// accumulator (adjacent TMEM columns) instead of two N = 64 MMAs (100 clk); phase LO adds A_lo x W_hi into MAIN; the epilogue
// reads MAIN + AUX.  Two accumulators per tile limit an item to T = 2 tiles (2 sets x 2 tiles x 128 columns = 512).
#pragma once
#include "conv_tc_kernels.cuh"

namespace udh {
namespace tc {

constexpr int kX3MaxStages = 6;

template <int N_OUT, int CB, int T, bool WIDE = false>
struct ConvX3Smem {
  static constexpr int kWStageBytes = N_OUT * 128 * (WIDE ? 2 : 1);
  // fixed part: alignment slack + both limbs of the A rows + epilogue staging + barriers
  static size_t fixed_bytes(int abuf_rows) { return 1024 + (size_t)2 * CB * abuf_rows * 128 + kEpiStageBytes + 256; }
  static int stages(int abuf_rows) {
    const long long left = 232448ll - (long long)fixed_bytes(abuf_rows);
    const int s = (int)(left / kWStageBytes);
    return s > kX3MaxStages ? kX3MaxStages : s;
  }
};

// STAGES > 0: the ring depth is a compile-time constant that divides the stages of an item, so every item starts at ring
// slot 0 and the MMA issue loop is fully unrolled with static slots, parities and tap offsets (ncu of the dynamic loop:
// the weights were never late, but ~90 bookkeeping instructions of the single issuing lane between two groups of MMAs let
// the tensor pipe drain — 54 % active where the issue mix allows 84 %).  STAGES == 0: runtime ring (any depth).  The WIDE
// kernels take the static ring and the other layers the runtime ring, so WIDE == (STAGES > 0).
// ROWS (W == 128 images, 64 -> 64 channels, T == 2: conv1_2).  An item is the interior of two consecutive image rows
// (2y, 2y+1): tile t starts at the first interior position of row 2y + t, i.e. the tiles are Wp (not 128) positions apart in
// the same staged rows, no border position is computed, and the epilogue thread of column x holds both rows of that column.
//   ROWS == 1: forward fused with the 2x2 max-pool — bias + ReLU, maximum (vertical in registers, horizontal with one lane
//              exchange), then the POOLED two-limb stream and the 3-bit routing codes of the max-pool backward are written; the
//              full-resolution activation (554 MB in this mode) is never written or re-read;
//   ROWS == 2: the ordinary epilogue (bias / ReLU-backward mask / limb split / TMA store) on row tiles (the dgrad).
template <int N_OUT, int CB, int T, bool WIDE = false, int STAGES = 0, int ROWS = 0>
__global__ void __launch_bounds__(384, 1)
tc_conv_x3_kernel(const __grid_constant__ CUtensorMap tmA128, const __grid_constant__ CUtensorMap tmAhh,
                  const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmOut, const ConvGeom g,
                  const int stages, const float* __restrict__ bias, const uint32_t* __restrict__ mask_bits,
                  uint32_t* __restrict__ mask_out, float* __restrict__ out_f32, const int relu, const float out_scale) {
  extern __shared__ uint8_t raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  const int abuf_bytes = g.abuf_rows * 128;                       // one 64-channel block of one limb
  uint8_t* sA = base;                                             // [2 limbs][CB][abuf_rows][128]
  uint8_t* sW = base + (size_t)2 * CB * abuf_bytes;               // [stages][N_OUT][128]
  static_assert(!WIDE || (N_OUT == 64 && T <= 2), "WIDE: 64 output channels, two accumulators per tile");
  static_assert(WIDE == (STAGES > 0), "WIDE kernels use the static ring, the others the runtime ring");
  static_assert(ROWS == 0 || (WIDE && CB == 1 && T == 2), "row tiles: the WIDE instance with two tiles");
  constexpr bool POOL = ROWS == 1;
  // first position of an item and distance between its tiles (in positions)
  auto item_q0 = [&](int item) { return ROWS ? ((item / (g.H >> 1)) * g.Hp + 2 * (item % (g.H >> 1)) + 1) * g.Wp + 1 : item * T * 128; };
  const int tstep = ROWS ? g.Wp : 128;
  constexpr int kAcc = WIDE ? 2 : 1;                              // accumulators per tile (MAIN | AUX)
  constexpr int kTileCols = N_OUT * kAcc;                         // TMEM columns per tile
  constexpr int kStageBytes = N_OUT * 128 * kAcc;                 // one ring stage: [W_hi] or [W_hi | W_lo]
  uint8_t* sEpi = sW + (size_t)stages * kStageBytes;              // [4 quarters][32 rows][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sEpi + kEpiStageBytes);
  uint64_t* a_full = bars;            // [2] per limb (0 = hi, 1 = lo)
  uint64_t* a_empty = bars + 2;       // [2]
  uint64_t* t_full = bars + 4;        // [2] per accumulator set
  uint64_t* t_empty = bars + 6;       // [2]
  uint64_t* w_full = bars + 8;        // [kX3MaxStages]
  uint64_t* w_empty = bars + 8 + kX3MaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8 + 2 * kX3MaxStages);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kTmemCols = (2 * T * kTileCols <= 32) ? 32 : (2 * T * kTileCols <= 64) ? 64 : (2 * T * kTileCols <= 128) ? 128
                            : (2 * T * kTileCols <= 256) ? 256 : 512;
  static_assert(2 * T * kTileCols <= 512, "accumulators exceed TMEM");
  static_assert(T <= 4, "mask prefetch registers are sized for T <= 4");

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1);
      mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 256);
    }
    for (int i = 0; i < kX3MaxStages; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { prefetch_tmap(&tmW); prefetch_tmap(&tmOut); }
  if (warp == 3 && lane == 0) { prefetch_tmap(&tmA128); prefetch_tmap(&tmAhh); }
  if (warp == 2) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int my_items = (g.num_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // items blockIdx.x + i*gridDim.x
  pdl_wait();                  // predecessor grid complete: global memory may be touched from here on
  pdl_trigger();

  if (warp == 3) {
    // ===================================== activation producer =====================================
    if (lane == 0) {
      for (int it = 0; it < my_items; ++it) {
        const int q0 = item_q0((int)blockIdx.x + it * (int)gridDim.x);
#pragma unroll 1
        for (int li = 0; li < 2; ++li) {
          const int l = li;                                       // consumption order: hi limb first
          mbar_wait(&a_empty[l], (it & 1) ^ 1);
          mbar_arrive_expect_tx(&a_full[l], (uint32_t)(CB * abuf_bytes));
          for (int cb = 0; cb < CB; ++cb) {
            uint8_t* dst = sA + (size_t)(l * CB + cb) * abuf_bytes;
            const int c0 = (l * CB + cb) * 64;                    // channel coordinate in the [hi | lo] stream
            tma_load_2d(dst, &tmAhh, c0, q0 - g.hh, &a_full[l]);
            for (int t = 0; t < T; ++t)
              tma_load_2d(dst + (size_t)(g.hh + t * 128) * 128, &tmA128, c0, q0 + t * 128, &a_full[l]);
            tma_load_2d(dst + (size_t)(g.hh + T * 128) * 128, &tmAhh, c0, q0 + T * 128, &a_full[l]);
          }
        }
      }
    }
  } else if (warp == 0) {
    // ===================================== weight-ring producer =====================================
    if (lane == 0) {
      uint32_t ws = 0, wpar = 1;                                  // first pass over the ring: the slots are free
      auto push = [&](int block, int nblocks) {                  // `nblocks` consecutive [N_OUT][64] blocks into one stage
        mbar_wait(&w_empty[ws], wpar);
        mbar_arrive_expect_tx(&w_full[ws], (uint32_t)(nblocks * N_OUT * 128));
        for (int i = 0; i < nblocks; ++i)
          tma_load_2d(sW + (size_t)ws * kStageBytes + (size_t)i * N_OUT * 128, &tmW, 0, (block + i) * N_OUT, &w_full[ws]);
        if (++ws == (uint32_t)stages) { ws = 0; wpar ^= 1u; }
      };
      for (int it = 0; it < my_items; ++it) {
        for (int kb = 0; kb < 9 * CB; ++kb) {                                     // phase HI: A_hi x W_hi, A_hi x W_lo
          if (WIDE) push(kb * 2, 2);
          else { push(kb * 2, 1); push(kb * 2 + 1, 1); }
        }
        for (int kb = 0; kb < 9 * CB; ++kb) push(kb * 2, 1);                      // phase LO: A_lo x W_hi
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =====================================
    // The whole warp stays converged (descriptors live in uniform registers); one elected lane issues.
    constexpr uint32_t idesc = make_idesc_bf16(128, N_OUT, 0, 0);
    constexpr uint32_t idesc_wide = make_idesc_bf16(128, 2 * N_OUT, 0, 0);
    const uint32_t a_addr0 = smem_u32(sA), w_addr0 = smem_u32(sW);
    // ring position as a running (stage, parity) pair and taps as running (ky, kx) counters: the issue loop of this single
    // warp is the serial resource of the kernel, so it carries no integer division and no per-block address rebuild
    uint32_t ws = 0, wpar = 0;
    const uint32_t w_stage_units = (uint32_t)kStageBytes >> 4;
    const uint32_t w_lo0 = desc_lo(w_addr0, 16);
    if constexpr (STAGES > 0) {
      constexpr int kHiStages = 9 * CB, kSPI = kHiStages + 9 * CB;                   // ring stages of phase HI / of an item
      static_assert(kSPI % STAGES == 0, "the static ring depth must divide the stages of an item");
      constexpr int kPasses = kSPI / STAGES;
      const uint32_t cb_units = (uint32_t)abuf_bytes >> 4;
      const uint32_t wp8 = (uint32_t)g.Wp * 8;                    // one image row of taps, in sixteen-byte units
      const uint32_t a_hi0 = desc_lo(a_addr0 + (uint32_t)(g.hh - g.Wp - 1) * 128, 16);
      const uint32_t a_lo0 = desc_lo(a_addr0 + (uint32_t)CB * abuf_bytes + (uint32_t)(g.hh - g.Wp - 1) * 128, 16);
      for (int it = 0; it < my_items; ++it) {
        const int b = it & 1;
        const uint32_t itpar = (kPasses & 1) ? (uint32_t)(it & 1) : 0u;
        mbar_wait(&t_empty[b], ((it >> 1) & 1) ^ 1);
        const uint32_t d0 = tmem_base + (uint32_t)(b * T * kTileCols);
        // ONE elected lane runs the whole item (waits included): no per-stage election / reconvergence between MMA groups
        if (elect_one()) {
          mbar_wait(&a_full[0], it & 1);
          tc_fence_after();
#pragma unroll
          for (int j = 0; j < kSPI; ++j) {
            const bool hi = j < kHiStages;
            const int jj = hi ? j : j - kHiStages;
            const int tap = jj / CB, cb = jj - tap * CB;
            const int ky = tap / 3, kx = tap - ky * 3;
            const int s = j % STAGES;
            if (j == kHiStages) {                                 // phase HI done: release the hi rows, take the lo rows
              umma_commit(&a_empty[0]);
              mbar_wait(&a_full[1], it & 1);
              tc_fence_after();
            }
            mbar_wait(&w_full[s], ((uint32_t)(j / STAGES) + itpar) & 1u);
            tc_fence_after();
            const uint32_t a_lo = (hi ? a_hi0 : a_lo0) + (uint32_t)ky * wp8 + (uint32_t)(kx * 8) + (uint32_t)cb * cb_units;
            const uint32_t w_lo = w_lo0 + (uint32_t)s * w_stage_units;
            const uint32_t id = hi ? idesc_wide : idesc;
#pragma unroll
            for (int t = 0; t < T; ++t) {
#pragma unroll
              for (int k = 0; k < 4; ++k)     // tiles are 128 rows (1024 units) apart, or one image row (Wp rows) on row tiles
                umma_bf16(d0 + (uint32_t)(t * kTileCols), desc_from_lo(a_lo + (ROWS ? (uint32_t)t * wp8 : (uint32_t)(t * 1024)) + k * 2),
                          desc_from_lo(w_lo + k * 2), id, (j > 0 || k > 0) ? 1u : 0u);
            }
            umma_commit(&w_empty[s]);
          }
          umma_commit(&a_empty[1]);
          umma_commit(&t_full[b]);
        }
        __syncwarp();
      }
    } else
    for (int it = 0; it < my_items; ++it) {
      const int b = it & 1;
      mbar_wait(&t_empty[b], ((it >> 1) & 1) ^ 1);
      const uint32_t d0 = tmem_base + (uint32_t)(b * T * kTileCols);
      const uint32_t ws0 = ws, wpar0 = wpar;
      if (elect_one()) {                                          // one elected lane runs the whole item (waits included)
#pragma unroll 1
        for (int ph = 0; ph < 2; ++ph) {
          const int l = ph;                                       // phase 0 consumes the hi limb, phase 1 the lo limb
          mbar_wait(&a_full[l], it & 1);
          tc_fence_after();
          // descriptor (low word) of tap (0,0), channel block 0 of this limb: rows start at hh - Wp - 1
          const uint32_t a_tap0 = desc_lo(a_addr0 + (uint32_t)(l * CB) * abuf_bytes + (uint32_t)(g.hh - g.Wp - 1) * 128, 16);
          const uint32_t cb_units = (uint32_t)abuf_bytes >> 4;
          uint32_t first = ph == 0 ? 0u : 1u;                     // the very first MMA of the item overwrites the accumulators
#pragma unroll 1
          for (int ky = 0; ky < 3; ++ky) {
#pragma unroll 1
            for (int kx = 0; kx < 3; ++kx) {
              const uint32_t a_tap = a_tap0 + (uint32_t)(ky * g.Wp + kx) * 8;      // 128-byte rows = 8 sixteen-byte units
#pragma unroll
              for (int cb = 0; cb < CB; ++cb) {
#pragma unroll
                for (int wl = 0; wl < 2; ++wl) {
                  if (wl == 1 && ph == 1) continue;               // phase LO multiplies with W_hi only
                  mbar_wait(&w_full[ws], wpar);
                  tc_fence_after();
                  const uint32_t a_lo = a_tap + (uint32_t)cb * cb_units;
                  const uint32_t w_lo = w_lo0 + ws * w_stage_units;
#pragma unroll
                  for (int t = 0; t < T; ++t) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)     // +1024 sixteen-byte units per tile, +2 per 32-byte k-step
                      umma_bf16(d0 + (uint32_t)(t * kTileCols), desc_from_lo(a_lo + t * 1024 + k * 2), desc_from_lo(w_lo + k * 2), idesc,
                                (first | (uint32_t)(k > 0)) ? 1u : 0u);
                  }
                  umma_commit(&w_empty[ws]);
                  first = 1u;
                  if (++ws == (uint32_t)stages) { ws = 0; wpar ^= 1u; }
                }
              }
            }
          }
          umma_commit(&a_empty[l]);                               // this limb's rows are no longer read -> producer
          if (ph == 1) umma_commit(&t_full[b]);                   // accumulators of this item complete -> epilogue
        }
      }
      __syncwarp();
      // the elected lane advanced its private copy of the ring position: every lane recomputes it (once per item)
      {
        constexpr uint32_t kSPI = (uint32_t)(27 * CB);
        const uint32_t tot = ws0 + kSPI;
        ws = tot % (uint32_t)stages;
        wpar = wpar0 ^ ((tot / (uint32_t)stages) & 1u);
      }
    }
  } else if (warp >= 4) {
    // ===================================== epilogue =====================================
    // Two warps per TMEM lane quarter (warps 4-7 and 8-11): warp group eg owns the 32-column chunk eg of every 64-channel
    // half.  Both warps of a quarter fill their halves of the quarter's 32 x 128 B staging block, meet at a 64-thread named
    // barrier, and one lane issues the TMA store; the hi block and the lo block of a half go through the same staging block.
    const int eg = (warp - 4) >> 2;
    const int ew = (warp - 4) & 3;
    const int HpWp = g.Hp * g.Wp;
    if constexpr (POOL) {
      // thread = image column x (W == 128 == tile rows); warp group eg pools the 32-channel chunk eg
      const int OH = g.H >> 1, OW = g.W >> 1;
      const int x = ew * 32 + lane;
      const int px = x >> 1, odd = x & 1;
      uint16_t* out_pool = reinterpret_cast<uint16_t*>(out_f32);             // pooled two-limb stream [B][OH+2][OW+2][hi 64 | lo 64]
      for (int it = 0; it < my_items; ++it) {
        const int b = it & 1;
        const int item = (int)blockIdx.x + it * (int)gridDim.x;
        const int n = item / OH, yy = item - n * OH;
        mbar_wait(&t_full[b], (it >> 1) & 1);
        tc_fence_after();
        uint16_t* prow = out_pool + (((size_t)n * (OH + 2) + yy + 1) * (OW + 2) + px + 1) * 128;
        uint32_t* crow = mask_out + (((size_t)n * OH + yy) * OW + px) * 8;
        const int c = eg;
        float v0[32], v1[32], u[32];
        const uint32_t tl = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(b * T * kTileCols + c * 32);
        tmem_ld32(tl, v0);                  tmem_ld32(tl + N_OUT, u);
#pragma unroll
        for (int j = 0; j < 32; ++j) v0[j] += u[j];
        tmem_ld32(tl + kTileCols, v1);      tmem_ld32(tl + kTileCols + N_OUT, u);
#pragma unroll
        for (int j = 0; j < 32; ++j) v1[j] += u[j];
        tc_fence_before();
        mbar_arrive(&t_empty[b]);           // the accumulators are in registers: the MMA warp may overwrite this set
        uint32_t code[4] = {0u, 0u, 0u, 0u};
        float m[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float bj = __ldg(bias + c * 32 + j);
          const float a = fmaxf(v0[j] + bj, 0.f), d = fmaxf(v1[j] + bj, 0.f);
          // scan order of the 2x2 window: (row 0, x even)=0, (row 0, x odd)=1, (row 1, even)=2, (row 1, odd)=3;
          // the first maximum wins: larger value, ties to the smaller index
          float vs = a; uint32_t ks = (uint32_t)odd;
          if (d > a) { vs = d; ks = 2u + (uint32_t)odd; }
          const float vo = __shfl_xor_sync(0xffffffffu, vs, 1);
          const uint32_t ko = __shfl_xor_sync(0xffffffffu, ks, 1);
          const bool other = vo > vs || (vo == vs && ko < ks);
          const float mv = other ? vo : vs;
          const uint32_t mk = other ? ko : ks;
          m[j] = mv;
          code[j >> 3] |= (mv > 0.f ? mk : 4u) << (3 * (j & 7));
        }
        // both lanes of a pair hold the pooled pixel: the even lane stores channels 0-15 of this chunk, the odd 16-31
        uint32_t ph_[8], pl_[8];
#pragma unroll
        for (int h = 0; h < 8; ++h) split2(odd ? m[16 + 2 * h] : m[2 * h], odd ? m[17 + 2 * h] : m[2 * h + 1], ph_[h], pl_[h]);
        uint4* oh = reinterpret_cast<uint4*>(prow + c * 32 + odd * 16);
        oh[0] = make_uint4(ph_[0], ph_[1], ph_[2], ph_[3]); oh[1] = make_uint4(ph_[4], ph_[5], ph_[6], ph_[7]);
        uint4* ol = reinterpret_cast<uint4*>(prow + 64 + c * 32 + odd * 16);
        ol[0] = make_uint4(pl_[0], pl_[1], pl_[2], pl_[3]); ol[1] = make_uint4(pl_[4], pl_[5], pl_[6], pl_[7]);
        *reinterpret_cast<uint2*>(crow + c * 4 + odd * 2) = odd ? make_uint2(code[2], code[3]) : make_uint2(code[0], code[1]);
      }
    } else {
    uint8_t* stg = sEpi + ew * 4096;
    const uint32_t my_row = smem_u32(stg) + lane * 128;
    const int sw = lane & 7;
    const bool issuer = eg == 0 && lane == 0;
    auto pair_sync = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(1 + ew) : "memory"); };
    bool store_pending = false;
    for (int it = 0; it < my_items; ++it) {
      const int b = it & 1;
      const int item = (int)blockIdx.x + it * (int)gridDim.x;
      const int q0w0 = item_q0(item) + ew * 32;
      // ReLU-backward mask words (1 bit / element) of all T tiles, requested before the accumulator wait
      uint32_t mbt[T][2];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int qt = q0w0 + t * tstep + lane;
        const bool ok = mask_bits && qt < g.Q;
        if (N_OUT == 64) {
          mbt[t][0] = ok ? __ldg(mask_bits + (size_t)qt * 2 + eg) : 0u; mbt[t][1] = 0u;
        } else {
          mbt[t][0] = ok ? __ldg(mask_bits + (size_t)qt * 4 + eg) : 0u;
          mbt[t][1] = ok ? __ldg(mask_bits + (size_t)qt * 4 + 2 + eg) : 0u;
        }
      }
      mbar_wait(&t_full[b], (it >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int q0w = q0w0 + t * tstep;
        const int q = q0w + lane;
        const int n = q / HpWp, rem = q - n * HpWp;
        const int yp = rem / g.Wp, xp = rem - yp * g.Wp;
        const bool valid = q < g.Q && xp >= 1 && xp <= g.W && yp >= 1 && yp <= g.H;
        const size_t o_f32 = (((size_t)n * g.H + (yp - 1)) * g.W + (xp - 1)) * N_OUT;
        uint32_t mo[N_OUT / 64];
#pragma unroll
        for (int hf = 0; hf < N_OUT / 64; ++hf) {
          const int c = hf * 2 + eg;
          float v[32];
          tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)((b * T + t) * kTileCols + c * 32), v);
          if (WIDE) {                                             // MAIN (A.W_hi terms) + AUX (A_hi.W_lo)
            float u[32];
            tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)((b * T + t) * kTileCols + N_OUT + c * 32), u);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += u[j];
          }
          if (out_scale != 1.0f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= out_scale;
          }
          if (bias) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + c * 32 + j));
              v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
            }
          }
          if (relu) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          if (mask_bits) {
            const uint32_t w = mbt[t][hf];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = ((w >> j) & 1u) ? v[j] : 0.f;
          }
          mo[hf] = 0u;
          if (mask_out) {
            uint32_t w = 0;
#pragma unroll
            for (int j = 0; j < 32; ++j) w |= (v[j] > 0.f ? 1u : 0u) << j;
            mo[hf] = w;
          }
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            if (valid) split2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
            else { hi[j] = 0u; lo[j] = 0u; }                       // border / out-of-range positions store zeros
          }
#pragma unroll
          for (int limb = 0; limb < 2; ++limb) {
            // the staging block may still be read by the previous TMA store
            if (store_pending) { if (issuer) bulk_wait_read0(); pair_sync(); }
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const uint32_t addr = my_row + (uint32_t)(((eg * 4 + j4) ^ sw) << 4);
              const uint32_t* src = limb ? lo : hi;
              asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(src[j4 * 4]), "r"(src[j4 * 4 + 1]),
                           "r"(src[j4 * 4 + 2]), "r"(src[j4 * 4 + 3]) : "memory");
            }
            fence_proxy_async();                    // generic-proxy smem writes -> visible to the TMA engine
            pair_sync();                            // both 64-byte halves of every row are in place
            if (issuer && q0w < g.Q) { tma_store_2d(&tmOut, stg, limb * N_OUT + hf * 64, q0w); bulk_commit(); }
            store_pending = true;
          }
          if (out_f32 && valid) {
            float4* fp = reinterpret_cast<float4*>(out_f32 + o_f32 + c * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j) fp[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
        }
        if (mask_out && q < g.Q) {
#pragma unroll
          for (int hf = 0; hf < N_OUT / 64; ++hf) mask_out[(size_t)q * (N_OUT / 32) + hf * 2 + eg] = valid ? mo[hf] : 0u;
        }
      }
      tc_fence_before();
      mbar_arrive(&t_empty[b]);
    }
    if (issuer) bulk_wait0();
    __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
}

}  // namespace tc
}  // namespace udh
