// UDH_NUMERIC_BF16X3: the regressor on tcgen05 tensor cores with fp32-grade results.  Every fp32 value (activations,
// activation gradients, weights) travels as two 16-bit limbs, x = hi + lo, and every product is evaluated as
// lo.hi + hi.hi + hi.lo with fp32 TMEM accumulation (conv_x3_kernels.cuh, wgrad_x3_kernels.cuh, conv1_x3_kernels.cuh, and
// the segment mechanism of gemm_tc_kernels.cuh for fc1).  Bias, ReLU, masks, pooling decisions, dropout, fc2, losses,
// DLT, warp and Adam are fp32 exactly as in the other modes.  Reference arithmetic matched: fp32 everywhere,
// code/homography_model.py:67,88-133.
#include "conv_tc.cuh"

#include "cnn_kernels.cuh"
#include "conv_x3_kernels.cuh"
#include "wgrad_x3_kernels.cuh"
#include "gemm_tc_kernels.cuh"
#include "conv1_x3_kernels.cuh"
#include "tc_layout.cuh"

namespace udh {

namespace {

using namespace tcl;
#define TRY UDH_TRY

__device__ __forceinline__ void split1(float v, uint16_t& hi, uint16_t& lo) {
  uint32_t h, l;
  tc::split2(v, 0.f, h, l);
  hi = (uint16_t)(h & 0xFFFFu); lo = (uint16_t)(l & 0xFFFFu);
}

// ---------------------------------------------------------------------------------------------------- small kernels
// dst[tap][cb][limb][n][k] 16-bit <- fp32 HWIO w[tap][ci][co]; forward: n = co, k-channel = ci; dgrad: n = ci, k-channel = co,
// tap mirrored.  All seven tensor-core layers, both directions, in one launch: blockIdx.y = layer-1, blockIdx.z = direction.
struct PackTableX3 { const float* w[7]; uint16_t* fwd[7]; uint16_t* dgr[7]; int cin[7], cout[7]; };
__global__ void pack_all_weights_x3_kernel(PackTableX3 t) {
  pdl_wait(); pdl_trigger();
  const int L = blockIdx.y, dgrad = blockIdx.z;
  const int Cin = t.cin[L], Cout = t.cout[L];
  const int K = dgrad ? Cout : Cin, N = dgrad ? Cin : Cout, CBk = K / 64, total = 9 * K * N;
  const float* __restrict__ w = t.w[L];
  uint16_t* __restrict__ dst = dgrad ? t.dgr[L] : t.fwd[L];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i & 63;
    int r = i >> 6;
    const int n = r % N; r /= N;
    const int cb = r % CBk;
    const int tap = r / CBk;
    const int kc = cb * 64 + k;
    const float v = dgrad ? w[((size_t)(8 - tap) * Cin + n) * Cout + kc] : w[((size_t)tap * Cin + kc) * Cout + n];
    uint16_t hi, lo;
    split1(v, hi, lo);
    const size_t blk = (size_t)(tap * CBk + cb) * 2;
    dst[(blk * N + n) * 64 + k] = hi;
    dst[((blk + 1) * N + n) * 64 + k] = lo;
  }
}

// fp32 [B,H,W,C] -> limb stream [B,H+2,W+2,2C] interior (borders untouched = zero)
__global__ void pad_cast_x3_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, int B, int H, int W, int C) {
  pdl_wait(); pdl_trigger();
  const int C4 = C >> 2;
  const size_t total = (size_t)B * H * W * C4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c4 = i % C4;
    size_t r = i / C4;
    const int x = r % W; r /= W;
    const int y = r % H;
    const int n = r / H;
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    uint2 hi, lo;
    tc::split2(v.x, v.y, hi.x, lo.x);
    tc::split2(v.z, v.w, hi.y, lo.y);
    uint16_t* p = dst + (((size_t)n * (H + 2) + y + 1) * (W + 2) + x + 1) * (2 * C) + c4 * 4;
    *reinterpret_cast<uint2*>(p) = hi;
    *reinterpret_cast<uint2*>(p + C) = lo;
  }
}

// limb stream interior -> fp32 [B,H,W,C] (debug / tests)
__global__ void unpad_cast_x3_kernel(const uint16_t* __restrict__ src, float* __restrict__ dst, int B, int H, int W, int C) {
  const int C4 = C >> 2;
  const size_t total = (size_t)B * H * W * C4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c4 = i % C4;
    size_t r = i / C4;
    const int x = r % W; r /= W;
    const int y = r % H;
    const int n = r / H;
    const uint16_t* p = src + (((size_t)n * (H + 2) + y + 1) * (W + 2) + x + 1) * (2 * C) + c4 * 4;
    const uint2 hi = __ldg(reinterpret_cast<const uint2*>(p)), lo = __ldg(reinterpret_cast<const uint2*>(p + C));
    const float2 a = tc::join2(hi.x, lo.x), b = tc::join2(hi.y, lo.y);
    reinterpret_cast<float4*>(dst)[i] = make_float4(a.x, a.y, b.x, b.y);
  }
}

// fp32 [rows][cols] -> [rows][hi(cols) | lo(cols)]
__global__ void cast_x3_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, size_t rows, int cols) {
  pdl_wait(); pdl_trigger();
  const int C4 = cols >> 2;
  const size_t total = rows * C4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / C4;
    const int c4 = (int)(i - r * C4);
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    uint2 hi, lo;
    tc::split2(v.x, v.y, hi.x, lo.x);
    tc::split2(v.z, v.w, hi.y, lo.y);
    uint16_t* p = dst + r * (size_t)(2 * cols) + c4 * 4;
    *reinterpret_cast<uint2*>(p) = hi;
    *reinterpret_cast<uint2*>(p + cols) = lo;
  }
}

// fp32 [n] -> hi[n], lo[n] (fc1's weight mirror: W_hi rows then W_lo rows)
__global__ void cast_planes_x3_kernel(const float* __restrict__ src, uint16_t* __restrict__ hi_dst, uint16_t* __restrict__ lo_dst, size_t n4) {
  pdl_wait(); pdl_trigger();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    uint2 hi, lo;
    tc::split2(v.x, v.y, hi.x, lo.x);
    tc::split2(v.z, v.w, hi.y, lo.y);
    reinterpret_cast<uint2*>(hi_dst)[i] = hi;
    reinterpret_cast<uint2*>(lo_dst)[i] = lo;
  }
}

__device__ __forceinline__ void join8(const uint4& h, const uint4& l, float (&f)[8]) {
  const float2 a = tc::join2(h.x, l.x), b = tc::join2(h.y, l.y), c = tc::join2(h.z, l.z), d = tc::join2(h.w, l.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint16_t half_of(uint32_t w, int odd) { return (uint16_t)(odd ? (w >> 16) : (w & 0xFFFFu)); }

// 2x2/2 max pool on limb streams.  The decision uses the value hi + lo; the winner's limbs are copied unchanged, so pooling
// adds no rounding.  Routing codes as in pool_fwd_bf16_kernel (3 bits per channel, 4 = maximum not positive).
__global__ void pool_fwd_x3_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, uint32_t* __restrict__ codes,
                                   int B, int H, int W, int C) {
  pdl_wait(); pdl_trigger();
  const int C8 = C >> 3, OH = H >> 1, OW = W >> 1;
  const size_t total = (size_t)B * OH * OW * C8;
  const size_t pix = 2 * (size_t)C;                               // elements per stream position
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c8 = i % C8;
    size_t r = i / C8;
    const int ox = r % OW; r /= OW;
    const int oy = r % OH;
    const int n = r / OH;
    const uint16_t* p = in + (((size_t)n * (H + 2) + 2 * oy + 1) * (W + 2) + 2 * ox + 1) * pix + c8 * 8;
    const size_t rowp = (size_t)(W + 2) * pix;
    uint4 h[4], l[4];
    h[0] = __ldg(reinterpret_cast<const uint4*>(p));               l[0] = __ldg(reinterpret_cast<const uint4*>(p + C));
    h[1] = __ldg(reinterpret_cast<const uint4*>(p + pix));         l[1] = __ldg(reinterpret_cast<const uint4*>(p + pix + C));
    h[2] = __ldg(reinterpret_cast<const uint4*>(p + rowp));        l[2] = __ldg(reinterpret_cast<const uint4*>(p + rowp + C));
    h[3] = __ldg(reinterpret_cast<const uint4*>(p + rowp + pix));  l[3] = __ldg(reinterpret_cast<const uint4*>(p + rowp + pix + C));
    float f[4][8];
#pragma unroll
    for (int k = 0; k < 4; ++k) join8(h[k], l[k], f[k]);
    uint32_t code = 0;
    uint32_t oh[4] = {0, 0, 0, 0}, ol[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = f[0][j]; uint32_t k = 0;
      if (f[1][j] > v) { v = f[1][j]; k = 1; }
      if (f[2][j] > v) { v = f[2][j]; k = 2; }
      if (f[3][j] > v) { v = f[3][j]; k = 3; }
      code |= (v > 0.f ? k : 4u) << (3 * j);
      const uint4 hs = k == 0 ? h[0] : k == 1 ? h[1] : k == 2 ? h[2] : h[3];
      const uint4 ls = k == 0 ? l[0] : k == 1 ? l[1] : k == 2 ? l[2] : l[3];
      const uint32_t hw = (j >> 1) == 0 ? hs.x : (j >> 1) == 1 ? hs.y : (j >> 1) == 2 ? hs.z : hs.w;
      const uint32_t lw = (j >> 1) == 0 ? ls.x : (j >> 1) == 1 ? ls.y : (j >> 1) == 2 ? ls.z : ls.w;
      oh[j >> 1] |= (uint32_t)half_of(hw, j & 1) << (16 * (j & 1));
      ol[j >> 1] |= (uint32_t)half_of(lw, j & 1) << (16 * (j & 1));
    }
    uint16_t* o = out + (((size_t)n * (OH + 2) + oy + 1) * (OW + 2) + ox + 1) * pix + c8 * 8;
    *reinterpret_cast<uint4*>(o) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
    *reinterpret_cast<uint4*>(o + C) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
    codes[i] = code;
  }
}

// gradient routing of the above + ReLU mask of the producer, from the forward's routing codes (limbs are moved, not re-split)
__global__ void pool_bwd_x3_kernel(const uint32_t* __restrict__ codes, const uint16_t* __restrict__ gout, uint16_t* __restrict__ gin,
                                   int B, int H, int W, int C) {
  pdl_wait(); pdl_trigger();
  const int C8 = C >> 3, OH = H >> 1, OW = W >> 1;
  const size_t total = (size_t)B * OH * OW * C8;
  const size_t pix = 2 * (size_t)C;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c8 = i % C8;
    size_t r = i / C8;
    const int ox = r % OW; r /= OW;
    const int oy = r % OH;
    const int n = r / OH;
    const size_t base = (((size_t)n * (H + 2) + 2 * oy + 1) * (W + 2) + 2 * ox + 1) * pix + c8 * 8;
    const size_t rowp = (size_t)(W + 2) * pix;
    const uint32_t code = __ldg(codes + i);
    const uint16_t* gp = gout + (((size_t)n * (OH + 2) + oy + 1) * (OW + 2) + ox + 1) * pix + c8 * 8;
    const uint4 gh = __ldg(reinterpret_cast<const uint4*>(gp)), gl = __ldg(reinterpret_cast<const uint4*>(gp + C));
    const uint32_t ghw[4] = {gh.x, gh.y, gh.z, gh.w}, glw[4] = {gl.x, gl.y, gl.z, gl.w};
    uint32_t oh[4][4], ol[4][4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int w = 0; w < 4; ++w) { oh[k][w] = 0u; ol[k][w] = 0u; }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t k = (code >> (3 * j)) & 7u;
      const uint32_t hm = ghw[j >> 1] & (0xFFFFu << (16 * (j & 1))), lm = glw[j >> 1] & (0xFFFFu << (16 * (j & 1)));
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        if (k == (uint32_t)kk) { oh[kk][j >> 1] |= hm; ol[kk][j >> 1] |= lm; }
      }
    }
    const size_t offs[4] = {0, pix, rowp, rowp + pix};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      *reinterpret_cast<uint4*>(gin + base + offs[k]) = make_uint4(oh[k][0], oh[k][1], oh[k][2], oh[k][3]);
      *reinterpret_cast<uint4*>(gin + base + offs[k] + C) = make_uint4(ol[k][0], ol[k][1], ol[k][2], ol[k][3]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------- launchers
template <int N_OUT, int CB, int T, bool WIDE, int STAGES>
int launch_conv_x3_impl(const CUtensorMap& tmA128, const CUtensorMap& tmAhh, const CUtensorMap& tmW, const CUtensorMap& tmOut, const tc::ConvGeom& g,
                        int stages, size_t smem, const float* bias, const uint32_t* mask_bits, uint32_t* mask_out, float* out_f32, int relu,
                        float out_scale, cudaStream_t st) {
  auto kern = tc::tc_conv_x3_kernel<N_OUT, CB, T, WIDE, STAGES>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = persistent_ctas();
  const int grid = g.num_items < sms ? g.num_items : sms;
  launch_chain(kern, dim3(grid), dim3(384), smem, st, tmA128, tmAhh, tmW, tmOut, g, stages, bias, mask_bits, mask_out, out_f32, relu, out_scale);
  return check_launch("tc_conv_x3_kernel");
}

template <int N_OUT, int CB, int T, bool WIDE = false>
int launch_conv_x3(const uint16_t* x, const uint16_t* wpk, const float* bias, const uint32_t* mask_bits, uint32_t* mask_out,
                   uint16_t* out_limbs, float* out_f32, int relu, int B, int H, int W, float out_scale, cudaStream_t st) {
  tc::ConvGeom g;
  g.B = B; g.H = H; g.W = W; g.Hp = H + 2; g.Wp = W + 2;
  g.Q = B * g.Hp * g.Wp;
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  const int tiles = (g.Q + 127) / 128;
  g.num_items = (tiles + T - 1) / T;
  g.abuf_rows = T * 128 + 2 * g.hh;
  const int Cin2 = 2 * CB * 64;
  CUtensorMap tmA128, tmAhh, tmW, tmOut;
  uint64_t dimsA[2] = {(uint64_t)Cin2, (uint64_t)g.Q}, strA[2] = {2, (uint64_t)Cin2 * 2};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh};
  TRY(tc::make_tmap_bf16(&tmA128, x, 2, dimsA, strA, box128));
  TRY(tc::make_tmap_bf16(&tmAhh, x, 2, dimsA, strA, boxhh));
  uint64_t dimsW[2] = {64, (uint64_t)18 * CB * N_OUT}, strW[2] = {2, 128};
  uint32_t boxW[2] = {64, (uint32_t)N_OUT};
  TRY(tc::make_tmap_bf16(&tmW, wpk, 2, dimsW, strW, boxW));
  uint64_t dimsO[2] = {(uint64_t)2 * N_OUT, (uint64_t)g.Q}, strO[2] = {2, (uint64_t)2 * N_OUT * 2};
  uint32_t boxO[2] = {64, 32};
  TRY(tc::make_tmap_bf16(&tmOut, out_limbs, 2, dimsO, strO, boxO));
  using S = tc::ConvX3Smem<N_OUT, CB, T, WIDE>;
  int stages = S::stages(g.abuf_rows);
  // WIDE: static ring (unrolled issue loop) of depth 6 when it fits, else 3 (both divide the 18 stages of an item; at W = 64
  // six fit, at W = 128 four).  The other instances are better off with the deepest runtime ring that fits (measured).
  UDH_REQUIRE(stages >= (WIDE ? 3 : 2), "tc conv x3: activation rows (%d x %d blocks) leave no room for the weight ring", g.abuf_rows, 2 * CB);
  if constexpr (WIDE) stages = stages >= 6 ? 6 : 3;
  const size_t smem = S::fixed_bytes(g.abuf_rows) + (size_t)stages * S::kWStageBytes;
  if constexpr (WIDE) {
    if (stages == 6)
      return launch_conv_x3_impl<N_OUT, CB, T, true, 6>(tmA128, tmAhh, tmW, tmOut, g, stages, smem, bias, mask_bits, mask_out, out_f32, relu, out_scale, st);
    return launch_conv_x3_impl<N_OUT, CB, T, true, 3>(tmA128, tmAhh, tmW, tmOut, g, stages, smem, bias, mask_bits, mask_out, out_f32, relu, out_scale, st);
  } else {
    return launch_conv_x3_impl<N_OUT, CB, T, false, 0>(tmA128, tmAhh, tmW, tmOut, g, stages, smem, bias, mask_bits, mask_out, out_f32, relu, out_scale, st);
  }
}

// conv1_2 on row tiles (64 -> 64 channels, 128-wide images): ROWS = 1 forward fused with pool1 (writes the pooled two-limb
// stream + routing codes), ROWS = 2 the dgrad (ordinary epilogue).  See conv_x3_kernels.cuh.
template <int ROWS>
int launch_conv_x3_rows(const uint16_t* x, const uint16_t* wpk, const float* bias, const uint32_t* mask_bits, uint32_t* codes_or_mask,
                        uint16_t* out_limbs, int relu, int B, int H, int W, cudaStream_t st) {
  UDH_REQUIRE(W == 128 && H % 2 == 0 && out_limbs, "tc conv x3 rows: needs W == 128, an even height and an output stream");
  tc::ConvGeom g;
  g.B = B; g.H = H; g.W = W; g.Hp = H + 2; g.Wp = W + 2;
  g.Q = B * g.Hp * g.Wp;
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  g.num_items = B * (H / 2);
  g.abuf_rows = 2 * 128 + 2 * g.hh;
  UDH_REQUIRE(g.hh + g.Wp + 128 + g.Wp + 1 <= g.abuf_rows, "tc conv x3 rows: halo does not cover the second row tile");
  CUtensorMap tmA128, tmAhh, tmW, tmOut;
  uint64_t dimsA[2] = {128, (uint64_t)g.Q}, strA[2] = {2, 256};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh}, boxO[2] = {64, 32};
  TRY(tc::make_tmap_bf16(&tmA128, x, 2, dimsA, strA, box128));
  TRY(tc::make_tmap_bf16(&tmAhh, x, 2, dimsA, strA, boxhh));
  uint64_t dimsW[2] = {64, (uint64_t)18 * 64}, strW[2] = {2, 128};
  uint32_t boxW[2] = {64, 64};
  TRY(tc::make_tmap_bf16(&tmW, wpk, 2, dimsW, strW, boxW));
  // ROWS = 1 stores the pooled stream with plain vector stores (the map is only a placeholder there)
  TRY(tc::make_tmap_bf16(&tmOut, ROWS == 2 ? out_limbs : const_cast<uint16_t*>(x), 2, dimsA, strA, boxO));
  using S = tc::ConvX3Smem<64, 1, 2, true>;
  constexpr int kStages = 3;
  const size_t smem = S::fixed_bytes(g.abuf_rows) + (size_t)kStages * S::kWStageBytes;
  UDH_REQUIRE(smem <= 232448, "tc conv x3 rows: %zu bytes of shared memory exceed the 227 KiB limit", smem);
  auto kern = tc::tc_conv_x3_kernel<64, 1, 2, true, kStages, ROWS>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = persistent_ctas();
  const int grid = g.num_items < sms ? g.num_items : sms;
  // ROWS = 1: `out_f32` carries the pooled stream pointer and `mask_out` the routing codes
  launch_chain(kern, dim3(grid), dim3(384), smem, st, tmA128, tmAhh, tmW, tmOut, g, kStages, bias, mask_bits, codes_or_mask,
               ROWS == 1 ? reinterpret_cast<float*>(out_limbs) : (float*)nullptr, relu, 1.0f);
  return check_launch("tc_conv_x3_kernel(rows)");
}

// one 3x3 conv on limb streams; (cin -> cout) selects the kernel instance
int tc_conv_x3(const uint16_t* x, const uint16_t* wpk, const float* bias, const uint32_t* mask_bits, uint32_t* mask_out,
               uint16_t* out_limbs, float* out_f32, int relu, int B, int H, int W, int cin, int cout, cudaStream_t st) {
  if (cin == 64 && cout == 64) return launch_conv_x3<64, 1, 2, true>(x, wpk, bias, mask_bits, mask_out, out_limbs, out_f32, relu, B, H, W, 1.0f, st);
  if (cin == 64 && cout == 128) return launch_conv_x3<128, 1, 2>(x, wpk, bias, mask_bits, mask_out, out_limbs, out_f32, relu, B, H, W, 1.0f, st);
  if (cin == 128 && cout == 64) return launch_conv_x3<64, 2, 2>(x, wpk, bias, mask_bits, mask_out, out_limbs, out_f32, relu, B, H, W, 1.0f, st);
  if (cin == 128 && cout == 128) return launch_conv_x3<128, 2, 2>(x, wpk, bias, mask_bits, mask_out, out_limbs, out_f32, relu, B, H, W, 1.0f, st);
  set_error("tc_conv_x3: unsupported channel combination %d -> %d", cin, cout);
  return UDH_ENOSUP;
}

template <int N_OUT, int CBX, int T>
int launch_wgrad_x3(const uint16_t* x, const uint16_t* gsrc, float* dW, float* db, int B, int H, int W, cudaStream_t st) {
  tc::WgradGeom g;
  g.Wp = W + 2;
  g.Q = B * (H + 2) * (W + 2);
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  const int tiles = (g.Q + 127) / 128;
  g.num_items = (tiles + T - 1) / T;
  g.xrows = T * 128 + 2 * g.hh;
  g.num_groups = CBX == 1 ? 5 : 10;
  const int sms = persistent_ctas();
  const int max_groups = 512 / N_OUT;                              // accumulators of one slice fit TMEM
  g.num_slices = (g.num_groups + max_groups - 1) / max_groups;
  g.slice_group[0] = 0; g.slice_cta[0] = 0;
  for (int s = 0; s < g.num_slices; ++s) {
    g.slice_group[s + 1] = g.slice_group[s] + g.num_groups / g.num_slices + (s < g.num_groups % g.num_slices ? 1 : 0);
    g.slice_cta[s + 1] = (int)((long long)sms * g.slice_group[s + 1] / g.num_groups);
    if (g.slice_cta[s + 1] <= g.slice_cta[s]) g.slice_cta[s + 1] = g.slice_cta[s] + 1;
  }
  constexpr int CBO = N_OUT / 64;
  const int Cin2 = 2 * CBX * 64;
  CUtensorMap tmX128, tmXhh, tmG;
  uint64_t dimsX[2] = {(uint64_t)Cin2, (uint64_t)g.Q}, strX[2] = {2, (uint64_t)Cin2 * 2};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh};
  TRY(tc::make_tmap_bf16(&tmX128, x, 2, dimsX, strX, box128));
  TRY(tc::make_tmap_bf16(&tmXhh, x, 2, dimsX, strX, boxhh));
  uint64_t dimsG[2] = {(uint64_t)2 * N_OUT, (uint64_t)g.Q}, strG[2] = {2, (uint64_t)2 * N_OUT * 2};
  TRY(tc::make_tmap_bf16(&tmG, gsrc, 2, dimsG, strG, box128));
  const size_t smem = 1024 + 2 * ((size_t)CBX * g.xrows * 128 + (size_t)CBO * T * 16384) + 2 * tc::kConstBlockBytes + 256;
  UDH_REQUIRE(smem <= 232448, "tc wgrad x3: %zu bytes of shared memory exceed the 227 KiB limit", smem);
  auto kern = tc::tc_wgrad_x3_kernel<N_OUT, CBX, T>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_chain(kern, dim3(g.slice_cta[g.num_slices]), dim3(256), smem, st, tmX128, tmXhh, tmG, g, dW, db);
  return check_launch("tc_wgrad_x3_kernel");
}

int launch_wgrad64_x3(const uint16_t* x, const uint16_t* gsrc, float* dW, float* db, int B, int H, int W, cudaStream_t st) {
  constexpr int T = 2;
  tc::Wgrad64Geom g;
  g.Wp = W + 2;
  g.Q = B * (H + 2) * (W + 2);
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  const int tiles = (g.Q + 127) / 128;
  g.num_items = (tiles + T - 1) / T;
  g.xrows = T * 128 + 2 * g.hh;
  CUtensorMap tmX128, tmXhh, tmG136;
  uint64_t dims[2] = {128, (uint64_t)g.Q}, str[2] = {2, 256};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh}, box136[2] = {64, 136};
  TRY(tc::make_tmap_bf16(&tmX128, x, 2, dims, str, box128));
  TRY(tc::make_tmap_bf16(&tmXhh, x, 2, dims, str, boxhh));
  TRY(tc::make_tmap_bf16(&tmG136, gsrc, 2, dims, str, box136));
  const size_t smem = 1024 + 2 * ((size_t)g.xrows * 128 + (size_t)(T * 128 + 16) * 128) + 2 * tc::kConstBlockBytes + 256;
  UDH_REQUIRE(smem <= 232448, "tc wgrad64 x3: %zu bytes of shared memory exceed the 227 KiB limit", smem);
  auto kern = tc::tc_wgrad64_x3_kernel<T>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = persistent_ctas();
  launch_chain(kern, dim3(g.num_items < sms ? g.num_items : sms), dim3(256), smem, st, tmX128, tmXhh, tmG136, g, dW, db);
  return check_launch("tc_wgrad64_x3_kernel");
}

int tc_wgrad_x3(const uint16_t* x, const uint16_t* gsrc, float* dW, float* db, int B, int H, int W, int cin, int cout, cudaStream_t st) {
  if (cin == 64 && cout == 64) return launch_wgrad64_x3(x, gsrc, dW, db, B, H, W, st);
  if (cin == 64 && cout == 128) return launch_wgrad_x3<128, 1, 1>(x, gsrc, dW, db, B, H, W, st);
  if (cin == 128 && cout == 128) return launch_wgrad_x3<128, 2, 1>(x, gsrc, dW, db, B, H, W, st);
  set_error("tc_wgrad_x3: unsupported channel combination %d -> %d", cin, cout);
  return UDH_ENOSUP;
}

int pad_cast_x3(const float* src, uint16_t* dst, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * H * W * (C / 4);
  launch_chain(pad_cast_x3_kernel, dim3(grid1d((total + 255) / 256, 148 * 32)), dim3(256), 0, st, src, dst, B, H, W, C);
  return check_launch("pad_cast_x3");
}
int unpad_cast_x3(const uint16_t* src, float* dst, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * H * W * (C / 4);
  unpad_cast_x3_kernel<<<grid1d((total + 255) / 256, 148 * 32), 256, 0, st>>>(src, dst, B, H, W, C);
  return check_launch("unpad_cast_x3");
}
int cast_x3(const float* src, uint16_t* dst, size_t rows, int cols, cudaStream_t st) {
  const size_t total = rows * (cols / 4);
  launch_chain(cast_x3_kernel, dim3(grid1d((total + 255) / 256, 148 * 16)), dim3(256), 0, st, src, dst, rows, cols);
  return check_launch("cast_x3");
}
int pool_fwd_x3(const uint16_t* in, uint16_t* out, uint32_t* codes, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * (H / 2) * (W / 2) * (C / 8);
  launch_chain(pool_fwd_x3_kernel, dim3(grid1d((total + 255) / 256, 148 * 32)), dim3(256), 0, st, in, out, codes, B, H, W, C);
  return check_launch("pool_fwd_x3");
}
int pool_bwd_x3(const uint32_t* codes, const uint16_t* gout, uint16_t* gin, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * (H / 2) * (W / 2) * (C / 8);
  launch_chain(pool_bwd_x3_kernel, dim3(grid1d((total + 255) / 256, 148 * 32)), dim3(256), 0, st, codes, gout, gin, B, H, W, C);
  return check_launch("pool_bwd_x3");
}

int conv1_x3_fwd(const float* I1, const float* I2, const float* w, const float* bias, uint16_t* out_limbs, uint32_t* mask_out, int B,
                 int H, int W, cudaStream_t st) {
  UDH_REQUIRE(W % 128 == 0, "conv1_x3_fwd: image width must be a multiple of 128");
  tc::Conv1Geom g{B, H, W, B * H * (W / 128)};
  CUtensorMap tmOut;
  const uint64_t Q = (uint64_t)B * (H + 2) * (W + 2);
  uint64_t dims[2] = {128, Q}, str[2] = {2, 256};
  uint32_t box[2] = {64, 32};
  TRY(tc::make_tmap_bf16(&tmOut, out_limbs, 2, dims, str, box));
  const size_t smem = 1024 + 2 * 16384 + 16384 + 16384 + 256;
  auto kern = tc::conv1_x3_fwd_kernel;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int want = tc::kConv1X3CtasPerSm * persistent_ctas();
  const int grid = g.tiles < want ? g.tiles : want;
  launch_chain(kern, dim3(grid), dim3(160), smem, st, tmOut, g, I1, I2, w, bias, mask_out);
  return check_launch("conv1_x3_fwd_kernel");
}

int conv1_x3_wgrad(const float* I1, const float* I2, const uint16_t* G_limbs, float* dW, float* db, int B, int H, int W, cudaStream_t st) {
  UDH_REQUIRE(W % 128 == 0, "conv1_x3_wgrad: image width must be a multiple of 128");
  tc::Conv1Geom g{B, H, W, B * H * (W / 128)};
  CUtensorMap tmG;
  const uint64_t Q = (uint64_t)B * (H + 2) * (W + 2);
  uint64_t dims[2] = {128, Q}, str[2] = {2, 256};
  uint32_t box[2] = {64, 128};
  TRY(tc::make_tmap_bf16(&tmG, G_limbs, 2, dims, str, box));
  const size_t smem = 1024 + 2 * 16384 + 4 * 16384 + 256;
  auto kern = tc::conv1_x3_wgrad_kernel;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int want = tc::kConv1X3WgradCtasPerSm * persistent_ctas();
  const int grid = g.tiles < want ? g.tiles : want;
  launch_chain(kern, dim3(grid), dim3(160), smem, st, tmG, g, I1, I2, dW, db);
  return check_launch("conv1_x3_wgrad_kernel");
}

inline uint16_t* U16(char* base, size_t off) { return reinterpret_cast<uint16_t*>(base + off); }

// conv1_2 on row tiles (forward fused with pool1, row-tile dgrad): on by default, udh_debug_x3_set_rows(0) selects the
// generic flattened-tile kernels + the separate pool kernel (tests compare the two)
int g_x3_rows = 1;

}  // namespace

int x3_cnn_fwd_convs(const float* params, const size_t* poff, const float* I1, const float* I2, void* ws, const size_t* act_off,
                     size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P, 2);
  char* tcw = at<char>(ws, tc_off);
  {
    // forward AND mirrored (dgrad) limb packs of the seven tensor-core layers, one launch per step
    ProfScope ps(PROF_TC_PREP, st);
    PackTableX3 t;
    for (int i = 1; i < 8; ++i) {
      t.w[i - 1] = params + poff[2 * i];
      t.fwd[i - 1] = U16(tcw, L.wf[i]);
      t.dgr[i - 1] = U16(tcw, L.wd[i]);
      t.cin[i - 1] = kConv[i].cin; t.cout[i - 1] = kConv[i].cout;
    }
    launch_chain(pack_all_weights_x3_kernel, dim3(72, 7, 2), dim3(256), 0, st, t);
    TRY(check_launch("pack_all_weights_x3"));
  }
  {
    ProfScope ps(PROF_CONV_FWD0, st);
    TRY(conv1_x3_fwd(I1, I2, params + poff[0], params + poff[1], U16(tcw, L.P[0]), reinterpret_cast<uint32_t*>(tcw + L.Mb[0]), B, P, P, st));
  }
  const bool fuse_pool1 = g_x3_rows && P == 128;            // conv1_2 + pool1 in one kernel (row tiles need 128-wide images)
  for (int i = 1; i < 8; ++i) {
    const int s = P / kConv[i].div;
    if (i == 1 && fuse_pool1) {
      ProfScope ps(PROF_CONV_FWD0 + i, st);
      TRY((launch_conv_x3_rows<1>(U16(tcw, L.P[0]), U16(tcw, L.wf[1]), params + poff[3], nullptr,
                                  reinterpret_cast<uint32_t*>(tcw + L.Px[0]), U16(tcw, L.P[8]), 1, B, s, s, st)));
      continue;
    }
    {
      ProfScope ps(PROF_CONV_FWD0 + i, st);
      TRY(tc_conv_x3(U16(tcw, L.P[input_of(i)]), U16(tcw, L.wf[i]), params + poff[2 * i + 1], nullptr,
                     (i % 2 == 0) ? reinterpret_cast<uint32_t*>(tcw + L.Mb[i]) : nullptr, U16(tcw, L.P[i]),
                     i == 7 ? at<float>(ws, act_off[7]) : nullptr, 1, B, s, s, kConv[i].cin, kConv[i].cout, st));
    }
    if (i == 1 || i == 3 || i == 5) {
      ProfScope ps(PROF_POOL_FWD, st);
      TRY(pool_fwd_x3(U16(tcw, L.P[i]), U16(tcw, L.P[8 + i / 2]), reinterpret_cast<uint32_t*>(tcw + L.Px[i / 2]), B, s, s, kConv[i].cout, st));
    }
  }
  return UDH_OK;
}

int x3_cnn_bwd_convs(const float* params, const size_t* poff, const float* I1, const float* I2, float* grads, float* gA, void* ws,
                     size_t tc_off, int B, int P, cudaStream_t st) {
  (void)params;
  TcLayout L(B, P, 2);
  char* tcw = at<char>(ws, tc_off);
  {
    ProfScope ps(PROF_TC_PREP, st);        // (the mirrored weight packs were made by the forward of this step)
    TRY(pad_cast_x3(gA, U16(tcw, L.G[7]), B, P / 8, P / 8, 128, st));
  }
  struct RestoreReserve { ~RestoreReserve() { g_sm_reserve = 0; } } restore_reserve;   // outside the conv backward every SM is used
  for (int i = 7; i >= 0; --i) {
    TRY(bwd_marker_record(i, st));
    const int s = P / kConv[i].div;
    const int cin = kConv[i].cin, cout = kConv[i].cout;
    g_sm_reserve = bwd_sm_reserve(i);   // see udh_set_sm_reserve_top
    {
      ProfScope ps(PROF_CONV_WGRAD0 + i, st);
      if (i == 0) TRY(conv1_x3_wgrad(I1, I2, U16(tcw, L.G[0]), grads + poff[0], grads + poff[1], B, s, s, st));
      else TRY(tc_wgrad_x3(U16(tcw, L.P[input_of(i)]), U16(tcw, L.G[i]), grads + poff[2 * i], grads + poff[2 * i + 1], B, s, s, cin, cout, st));
    }
    if (i == 0) break;
    const bool below_is_pool = (i == 2 || i == 4 || i == 6);
    const int below = input_of(i);
    if (i == 1 && g_x3_rows && P == 128) {
      ProfScope ps(PROF_CONV_DGRAD0 + i, st);                 // conv1_2 dgrad on row tiles, ReLU mask of conv1_1 fused
      TRY((launch_conv_x3_rows<2>(U16(tcw, L.G[1]), U16(tcw, L.wd[1]), nullptr, reinterpret_cast<const uint32_t*>(tcw + L.Mb[0]),
                                  nullptr, U16(tcw, L.G[0]), 0, B, s, s, st)));
      continue;
    }
    {
      ProfScope ps(PROF_CONV_DGRAD0 + i, st);
      // dgrad = conv of G[i] with the mirrored kernel; ReLU mask of the layer below fused unless a pool sits between
      TRY(tc_conv_x3(U16(tcw, L.G[i]), U16(tcw, L.wd[i]), nullptr,
                     below_is_pool ? nullptr : reinterpret_cast<const uint32_t*>(tcw + L.Mb[below]), nullptr,
                     U16(tcw, L.G[below]), nullptr, 0, B, s, s, cout, cin, st));
    }
    if (below_is_pool) {
      ProfScope ps(PROF_POOL_BWD, st);
      TRY(pool_bwd_x3(reinterpret_cast<const uint32_t*>(tcw + L.Px[i / 2 - 1]), U16(tcw, L.G[below]), U16(tcw, L.G[i - 1]), B, 2 * s, 2 * s, cin, st));
    }
  }
  return UDH_OK;
}

// tests: write fp32 copies (hi + lo) of the saved conv / pool activations into the fp32 activation slots of the workspace
// (the slots the CUDA-core mode uses), so that a test can read them or run the fp32 backward on this mode's forward state
int x3_materialize_acts(void* ws, const size_t* act_off, size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P, 2);
  char* tcw = at<char>(ws, tc_off);
  for (int i = 0; i < 11; ++i) {
    if (i == 7) continue;                                    // conv4_2 is written in fp32 by the forward itself
    if (i == 1 && P == 128 && g_x3_rows) continue;           // conv1_2 is fused with pool1: its full-resolution output is never stored
    const int s = i < 8 ? P / kConv[i].div : P >> (i - 7);
    const int c = i < 8 ? kConv[i].cout : (i == 10 ? 128 : 64);
    TRY(unpad_cast_x3(U16(tcw, L.P[i]), at<float>(ws, act_off[i]), B, s, s, c, st));
  }
  return UDH_OK;
}

size_t x3_workspace_bytes(int B, int P) { return TcLayout(B, P, 2).total; }

int x3_workspace_init(void* ws, size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P, 2);
  UDH_CUDA(cudaMemsetAsync(at<char>(ws, tc_off), 0, L.total, st));
  return UDH_OK;
}

void* x3_fc1_mirror(void* ws, size_t tc_off, int B, int P) {
  TcLayout L(B, P, 2);
  return at<char>(ws, tc_off) + L.fc_w;
}

// fc1 forward: acc[B,1024] (zeroed by the caller) += x[B,F] . W[F,1024] as lo.hi + hi.hi + hi.lo over three K segments
int x3_fc1_fwd(const float* x, const float* w, float* acc, void* ws, size_t tc_off, int B, int P, bool w_mirror_current, cudaStream_t st) {
  TcLayout L(B, P, 2);
  char* tcw = at<char>(ws, tc_off);
  const size_t feat = (size_t)(P / 8) * (P / 8) * 128;
  uint16_t* xb = U16(tcw, L.fc_x);
  uint16_t* wb = U16(tcw, L.fc_w);
  TRY(cast_x3(x, xb, (size_t)B, (int)feat, st));
  if (!w_mirror_current) {
    const size_t n4 = feat * 1024 / 4;
    launch_chain(cast_planes_x3_kernel, dim3(grid1d((n4 + 255) / 256, 148 * 16)), dim3(256), 0, st, w, wb, wb + feat * 1024, n4);
    TRY(check_launch("cast_planes_x3"));
  }
  const int kb = 3 * (int)(feat / 64);
  int splits = 32;
  while (kb % splits) splits >>= 1;
  tc::GemmSegments seg = {3, {(int)feat, 0, 0}, {0, 0, 0}, {0, 0, (int)feat}, {0, 0, 0}};
  return tc::launch_gemm<false, true, true>(xb, 2 * feat, (uint64_t)B, wb, 1024, 2 * feat, acc, 1024, B, 1024, (int)feat, splits, &seg, st);
}

// fc1 backward: dW[F,1024] = x^T . dy (stored), dx[B,F] = dy . W^T, from the limb copies of x and W made by the forward
int x3_fc1_bwd(const float* dy, float* dW, float* dx, void* ws, size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P, 2);
  char* tcw = at<char>(ws, tc_off);
  const size_t feat = (size_t)(P / 8) * (P / 8) * 128;
  uint16_t* xb = U16(tcw, L.fc_x);
  uint16_t* wb = U16(tcw, L.fc_w);
  uint16_t* dyb = U16(tcw, L.fc_dy);
  TRY(cast_x3(dy, dyb, (size_t)B, 1024, st));
  // dW = x^T . dy: A = x limbs read MN-major (m = feature), B = dy limbs MN-major (n = output); K = batch
  tc::GemmSegments sw = {3, {0, 0, 0}, {(int)feat, 0, 0}, {0, 0, 0}, {0, 0, 1024}};
  TRY((tc::launch_gemm<true, true, false>(xb, 2 * feat, (uint64_t)B, dyb, 2048, (uint64_t)B, dW, 1024, (int)feat, 1024, B, 1, &sw, st)));
  // dx = dy . W^T: A = dy limbs K-major, B = W limbs as [n = feature][k = 1024] K-major (W_lo rows start at row F)
  tc::GemmSegments sx = {3, {1024, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, (int)feat}};
  return tc::launch_gemm<false, false, false>(dyb, 2048, (uint64_t)B, wb, 1024, 2 * feat, dx, (int64_t)feat, B, (int)feat, 1024, 1, &sx, st);
}

// ---- debug / test entries: one x3 layer on fp32 NHWC tensors (splits into limbs internally) --------------------------
size_t x3_debug_scratch_bytes(int B, int H, int W, int cin, int cout) {
  return al256((size_t)B * (H + 2) * (W + 2) * cin * 4) + al256((size_t)B * (H + 2) * (W + 2) * cout * 4) + al256((size_t)9 * cin * cout * 4);
}

__global__ void pack_one_x3_kernel(const float* __restrict__ w, uint16_t* __restrict__ dst, int Cin, int Cout, int dgrad) {
  const int K = dgrad ? Cout : Cin, N = dgrad ? Cin : Cout, CBk = K / 64, total = 9 * K * N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i & 63;
    int r = i >> 6;
    const int n = r % N; r /= N;
    const int cb = r % CBk;
    const int tap = r / CBk;
    const int kc = cb * 64 + k;
    const float v = dgrad ? w[((size_t)(8 - tap) * Cin + n) * Cout + kc] : w[((size_t)tap * Cin + kc) * Cout + n];
    uint16_t hi, lo;
    split1(v, hi, lo);
    const size_t blk = (size_t)(tap * CBk + cb) * 2;
    dst[(blk * N + n) * 64 + k] = hi;
    dst[((blk + 1) * N + n) * 64 + k] = lo;
  }
}

int x3_debug_conv(const float* x, const float* w, const float* bias, float* out, void* scratch, int B, int H, int W, int cin, int cout,
                  int relu, int dgrad, cudaStream_t st) {
  const int kin = dgrad ? cout : cin, kout = dgrad ? cin : cout;
  char* s = reinterpret_cast<char*>(scratch);
  uint16_t* xp = reinterpret_cast<uint16_t*>(s);
  uint16_t* op = reinterpret_cast<uint16_t*>(s + al256((size_t)B * (H + 2) * (W + 2) * kin * 4));
  uint16_t* wp = reinterpret_cast<uint16_t*>(s + al256((size_t)B * (H + 2) * (W + 2) * kin * 4) + al256((size_t)B * (H + 2) * (W + 2) * kout * 4));
  UDH_CUDA(cudaMemsetAsync(scratch, 0, x3_debug_scratch_bytes(B, H, W, cin, cout), st));
  TRY(pad_cast_x3(x, xp, B, H, W, kin, st));
  pack_one_x3_kernel<<<(9 * cin * cout + 255) / 256, 256, 0, st>>>(w, wp, cin, cout, dgrad);
  TRY(check_launch("pack_one_x3"));
  TRY(tc_conv_x3(xp, wp, bias, nullptr, nullptr, op, nullptr, relu, B, H, W, kin, kout, st));
  return unpad_cast_x3(op, out, B, H, W, kout, st);
}

int x3_debug_wgrad(const float* x, const float* gsrc, float* dW, float* db, void* scratch, int B, int H, int W, int cin, int cout, cudaStream_t st) {
  char* s = reinterpret_cast<char*>(scratch);
  uint16_t* xp = reinterpret_cast<uint16_t*>(s);
  uint16_t* gp = reinterpret_cast<uint16_t*>(s + al256((size_t)B * (H + 2) * (W + 2) * cin * 4));
  UDH_CUDA(cudaMemsetAsync(scratch, 0, x3_debug_scratch_bytes(B, H, W, cin, cout), st));
  TRY(pad_cast_x3(x, xp, B, H, W, cin, st));
  TRY(pad_cast_x3(gsrc, gp, B, H, W, cout, st));
  return tc_wgrad_x3(xp, gp, dW, db, B, H, W, cin, cout, st);
}

int x3_debug_conv1(const float* I1, const float* I2, const float* w, const float* bias, float* out, const float* g, float* dW, float* db,
                   void* scratch, int B, int H, int W, cudaStream_t st) {
  // forward (out != nullptr): out [B,H,W,64] = relu(conv1_1(I1, I2)); wgrad (g != nullptr): dW [3,3,2,64], db [64] accumulated
  char* s = reinterpret_cast<char*>(scratch);
  uint16_t* op = reinterpret_cast<uint16_t*>(s);
  const size_t sbytes = al256((size_t)B * (H + 2) * (W + 2) * 64 * 4);
  UDH_CUDA(cudaMemsetAsync(scratch, 0, sbytes, st));
  if (out) {
    TRY(conv1_x3_fwd(I1, I2, w, bias, op, nullptr, B, H, W, st));
    TRY(unpad_cast_x3(op, out, B, H, W, 64, st));
  }
  if (g) {
    UDH_CUDA(cudaMemsetAsync(scratch, 0, sbytes, st));
    TRY(pad_cast_x3(g, op, B, H, W, 64, st));
    TRY(conv1_x3_wgrad(I1, I2, op, dW, db, B, H, W, st));
  }
  return UDH_OK;
}

}  // namespace udh

extern "C" int udh_debug_x3_set_rows(int on) {
  udh::g_x3_rows = on != 0;
  return UDH_OK;
}

extern "C" size_t udh_debug_x3_scratch_bytes(int B, int H, int W, int cin, int cout) { return udh::x3_debug_scratch_bytes(B, H, W, cin, cout); }

extern "C" int udh_debug_x3_conv(const float* x, const float* w, const float* bias, float* out, void* scratch, int B, int H, int W,
                                 int cin, int cout, int relu, int dgrad, void* stream) {
  UDH_REQUIRE(x && w && out && scratch, "udh_debug_x3_conv: null pointer");
  return udh::x3_debug_conv(x, w, bias, out, scratch, B, H, W, cin, cout, relu, dgrad, udh::as_stream(stream));
}

extern "C" int udh_debug_x3_wgrad(const float* x, const float* g, float* dW, float* db, void* scratch, int B, int H, int W, int cin,
                                  int cout, void* stream) {
  UDH_REQUIRE(x && g && dW && scratch, "udh_debug_x3_wgrad: null pointer");
  return udh::x3_debug_wgrad(x, g, dW, db, scratch, B, H, W, cin, cout, udh::as_stream(stream));
}

extern "C" int udh_debug_x3_conv1(const float* I1, const float* I2, const float* w, const float* bias, float* out, const float* g,
                                  float* dW, float* db, void* scratch, int B, int H, int W, void* stream) {
  UDH_REQUIRE(I1 && I2 && scratch && (out || g), "udh_debug_x3_conv1: null pointer");
  UDH_REQUIRE(!out || (w && bias), "udh_debug_x3_conv1: forward needs weights and bias");
  UDH_REQUIRE(!g || (dW && db), "udh_debug_x3_conv1: wgrad needs dW and db");
  return udh::x3_debug_conv1(I1, I2, w, bias, out, g, dW, db, scratch, B, H, W, udh::as_stream(stream));
}
