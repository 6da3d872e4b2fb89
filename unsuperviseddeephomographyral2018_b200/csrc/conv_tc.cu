// UDH_NUMERIC_BF16: the regressor's conv stack on tcgen05 tensor cores (see conv_tc_kernels.cuh for the kernel design).
// Activations and activation gradients are zero-bordered NHWC bf16 ("padded streams"); parameters, parameter gradients,
// the fully connected head and all reductions stay fp32.
#include "conv_tc.cuh"

#include "cnn_kernels.cuh"
#include "conv_tc_kernels.cuh"
#include "wgrad_tc_kernels.cuh"
#include "gemm_tc_kernels.cuh"
#include "conv1_tc_kernels.cuh"
#include "tc_layout.cuh"

namespace udh {

namespace {

using namespace tcl;
#define TRY UDH_TRY

// ---------------------------------------------------------------------------------------------------- small kernels
// dst[tap][cb][n][k] bf16 <- fp32 HWIO w[tap][ci][co].
//   forward: n = co, k-channel = ci.   dgrad: n = ci, k-channel = co, tap mirrored (w[8-tap]).
// rowtile != 0: block p of dst holds tap (ky, kx) = (2 - p % 3, p / 3), i.e. for every kx the three ky taps are adjacent in
// the order +1, 0, -1 — the row-tile conv kernels read two adjacent blocks as one N = 128 operand.
__device__ __forceinline__ int packed_src_tap(int p, int rowtile) { return rowtile ? (2 - p % 3) * 3 + p / 3 : p; }

__global__ void pack_weights_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst, int Cin, int Cout, int dgrad, int rowtile) {
  const int K = dgrad ? Cout : Cin, N = dgrad ? Cin : Cout;      // contraction channels, output channels of the packed conv
  const int CBk = K / 64;
  const int total = 9 * K * N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i & 63;
    int r = i >> 6;
    const int n = r % N; r /= N;
    const int cb = r % CBk;
    const int tap = packed_src_tap(r / CBk, rowtile);
    const int kc = cb * 64 + k;
    const float v = dgrad ? w[((size_t)(8 - tap) * Cin + n) * Cout + kc] : w[((size_t)tap * Cin + kc) * Cout + n];
    dst[i] = __float2bfloat16_rn(v);
  }
}

// all seven tensor-core layers in one launch (both directions): blockIdx.y = layer-1, blockIdx.z = direction
struct PackTable { const float* w[7]; __nv_bfloat16* fwd[7]; __nv_bfloat16* dgr[7]; int cin[7], cout[7]; int rowtile_fwd[7], rowtile_dgr[7]; };
__global__ void pack_all_weights_kernel(PackTable t, int do_fwd, int do_dgrad) {
  pdl_wait(); pdl_trigger();
  const int L = blockIdx.y, dgrad = blockIdx.z;
  if ((dgrad && !do_dgrad) || (!dgrad && !do_fwd)) return;
  const int Cin = t.cin[L], Cout = t.cout[L];
  const int K = dgrad ? Cout : Cin, N = dgrad ? Cin : Cout, CBk = K / 64, total = 9 * K * N;
  const float* __restrict__ w = t.w[L];
  __nv_bfloat16* __restrict__ dst = dgrad ? t.dgr[L] : t.fwd[L];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i & 63;
    int r = i >> 6;
    const int n = r % N; r /= N;
    const int cb = r % CBk;
    const int tap = packed_src_tap(r / CBk, dgrad ? t.rowtile_dgr[L] : t.rowtile_fwd[L]);
    const int kc = cb * 64 + k;
    dst[i] = __float2bfloat16_rn(dgrad ? w[((size_t)(8 - tap) * Cin + n) * Cout + kc] : w[((size_t)tap * Cin + kc) * Cout + n]);
  }
}

// fp32 [B,H,W,C] -> bf16 padded [B,H+2,W+2,C] interior (borders untouched = zero)
__global__ void pad_cast_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int B, int H, int W, int C) {
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
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&a); pk.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(dst + (((size_t)n * (H + 2) + y + 1) * (W + 2) + x + 1) * C + c4 * 4) = pk;
  }
}

// bf16 padded -> fp32 [B,H,W,C]
__global__ void unpad_cast_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int B, int H, int W, int C) {
  const int C4 = C >> 2;
  const size_t total = (size_t)B * H * W * C4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c4 = i % C4;
    size_t r = i / C4;
    const int x = r % W; r /= W;
    const int y = r % H;
    const int n = r / H;
    const uint2 pk = __ldg(reinterpret_cast<const uint2*>(src + (((size_t)n * (H + 2) + y + 1) * (W + 2) + x + 1) * C + c4 * 4));
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&pk.x), b = *reinterpret_cast<const __nv_bfloat162*>(&pk.y);
    reinterpret_cast<float4*>(dst)[i] = make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
  }
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&w[i]);
    f[2 * i] = __low2float(p); f[2 * i + 1] = __high2float(p);
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 p = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&p);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// 2x2/2 max pool on padded bf16 streams: in [B,H+2,W+2,C] -> out [B,H/2+2,W/2+2,C]
// Also records, per channel, which of the four inputs won (first maximum in scan order) or 4 when the maximum is not
// positive (the producer's ReLU passes no gradient): 3 bits per channel, 8 channels per uint32 -> the backward pass routes
// gradients from these codes and never re-reads the pre-pool activations.
__global__ void pool_fwd_bf16_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, uint32_t* __restrict__ codes,
                                     int B, int H, int W, int C) {
  pdl_wait(); pdl_trigger();
  const int C8 = C >> 3, OH = H >> 1, OW = W >> 1;
  const size_t total = (size_t)B * OH * OW * C8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c8 = i % C8;
    size_t r = i / C8;
    const int ox = r % OW; r /= OW;
    const int oy = r % OH;
    const int n = r / OH;
    const __nv_bfloat16* p = in + (((size_t)n * (H + 2) + 2 * oy + 1) * (W + 2) + 2 * ox + 1) * C + c8 * 8;
    float a[8], b[8], c[8], d[8], m[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p)), a);
    unpack8(__ldg(reinterpret_cast<const uint4*>(p + C)), b);
    unpack8(__ldg(reinterpret_cast<const uint4*>(p + (size_t)(W + 2) * C)), c);
    unpack8(__ldg(reinterpret_cast<const uint4*>(p + (size_t)(W + 2) * C + C)), d);
#pragma unroll
    uint32_t code = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = a[j]; uint32_t k = 0;
      if (b[j] > v) { v = b[j]; k = 1; }
      if (c[j] > v) { v = c[j]; k = 2; }
      if (d[j] > v) { v = d[j]; k = 3; }
      m[j] = v;
      code |= (v > 0.f ? k : 4u) << (3 * j);
    }
    *reinterpret_cast<uint4*>(out + (((size_t)n * (OH + 2) + oy + 1) * (OW + 2) + ox + 1) * C + c8 * 8) = pack8(m);
    codes[i] = code;
  }
}

// gradient routing of the above + ReLU mask of the producer, from the forward's routing codes
__global__ void pool_bwd_bf16_kernel(const uint32_t* __restrict__ codes, const __nv_bfloat16* __restrict__ gout,
                                     __nv_bfloat16* __restrict__ gin, int B, int H, int W, int C) {
  pdl_wait(); pdl_trigger();
  const int C8 = C >> 3, OH = H >> 1, OW = W >> 1;
  const size_t total = (size_t)B * OH * OW * C8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c8 = i % C8;
    size_t r = i / C8;
    const int ox = r % OW; r /= OW;
    const int oy = r % OH;
    const int n = r / OH;
    const size_t base = (((size_t)n * (H + 2) + 2 * oy + 1) * (W + 2) + 2 * ox + 1) * C + c8 * 8;
    const size_t rowp = (size_t)(W + 2) * C;
    const uint32_t code = __ldg(codes + i);
    float g[8], oa[8], ob[8], oc[8], od[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(gout + (((size_t)n * (OH + 2) + oy + 1) * (OW + 2) + ox + 1) * C + c8 * 8)), g);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t k = (code >> (3 * j)) & 7u;
      oa[j] = k == 0 ? g[j] : 0.f; ob[j] = k == 1 ? g[j] : 0.f; oc[j] = k == 2 ? g[j] : 0.f; od[j] = k == 3 ? g[j] : 0.f;
    }
    *reinterpret_cast<uint4*>(gin + base) = pack8(oa);
    *reinterpret_cast<uint4*>(gin + base + C) = pack8(ob);
    *reinterpret_cast<uint4*>(gin + base + rowp) = pack8(oc);
    *reinterpret_cast<uint4*>(gin + base + rowp + C) = pack8(od);
  }
}

// ---------------------------------------------------------------------------------------------------- launchers
template <int N_OUT, int CB, int T, bool WRES, bool TMA_EPI, int ROWS = 0>
int launch_conv_impl(const CUtensorMap& tmA128, const CUtensorMap& tmAhh, const CUtensorMap& tmW, const CUtensorMap& tmOut,
                     const tc::ConvGeom& g, const float* bias, const __nv_bfloat16* mask_src, const uint32_t* mask_bits,
                     uint32_t* mask_out, __nv_bfloat16* out_bf, float* out_f32, int relu, size_t smem, cudaStream_t st) {
  auto kern = tc::tc_conv_kernel<N_OUT, CB, T, WRES, TMA_EPI, ROWS>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = persistent_ctas();
  const int grid = g.num_items < sms ? g.num_items : sms;
  launch_chain(kern, dim3(grid), dim3(tc::conv_threads<TMA_EPI>()), smem, st, tmA128, tmAhh, tmW, tmOut, g, bias, mask_src, mask_bits, mask_out, out_bf, out_f32, relu);
  return check_launch("tc_conv_kernel");
}

template <int N_OUT, int CB, int T, bool WRES>
int launch_conv(const __nv_bfloat16* x, const __nv_bfloat16* wpk, const float* bias, const __nv_bfloat16* mask_src,
                const uint32_t* mask_bits, uint32_t* mask_out, __nv_bfloat16* out_bf, float* out_f32, int relu, int B, int H, int W,
                cudaStream_t st) {
  tc::ConvGeom g;
  g.B = B; g.H = H; g.W = W; g.Hp = H + 2; g.Wp = W + 2;
  g.Q = B * g.Hp * g.Wp;
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  const int tiles = (g.Q + 127) / 128;
  g.num_items = (tiles + T - 1) / T;
  g.abuf_rows = T * 128 + 2 * g.hh;
  const int Cin = CB * 64;
  CUtensorMap tmA128, tmAhh, tmW, tmOut;
  uint64_t dimsA[2] = {(uint64_t)Cin, (uint64_t)g.Q}, strA[2] = {2, (uint64_t)Cin * 2};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh};
  TRY(tc::make_tmap_bf16(&tmA128, x, 2, dimsA, strA, box128));
  TRY(tc::make_tmap_bf16(&tmAhh, x, 2, dimsA, strA, boxhh));
  uint64_t dimsW[2] = {64, (uint64_t)9 * CB * N_OUT}, strW[2] = {2, 128};
  uint32_t boxW[2] = {64, (uint32_t)N_OUT};
  TRY(tc::make_tmap_bf16(&tmW, wpk, 2, dimsW, strW, boxW));
  uint64_t dimsO[2] = {(uint64_t)N_OUT, (uint64_t)g.Q}, strO[2] = {2, (uint64_t)N_OUT * 2};
  uint32_t boxO[2] = {64, 32};
  TRY(tc::make_tmap_bf16(&tmOut, out_bf, 2, dimsO, strO, boxO));
  // TMA-store epilogue when its 16 KiB staging block still fits next to the operand buffers
  const size_t smem_tma = tc::ConvSmem<N_OUT, CB, T, WRES>::bytes(g.abuf_rows, true);
  if (out_bf && !mask_src && smem_tma <= 232448)
    return launch_conv_impl<N_OUT, CB, T, WRES, true>(tmA128, tmAhh, tmW, tmOut, g, bias, mask_src, mask_bits, mask_out, out_bf, out_f32, relu,
                                                      smem_tma, st);
  const size_t smem = tc::ConvSmem<N_OUT, CB, T, WRES>::bytes(g.abuf_rows, false);
  UDH_REQUIRE(smem <= 232448, "tc conv: %zu bytes of shared memory exceed the 227 KiB limit", smem);
  return launch_conv_impl<N_OUT, CB, T, WRES, false>(tmA128, tmAhh, tmW, tmOut, g, bias, mask_src, mask_bits, mask_out, out_bf, out_f32, relu,
                                                     smem, st);
}

// conv (64 -> 64, W == 128) + bias + ReLU + 2x2 max-pool in one kernel: writes the pooled padded stream and the routing codes
int tc_conv_pool(const __nv_bfloat16* x, const __nv_bfloat16* wpk, const float* bias, __nv_bfloat16* pooled, uint32_t* codes, int B, int H,
                 int W, cudaStream_t st) {
  UDH_REQUIRE(W == 128 && H % 2 == 0, "tc_conv_pool: needs W == 128 and an even height (got %d x %d)", H, W);
  tc::ConvGeom g;
  g.B = B; g.H = H; g.W = W; g.Hp = H + 2; g.Wp = W + 2;
  g.Q = B * g.Hp * g.Wp;
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  g.num_items = B * (H / 2);
  g.abuf_rows = 2 * 128 + 2 * g.hh;
  UDH_REQUIRE(g.hh + g.Wp + 128 + g.Wp + 1 <= g.abuf_rows, "tc_conv_pool: halo does not cover the second row tile");
  CUtensorMap tmA128, tmAhh, tmW;
  uint64_t dimsA[2] = {64, (uint64_t)g.Q}, strA[2] = {2, 128};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh};
  TRY(tc::make_tmap_bf16(&tmA128, x, 2, dimsA, strA, box128));
  TRY(tc::make_tmap_bf16(&tmAhh, x, 2, dimsA, strA, boxhh));
  uint64_t dimsW[2] = {64, (uint64_t)9 * 64}, strW[2] = {2, 128};
  uint32_t boxW[2] = {64, 64};
  TRY(tc::make_tmap_bf16(&tmW, wpk, 2, dimsW, strW, boxW));
  const size_t smem = tc::ConvSmem<64, 1, 2, true>::bytes(g.abuf_rows, false);
  return launch_conv_impl<64, 1, 2, true, false, 1>(tmA128, tmAhh, tmW, tmW, g, bias, nullptr, nullptr, codes, pooled, nullptr, 1, smem, st);
}

// conv (64 -> 64, W == 128) on row tiles with the plain epilogue (bias / ReLU / 1-bit mask / TMA store); weights must be
// packed in row-tile block order.  Used for the dgrad of conv1_2.
int tc_conv_rows(const __nv_bfloat16* x, const __nv_bfloat16* wpk, const float* bias, const uint32_t* mask_bits, uint32_t* mask_out,
                 __nv_bfloat16* out_bf, int relu, int B, int H, int W, cudaStream_t st) {
  UDH_REQUIRE(W == 128 && H % 2 == 0 && out_bf, "tc_conv_rows: needs W == 128, an even height and an output stream");
  tc::ConvGeom g;
  g.B = B; g.H = H; g.W = W; g.Hp = H + 2; g.Wp = W + 2;
  g.Q = B * g.Hp * g.Wp;
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  g.num_items = B * (H / 2);
  g.abuf_rows = 2 * 128 + 2 * g.hh;
  UDH_REQUIRE(g.hh + g.Wp + 128 + g.Wp + 1 <= g.abuf_rows, "tc_conv_rows: halo does not cover the second row tile");
  CUtensorMap tmA128, tmAhh, tmW, tmOut;
  uint64_t dimsA[2] = {64, (uint64_t)g.Q}, strA[2] = {2, 128};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh}, boxO[2] = {64, 32};
  TRY(tc::make_tmap_bf16(&tmA128, x, 2, dimsA, strA, box128));
  TRY(tc::make_tmap_bf16(&tmAhh, x, 2, dimsA, strA, boxhh));
  uint64_t dimsW[2] = {64, (uint64_t)9 * 64}, strW[2] = {2, 128};
  uint32_t boxW[2] = {64, 64};
  TRY(tc::make_tmap_bf16(&tmW, wpk, 2, dimsW, strW, boxW));
  TRY(tc::make_tmap_bf16(&tmOut, out_bf, 2, dimsA, strA, boxO));
  const size_t smem = tc::ConvSmem<64, 1, 2, true>::bytes(g.abuf_rows, true);
  UDH_REQUIRE(smem <= 232448, "tc_conv_rows: %zu bytes of shared memory exceed the 227 KiB limit", smem);
  return launch_conv_impl<64, 1, 2, true, true, 2>(tmA128, tmAhh, tmW, tmOut, g, bias, nullptr, mask_bits, mask_out, out_bf, nullptr, relu, smem, st);
}

// one 3x3 conv on padded bf16 streams; (cin -> cout) selects the kernel instance
int tc_conv(const __nv_bfloat16* x, const __nv_bfloat16* wpk, const float* bias, const __nv_bfloat16* mask_src,
            const uint32_t* mask_bits, uint32_t* mask_out, __nv_bfloat16* out_bf, float* out_f32, int relu, int B, int H, int W, int cin,
            int cout, cudaStream_t st) {
  if (cin == 64 && cout == 64) return launch_conv<64, 1, 2, true>(x, wpk, bias, mask_src, mask_bits, mask_out, out_bf, out_f32, relu, B, H, W, st);
  if (cin == 64 && cout == 128) return launch_conv<128, 1, 1, true>(x, wpk, bias, mask_src, mask_bits, mask_out, out_bf, out_f32, relu, B, H, W, st);
  if (cin == 128 && cout == 64) return launch_conv<64, 2, 2, false>(x, wpk, bias, mask_src, mask_bits, mask_out, out_bf, out_f32, relu, B, H, W, st);
  if (cin == 128 && cout == 128) return launch_conv<128, 2, 2, false>(x, wpk, bias, mask_src, mask_bits, mask_out, out_bf, out_f32, relu, B, H, W, st);
  set_error("tc_conv: unsupported channel combination %d -> %d", cin, cout);
  return UDH_ENOSUP;
}

int pack_weights(const float* w, __nv_bfloat16* dst, int cin, int cout, int dgrad, cudaStream_t st, int rowtile = 0) {
  const int total = 9 * cin * cout;
  pack_weights_kernel<<<(total + 255) / 256, 256, 0, st>>>(w, dst, cin, cout, dgrad, rowtile);
  return check_launch("pack_weights");
}
int pad_cast(const float* src, __nv_bfloat16* dst, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * H * W * (C / 4);
  launch_chain(pad_cast_kernel, dim3(grid1d((total + 255) / 256, 148 * 32)), dim3(256), 0, st, src, dst, B, H, W, C);
  return check_launch("pad_cast");
}
int unpad_cast(const __nv_bfloat16* src, float* dst, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * H * W * (C / 4);
  unpad_cast_kernel<<<grid1d((total + 255) / 256, 148 * 32), 256, 0, st>>>(src, dst, B, H, W, C);
  return check_launch("unpad_cast");
}
int pool_fwd_bf16(const __nv_bfloat16* in, __nv_bfloat16* out, uint32_t* codes, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * (H / 2) * (W / 2) * (C / 8);
  launch_chain(pool_fwd_bf16_kernel, dim3(grid1d((total + 255) / 256, 148 * 32)), dim3(256), 0, st, in, out, codes, B, H, W, C);
  return check_launch("pool_fwd_bf16");
}
int pool_bwd_bf16(const uint32_t* codes, const __nv_bfloat16* gout, __nv_bfloat16* gin, int B, int H, int W, int C, cudaStream_t st) {
  const size_t total = (size_t)B * (H / 2) * (W / 2) * (C / 8);
  launch_chain(pool_bwd_bf16_kernel, dim3(grid1d((total + 255) / 256, 148 * 32)), dim3(256), 0, st, codes, gout, gin, B, H, W, C);
  return check_launch("pool_bwd_bf16");
}

template <int N_OUT, int CBX, int T>
int launch_wgrad(const __nv_bfloat16* x, const __nv_bfloat16* gsrc, float* dW, float* db, int B, int H, int W, cudaStream_t st) {
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
  const int Cin = CBX * 64;
  CUtensorMap tmX128, tmXhh, tmG;
  uint64_t dimsX[2] = {(uint64_t)Cin, (uint64_t)g.Q}, strX[2] = {2, (uint64_t)Cin * 2};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh};
  TRY(tc::make_tmap_bf16(&tmX128, x, 2, dimsX, strX, box128));
  TRY(tc::make_tmap_bf16(&tmXhh, x, 2, dimsX, strX, boxhh));
  uint64_t dimsG[2] = {(uint64_t)N_OUT, (uint64_t)g.Q}, strG[2] = {2, (uint64_t)N_OUT * 2};
  TRY(tc::make_tmap_bf16(&tmG, gsrc, 2, dimsG, strG, box128));
  const size_t stage = (size_t)CBX * g.xrows * 128 + (size_t)CBO * T * 16384;
  const size_t smem = 1024 + 2 * stage + 16384 + 256;
  UDH_REQUIRE(smem <= 232448, "tc wgrad: %zu bytes of shared memory exceed the 227 KiB limit", smem);
  auto kern = tc::tc_wgrad_kernel<N_OUT, CBX, T>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_chain(kern, dim3(g.slice_cta[g.num_slices]), dim3(256), smem, st, tmX128, tmXhh, tmG, g, dW, db);
  return check_launch("tc_wgrad_kernel");
}

// 64 -> 64 layers: the N = 192 kernel (see wgrad_tc_kernels.cuh)
int launch_wgrad64(const __nv_bfloat16* x, const __nv_bfloat16* gsrc, float* dW, float* db, int B, int H, int W, cudaStream_t st) {
  constexpr int T = 2;
  tc::Wgrad64Geom g;
  g.Wp = W + 2;
  g.Q = B * (H + 2) * (W + 2);
  g.hh = (g.Wp + 1 + 7) / 8 * 8;
  const int tiles = (g.Q + 127) / 128;
  g.num_items = (tiles + T - 1) / T;
  g.xrows = T * 128 + 2 * g.hh;
  CUtensorMap tmX128, tmXhh, tmG136;
  uint64_t dims[2] = {64, (uint64_t)g.Q}, str[2] = {2, 128};
  uint32_t box128[2] = {64, 128}, boxhh[2] = {64, (uint32_t)g.hh}, box136[2] = {64, 136};
  TRY(tc::make_tmap_bf16(&tmX128, x, 2, dims, str, box128));
  TRY(tc::make_tmap_bf16(&tmXhh, x, 2, dims, str, boxhh));
  TRY(tc::make_tmap_bf16(&tmG136, gsrc, 2, dims, str, box136));
  const size_t stage = (size_t)g.xrows * 128 + (size_t)(T * 128 + 16) * 128;
  const size_t smem = 1024 + 2 * stage + 16384 + 256;
  UDH_REQUIRE(smem <= 232448, "tc wgrad64: %zu bytes of shared memory exceed the 227 KiB limit", smem);
  auto kern = tc::tc_wgrad64_kernel<T>;
  UDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = persistent_ctas();
  launch_chain(kern, dim3(g.num_items < sms ? g.num_items : sms), dim3(256), smem, st, tmX128, tmXhh, tmG136, g, dW, db);
  return check_launch("tc_wgrad64_kernel");
}

// dW (HWIO fp32) += X^T-shifted . G ; db += sum G   for one layer, on padded bf16 streams
int tc_wgrad(const __nv_bfloat16* x, const __nv_bfloat16* gsrc, float* dW, float* db, int B, int H, int W, int cin, int cout,
             cudaStream_t st) {
  if (cin == 64 && cout == 64) return launch_wgrad64(x, gsrc, dW, db, B, H, W, st);
  if (cin == 64 && cout == 128) return launch_wgrad<128, 1, 1>(x, gsrc, dW, db, B, H, W, st);
  if (cin == 128 && cout == 128) return launch_wgrad<128, 2, 1>(x, gsrc, dW, db, B, H, W, st);
  set_error("tc_wgrad: unsupported channel combination %d -> %d", cin, cout);
  return UDH_ENOSUP;
}

__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n4) {
  pdl_wait(); pdl_trigger();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&a); pk.y = *reinterpret_cast<uint32_t*>(&b);
    reinterpret_cast<uint2*>(dst)[i] = pk;
  }
}
int cast_bf16(const float* src, __nv_bfloat16* dst, size_t n, cudaStream_t st) {
  launch_chain(cast_bf16_kernel, dim3(grid1d((n / 4 + 255) / 256, 148 * 16)), dim3(256), 0, st, src, dst, n / 4);
  return check_launch("cast_bf16");
}

// conv1_1 on the tensor pipe (im2col tile built in shared memory), see conv1_tc_kernels.cuh
int conv1_tc_fwd(const float* I1, const float* I2, const float* w, const float* bias, __nv_bfloat16* out_pad, uint32_t* mask_out, int B,
                 int H, int W, cudaStream_t st) {
  UDH_REQUIRE(W % 128 == 0, "conv1_tc_fwd: image width must be a multiple of 128");
  tc::Conv1Geom g{B, H, W, B * H * (W / 128)};
  CUtensorMap tmOut;
  const uint64_t Q = (uint64_t)B * (H + 2) * (W + 2);
  uint64_t dims[2] = {64, Q}, str[2] = {2, 128};
  uint32_t box[2] = {64, 32};
  TRY(tc::make_tmap_bf16(&tmOut, out_pad, 2, dims, str, box));
  const size_t smem = 1024 + 2 * 16384 + 8192 + 16384 + 256;
  UDH_CUDA(cudaFuncSetAttribute(tc::conv1_tc_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int want = tc::kConv1CtasPerSm * persistent_ctas();
  const int grid = g.tiles < want ? g.tiles : want;
  launch_chain(tc::conv1_tc_fwd_kernel, dim3(grid), dim3(160), smem, st, tmOut, g, I1, I2, w, bias, mask_out);
  return check_launch("conv1_tc_fwd_kernel");
}

int conv1_tc_wgrad(const float* I1, const float* I2, const __nv_bfloat16* G_pad, float* dW, float* db, int B, int H, int W,
                   cudaStream_t st) {
  UDH_REQUIRE(W % 128 == 0, "conv1_tc_wgrad: image width must be a multiple of 128");
  tc::Conv1Geom g{B, H, W, B * H * (W / 128)};
  CUtensorMap tmG;
  const uint64_t Q = (uint64_t)B * (H + 2) * (W + 2);
  uint64_t dims[2] = {64, Q}, str[2] = {2, 128};
  uint32_t box[2] = {64, 128};
  TRY(tc::make_tmap_bf16(&tmG, G_pad, 2, dims, str, box));
  const size_t smem = 1024 + 4 * 16384 + 256;
  UDH_CUDA(cudaFuncSetAttribute(tc::conv1_tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int want = tc::kConv1CtasPerSm * persistent_ctas();
  const int grid = g.tiles < want ? g.tiles : want;
  launch_chain(tc::conv1_tc_wgrad_kernel, dim3(grid), dim3(160), smem, st, tmG, g, I1, I2, dW, db);
  return check_launch("conv1_tc_wgrad_kernel");
}

}  // namespace

size_t tc_workspace_bytes(int B, int P, int numeric_mode) {
  if (numeric_mode != UDH_NUMERIC_BF16) return 0;
  return TcLayout(B, P).total;
}

int tc_workspace_init(void* ws, size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P);
  // borders of every padded stream must be zero and are never written afterwards
  UDH_CUDA(cudaMemsetAsync(at<char>(ws, tc_off), 0, L.total, st));
  return UDH_OK;
}

int tc_cnn_fwd_convs(const float* params, const size_t* poff, const float* I1, const float* I2, void* ws, const size_t* act_off,
                     size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P);
  char* tcw = at<char>(ws, tc_off);
  auto Pb = [&](int i) { return reinterpret_cast<__nv_bfloat16*>(tcw + L.P[i]); };
  {
    // forward AND mirrored (dgrad) bf16 weight packs of the seven tensor-core layers, one launch per step
    ProfScope ps(PROF_TC_PREP, st);
    PackTable t;
    for (int i = 1; i < 8; ++i) {
      t.w[i - 1] = params + poff[2 * i];
      t.fwd[i - 1] = reinterpret_cast<__nv_bfloat16*>(tcw + L.wf[i]);
      t.dgr[i - 1] = reinterpret_cast<__nv_bfloat16*>(tcw + L.wd[i]);
      t.cin[i - 1] = kConv[i].cin; t.cout[i - 1] = kConv[i].cout;
      t.rowtile_fwd[i - 1] = (i == 1 && P == 128) ? 1 : 0;          // conv1_2 forward runs on row tiles (fused with pool1)
      t.rowtile_dgr[i - 1] = (i == 1 && P == 128) ? 1 : 0;          // ... and so does its dgrad
    }
    launch_chain(pack_all_weights_kernel, dim3(72, 7, 2), dim3(256), 0, st, t, 1, 1);
    TRY(check_launch("pack_all_weights"));
  }
  {
    // conv1_1 (K = 18): im2col tile in shared memory + tcgen05, writing the padded bf16 stream and its 1-bit ReLU mask
    ProfScope ps(PROF_CONV_FWD0, st);
    TRY(conv1_tc_fwd(I1, I2, params + poff[0], params + poff[1], Pb(0), reinterpret_cast<uint32_t*>(tcw + L.Mb[0]), B, P, P, st));
  }
  const bool fuse_pool1 = (P == 128);      // conv1_2 + pool1 in one kernel (its row tiling needs 128-wide images)
  for (int i = 1; i < 8; ++i) {
    const int s = P / kConv[i].div;
    if (i == 1 && fuse_pool1) {
      ProfScope ps(PROF_CONV_FWD0 + i, st);
      TRY(tc_conv_pool(Pb(0), reinterpret_cast<__nv_bfloat16*>(tcw + L.wf[1]), params + poff[3], Pb(8),
                       reinterpret_cast<uint32_t*>(tcw + L.Px[0]), B, s, s, st));
      continue;
    }
    {
      ProfScope ps(PROF_CONV_FWD0 + i, st);
      TRY(tc_conv(Pb(input_of(i)), reinterpret_cast<__nv_bfloat16*>(tcw + L.wf[i]), params + poff[2 * i + 1], nullptr, nullptr,
                  (i % 2 == 0) ? reinterpret_cast<uint32_t*>(tcw + L.Mb[i]) : nullptr, Pb(i),
                  i == 7 ? at<float>(ws, act_off[7]) : nullptr, 1, B, s, s, kConv[i].cin, kConv[i].cout, st));
    }
    if ((i == 3 || i == 5) || (i == 1 && !fuse_pool1)) {
      ProfScope ps(PROF_POOL_FWD, st);
      TRY(pool_fwd_bf16(Pb(i), Pb(8 + i / 2), reinterpret_cast<uint32_t*>(tcw + L.Px[i / 2]), B, s, s, kConv[i].cout, st));
    }
  }
  return UDH_OK;
}

int tc_cnn_bwd_convs(const float* params, const size_t* poff, const float* I1, const float* I2, float* grads, float* gA, float* gB,
                     void* ws, const size_t* act_off, size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P);
  char* tcw = at<char>(ws, tc_off);
  auto Pb = [&](int i) { return reinterpret_cast<__nv_bfloat16*>(tcw + L.P[i]); };
  auto Gb = [&](int i) { return reinterpret_cast<__nv_bfloat16*>(tcw + L.G[i]); };
  {
    ProfScope ps(PROF_TC_PREP, st);        // (the mirrored weight packs were made by the forward of this step)
    TRY(pad_cast(gA, Gb(7), B, P / 8, P / 8, 128, st));
  }
  struct RestoreReserve { ~RestoreReserve() { g_sm_reserve = 0; } } restore_reserve;   // outside the conv backward every SM is used
  for (int i = 7; i >= 0; --i) {
    TRY(bwd_marker_record(i, st));
    const int s = P / kConv[i].div;
    const int cin = kConv[i].cin, cout = kConv[i].cout;
    g_sm_reserve = bwd_sm_reserve(i);   // see udh_set_sm_reserve_top
    {
      ProfScope ps(PROF_CONV_WGRAD0 + i, st);
      if (i == 0) {
        // conv1_1 (Cin = 2): im2col tile (MN-major A, M = 64) x gradient rows by TMA, bias gradient from the ones column
        TRY(conv1_tc_wgrad(I1, I2, Gb(0), grads + poff[0], grads + poff[1], B, s, s, st));
      } else {
        TRY(tc_wgrad(Pb(input_of(i)), Gb(i), grads + poff[2 * i], grads + poff[2 * i + 1], B, s, s, cin, cout, st));
      }
    }
    if (i == 0) break;
    const bool below_is_pool = (i == 2 || i == 4 || i == 6);
    const int below = input_of(i);
    if (i == 1 && P == 128) {
      // conv1_2 dgrad on row tiles (weights were packed in row-tile order by the forward), ReLU mask of conv1_1 fused
      ProfScope ps(PROF_CONV_DGRAD0 + i, st);
      TRY(tc_conv_rows(Gb(1), reinterpret_cast<__nv_bfloat16*>(tcw + L.wd[1]), nullptr, reinterpret_cast<const uint32_t*>(tcw + L.Mb[0]),
                       nullptr, Gb(0), 0, B, s, s, st));
      continue;
    }
    {
      ProfScope ps(PROF_CONV_DGRAD0 + i, st);
      // dgrad = conv of G[i] with the mirrored kernel; ReLU mask of the layer below fused unless a pool sits between
      TRY(tc_conv(Gb(i), reinterpret_cast<__nv_bfloat16*>(tcw + L.wd[i]), nullptr, nullptr,
                  below_is_pool ? nullptr : reinterpret_cast<const uint32_t*>(tcw + L.Mb[below]), nullptr, Gb(below), nullptr, 0, B, s, s,
                  cout, cin, st));
    }
    if (below_is_pool) {
      ProfScope ps(PROF_POOL_BWD, st);
      TRY(pool_bwd_bf16(reinterpret_cast<const uint32_t*>(tcw + L.Px[i / 2 - 1]), Gb(below), Gb(i - 1), B, 2 * s, 2 * s, cin, st));
    }
  }
  return UDH_OK;
}

// fc1 forward on tensor cores: acc[B,1024] (zeroed by the caller) += x[B,F] . W[F,1024]
void* tc_fc1_mirror(void* ws, size_t tc_off, int B, int P) {
  TcLayout L(B, P);
  return at<char>(ws, tc_off) + L.fc_w;
}

int tc_fc1_fwd(const float* x, const float* w, float* acc, void* ws, size_t tc_off, int B, int P, bool w_mirror_current, cudaStream_t st) {
  TcLayout L(B, P);
  char* tcw = at<char>(ws, tc_off);
  const size_t feat = (size_t)(P / 8) * (P / 8) * 128;
  __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(tcw + L.fc_x);
  __nv_bfloat16* wb = reinterpret_cast<__nv_bfloat16*>(tcw + L.fc_w);
  TRY(cast_bf16(x, xb, (size_t)B * feat, st));
  if (!w_mirror_current) TRY(cast_bf16(w, wb, feat * 1024, st));
  const int kb = (int)(feat / 64);
  int splits = 32;
  while (kb % splits) splits >>= 1;
  return tc::launch_gemm<false, true, true>(xb, feat, (uint64_t)B, wb, 1024, feat, acc, 1024, B, 1024, (int)feat, splits, nullptr, st);
}

// fc1 backward: dW[F,1024] = x^T . dy (stored: the gradient buffer is zero on entry), dx[B,F] = dy . W^T.
// Uses the bf16 copies of x and W made by the forward of the same step.
int tc_fc1_bwd(const float* dy, float* dW, float* dx, void* ws, size_t tc_off, int B, int P, cudaStream_t st) {
  TcLayout L(B, P);
  char* tcw = at<char>(ws, tc_off);
  const size_t feat = (size_t)(P / 8) * (P / 8) * 128;
  __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(tcw + L.fc_x);
  __nv_bfloat16* wb = reinterpret_cast<__nv_bfloat16*>(tcw + L.fc_w);
  __nv_bfloat16* dyb = reinterpret_cast<__nv_bfloat16*>(tcw + L.fc_dy);
  TRY(cast_bf16(dy, dyb, (size_t)B * 1024, st));
  TRY((tc::launch_gemm<true, true, false>(xb, feat, (uint64_t)B, dyb, 1024, (uint64_t)B, dW, 1024, (int)feat, 1024, B, 1, nullptr, st)));
  return tc::launch_gemm<false, false, false>(dyb, 1024, (uint64_t)B, wb, 1024, feat, dx, (int64_t)feat, B, (int)feat, 1024, 1, nullptr, st);
}

// Debug / test entry: one tensor-core conv layer on fp32 NHWC tensors (pads + casts internally).
// x [B,H,W,cin], w HWIO [3,3,cin,cout], bias [cout] (nullable), out [B,H,W,cout]; scratch: device buffer of
// udh_debug_tc_conv_scratch_bytes().  dgrad != 0 runs the mirrored-kernel convolution (cout -> cin channels).
size_t tc_debug_scratch_bytes(int B, int H, int W, int cin, int cout) {
  return al256((size_t)B * (H + 2) * (W + 2) * cin * 2) + al256((size_t)B * (H + 2) * (W + 2) * cout * 2) + al256((size_t)9 * cin * cout * 2);
}

int tc_debug_conv(const float* x, const float* w, const float* bias, float* out, void* scratch, int B, int H, int W, int cin, int cout,
                  int relu, int dgrad, cudaStream_t st) {
  const int kin = dgrad ? cout : cin, kout = dgrad ? cin : cout;      // channels of the convolution actually run
  char* s = reinterpret_cast<char*>(scratch);
  __nv_bfloat16* xp = reinterpret_cast<__nv_bfloat16*>(s);
  __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(s + al256((size_t)B * (H + 2) * (W + 2) * kin * 2));
  __nv_bfloat16* wp = reinterpret_cast<__nv_bfloat16*>(s + al256((size_t)B * (H + 2) * (W + 2) * kin * 2) + al256((size_t)B * (H + 2) * (W + 2) * kout * 2));
  UDH_CUDA(cudaMemsetAsync(scratch, 0, tc_debug_scratch_bytes(B, H, W, cin, cout), st));
  TRY(pad_cast(x, xp, B, H, W, kin, st));
  TRY(pack_weights(w, wp, cin, cout, dgrad, st));
  TRY(tc_conv(xp, wp, bias, nullptr, nullptr, nullptr, op, out, relu, B, H, W, kin, kout, st));
  return UDH_OK;
}

// Debug / test entry: fused conv (64 -> 64) + bias + ReLU + 2x2 max-pool.  x [B,H,128,64] fp32 -> pooled [B,H/2,64,64] fp32 and
// routing codes [B,H/2,64,8] uint32 (3 bits per channel: 0..3 = winner in scan order, 4 = maximum not positive).
int tc_debug_conv_pool(const float* x, const float* w, const float* bias, float* pooled, uint32_t* codes, void* scratch, int B, int H, int W,
                       cudaStream_t st) {
  char* s = reinterpret_cast<char*>(scratch);
  const size_t in_bytes = al256((size_t)B * (H + 2) * (W + 2) * 64 * 2);
  __nv_bfloat16* xp = reinterpret_cast<__nv_bfloat16*>(s);
  __nv_bfloat16* pp = reinterpret_cast<__nv_bfloat16*>(s + in_bytes);
  __nv_bfloat16* wp = reinterpret_cast<__nv_bfloat16*>(s + 2 * in_bytes);
  UDH_CUDA(cudaMemsetAsync(scratch, 0, tc_debug_scratch_bytes(B, H, W, 64, 64), st));
  TRY(pad_cast(x, xp, B, H, W, 64, st));
  TRY(pack_weights(w, wp, 64, 64, 0, st, 1));
  TRY(tc_conv_pool(xp, wp, bias, pp, codes, B, H, W, st));
  return unpad_cast(pp, pooled, B, H / 2, W / 2, 64, st);
}

// Debug / test entry: tensor-core weight gradient on fp32 NHWC tensors x [B,H,W,cin], g [B,H,W,cout] -> dW HWIO, db (accumulated).
int tc_debug_wgrad(const float* x, const float* gsrc, float* dW, float* db, void* scratch, int B, int H, int W, int cin, int cout,
                   cudaStream_t st) {
  char* s = reinterpret_cast<char*>(scratch);
  __nv_bfloat16* xp = reinterpret_cast<__nv_bfloat16*>(s);
  __nv_bfloat16* gp = reinterpret_cast<__nv_bfloat16*>(s + al256((size_t)B * (H + 2) * (W + 2) * cin * 2));
  UDH_CUDA(cudaMemsetAsync(scratch, 0, tc_debug_scratch_bytes(B, H, W, cin, cout), st));
  TRY(pad_cast(x, xp, B, H, W, cin, st));
  TRY(pad_cast(gsrc, gp, B, H, W, cout, st));
  return tc_wgrad(xp, gp, dW, db, B, H, W, cin, cout, st);
}

}  // namespace udh

extern "C" int udh_debug_tc_wgrad(const float* x, const float* g, float* dW, float* db, void* scratch, int B, int H, int W, int cin,
                                  int cout, void* stream) {
  UDH_REQUIRE(x && g && dW && scratch, "udh_debug_tc_wgrad: null pointer");
  return udh::tc_debug_wgrad(x, g, dW, db, scratch, B, H, W, cin, cout, udh::as_stream(stream));
}

extern "C" int udh_debug_tc_conv_pool(const float* x, const float* w, const float* bias, float* pooled, uint32_t* codes, void* scratch,
                                      int B, int H, int W, void* stream) {
  UDH_REQUIRE(x && w && bias && pooled && codes && scratch, "udh_debug_tc_conv_pool: null pointer");
  return udh::tc_debug_conv_pool(x, w, bias, pooled, codes, scratch, B, H, W, udh::as_stream(stream));
}

extern "C" size_t udh_debug_tc_conv_scratch_bytes(int B, int H, int W, int cin, int cout) {
  return udh::tc_debug_scratch_bytes(B, H, W, cin, cout);
}

extern "C" int udh_debug_tc_conv(const float* x, const float* w, const float* bias, float* out, void* scratch, int B, int H, int W,
                                 int cin, int cout, int relu, int dgrad, void* stream) {
  UDH_REQUIRE(x && w && out && scratch, "udh_debug_tc_conv: null pointer");
  return udh::tc_debug_conv(x, w, bias, out, scratch, B, H, W, cin, cout, relu, dgrad, udh::as_stream(stream));
}
