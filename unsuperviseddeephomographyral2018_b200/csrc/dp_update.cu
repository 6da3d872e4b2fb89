// Row G fused with the optimiser for the one large tensor (fc1's weights, 134 of the 137 MB of parameters):
//   gradient mean over the ranks  (code/utils/utils.py:380-403 get_average_grads, code/homography_CNN_synthetic.py:199-207)
//   -> TF-1 Adam                  (code/homography_CNN_synthetic.py:277-284 apply_gradients)
//   -> the updated weights (fp32 master + tensor-core limbs) back to every replica,
// as ONE kernel over NVSwitch multicast memory.  Each rank owns a contiguous shard of the tensor:
//   multimem.ld_reduce  pulls the shard's gradient from all ranks, summed inside the switch (no staging copy, no ring);
//   Adam runs on the shard only (m and v of a shard live on its owner: 1/N of the optimiser traffic per GPU);
//   multimem.st         pushes the new fp32 weights and their bf16 limb planes to all replicas at once.
// Per GPU and step this moves 134 MB (gradient read by the switch) + 1035/N MB (Adam) + 268 MB (incoming weights) through
// HBM, against ~650 MB (ring allreduce with staging) + 1035 MB (replicated Adam) of the NCCL path it replaces.
// The cross-rank ordering (all gradients final before the first ld_reduce; all stores landed before the next forward) is
// two symmetric-memory barriers enqueued by the host around this launch (engine.py); the kernel itself never waits on a peer.
#include "common.cuh"
#include "tc_common.cuh"

namespace udh {

__device__ __forceinline__ float4 mm_ld_reduce_add(const float4* mc) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(mc) : "memory");
  return r;
}
__device__ __forceinline__ void mm_st(float4* mc, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
               :: "l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void mm_st(uint2* mc, const uint2& v) {
  asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};"
               :: "l"(mc), "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)) : "memory");
}

constexpr int kDpUnroll = 4;   // multicast loads in flight per thread (a switch round trip is a few microseconds)
// The kernel takes turns on the SMs with the conv kernels next to it (a conv CTA owns its SM outright): large CTAs with every
// load of an iteration issued up front, so that each SM it gets keeps enough bytes in flight.
constexpr int kDpThreads = 512;

// LIMBS: 0 = no mirror (fp32 mode), 1 = one bf16 plane, 2 = hi + lo planes (p = hi + lo)
template <int LIMBS>
__global__ void __launch_bounds__(kDpThreads) dp_shard_update_kernel(const float4* __restrict__ mc_g, const float4* p,
                                                              float4* __restrict__ mc_p, float4* __restrict__ m,
                                                              float4* __restrict__ v, uint2* __restrict__ mc_hi,
                                                              uint2* __restrict__ mc_lo, size_t begin4, size_t end4, size_t mb4,
                                                              float alpha, float b1, float b2, float eps, float gs) {
  const float c1 = 1.0f - b1, c2 = 1.0f - b2;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i0 = begin4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < end4; i0 += kDpUnroll * stride) {
    // every load of the kDpUnroll elements is issued before the first use: the few SMs this kernel owns keep
    // kDpThreads x kDpUnroll x 4 streams x 16 B (128 KB) in flight each
    float4 g[kDpUnroll], pv[kDpUnroll], mv[kDpUnroll], vv[kDpUnroll];
#pragma unroll
    for (int u = 0; u < kDpUnroll; ++u) {
      const size_t i = i0 + u * stride;
      if (i < end4) { g[u] = mm_ld_reduce_add(mc_g + i); pv[u] = p[i]; mv[u] = m[i]; vv[u] = v[i]; }
    }
#pragma unroll
    for (int u = 0; u < kDpUnroll; ++u) {
      const size_t i = i0 + u * stride;
      if (i < end4) {
        float4 gv = g[u], P = pv[u], M = mv[u], V = vv[u];
        gv.x *= gs; gv.y *= gs; gv.z *= gs; gv.w *= gs;
        M.x = b1 * M.x + c1 * gv.x; M.y = b1 * M.y + c1 * gv.y; M.z = b1 * M.z + c1 * gv.z; M.w = b1 * M.w + c1 * gv.w;
        V.x = b2 * V.x + c2 * gv.x * gv.x; V.y = b2 * V.y + c2 * gv.y * gv.y;
        V.z = b2 * V.z + c2 * gv.z * gv.z; V.w = b2 * V.w + c2 * gv.w * gv.w;
        P.x -= alpha * M.x / (sqrtf(V.x) + eps); P.y -= alpha * M.y / (sqrtf(V.y) + eps);
        P.z -= alpha * M.z / (sqrtf(V.z) + eps); P.w -= alpha * M.w / (sqrtf(V.w) + eps);
        m[i] = M; v[i] = V;
        mm_st(mc_p + i, P);
        if (LIMBS == 2) {
          uint2 h, l;
          tc::split2(P.x, P.y, h.x, l.x);
          tc::split2(P.z, P.w, h.y, l.y);
          mm_st(mc_hi + (i - mb4), h);
          mm_st(mc_lo + (i - mb4), l);
        } else if (LIMBS == 1) {
          const __nv_bfloat162 lo = __floats2bfloat162_rn(P.x, P.y), hi = __floats2bfloat162_rn(P.z, P.w);
          uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&lo); pk.y = *reinterpret_cast<const uint32_t*>(&hi);
          mm_st(mc_hi + (i - mb4), pk);
        }
      }
    }
  }
}

}  // namespace udh

extern "C" int udh_dp_shard_update(const void* mc_grads, const float* params, void* mc_params, float* adam_m, float* adam_v,
                                   void* mc_mirror, size_t shard_begin, size_t shard_count, size_t mirror_begin,
                                   size_t mirror_count, int mirror_limbs, float alpha_t, float beta1, float beta2, float eps,
                                   float grad_scale, int grid, void* stream) {
  UDH_REQUIRE(mc_grads && params && mc_params && adam_m && adam_v, "udh_dp_shard_update: null pointer");
  UDH_REQUIRE(mirror_limbs >= 0 && mirror_limbs <= 2 && (mirror_limbs == 0) == (mc_mirror == nullptr),
              "udh_dp_shard_update: mirror_limbs must be 0 (no mirror), 1 or 2 and agree with mc_mirror");
  UDH_REQUIRE(shard_begin % 4 == 0 && shard_count % 4 == 0 && mirror_begin % 4 == 0 && mirror_count % 4 == 0,
              "udh_dp_shard_update: ranges must be 4-float aligned");
  UDH_REQUIRE(((uintptr_t)mc_grads | (uintptr_t)params | (uintptr_t)mc_params | (uintptr_t)adam_m | (uintptr_t)adam_v) % 16 == 0 &&
                  (uintptr_t)mc_mirror % 8 == 0, "udh_dp_shard_update: buffers must be 16-byte aligned");
  UDH_REQUIRE(!mc_mirror || (shard_begin >= mirror_begin && shard_begin + shard_count <= mirror_begin + mirror_count),
              "udh_dp_shard_update: the shard must lie inside the mirrored tensor");
  UDH_REQUIRE(grid >= 0 && grid <= 148 * 2, "udh_dp_shard_update: grid must be in 0..296");
  if (shard_count == 0) return UDH_OK;
  const size_t n4 = shard_count / 4, per = (size_t)udh::kDpThreads * udh::kDpUnroll;
  const size_t full = (n4 + per - 1) / per, cap = grid > 0 ? (size_t)grid : (size_t)148;
  const unsigned blocks = (unsigned)(full < cap ? full : cap);
  cudaStream_t st = udh::as_stream(stream);
  udh::ProfScope ps(udh::PROF_ADAM, st);
  const size_t b4 = shard_begin / 4, e4 = b4 + n4, mb4 = mirror_begin / 4;
  uint2* hi = (uint2*)mc_mirror;
  uint2* lo = mirror_limbs == 2 ? (uint2*)((char*)mc_mirror + mirror_count * 2) : nullptr;
#define UDH_DP_LAUNCH(L)                                                                                                       \
  udh::dp_shard_update_kernel<L><<<blocks, udh::kDpThreads, 0, st>>>((const float4*)mc_grads, (const float4*)params, (float4*)mc_params, \
                                                         (float4*)adam_m, (float4*)adam_v, hi, lo, b4, e4, mb4, alpha_t, beta1, \
                                                         beta2, eps, grad_scale)
  if (mirror_limbs == 2) UDH_DP_LAUNCH(2);
  else if (mirror_limbs == 1) UDH_DP_LAUNCH(1);
  else UDH_DP_LAUNCH(0);
#undef UDH_DP_LAUNCH
  return udh::check_launch("udh_dp_shard_update");
}
