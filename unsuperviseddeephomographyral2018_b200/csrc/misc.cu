// Small entry points: error reporting, h4p losses / test metrics (Row L), TF-1 Adam (Row O).
#include <cuda_bf16.h>
#include <string.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace udh {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

unsigned long long g_launches = 0;
int g_sm_reserve = 0;
int g_sm_reserve_top = 0;
int g_bwd_marker_layer = -1;   // udh_set_bwd_marker
static cudaEvent_t g_bwd_marker_ev = nullptr;
static bool g_bwd_marker_recorded = false;

namespace {
const char* kTagNames[PROF_NUM_TAGS] = {
    "conv1_1.fwd", "conv1_2.fwd", "conv2_1.fwd", "conv2_2.fwd", "conv3_1.fwd", "conv3_2.fwd", "conv4_1.fwd", "conv4_2.fwd",
    "conv1_1.dgrad", "conv1_2.dgrad", "conv2_1.dgrad", "conv2_2.dgrad", "conv3_1.dgrad", "conv3_2.dgrad", "conv4_1.dgrad", "conv4_2.dgrad",
    "conv1_1.wgrad", "conv1_2.wgrad", "conv2_1.wgrad", "conv2_2.wgrad", "conv3_1.wgrad", "conv3_2.wgrad", "conv4_1.wgrad", "conv4_2.wgrad",
    "pool.fwd", "pool.bwd", "fc.fwd", "fc.bwd", "dlt", "warp_loss.fwd", "warp_loss.bwd", "ssim", "h4p_loss", "adam", "eltwise", "tc_prep"};
constexpr int kMaxPairs = 2048;
struct TagState { cudaEvent_t ev[kMaxPairs][2]; int created = 0, used = 0; bool open = false; };
bool g_prof_on = false;
TagState* g_tags = nullptr;
}  // namespace

void prof_begin(int tag, cudaStream_t st) {
  if (!g_prof_on || tag < 0 || tag >= PROF_NUM_TAGS) return;
  TagState& t = g_tags[tag];
  if (t.used >= kMaxPairs) return;
  if (t.used >= t.created) {
    if (cudaEventCreate(&t.ev[t.created][0]) != cudaSuccess || cudaEventCreate(&t.ev[t.created][1]) != cudaSuccess) return;
    ++t.created;
  }
  cudaEventRecord(t.ev[t.used][0], st);
  t.open = true;
}

void prof_end(int tag, cudaStream_t st) {
  if (!g_prof_on || tag < 0 || tag >= PROF_NUM_TAGS) return;
  TagState& t = g_tags[tag];
  if (!t.open) return;
  cudaEventRecord(t.ev[t.used][1], st);
  ++t.used;
  t.open = false;
}

// h_loss = sqrt(mean_{B x 8}(pred-gt)^2) (homography_model.py:288); test metrics (:274-281):
// batch_h_loss_b = sqrt(mean_8 (pred-gt)^2), identity_b = sqrt(mean_8 gt^2), failure = batch >= identity,
// bounded = mean_b(failure ? identity : batch).  One CTA; B is small (<= a few thousand).
__global__ void __launch_bounds__(256) h4p_loss_kernel(const float* __restrict__ pred, const float* __restrict__ gt, int B,
                                                       float* __restrict__ metrics, float* __restrict__ per_sample,
                                                       float* __restrict__ dpred) {
  pdl_wait(); pdl_trigger();   // launched through launch_chain (common.cuh)
  __shared__ double red[4 * 32];
  __shared__ float s_hloss;
  double acc[4] = {0, 0, 0, 0};   // sum sq, sum bounded, num fail, sum corner distance
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float sq = 0.f, id = 0.f, dist = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float dx = pred[b * 8 + 2 * i] - gt[b * 8 + 2 * i], dy = pred[b * 8 + 2 * i + 1] - gt[b * 8 + 2 * i + 1];
      sq += dx * dx + dy * dy;
      id += gt[b * 8 + 2 * i] * gt[b * 8 + 2 * i] + gt[b * 8 + 2 * i + 1] * gt[b * 8 + 2 * i + 1];
      dist += sqrtf(dx * dx + dy * dy);
    }
    const float bh = sqrtf(sq / 8.0f), ih = sqrtf(id / 8.0f);
    const bool fail = bh >= ih;
    if (per_sample) per_sample[b] = bh;
    acc[0] += sq; acc[1] += fail ? ih : bh; acc[2] += fail ? 1.0 : 0.0; acc[3] += dist * 0.25f;
  }
  block_sum<double, 4>(acc, red);
  if (threadIdx.x == 0) {
    const float hl = (float)sqrt(acc[0] / (8.0 * B));
    metrics[UDH_M_H_LOSS] = hl;
    metrics[UDH_M_BOUNDED_H_LOSS] = (float)(acc[1] / B);
    metrics[UDH_M_NUM_FAIL] = (float)acc[2];
    metrics[UDH_M_ACE] = (float)(acc[3] / B);
    s_hloss = hl;
  }
  __syncthreads();
  if (dpred) {
    // d sqrt(mean d^2) / d pred = d / (N * h_loss)
    const float k = s_hloss > 0.f ? 1.0f / (8.0f * (float)B * s_hloss) : 0.f;
    for (int i = threadIdx.x; i < B * 8; i += blockDim.x) dpred[i] = (pred[i] - gt[i]) * k;
  }
}

__global__ void __launch_bounds__(256) adam_kernel(float4* __restrict__ p, float4* __restrict__ g, float4* __restrict__ m,
                                                   float4* __restrict__ v, size_t n4, float alpha, float b1, float b2,
                                                   float eps, float gs, int zero_grad, uint2* __restrict__ mirror,
                                                   size_t mb4, size_t me4, int keep_grad, uint2* __restrict__ mirror_lo) {
  pdl_wait(); pdl_trigger();   // launched through launch_chain (common.cuh)
  const float c1 = 1.0f - b1, c2 = 1.0f - b2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 pv = p[i], gv = g[i], mv = m[i], vv = v[i];
    gv.x *= gs; gv.y *= gs; gv.z *= gs; gv.w *= gs;
    mv.x = b1 * mv.x + c1 * gv.x; mv.y = b1 * mv.y + c1 * gv.y; mv.z = b1 * mv.z + c1 * gv.z; mv.w = b1 * mv.w + c1 * gv.w;
    vv.x = b2 * vv.x + c2 * gv.x * gv.x; vv.y = b2 * vv.y + c2 * gv.y * gv.y;
    vv.z = b2 * vv.z + c2 * gv.z * gv.z; vv.w = b2 * vv.w + c2 * gv.w * gv.w;
    pv.x -= alpha * mv.x / (sqrtf(vv.x) + eps); pv.y -= alpha * mv.y / (sqrtf(vv.y) + eps);
    pv.z -= alpha * mv.z / (sqrtf(vv.z) + eps); pv.w -= alpha * mv.w / (sqrtf(vv.w) + eps);
    p[i] = pv; m[i] = mv; v[i] = vv;
    const bool in_mirror = i >= mb4 && i < me4;
    if (in_mirror) {
      if (mirror_lo) {             // two-limb mirror (UDH_NUMERIC_BF16X3): p = hi + lo
        uint2 h, l;
        tc::split2(pv.x, pv.y, h.x, l.x);
        tc::split2(pv.z, pv.w, h.y, l.y);
        mirror[i - mb4] = h;
        mirror_lo[i - mb4] = l;
      } else {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(pv.x, pv.y), hi = __floats2bfloat162_rn(pv.z, pv.w);
        uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&lo); pk.y = *reinterpret_cast<const uint32_t*>(&hi);
        mirror[i - mb4] = pk;
      }
    }
    if (zero_grad && !(in_mirror && keep_grad)) g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

}  // namespace udh

extern "C" int udh_version(void) { return 100; }

extern "C" const char* udh_last_error(void) { return udh::g_err; }

extern "C" int udh_device_available(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) { cudaGetLastError(); return 0; }
  return n > 0 ? 1 : 0;
}

extern "C" unsigned long long udh_launch_count(void) { return udh::g_launches; }

namespace udh {
int bwd_marker_record(int layer, cudaStream_t st) {
  if (layer != g_bwd_marker_layer) return UDH_OK;
  if (!g_bwd_marker_ev) UDH_CUDA(cudaEventCreateWithFlags(&g_bwd_marker_ev, cudaEventDisableTiming));
  UDH_CUDA(cudaEventRecord(g_bwd_marker_ev, st));
  g_bwd_marker_recorded = true;
  return UDH_OK;
}
}  // namespace udh

extern "C" int udh_set_bwd_marker(int layer) {
  UDH_REQUIRE(layer >= -1 && layer <= 7, "udh_set_bwd_marker: layer must be -1 (off) or 0..7");
  udh::g_bwd_marker_layer = layer;
  return UDH_OK;
}

extern "C" int udh_bwd_marker_wait(void* stream) {
  if (!udh::g_bwd_marker_recorded) return UDH_OK;      // nothing recorded yet: no dependency to add
  UDH_CUDA(cudaStreamWaitEvent(udh::as_stream(stream), udh::g_bwd_marker_ev, 0));
  return UDH_OK;
}

extern "C" int udh_set_sm_reserve_top(int n) {
  UDH_REQUIRE(n >= 0 && n < 128, "udh_set_sm_reserve_top: bad value %d", n);
  udh::g_sm_reserve_top = n;
  return UDH_OK;
}

extern "C" int udh_prof_enable(int on) {
  if (on && !udh::g_tags) udh::g_tags = new udh::TagState[udh::PROF_NUM_TAGS];
  udh::g_prof_on = on != 0;
  return UDH_OK;
}

extern "C" int udh_prof_reset(void) {
  if (udh::g_tags)
    for (int i = 0; i < udh::PROF_NUM_TAGS; ++i) { udh::g_tags[i].used = 0; udh::g_tags[i].open = false; }
  return UDH_OK;
}

extern "C" int udh_prof_num_tags(void) { return udh::PROF_NUM_TAGS; }

extern "C" const char* udh_prof_tag_name(int tag) { return (tag >= 0 && tag < udh::PROF_NUM_TAGS) ? udh::kTagNames[tag] : ""; }

extern "C" int udh_prof_read(int tag, float* total_ms, int* count) {
  UDH_REQUIRE(tag >= 0 && tag < udh::PROF_NUM_TAGS && total_ms && count, "udh_prof_read: bad arguments");
  *total_ms = 0.f; *count = 0;
  if (!udh::g_tags) return UDH_OK;
  udh::TagState& t = udh::g_tags[tag];
  for (int i = 0; i < t.used; ++i) {
    float ms = 0.f;
    UDH_CUDA(cudaEventSynchronize(t.ev[i][1]));
    UDH_CUDA(cudaEventElapsedTime(&ms, t.ev[i][0], t.ev[i][1]));
    *total_ms += ms;
  }
  *count = t.used;
  return UDH_OK;
}

extern "C" int udh_h4p_loss(const float* pred, const float* gt, int B, float* metrics, float* per_sample, float* dpred,
                            void* stream) {
  UDH_REQUIRE(pred && gt && metrics && B >= 1, "udh_h4p_loss: bad arguments");
  udh::ProfScope ps(udh::PROF_H4P_LOSS, udh::as_stream(stream));
  udh::launch_chain(udh::h4p_loss_kernel, dim3(1), dim3(256), 0, udh::as_stream(stream), pred, gt, B, metrics, per_sample, dpred);
  return udh::check_launch("udh_h4p_loss");
}

extern "C" int udh_adam_step(float* p, float* g, float* m, float* v, size_t n, float alpha_t, float beta1, float beta2,
                             float eps, float grad_scale, int zero_grad, void* stream) {
  return udh_adam_step_mirror(p, g, m, v, n, alpha_t, beta1, beta2, eps, grad_scale, zero_grad, nullptr, 0, 0, 0, stream);
}

extern "C" int udh_adam_step_mirror(float* p, float* g, float* m, float* v, size_t n, float alpha_t, float beta1, float beta2,
                                    float eps, float grad_scale, int zero_grad, void* mirror, size_t mirror_begin,
                                    size_t mirror_count, int mirror_keep_grad, void* stream) {
  return udh_adam_step_mirror_ex(p, g, m, v, n, alpha_t, beta1, beta2, eps, grad_scale, zero_grad, mirror, mirror_begin, mirror_count,
                                 mirror_keep_grad, 1, stream);
}

extern "C" int udh_adam_step_mirror_ex(float* p, float* g, float* m, float* v, size_t n, float alpha_t, float beta1, float beta2,
                                       float eps, float grad_scale, int zero_grad, void* mirror, size_t mirror_begin,
                                       size_t mirror_count, int mirror_keep_grad, int mirror_limbs, void* stream) {
  UDH_REQUIRE(mirror_limbs == 1 || mirror_limbs == 2, "udh_adam_step_mirror_ex: mirror_limbs must be 1 or 2");
  UDH_REQUIRE(p && g && m && v, "udh_adam_step: null pointer");
  if (!mirror) mirror_begin = mirror_count = 0;
  UDH_REQUIRE(mirror_begin % 4 == 0 && mirror_count % 4 == 0 && mirror_begin + mirror_count <= n && (uintptr_t)mirror % 8 == 0,
              "udh_adam_step_mirror: mirror range must be 4-float aligned and inside the buffer");
  UDH_REQUIRE(n % 4 == 0, "udh_adam_step: n must be a multiple of 4 (flat buffers are padded to 32 floats)");
  UDH_REQUIRE(((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) % 16 == 0, "udh_adam_step: buffers must be 16-byte aligned");
  if (n == 0) return UDH_OK;
  const size_t n4 = n / 4;
  const size_t full = (n4 + 255) / 256, cap = (size_t)148 * 16;
  const unsigned blocks = (unsigned)(full < cap ? full : cap);
  udh::ProfScope ps(udh::PROF_ADAM, udh::as_stream(stream));
  udh::launch_chain(udh::adam_kernel, dim3(blocks), dim3(256), 0, udh::as_stream(stream), (float4*)p, (float4*)g, (float4*)m, (float4*)v, n4, alpha_t,
                                                              beta1, beta2, eps, grad_scale, zero_grad, (uint2*)mirror,
                                                              mirror_begin / 4, (mirror_begin + mirror_count) / 4, mirror_keep_grad,
                                                              (mirror && mirror_limbs == 2) ? (uint2*)((char*)mirror + mirror_count * 2) : (uint2*)nullptr);
  return udh::check_launch("udh_adam_step");
}
