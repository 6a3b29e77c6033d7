// Shared device helpers for the dan_b200 kernels (sm_100a).
//
// Numerics contract: the reference computes this path with TensorFlow's unfused
// Eigen elementwise kernels, i.e. every fp32 +,-,*,/ is one separately rounded
// IEEE-754 operation.  All arithmetic that can reach an index / label / keep-list
// therefore goes through the __f*_rn intrinsics below, which the compiler may not
// contract into FMA (the build also passes -fmad=false as a second guard).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dan_b200.h"

#define DAN_HD __host__ __device__ __forceinline__
#define DAN_D __device__ __forceinline__

namespace dan {

// host side error plumbing -------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define DAN_REQUIRE(cond, code, ...)      \
  do {                                    \
    if (!(cond)) {                        \
      ::dan::set_error(__VA_ARGS__);      \
      return (code);                      \
    }                                     \
  } while (0)

#define DAN_CUDA(expr)                                         \
  do {                                                         \
    cudaError_t e__ = (expr);                                  \
    if (e__ != cudaSuccess) return ::dan::cuda_fail(e__, #expr); \
  } while (0)

#define DAN_LAUNCH_CHECK(name)                                       \
  do {                                                               \
    cudaError_t e__ = cudaGetLastError();                            \
    if (e__ != cudaSuccess) return ::dan::cuda_fail(e__, name);      \
  } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
// grid for a grid-stride streaming kernel: enough CTAs to fill 148 SMs x 16 resident CTAs
static inline int grid_for(int64_t n, int block = 256) {
  int64_t g = (n + block - 1) / block;
  const int64_t cap = 148 * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// exact fp32 ops -----------------------------------------------------------
DAN_D float fadd(float a, float b) { return __fadd_rn(a, b); }
DAN_D float fsub(float a, float b) { return __fsub_rn(a, b); }
DAN_D float fmul(float a, float b) { return __fmul_rn(a, b); }
DAN_D float fdiv(float a, float b) { return __fdiv_rn(a, b); }

// point2center, anchor_manipulator.py:129-132
DAN_D void point2center(float ymin, float xmin, float ymax, float xmax, float& cy, float& cx, float& h,
                        float& w) {
  h = fadd(fsub(ymax, ymin), 1.f);
  w = fadd(fsub(xmax, xmin), 1.f);
  // x / 2 == x * 0.5 exactly (a power-of-two scaling rounds identically, also into the denormals): one FMUL instead of
  // the IEEE division sequence
  cy = fmul(fadd(ymin, ymax), 0.5f);
  cx = fmul(fadd(xmin, xmax), 0.5f);
}

// center2point, anchor_manipulator.py:125-127
DAN_D void center2point(float cy, float cx, float h, float w, float& ymin, float& xmin, float& ymax,
                        float& xmax) {
  const float hh = fmul(fsub(h, 1.f), 0.5f);
  const float hw = fmul(fsub(w, 1.f), 0.5f);
  ymin = fsub(cy, hh);
  xmin = fsub(cx, hw);
  ymax = fadd(cy, hh);
  xmax = fadd(cx, hw);
}

// area with the +1 convention, anchor_manipulator.py:24-27
DAN_D float box_area(float ymin, float xmin, float ymax, float xmax) {
  return fmul(fadd(fsub(xmax, xmin), 1.f), fadd(fsub(ymax, ymin), 1.f));
}

// One anchor x GT overlap, anchor_manipulator.py:29-52 in the reference's
// association order.  `hit` reports a non-empty intersection (h>0 && w>0); when
// it is false the overlap is exactly 0 and the division is skipped.
DAN_D float pair_iou(float ay0, float ax0, float ay1, float ax1, float a_area, float gy0, float gx0,
                     float gy1, float gx1, float g_area, bool& hit) {
  const float iy0 = fmaxf(ay0, gy0);
  const float ix0 = fmaxf(ax0, gx0);
  const float iy1 = fminf(ay1, gy1);
  const float ix1 = fminf(ax1, gx1);
  const float h = fmaxf(fadd(fsub(iy1, iy0), 1.f), 0.f);
  const float w = fmaxf(fadd(fsub(ix1, ix0), 1.f), 0.f);
  hit = (h > 0.f) && (w > 0.f);
  if (!hit) return 0.f;
  const float inter = fmul(h, w);
  const float uni = fsub(fadd(a_area, g_area), inter);
  return (uni == 0.f) ? 0.f : fdiv(inter, uni);
}

// Cephes expf / logf in the op order of Eigen's pexp / plog with pmadd = mul,add
// (oracle/reference_np.py expf/logf are the same sequence in numpy).
DAN_D float cephes_expf(float x) {
  x = fminf(fmaxf(x, -88.3762626647949f), 88.3762626647950f);
  const float fx = floorf(fadd(fmul(x, 1.44269504088896341f), 0.5f));
  const float tmp = fmul(fx, 0.693359375f);
  float z = fmul(fx, -2.12194440e-4f);
  x = fsub(x, tmp);
  x = fsub(x, z);
  z = fmul(x, x);
  float y = 1.9875691500e-4f;
  y = fadd(fmul(y, x), 1.3981999507e-3f);
  y = fadd(fmul(y, x), 8.3334519073e-3f);
  y = fadd(fmul(y, x), 4.1665795894e-2f);
  y = fadd(fmul(y, x), 1.6666665459e-1f);
  y = fadd(fmul(y, x), 5.0000001201e-1f);
  y = fadd(fmul(y, z), x);
  y = fadd(y, 1.f);
  // 2^n built in ONE step, (n + 127) << 23, as Eigen's pexp does: n = -127 (x - max below about -87.7) gives the
  // factor +0 and the result 0, not a denormal; n = 128 gives inf
  const int n = (int)fx;
  return fmul(y, __int_as_float((n + 127) << 23));
}

DAN_D float cephes_logf(float x) {
  const bool invalid = x < 0.f;
  const bool iszero = x == 0.f;
  x = fmaxf(x, 1.17549435e-38f);
  const uint32_t bits = __float_as_uint(x);
  float e = (float)((int)(bits >> 23) - 126);
  float m = __uint_as_float((bits & 0x807FFFFFu) | 0x3F000000u);
  const bool small = m < 0.707106781186547524f;
  const float tmp0 = small ? m : 0.f;
  m = fsub(m, 1.f);
  e = fsub(e, small ? 1.f : 0.f);
  m = fadd(m, tmp0);
  const float x2 = fmul(m, m);
  const float x3 = fmul(x2, m);
  float y = fadd(fmul(7.0376836292e-2f, m), -1.1514610310e-1f);
  float y1 = fadd(fmul(-1.2420140846e-1f, m), 1.4249322787e-1f);
  float y2 = fadd(fmul(2.0000714765e-1f, m), -2.4999993993e-1f);
  y = fadd(fmul(y, m), 1.1676998740e-1f);
  y1 = fadd(fmul(y1, m), -1.6668057665e-1f);
  y2 = fadd(fmul(y2, m), 3.3333331174e-1f);
  y = fadd(fmul(y, x3), y1);
  y = fadd(fmul(y, x3), y2);
  y = fmul(y, x3);
  y1 = fmul(e, -2.12194440e-4f);
  const float tmp = fmul(x2, 0.5f);
  y = fadd(y, y1);
  m = fsub(m, tmp);
  y2 = fmul(e, 0.693359375f);
  m = fadd(m, y);
  m = fadd(m, y2);
  if (iszero) m = __int_as_float(0xff800000);  // -inf
  if (invalid) m = __int_as_float(0x7fc00000); // nan
  return m;
}

// tf.nn.softmax of two logits, column 1 (the face probability): exp(x - max) * (1 / sum(exp(x - max))), sum in class
// order - bit for bit the column 1 of dan_softmax with two classes
DAN_D float softmax2_face(float x0, float x1) {
  const float mx = fmaxf(x0, x1);
  const float e0 = cephes_expf(fsub(x0, mx));
  const float e1 = cephes_expf(fsub(x1, mx));
  return fmul(e1, fdiv(1.f, fadd(e0, e1)));
}

// decode one box, anchor_manipulator.py:399-408 / :417-424
DAN_D float4 decode_box(float4 p, float ay0, float ax0, float ay1, float ax1, float ps0, float ps1,
                        float ps2, float ps3) {
  float acy, acx, ah, aw;
  point2center(ay0, ax0, ay1, ax1, acy, acx, ah, aw);
  const float ph = fmul(cephes_expf(fmul(p.z, ps2)), ah);
  const float pw = fmul(cephes_expf(fmul(p.w, ps3)), aw);
  const float pcy = fadd(fmul(fmul(p.x, ps0), ah), acy);
  const float pcx = fadd(fmul(fmul(p.y, ps1), aw), acx);
  float4 o;
  center2point(pcy, pcx, ph, pw, o.x, o.y, o.z, o.w);
  return o;
}

// prediction element types (DAN_DTYPE_*) ---------------------------------------
// fp16 and bf16 predictions are widened to fp32 where they are loaded.  The widening is exact, so everything after the
// load is the fp32 code and its results are those of the fp32 path on the widened inputs.
static inline int dtype_bytes(int32_t dtype) {
  return dtype == DAN_DTYPE_F32 ? 4 : (dtype == DAN_DTYPE_F16 || dtype == DAN_DTYPE_BF16) ? 2 : 0;
}

DAN_D float widen(float v) { return v; }
DAN_D float widen(__half v) { return __half2float(v); }
DAN_D float widen(__nv_bfloat16 v) { return __uint_as_float((uint32_t)__bfloat16_as_ushort(v) << 16); }

// two packed 16-bit values (the lower one first in memory)
template <typename T> DAN_D float2 widen2(uint32_t bits);
template <> DAN_D float2 widen2<__half>(uint32_t bits) { return __half22float2(*reinterpret_cast<const __half2*>(&bits)); }
template <> DAN_D float2 widen2<__nv_bfloat16>(uint32_t bits) {
  return make_float2(__uint_as_float(bits << 16), __uint_as_float(bits & 0xffff0000u));
}

// one anchor's four box values: a 16-byte row (fp32) or an 8-byte row (fp16 / bf16)
template <typename T> struct PredRow {
  typedef uint2 type;
  DAN_D static float4 widen(uint2 r) {
    const float2 lo = widen2<T>(r.x), hi = widen2<T>(r.y);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
  }
};
template <> struct PredRow<float> {
  typedef float4 type;
  DAN_D static float4 widen(float4 r) { return r; }
};

// the two logits of one anchor (two classes); x must be aligned to 2 * sizeof(T)
DAN_D float2 ld_pair(const float* x) { return *reinterpret_cast<const float2*>(x); }
template <typename T> DAN_D float2 ld_pair(const T* x) { return widen2<T>(*reinterpret_cast<const uint32_t*>(x)); }

// logit pair j of a 16-byte vector of four fp16 / bf16 anchors
template <typename T> DAN_D float2 vec_pair(const float4& q, int j) {
  const float w = j == 0 ? q.x : j == 1 ? q.y : j == 2 ? q.z : q.w;
  return widen2<T>(__float_as_uint(w));
}

// warp helpers ---------------------------------------------------------------
// monotone float -> int32 map (total order on non-NaN floats)
DAN_D int float_to_ordered(float f) {
  const int i = __float_as_int(f);
  return i ^ ((i >> 31) & 0x7fffffff);
}
DAN_D float ordered_to_float(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

DAN_D float warp_min_f(float v) { return ordered_to_float(__reduce_min_sync(0xffffffffu, float_to_ordered(v))); }
DAN_D float warp_max_f(float v) { return ordered_to_float(__reduce_max_sync(0xffffffffu, float_to_ordered(v))); }

}  // namespace dan
