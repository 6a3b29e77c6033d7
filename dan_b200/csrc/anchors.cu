// K1 anchor generation, materialised IoU matrix, decode and the elementwise
// bbox_util helpers.  All HBM-bound streaming kernels: one element per thread,
// 128-bit accesses where the layout allows it.
#include "common.cuh"

namespace dan {

// ---------------------------------------------------------------------------
// K1: AnchorEncoder.get_all_anchors, utility/anchor_manipulator.py:163-198,213-273.
// Anchor order inside a layer is y-major, x, depth-minor (reshape [-1, depth] of a
// [H, W, depth] tensor, :192-195); layers are concatenated in list order (:262-266).
// ---------------------------------------------------------------------------
struct PyramidDev {
  dan_pyramid p;
  int64_t layer_base[DAN_MAX_LAYERS + 1];
  int32_t depth_base[DAN_MAX_LAYERS];
};

__global__ void __launch_bounds__(256) anchor_gen_kernel(const __grid_constant__ PyramidDev pd, float* __restrict__ o_ymin,
                                                         float* __restrict__ o_xmin, float* __restrict__ o_ymax,
                                                         float* __restrict__ o_xmax, uint8_t* __restrict__ o_mask) {
  const int64_t total = pd.layer_base[pd.p.num_layers];
  const float img_h = (float)pd.p.image_h;
  const float img_w = (float)pd.p.image_w;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int l = 0;
    while (l + 1 < pd.p.num_layers && i >= pd.layer_base[l + 1]) ++l;
    const int64_t r = i - pd.layer_base[l];
    const int depth = pd.p.depth[l];
    const int d = (int)(r % depth);
    const int64_t cell = r / depth;
    const int x = (int)(cell % pd.p.layer_w[l]);
    const int y = (int)(cell / pd.p.layer_w[l]);
    const float stride = pd.p.stride[l];
    // :186-187  (to_float(y) + offset) * feat_stride
    const float cy = fmul(fadd((float)y, pd.p.offset_h[l]), stride);
    const float cx = fmul(fadd((float)x, pd.p.offset_w[l]), stride);
    float ymin, xmin, ymax, xmax;
    center2point(cy, cx, pd.p.anchor_h[pd.depth_base[l] + d], pd.p.anchor_w[pd.depth_base[l] + d], ymin, xmin, ymax, xmax);
    if (pd.p.clip[l]) {  // :240-244 tf.clip_by_value(v, 0, dim - 1)
      const float hy = fsub(img_h, 1.f), hx = fsub(img_w, 1.f);
      ymin = fminf(fmaxf(ymin, 0.f), hy);
      xmin = fminf(fmaxf(xmin, 0.f), hx);
      ymax = fminf(fmaxf(ymax, 0.f), hy);
      xmax = fminf(fmaxf(xmax, 0.f), hx);
    }
    o_ymin[i] = ymin;
    o_xmin[i] = xmin;
    o_ymax[i] = ymax;
    o_xmax[i] = xmax;
    if (o_mask != nullptr) {  // :268-271
      const float b = fmul(1.f, pd.p.border[l]);
      const bool in = (ymin > -b) && (xmin > -b) && (ymax < fadd(fsub(img_h, 1.f), b)) &&
                      (xmax < fadd(fsub(img_w, 1.f), b));
      o_mask[i] = in ? 1 : 0;
    }
  }
}

static int build_pyramid(const dan_pyramid* h, PyramidDev& pd) {
  DAN_REQUIRE(h != nullptr, DAN_ERR_INVALID_ARGUMENT, "pyramid is NULL");
  DAN_REQUIRE(h->num_layers >= 1 && h->num_layers <= DAN_MAX_LAYERS, DAN_ERR_INVALID_ARGUMENT,
              "num_layers must be in [1, %d], got %d", DAN_MAX_LAYERS, h->num_layers);
  DAN_REQUIRE(h->image_h > 0 && h->image_w > 0, DAN_ERR_INVALID_ARGUMENT, "image shape must be positive");
  pd.p = *h;
  int64_t base = 0;
  int dbase = 0;
  for (int l = 0; l < h->num_layers; ++l) {
    DAN_REQUIRE(h->layer_h[l] >= 0 && h->layer_w[l] >= 0 && h->depth[l] >= 1, DAN_ERR_INVALID_ARGUMENT,
                "layer %d: bad shape (%d,%d) or depth %d", l, h->layer_h[l], h->layer_w[l], h->depth[l]);
    pd.layer_base[l] = base;
    pd.depth_base[l] = dbase;
    base += (int64_t)h->layer_h[l] * h->layer_w[l] * h->depth[l];
    dbase += h->depth[l];
    DAN_REQUIRE(dbase <= DAN_MAX_DEPTH_TOTAL, DAN_ERR_UNSUPPORTED, "sum of anchor depths exceeds %d", DAN_MAX_DEPTH_TOTAL);
  }
  for (int l = h->num_layers; l <= DAN_MAX_LAYERS; ++l) pd.layer_base[l] = base;
  return DAN_OK;
}

// ---------------------------------------------------------------------------
// iou_matrix, anchor_manipulator.py:44-52 (+ the inside-mask multiply of :287)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) iou_matrix_kernel(const float* __restrict__ ay0, const float* __restrict__ ax0,
                                                         const float* __restrict__ ay1, const float* __restrict__ ax1,
                                                         const uint8_t* __restrict__ mask, int n, const float4* __restrict__ gt,
                                                         int m, int mode, float* __restrict__ out) {
  const int64_t total = (int64_t)n * m;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int a = (int)(i / m);
    const int j = (int)(i % m);
    const float y0 = ay0[a], x0 = ax0[a], y1 = ay1[a], x1 = ax1[a];
    const float4 g = __ldg(gt + j);
    float v;
    if (mode == 1) {  // intersection(), anchor_manipulator.py:29-43
      const float h = fmaxf(fadd(fsub(fminf(y1, g.z), fmaxf(y0, g.x)), 1.f), 0.f);
      const float w = fmaxf(fadd(fsub(fminf(x1, g.w), fmaxf(x0, g.y)), 1.f), 0.f);
      v = fmul(h, w);
    } else {
      bool hit;
      v = pair_iou(y0, x0, y1, x1, box_area(y0, x0, y1, x1), g.x, g.y, g.z, g.w, box_area(g.x, g.y, g.z, g.w), hit);
    }
    if (mask != nullptr) v = fmul(v, mask[a] ? 1.f : 0.f);
    out[i] = v;
  }
}

// ---------------------------------------------------------------------------
// decode_anchors / batch_decode_anchors, anchor_manipulator.py:389-424
// ---------------------------------------------------------------------------
// T: element type of pred (float, __half, __nv_bfloat16), widened to fp32 at the load
template <typename T>
__global__ void __launch_bounds__(256) decode_kernel(const typename PredRow<T>::type* __restrict__ pred, const float* __restrict__ ay0,
                                                     const float* __restrict__ ax0, const float* __restrict__ ay1,
                                                     const float* __restrict__ ax1, int n, int64_t total, float ps0, float ps1,
                                                     float ps2, float ps3, float4* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int a = (int)(i % n);
    out[i] = decode_box(PredRow<T>::widen(pred[i]), ay0[a], ax0[a], ay1[a], ax1[a], ps0, ps1, ps2, ps3);
  }
}

// ---------------------------------------------------------------------------
// bbox_util elementwise helpers
// ---------------------------------------------------------------------------
// tf.nn.softmax (bbox_util.py:105): exp(x - max) * (1 / sum), class sum in index order.
__global__ void __launch_bounds__(256) softmax_kernel(const float* __restrict__ logits, int64_t rows, int c, float* __restrict__ out) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
    const float* x = logits + r * c;
    float mx = x[0];
    for (int k = 1; k < c; ++k) mx = fmaxf(mx, x[k]);
    float s = 0.f;
    for (int k = 0; k < c; ++k) {
      const float e = cephes_expf(fsub(x[k], mx));
      out[r * c + k] = e;
      s = (k == 0) ? e : fadd(s, e);
    }
    const float inv = fdiv(1.f, s);
    for (int k = 0; k < c; ++k) out[r * c + k] = fmul(out[r * c + k], inv);
  }
}

// select_bboxes, bbox_util.py:24-36 (one class column)
__global__ void __launch_bounds__(256) select_kernel(const float* __restrict__ scores, int c, int cls, const float4* __restrict__ boxes,
                                                     int64_t n, float thr, float4* __restrict__ o_boxes, float* __restrict__ o_scores) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float s = scores[i * c + cls];
    const float m = (s > thr) ? 1.f : 0.f;
    const float4 b = boxes[i];
    o_boxes[i] = make_float4(fmul(b.x, m), fmul(b.y, m), fmul(b.z, m), fmul(b.w, m));
    o_scores[i] = fmul(s, m);
  }
}

// clip_bboxes, bbox_util.py:38-48
DAN_D float4 clip_box(float4 b, float height, float width) {
  float ymin = fmaxf(b.x, 0.f);
  float xmin = fmaxf(b.y, 0.f);
  const float ymax = fminf(b.z, fsub(height, 1.f));
  const float xmax = fminf(b.w, fsub(width, 1.f));
  ymin = fminf(ymin, ymax);
  xmin = fminf(xmin, xmax);
  return make_float4(ymin, xmin, ymax, xmax);
}

__global__ void __launch_bounds__(256) clip_kernel(const float4* __restrict__ boxes, int64_t n, float height, float width,
                                                   float4* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = clip_box(boxes[i], height, width);
}

// filter_bboxes, bbox_util.py:50-59
__global__ void __launch_bounds__(256) filter_kernel(const float* __restrict__ scores, const float4* __restrict__ boxes, int64_t n,
                                                     float thr, float* __restrict__ o_scores, float4* __restrict__ o_boxes) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 b = boxes[i];
    const float w = fadd(fsub(b.w, b.y), 1.f);
    const float h = fadd(fsub(b.z, b.x), 1.f);
    const float m = ((w > thr) && (h > thr)) ? 1.f : 0.f;
    o_scores[i] = fmul(scores[i], m);
    o_boxes[i] = make_float4(fmul(b.x, m), fmul(b.y, m), fmul(b.z, m), fmul(b.w, m));
  }
}

// bbox_point2center :92-96 / bbox_center2point :98-101 / areas (anchor_manipulator.py:24-27, mode 2: area in .x)
__global__ void __launch_bounds__(256) convert_kernel(const float4* __restrict__ boxes, int64_t n, int mode, float4* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 b = boxes[i];
    float4 o;
    if (mode == 0) point2center(b.x, b.y, b.z, b.w, o.x, o.y, o.z, o.w);
    else if (mode == 1) center2point(b.x, b.y, b.z, b.w, o.x, o.y, o.z, o.w);
    else o = make_float4(box_area(b.x, b.y, b.z, b.w), 0.f, 0.f, 0.f);
    out[i] = o;
  }
}

template <typename T>
static int decode_launch(const void* pred, const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax,
                         int32_t num_anchors, int64_t total, const float* ps, float* out_boxes, cudaStream_t st) {
  decode_kernel<T><<<grid_for(total), 256, 0, st>>>(static_cast<const typename PredRow<T>::type*>(pred), a_ymin, a_xmin, a_ymax, a_xmax,
                                                    num_anchors, total, ps[0], ps[1], ps[2], ps[3], reinterpret_cast<float4*>(out_boxes));
  DAN_LAUNCH_CHECK("decode_kernel");
  return DAN_OK;
}

}  // namespace dan

using namespace dan;

extern "C" {

int64_t dan_anchor_count(const dan_pyramid* h_pyr) {
  PyramidDev pd;
  if (build_pyramid(h_pyr, pd) != DAN_OK) return -1;
  return pd.layer_base[h_pyr->num_layers];
}

int dan_generate_anchors(const dan_pyramid* h_pyr, float* out_ymin, float* out_xmin, float* out_ymax, float* out_xmax,
                         uint8_t* out_inside_mask, void* stream) {
  PyramidDev pd;
  int rc = build_pyramid(h_pyr, pd);
  if (rc != DAN_OK) return rc;
  DAN_REQUIRE(out_ymin && out_xmin && out_ymax && out_xmax, DAN_ERR_INVALID_ARGUMENT, "anchor outputs must be non-NULL");
  const int64_t total = pd.layer_base[h_pyr->num_layers];
  if (total == 0) return DAN_OK;
  anchor_gen_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(pd, out_ymin, out_xmin, out_ymax, out_xmax, out_inside_mask);
  DAN_LAUNCH_CHECK("anchor_gen_kernel");
  return DAN_OK;
}

static int pairwise_matrix(int mode, const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax,
                           const uint8_t* inside_mask, int32_t num_anchors, const float* gt_boxes, int32_t num_gt, float* out_overlaps,
                           void* stream) {
  DAN_REQUIRE(num_anchors >= 0 && num_gt >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  if (num_anchors == 0 || num_gt == 0) return DAN_OK;
  DAN_REQUIRE(a_ymin && a_xmin && a_ymax && a_xmax && gt_boxes && out_overlaps, DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  DAN_REQUIRE(aligned16(gt_boxes), DAN_ERR_INVALID_ARGUMENT, "gt_boxes must be 16-byte aligned");
  iou_matrix_kernel<<<grid_for((int64_t)num_anchors * num_gt), 256, 0, (cudaStream_t)stream>>>(
      a_ymin, a_xmin, a_ymax, a_xmax, inside_mask, num_anchors, reinterpret_cast<const float4*>(gt_boxes), num_gt, mode, out_overlaps);
  DAN_LAUNCH_CHECK("iou_matrix_kernel");
  return DAN_OK;
}

int dan_iou_matrix(const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax, const uint8_t* inside_mask,
                   int32_t num_anchors, const float* gt_boxes, int32_t num_gt, float* out_overlaps, void* stream) {
  return pairwise_matrix(0, a_ymin, a_xmin, a_ymax, a_xmax, inside_mask, num_anchors, gt_boxes, num_gt, out_overlaps, stream);
}

int dan_intersection_matrix(const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax, int32_t num_anchors,
                            const float* gt_boxes, int32_t num_gt, float* out_inter, void* stream) {
  return pairwise_matrix(1, a_ymin, a_xmin, a_ymax, a_xmax, nullptr, num_anchors, gt_boxes, num_gt, out_inter, stream);
}

int dan_decode_batch_typed(int32_t pred_dtype, const void* pred, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                           const float* a_xmax, int32_t num_anchors, int32_t batch, const float* h_prior_scaling, float* out_boxes,
                           void* stream) {
  const int esize = dtype_bytes(pred_dtype);
  DAN_REQUIRE(esize != 0, DAN_ERR_INVALID_ARGUMENT, "unknown pred_dtype %d", pred_dtype);
  DAN_REQUIRE(num_anchors >= 0 && batch >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  if (num_anchors == 0 || batch == 0) return DAN_OK;
  DAN_REQUIRE(pred && a_ymin && a_xmin && a_ymax && a_xmax && out_boxes && h_prior_scaling, DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  DAN_REQUIRE((reinterpret_cast<uintptr_t>(pred) & (uintptr_t)(4 * esize - 1)) == 0 && aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT,
              "pred must be %d-byte aligned, out_boxes 16-byte aligned", 4 * esize);
  const int64_t total = (int64_t)num_anchors * batch;
  cudaStream_t st = (cudaStream_t)stream;
  switch (pred_dtype) {
    case DAN_DTYPE_F16: return decode_launch<__half>(pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, total, h_prior_scaling, out_boxes, st);
    case DAN_DTYPE_BF16:
      return decode_launch<__nv_bfloat16>(pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, total, h_prior_scaling, out_boxes, st);
    default: return decode_launch<float>(pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, total, h_prior_scaling, out_boxes, st);
  }
}

int dan_decode_batch(const float* pred, const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax,
                     int32_t num_anchors, int32_t batch, const float* h_prior_scaling, float* out_boxes, void* stream) {
  return dan_decode_batch_typed(DAN_DTYPE_F32, pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch, h_prior_scaling, out_boxes,
                                stream);
}

int dan_softmax(const float* logits, int64_t rows, int32_t num_classes, float* out, void* stream) {
  DAN_REQUIRE(rows >= 0 && num_classes >= 1, DAN_ERR_INVALID_ARGUMENT, "bad shape");
  if (rows == 0) return DAN_OK;
  DAN_REQUIRE(logits && out, DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  softmax_kernel<<<grid_for(rows), 256, 0, (cudaStream_t)stream>>>(logits, rows, num_classes, out);
  DAN_LAUNCH_CHECK("softmax_kernel");
  return DAN_OK;
}

int dan_select_bboxes(const float* scores, int32_t num_classes, int32_t class_ind, const float* boxes, int64_t n,
                      float select_threshold, float* out_boxes, float* out_scores, void* stream) {
  DAN_REQUIRE(n >= 0 && num_classes >= 1 && class_ind >= 0 && class_ind < num_classes, DAN_ERR_INVALID_ARGUMENT, "bad shape / class index");
  if (n == 0) return DAN_OK;
  DAN_REQUIRE(scores && boxes && out_boxes && out_scores, DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  DAN_REQUIRE(aligned16(boxes) && aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT, "boxes must be 16-byte aligned");
  select_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(scores, num_classes, class_ind, reinterpret_cast<const float4*>(boxes), n,
                                                               select_threshold, reinterpret_cast<float4*>(out_boxes), out_scores);
  DAN_LAUNCH_CHECK("select_kernel");
  return DAN_OK;
}

int dan_clip_bboxes(const float* boxes, int64_t n, float height, float width, float* out_boxes, void* stream) {
  DAN_REQUIRE(n >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  if (n == 0) return DAN_OK;
  DAN_REQUIRE(boxes && out_boxes && aligned16(boxes) && aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT, "boxes NULL or not 16-byte aligned");
  clip_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(boxes), n, height, width,
                                                             reinterpret_cast<float4*>(out_boxes));
  DAN_LAUNCH_CHECK("clip_kernel");
  return DAN_OK;
}

int dan_filter_bboxes(const float* scores, const float* boxes, int64_t n, float min_size_plus_1, float* out_scores, float* out_boxes,
                      void* stream) {
  DAN_REQUIRE(n >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  if (n == 0) return DAN_OK;
  DAN_REQUIRE(scores && out_scores && boxes && out_boxes && aligned16(boxes) && aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT,
              "NULL pointer or boxes not 16-byte aligned");
  filter_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(scores, reinterpret_cast<const float4*>(boxes), n, min_size_plus_1,
                                                               out_scores, reinterpret_cast<float4*>(out_boxes));
  DAN_LAUNCH_CHECK("filter_kernel");
  return DAN_OK;
}

int dan_bbox_convert(const float* boxes, int64_t n, int32_t mode, float* out_boxes, void* stream) {
  DAN_REQUIRE(n >= 0 && mode >= 0 && mode <= 2, DAN_ERR_INVALID_ARGUMENT, "bad size or mode");
  if (n == 0) return DAN_OK;
  DAN_REQUIRE(boxes && out_boxes && aligned16(boxes) && aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT, "boxes NULL or not 16-byte aligned");
  convert_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(boxes), n, mode,
                                                                reinterpret_cast<float4*>(out_boxes));
  DAN_LAUNCH_CHECK("convert_kernel");
  return DAN_OK;
}

}  // extern "C"
