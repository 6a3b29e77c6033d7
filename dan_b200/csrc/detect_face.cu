// detect_face (eval_sfd.py:95-114) for B images of N anchors, in two kernels:
//   face_key_kernel     grid-wide over B x N: key = score bits << 32 | anchor (equal scores: higher anchor first), and a
//                       per-image histogram of the keys' face_bin() (shared-memory histogram per CTA, flushed with one
//                       global atomic per non-empty bin)
//   face_select_kernel  one CTA per image: the histogram gives the bin that holds the k-th key; one pass over the image's
//                       keys compacts those in that bin or above into shared memory, where they are sorted.  Only the k
//                       rows are read (or decoded from the offsets), divided by shrink and written.
//   face_select_large_kernel  the same steps for k > kSortCap (up to kFaceTopCap): the candidates are compacted into
//                       the workspace and sorted there with select_and_sort_large (face_large_plan).
// The score comes from the scores of decoded boxes (dan_detect_face_select) or from the two logits (the softmax in
// tf.nn.softmax's op order, dan_detect_face_batch); the box from a decoded row or from a decode of the offset row.
#include "common.cuh"

namespace dan {

#include "sort.cuh"

namespace {

constexpr int kFaceBins = 4096;             // histogram bins per image
constexpr int kFaceKeyThreads = 512;
constexpr int kFaceChunk = 8 * kFaceKeyThreads;   // anchors per CTA of the key kernel
// largest `top` of the _top entry points.  It equals bbox_vote's limit (kVoteLargeCap in vote.cu), so that the rows
// detect_face keeps per image always fit dan_bbox_vote_ws.
constexpr int kFaceTopCap = 1 << 20;

// A monotone map of a key to [0, kFaceBins): keys in a higher bin are larger.  Half of the bins cut the probabilities
// [0.5, 1) into steps of 2^-12 (confident detections crowd there), the other half cover [2^-17, 0.5) at 128 bins per
// octave; smaller scores (and negative ones) share bin 0, larger ones (and NaN) the last bin.
DAN_D int face_bin(unsigned long long key) {
  const uint32_t x = (uint32_t)(key >> 32);
  constexpr uint32_t kHalf = 0xBF000000u;                  // score_to_key(0.5f)
  if (x >= kHalf) return kFaceBins / 2 + (int)min((x - kHalf) >> 12, (uint32_t)(kFaceBins / 2 - 1));
  return max((int)(x >> 16) - (int)((kHalf >> 16) - kFaceBins / 2), 0);
}

struct FaceScores {                         // scores of decoded boxes, [B, N] fp32
  const float* s;
  DAN_D float score(int64_t row) const { return s[row]; }
};

template <typename T> struct FaceLogits {   // two logits per anchor, [B, N, 2]
  const T* x;
  bool pair_aligned;                        // false: a pair is not aligned for one load (read as two scalars)
  DAN_D float score(int64_t row) const {
    const float2 v = pair_aligned ? ld_pair(x + 2 * row) : make_float2(widen(x[2 * row]), widen(x[2 * row + 1]));
    return softmax2_face(v.x, v.y);
  }
};

struct FaceBoxes {                          // decoded boxes, [B, N, 4] (ymin, xmin, ymax, xmax)
  const float4* boxes;
  DAN_D float4 box(int64_t row, int) const { return boxes[row]; }
};

template <typename T> struct FaceOffsets {  // offsets [B, N, 4] (cy, cx, h, w), decoded like dan_decode_batch
  const typename PredRow<T>::type* loc;
  const float *ay0, *ax0, *ay1, *ax1;
  float ps0, ps1, ps2, ps3;
  DAN_D float4 box(int64_t row, int a) const {
    return decode_box(PredRow<T>::widen(loc[row]), ay0[a], ax0[a], ay1[a], ax1[a], ps0, ps1, ps2, ps3);
  }
};

struct FaceArgs {
  int n;                      // anchors per image
  int chunks;                 // CTAs of the key kernel per image
  float shrink;
  int top;                    // int(1.5 * max_per_image)
  int k;                      // rows per image: max(min(n - 1, top), 0)
  unsigned long long* keys;   // [B, n] workspace
  int* hist;                  // [B, kFaceBins] workspace, zeroed before the key kernel
  float* out;                 // [B, top, 5] zero padded
  int32_t* out_index;         // [B, top] optional, -1 padded
  int32_t* out_count;         // [1] optional (the single-image entry point)
};

template <class Score>
__global__ void __launch_bounds__(kFaceKeyThreads) face_key_kernel(const FaceArgs A, const Score S) {
  __shared__ int s_hist[kFaceBins];
  const int tid = threadIdx.x, lane = tid & 31;
  const int b = blockIdx.x / A.chunks;
  const int a0 = (blockIdx.x - b * A.chunks) * kFaceChunk;
  for (int i = tid; i < kFaceBins; i += kFaceKeyThreads) s_hist[i] = 0;
  __syncthreads();
  const int64_t row0 = (int64_t)b * A.n;
#pragma unroll 4
  for (int j = 0; j < kFaceChunk / kFaceKeyThreads; ++j) {
    const int a = a0 + j * kFaceKeyThreads + tid;
    int bin = -1;
    if (a < A.n) {
      const unsigned long long key = ((unsigned long long)score_to_key(S.score(row0 + a)) << 32) | (unsigned long long)(uint32_t)a;
      A.keys[row0 + a] = key;
      bin = face_bin(key);
    }
    const unsigned same = __match_any_sync(0xffffffffu, bin);         // one shared atomic per bin and warp
    if (bin >= 0 && lane == __ffs(same) - 1) atomicAdd(&s_hist[bin], __popc(same));
  }
  __syncthreads();
  int* hist = A.hist + (int64_t)b * kFaceBins;
  for (int i = tid; i < kFaceBins; i += kFaceKeyThreads)
    if (s_hist[i] != 0) atomicAdd(&hist[i], s_hist[i]);
}

// eval_sfd.py:101-112, one CTA per image, in the steps below (both select kernels run them).
struct FaceBin {
  int t;                      // the bin of the k-th largest key
  int ge;                     // keys in bin t or above (>= k)
};

// 1. the bin t of image b's k-th largest key (k = A.k > 0) and the keys in bin t or above, from the image's histogram:
// thread i holds bins 4i .. 4i + 3, `above` counts the keys in higher bins.  Also zeroes sc.fill for step 2.
// s_warp [32], s_bin and s_ge are the kernel's shared memory.  (The steps take the thread, lane and warp index from
// the kernel, which computes them first: face_select_kernel then compiles to the instructions it had as one function.)
DAN_D FaceBin face_kth_bin(const FaceArgs& A, int b, int tid, int lane, int warp, SortScratch& sc, int* s_warp, int& s_bin,
                           int& s_ge) {
  const int k = A.k;
  constexpr int kPer = kFaceBins / kSortThreads;
  const int* hist = A.hist + (int64_t)b * kFaceBins + kPer * tid;
  const int hb[kPer] = {hist[0], hist[1], hist[2], hist[3]};
  const int c = hb[0] + hb[1] + hb[2] + hb[3];
  int incl = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int v = __shfl_down_sync(0xffffffffu, incl, d);
    if (lane + d < 32) incl += v;
  }
  if (lane == 0) s_warp[warp] = incl;
  if (tid == 0) sc.fill = 0;
  __syncthreads();
  int above = incl - c;
  for (int w = warp + 1; w < kSortThreads / 32; ++w) above += s_warp[w];
  if (above < k && above + c >= k) {                       // exactly one thread: the bins hold all n > k keys
    int cum = above, t = kPer * tid;
    for (int j = kPer - 1; j >= 0; --j) {
      cum += hb[j];
      if (cum >= k) { t = kPer * tid + j; break; }
    }
    s_bin = t;
    s_ge = cum;
  }
  __syncthreads();
  return {s_bin, s_ge};
}

// 2. one pass over the image's n keys: the ge keys in bin t or above (a superset of the top k) into dst[0, ge) (shared
// memory or the workspace), in no particular order, one atomic on sc.fill per warp
DAN_D void face_compact(const unsigned long long* keys, int n, int t, unsigned long long* dst, int tid, int lane, SortScratch& sc) {
  for (int i0 = 0; i0 < n; i0 += 4 * kSortThreads) {
    unsigned long long q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * kSortThreads + tid;
      q[u] = i < n ? __ldcs(keys + i) : 0ull;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const bool keep = i0 + u * kSortThreads + tid < n && face_bin(q[u]) >= t;
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      if (m != 0u) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&sc.fill, __popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (keep) dst[base + __popc(m & ((1u << lane) - 1u))] = q[u];
      }
    }
  }
}

// 4. the top rows of image b from its k sorted keys (shared memory or the workspace): the box read or decoded, / shrink,
// columns (xmin, ymin, xmax, ymax, score); rows k .. top - 1 zero with index -1
template <class Box>
DAN_D void face_write_rows(const FaceArgs& A, const Box& src, int b, int k, const unsigned long long* sorted, int tid) {
  float* out = A.out + (int64_t)b * A.top * 5;
  for (int r = tid; r < A.top; r += kSortThreads) {
    float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f, o4 = 0.f;
    int idx = -1;
    if (r < k) {
      const unsigned long long key = sorted[r];
      idx = (int)(uint32_t)(key & 0xFFFFFFFFull);
      const float4 bx = src.box((int64_t)b * A.n + idx, idx);
      o0 = fdiv(bx.y, A.shrink); o1 = fdiv(bx.x, A.shrink); o2 = fdiv(bx.w, A.shrink); o3 = fdiv(bx.z, A.shrink);
      o4 = key_to_score((uint32_t)(key >> 32));           // the score's bits, NaN payloads included
    }
    out[r * 5] = o0; out[r * 5 + 1] = o1; out[r * 5 + 2] = o2; out[r * 5 + 3] = o3; out[r * 5 + 4] = o4;
    if (A.out_index) A.out_index[(int64_t)b * A.top + r] = idx;
  }
  if (tid == 0 && A.out_count) A.out_count[b] = k;
}

// k <= kSortCap: steps 2 and 3 in shared memory
template <class Box>
__global__ void __launch_bounds__(kSortThreads, 1) face_select_kernel(const FaceArgs A, const Box src) {
  extern __shared__ unsigned long long s_keys[];           // [kSortCap] keys | [kSortCap] merge buffer
  __shared__ SortScratch sc;
  __shared__ int s_warp[kSortThreads / 32];
  __shared__ int s_bin, s_ge;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  const int k = A.k;
  const unsigned long long* keys = A.keys + (int64_t)b * A.n;
  if (k > 0) {
    const FaceBin fb = face_kth_bin(A, b, tid, lane, warp, sc, s_warp, s_bin, s_ge);
    if (fb.ge <= kSortCap) {
      face_compact(keys, A.n, fb.t, s_keys, tid, lane, sc);
      __syncthreads();
      select_and_sort(keys, fb.ge, k, s_keys, sc, true, s_keys + kSortCap);     // 3. (the keys are staged)
    } else {
      // more keys share the k-th key's bin than shared memory holds: radix select over all of the image's keys
      select_and_sort(keys, A.n, k, s_keys, sc, false, s_keys + kSortCap);
    }
  }
  face_write_rows(A, src, b, k, s_keys, tid);
}

constexpr size_t kFaceSelectSmem = 2 * kSortCap * sizeof(unsigned long long);

static size_t face_hist_bytes(int32_t batch) { return align_up((size_t)batch * kFaceBins * sizeof(int), 256); }

// Workspace of face_select_large_kernel (k > kSortCap): one slice per image behind the histograms and the keys.  Offsets
// of the arrays are in bytes from the start of an image's slice (image * `image`); every array is 256-byte aligned.
struct FaceLargePlan {
  size_t region;              // start of the slices in the workspace (= dan_detect_face_batch_workspace_bytes(n, B))
  size_t image;               // workspace bytes per image
  size_t sorted;              // [k] u64: the top k keys, sorted (select_and_sort_large's buf_a)
  size_t merge;               // [k] u64: the sort's merge buffer (select_and_sort_large's buf_b)
  size_t cand;                // [cand_cap] u64: the keys in the k-th key's bin or above (step 2)
  int cand_cap;               // 2k: more candidates (ties in one bin) select over all n keys instead
};

static FaceLargePlan face_large_plan(int64_t n, int32_t batch, int k) {
  FaceLargePlan p = {};
  p.region = face_hist_bytes(batch) + align_up((size_t)n * (size_t)batch * 8, 256);
  p.cand_cap = 2 * k;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 256); return at; };
  p.sorted = take((size_t)k * 8);
  p.merge = take((size_t)k * 8);
  p.cand = take((size_t)p.cand_cap * 8);
  p.image = off;
  return p;
}

// k > kSortCap: the candidates are compacted into the workspace and sorted there (runs of kSortCap keys in shared
// memory, merged in the workspace); ws is the start of the plan's slices
template <class Box>
__global__ void __launch_bounds__(kSortThreads, 1) face_select_large_kernel(const FaceArgs A, const Box src, const FaceLargePlan P,
                                                                            unsigned char* ws) {
  extern __shared__ unsigned long long s_keys[];           // [kSortCap] the runs of the sort
  __shared__ SortScratch sc;
  __shared__ int s_warp[kSortThreads / 32];
  __shared__ int s_bin, s_ge;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  const int k = A.k;
  const unsigned long long* keys = A.keys + (int64_t)b * A.n;
  unsigned char* slice = ws + (size_t)b * P.image;
  unsigned long long* sorted = reinterpret_cast<unsigned long long*>(slice + P.sorted);
  unsigned long long* merge = reinterpret_cast<unsigned long long*>(slice + P.merge);
  unsigned long long* cand = reinterpret_cast<unsigned long long*>(slice + P.cand);
  const FaceBin fb = face_kth_bin(A, b, tid, lane, warp, sc, s_warp, s_bin, s_ge);
  // 3. the k largest of the candidates (or, with more keys in the k-th key's bin than the candidate area holds, of all
  // n keys), sorted into `sorted`
  const unsigned long long* from = keys;
  int cnt = A.n;
  if (fb.ge <= P.cand_cap) {
    face_compact(keys, A.n, fb.t, cand, tid, lane, sc);
    __syncthreads();
    from = cand;
    cnt = fb.ge;
  }
  select_and_sort_large(from, cnt, k, sorted, merge, s_keys, sc);
  face_write_rows(A, src, b, k, sorted, tid);
}

constexpr int kFaceLargeSmem = kSortCap * sizeof(unsigned long long);

template <class Score, class Box>
static int face_launch(const Score& score, const Box& box, int64_t n, int32_t batch, float shrink, int32_t top, float* out_det,
                       int32_t* out_index, int32_t* out_count, void* workspace, cudaStream_t st) {
  FaceArgs A = {};
  A.n = (int)n;
  A.chunks = (int)((n + kFaceChunk - 1) / kFaceChunk);
  A.shrink = shrink;
  A.top = top;
  A.k = (int)(n - 1 < top ? (n - 1 > 0 ? n - 1 : 0) : top);    // N == 0: the reference slices [:-1] of an empty array
  A.hist = static_cast<int*>(workspace);
  A.keys = reinterpret_cast<unsigned long long*>(static_cast<unsigned char*>(workspace) + face_hist_bytes(batch));
  A.out = out_det;
  A.out_index = out_index;
  A.out_count = out_count;
  if (A.k > 0) {
    DAN_CUDA(cudaMemsetAsync(A.hist, 0, (size_t)batch * kFaceBins * sizeof(int), st));
    face_key_kernel<Score><<<(unsigned)((int64_t)A.chunks * batch), kFaceKeyThreads, 0, st>>>(A, score);
    DAN_LAUNCH_CHECK("face_key_kernel");
  }
  if (A.k > kSortCap) {
    const FaceLargePlan P = face_large_plan(n, batch, A.k);
    DAN_CUDA(cudaFuncSetAttribute(face_select_large_kernel<Box>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFaceLargeSmem));
    face_select_large_kernel<Box><<<batch, kSortThreads, kFaceLargeSmem, st>>>(A, box, P, static_cast<unsigned char*>(workspace) + P.region);
    DAN_LAUNCH_CHECK("face_select_large_kernel");
    return DAN_OK;
  }
  DAN_CUDA(cudaFuncSetAttribute(face_select_kernel<Box>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFaceSelectSmem));
  face_select_kernel<Box><<<batch, kSortThreads, kFaceSelectSmem, st>>>(A, box);
  DAN_LAUNCH_CHECK("face_select_kernel");
  return DAN_OK;
}

template <typename T>
static int face_batch_launch(const void* cls_pred, const void* loc_pred, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                             const float* a_xmax, int64_t n, int32_t batch, const float* ps, float shrink, int32_t top, float* out_det,
                             int32_t* out_index, void* workspace, cudaStream_t st) {
  FaceLogits<T> score;
  score.x = static_cast<const T*>(cls_pred);
  score.pair_aligned = (reinterpret_cast<uintptr_t>(cls_pred) & (2 * sizeof(T) - 1)) == 0;
  FaceOffsets<T> box;
  box.loc = static_cast<const typename PredRow<T>::type*>(loc_pred);
  box.ay0 = a_ymin; box.ax0 = a_xmin; box.ay1 = a_ymax; box.ax1 = a_xmax;
  box.ps0 = ps[0]; box.ps1 = ps[1]; box.ps2 = ps[2]; box.ps3 = ps[3];
  return face_launch(score, box, n, batch, shrink, top, out_det, out_index, nullptr, workspace, st);
}

// dan_detect_face_select and dan_detect_face_select_top: the same checks, top in [1, top_cap]
static int face_select_checked(const float* bboxes, const float* scores, int64_t n, float shrink, int32_t top, int32_t top_cap,
                        float* out_det, int32_t* out_index, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream) {
  DAN_REQUIRE(n >= 0 && n < ((int64_t)1 << 31), DAN_ERR_INVALID_ARGUMENT, "bad n");
  DAN_REQUIRE(top >= 1 && top <= top_cap, DAN_ERR_UNSUPPORTED, "top must be in [1, %d]", top_cap);
  DAN_REQUIRE(out_det && out_count, DAN_ERR_INVALID_ARGUMENT, "NULL output");
  DAN_REQUIRE(n == 0 || (bboxes && scores && aligned16(bboxes)), DAN_ERR_INVALID_ARGUMENT, "NULL / misaligned input");
  const size_t need = dan_detect_face_top_workspace_bytes(n, 1, top);
  DAN_REQUIRE(n == 0 || (workspace != nullptr && workspace_bytes >= need), DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu",
              need, workspace_bytes);
  FaceScores score = {scores};
  FaceBoxes box = {reinterpret_cast<const float4*>(bboxes)};
  return face_launch(score, box, n, 1, shrink, top, out_det, out_index, out_count, workspace, (cudaStream_t)stream);
}

// dan_detect_face_batch and dan_detect_face_batch_top: the same checks, top in [1, top_cap]
static int face_batch_checked(int32_t pred_dtype, const void* cls_pred, const void* loc_pred, const float* a_ymin, const float* a_xmin,
                       const float* a_ymax, const float* a_xmax, int64_t num_anchors, int32_t batch, const float* h_prior_scaling,
                       float shrink, int32_t top, int32_t top_cap, float* out_det, int32_t* out_index, void* workspace,
                       size_t workspace_bytes, void* stream) {
  const int esize = dtype_bytes(pred_dtype);
  DAN_REQUIRE(esize != 0, DAN_ERR_INVALID_ARGUMENT, "unknown pred_dtype %d", pred_dtype);
  DAN_REQUIRE(num_anchors >= 0 && num_anchors < ((int64_t)1 << 31) && batch >= 0, DAN_ERR_INVALID_ARGUMENT, "bad num_anchors / batch");
  DAN_REQUIRE(top >= 1 && top <= top_cap, DAN_ERR_UNSUPPORTED, "top must be in [1, %d]", top_cap);
  if (batch == 0) return DAN_OK;
  DAN_REQUIRE(cls_pred && loc_pred && a_ymin && a_xmin && a_ymax && a_xmax && h_prior_scaling && out_det, DAN_ERR_INVALID_ARGUMENT,
              "NULL pointer");
  DAN_REQUIRE((reinterpret_cast<uintptr_t>(loc_pred) & (uintptr_t)(4 * esize - 1)) == 0, DAN_ERR_INVALID_ARGUMENT,
              "loc_pred must be %d-byte aligned", 4 * esize);
  const int64_t chunks = (num_anchors + kFaceChunk - 1) / kFaceChunk;
  DAN_REQUIRE(chunks * batch < ((int64_t)1 << 31), DAN_ERR_UNSUPPORTED, "batch x num_anchors too large");
  const size_t need = dan_detect_face_top_workspace_bytes(num_anchors, batch, top);
  DAN_REQUIRE(workspace != nullptr && workspace_bytes >= need, DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need,
              workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  switch (pred_dtype) {
    case DAN_DTYPE_F16:
      return face_batch_launch<__half>(cls_pred, loc_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch, h_prior_scaling, shrink, top,
                                       out_det, out_index, workspace, st);
    case DAN_DTYPE_BF16:
      return face_batch_launch<__nv_bfloat16>(cls_pred, loc_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch, h_prior_scaling, shrink,
                                              top, out_det, out_index, workspace, st);
    default:
      return face_batch_launch<float>(cls_pred, loc_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch, h_prior_scaling, shrink, top,
                                      out_det, out_index, workspace, st);
  }
}

}  // namespace

}  // namespace dan

using namespace dan;

extern "C" {

size_t dan_detect_face_batch_workspace_bytes(int64_t num_anchors, int32_t batch) {
  if (num_anchors < 0 || batch < 0) return 0;
  return face_hist_bytes(batch) + align_up((size_t)num_anchors * (size_t)batch * 8, 256);
}

size_t dan_detect_face_workspace_bytes(int64_t n) { return dan_detect_face_batch_workspace_bytes(n, 1); }

size_t dan_detect_face_top_workspace_bytes(int64_t num_anchors, int32_t batch, int32_t top) {
  if (num_anchors < 0 || batch < 0) return 0;
  const int64_t k = num_anchors - 1 < top ? (num_anchors - 1 > 0 ? num_anchors - 1 : 0) : top;
  const size_t base = dan_detect_face_batch_workspace_bytes(num_anchors, batch);
  if (top > kFaceTopCap) return 0;
  if (k <= kSortCap) return base;
  return base + (size_t)batch * face_large_plan(num_anchors, batch, (int)k).image;
}

int dan_detect_face_select(const float* bboxes, const float* scores, int64_t n, float shrink, int32_t top, float* out_det,
                           int32_t* out_index, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream) {
  return face_select_checked(bboxes, scores, n, shrink, top, kSortCap, out_det, out_index, out_count, workspace, workspace_bytes,
                             stream);
}

int dan_detect_face_select_top(const float* bboxes, const float* scores, int64_t n, float shrink, int32_t top, float* out_det,
                               int32_t* out_index, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream) {
  return face_select_checked(bboxes, scores, n, shrink, top, kFaceTopCap, out_det, out_index, out_count, workspace,
                             workspace_bytes, stream);
}

int dan_detect_face_batch(int32_t pred_dtype, const void* cls_pred, const void* loc_pred, const float* a_ymin, const float* a_xmin,
                          const float* a_ymax, const float* a_xmax, int64_t num_anchors, int32_t batch, const float* h_prior_scaling,
                          float shrink, int32_t top, float* out_det, int32_t* out_index, void* workspace, size_t workspace_bytes,
                          void* stream) {
  return face_batch_checked(pred_dtype, cls_pred, loc_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch, h_prior_scaling,
                            shrink, top, kSortCap, out_det, out_index, workspace, workspace_bytes, stream);
}

int dan_detect_face_batch_top(int32_t pred_dtype, const void* cls_pred, const void* loc_pred, const float* a_ymin,
                              const float* a_xmin, const float* a_ymax, const float* a_xmax, int64_t num_anchors, int32_t batch,
                              const float* h_prior_scaling, float shrink, int32_t top, float* out_det, int32_t* out_index,
                              void* workspace, size_t workspace_bytes, void* stream) {
  return face_batch_checked(pred_dtype, cls_pred, loc_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch, h_prior_scaling,
                            shrink, top, kFaceTopCap, out_det, out_index, workspace, workspace_bytes, stream);
}

}  // extern "C"
