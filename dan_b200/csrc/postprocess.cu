// K3-K5: the evaluation half of the path -- utility/bbox_util.py:103-119
// parse_by_class and its pieces, batched over images and classes.
//
//   pp_filter_kernel   (more than two classes; for two classes the NMS kernel filters its own image)
//                      softmax -> select(threshold) -> decode -> clip -> min-size;
//                      survivors are COMPACTED as 64-bit keys
//                      (ordered score bits << 32 | ~anchor index).  The reference
//                      instead multiplies by 0/1 masks and keeps all N rows
//                      (bbox_util.py:24-59); rows it zeroes can never precede a
//                      positive score in tf.nn.top_k, so dropping them is exact.
//   topk_sort_kernel   sort_bboxes alone (bbox_util.py:61-72): block radix select of the keep_topk largest keys
//                      when more survive, then the bitonic sort of sort.cuh.  Keys are unique, descending key
//                      order == descending score with ties broken by LOWER index, which is tf.nn.top_k's order.
//   nms_greedy_kernel  per (image, class): the same top-k + sort, decode of the survivors, and
//                      tf.image.non_max_suppression (no +1, corners min/max-normalised, strict >, area <= 0 never
//                      suppresses) as a chunked greedy sweep against the kept list, then the zero padded outputs
//                      (bbox_util.py:80-90).  One launch, one CTA per list.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace dan {

#include "sort.cuh"

// Dynamic shared memory of one nms_greedy_kernel launch (greedy_plan).  Offsets are in bytes from the start of the
// dynamic shared memory, 16-byte aligned; the candidate boxes start at 0, over the keys.
struct GreedyPlan {
  int where;            // the kernel's WHERE: 0 = candidates and kept list in shared memory, 1 = candidates in the
                        // workspace, 2 = both in the workspace (very long lists)
  int smem;             // dynamic shared memory of the launch
  int sort_bytes;       // bytes reserved for the keys while they are sorted
  int slots;            // candidate slots per list (cand_slots): also the per-list stride of the workspace arrays
  int wcap;             // 32-bit words per stripe bitset = ceil(nms_cap / 32)
  int cand_area, cand_mask;                      // where == 0
  int kept_box, kept_area, kept_rank, stripes;   // where <= 1; stripes: [2][32][wcap]
};

struct PpArgs {
  // inputs
  // inputs of element type T (float, __half or __nv_bfloat16: the T of the kernel templates)
  const void* cls;        // [B, N, C] logits
  const void* loc;        // [B, N, 4] offsets (or NULL)
  const void* boxes;      // [B, N, 4] decoded boxes (or NULL)
  const float* ay0;
  const float* ax0;
  const float* ay1;
  const float* ax1;
  int n, batch, num_classes;
  float img_h, img_w;
  float select_thr, min_size_p1;
  float reject_below;         // 2 classes: logit difference below which softmax <= threshold for sure (-inf: off)
  float ps0, ps1, ps2, ps3;
  int keep_topk, nms_topk;
  int nms_cap;                // kept-list capacity = min(nms_topk, keep_topk)
  float nms_thr;
  GreedyPlan plan;             // shared-memory plan of the NMS kernel
  // workspace
  unsigned long long* keys;   // [L, n]  L = batch * (C-1) lists
  int32_t* key_count;         // [L]
  int32_t* maybe;             // [L, n] anchors that pass the quick reject (fused filter; beyond shared memory)
  float4* stash;              // [B, n] decoded + clipped box of every anchor that passed the filter, or NULL.  Used when
                              // loc / boxes live in mapped HOST memory: a row then crosses PCIe once, not twice
  float* s_scores;            // sort_bboxes outputs [keep_topk]
  float4* s_boxes;
  int32_t* s_index;
  unsigned long long* s_key;  // [L, slots] sorted keys
  unsigned long long* s_key2; // [L, slots] merge buffer of lists longer than the in-shared-memory sort
  float4* s_box;              // [L, keep_topk] normalised corners (y0, x0, y1, x1), rank order (lists too long for shared memory)
  float* s_area;              // [L, keep_topk] (y1-y0)*(x1-x0)
  float4* g_kept_box;         // [L, keep_topk] kept list of the NMS when it does not fit shared memory
  float* g_kept_area;
  int32_t* g_kept_rank;
  uint2* s_mask;              // [L, keep_topk] stripe masks of the candidates
  uint32_t* g_stripes;        // [L, 64, ceil(keep_topk / 32)] stripe bitsets of the kept list
  // outputs
  float4* out_boxes;
  float* out_scores;
  int32_t* out_counts;
  int32_t* out_index;
  int32_t* out_keep;
  int filler;                 // fused parse_by_class: zero-score rows fill up the NMS selection
  // peer exchange (dan_postprocess_batch_peers): every output row of the slab is also stored into the receive buffers of
  // the other ranks over NVLink (mapped peer memory); the last CTA then raises this rank's flag in every peer
  int npeers;                                   // destinations besides out_* (0: no exchange)
  long long peer_delta[DAN_MAX_PEERS];          // byte offset from an address inside the own slab to its copy in destination q
  int32_t* peer_flag[DAN_MAX_PEERS];            // this rank's arrival flag inside destination q
  int32_t* peer_state;                          // [2] device words of this rank: CTAs done, step sequence number
};

// clip_bboxes, bbox_util.py:38-48
DAN_D float4 pp_clip(float4 b, float height, float width) {
  float ymin = fmaxf(b.x, 0.f);
  float xmin = fmaxf(b.y, 0.f);
  const float ymax = fminf(b.z, fsub(height, 1.f));
  const float xmax = fminf(b.w, fsub(width, 1.f));
  ymin = fminf(ymin, ymax);
  xmin = fminf(xmin, xmax);
  return make_float4(ymin, xmin, ymax, xmax);
}

// decode (when offsets are given) + clip for anchor `a` of image `b`, split into the global loads and the
// arithmetic so that a caller can put independent work between the two
struct RawBox {
  float4 v;        // offsets or decoded box
  float4 anchor;   // ymin, xmin, ymax, xmax (only when decoding)
};

template <typename T>
DAN_D RawBox pp_load(const PpArgs& A, int b, int a) {
  typedef typename PredRow<T>::type Row;
  const int64_t row = (int64_t)b * A.n + a;
  RawBox r;
  if (A.loc != nullptr) {
    r.v = PredRow<T>::widen(static_cast<const Row*>(A.loc)[row]);
    r.anchor = make_float4(A.ay0[a], A.ax0[a], A.ay1[a], A.ax1[a]);
  } else {
    r.v = PredRow<T>::widen(static_cast<const Row*>(A.boxes)[row]);
    r.anchor = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  return r;
}

DAN_D float4 pp_finish(const PpArgs& A, const RawBox& r) {
  float4 bx = r.v;
  if (A.loc != nullptr) bx = decode_box(r.v, r.anchor.x, r.anchor.y, r.anchor.z, r.anchor.w, A.ps0, A.ps1, A.ps2, A.ps3);
  return pp_clip(bx, A.img_h, A.img_w);
}

template <typename T>
DAN_D float4 pp_box(const PpArgs& A, int b, int a) { return pp_finish(A, pp_load<T>(A, b, a)); }

// ---------------------------------------------------------------------------
// K3: filter + compaction.  grid (ceil(N/256), B)
// ---------------------------------------------------------------------------
constexpr int kFilterPerThread = 4;     // anchors per thread: 4 independent logit loads in flight (memory-level parallelism)

// exact per-anchor path: softmax, threshold, decode + clip, min-size, warp-aggregated append of the survivors.
// STAGED (two classes = one list per image): the keys are collected in the CTA's shared memory and appended to the list
// with ONE global atomic per CTA; per-warp atomics on the same counter serialise in L2 (ncu: 20 % of the stall samples).
template <bool STAGED, typename T>
DAN_D void filter_one(const PpArgs& A, int b, int a, bool live, int lane, unsigned long long* s_keys, int* s_cnt) {
  const int C = A.num_classes;
  const T* x = static_cast<const T*>(A.cls) + ((int64_t)b * A.n + (live ? a : 0)) * C;
  // tf.nn.softmax: exp(x - max) * (1 / sum(exp(x - max))), sum in class order
  float mx = 0.f, inv = 0.f;
  if (live) {
    mx = widen(x[0]);
    for (int k = 1; k < C; ++k) mx = fmaxf(mx, widen(x[k]));
    float s = 0.f;
    for (int k = 0; k < C; ++k) {
      const float e = cephes_expf(fsub(widen(x[k]), mx));
      s = (k == 0) ? e : fadd(s, e);
    }
    inv = fdiv(1.f, s);
  }
  float4 box;
  bool have_box = false;
  for (int c = 1; c < C; ++c) {
    bool pass = false;
    float p = 0.f;
    if (live) {
      p = fmul(cephes_expf(fsub(widen(x[c]), mx)), inv);
      if (p > A.select_thr) {                       // select_bboxes :24-36
        if (!have_box) {
          box = pp_box<T>(A, b, a);
          have_box = true;
          if (A.stash != nullptr) A.stash[(int64_t)b * A.n + a] = box;
        }
        const float w = fadd(fsub(box.w, box.y), 1.f);   // filter_bboxes :50-59
        const float h = fadd(fsub(box.z, box.x), 1.f);
        pass = (w > A.min_size_p1) && (h > A.min_size_p1);
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, pass);
    if (m != 0u) {
      const int list = b * (C - 1) + (c - 1);
      const unsigned long long key = ((unsigned long long)score_to_key(p) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)a);
      int base = 0;
      if (lane == 0) base = STAGED ? atomicAdd(s_cnt, __popc(m)) : atomicAdd(A.key_count + list, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (pass) {
        const int pos = base + __popc(m & ((1u << lane) - 1u));
        if (STAGED) s_keys[pos] = key;
        else A.keys[(int64_t)list * A.n + pos] = key;
      }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256) pp_filter_kernel(const PpArgs A) {
  __shared__ unsigned long long s_keys[256 * kFilterPerThread];
  __shared__ int s_cnt, s_base;
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int a0 = blockIdx.x * (256 * kFilterPerThread) + threadIdx.x;
  const bool staged = A.num_classes == 2;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  // Two classes: softmax_1 = sigmoid(x1 - x0).  An anchor whose logit difference is more than 0.05 below
  // logit(threshold) cannot pass (the fp32 evaluation is accurate to ~1e-6 relative), so the ~98 % background anchors
  // leave after one subtraction.  The exact path runs per 32-anchor group when any of its lanes may pass.
  // Two classes come here only when cls_pred is not aligned to an anchor's pair of logits (the NMS kernel filters
  // aligned ones itself), so the pair is read as two scalars.
  bool maybe[kFilterPerThread];
  if (A.num_classes == 2) {
    float2 xx[kFilterPerThread];
#pragma unroll
    for (int u = 0; u < kFilterPerThread; ++u) {
      const int a = a0 + u * 256;
      const T* x = static_cast<const T*>(A.cls) + ((int64_t)b * A.n + (a < A.n ? a : 0)) * 2;
      xx[u] = (a < A.n) ? make_float2(widen(__ldcs(x)), widen(__ldcs(x + 1))) : make_float2(0.f, 0.f);   // read once: streaming
    }
#pragma unroll
    for (int u = 0; u < kFilterPerThread; ++u)
      maybe[u] = (a0 + u * 256 < A.n) &&
                 (!(fsub(xx[u].y, xx[u].x) < A.reject_below) || fabsf(xx[u].x) > 1e5f || fabsf(xx[u].y) > 1e5f);
  } else {
#pragma unroll
    for (int u = 0; u < kFilterPerThread; ++u) maybe[u] = a0 + u * 256 < A.n;
  }
  // compact the warp's few possibly-passing anchors (out of its 128) into dense lanes, then run the exact path on
  // full warps: without this ~60 % of the 32-anchor groups would run it for one or two live lanes
  __shared__ int s_list[8][32 * kFilterPerThread];
  int* mylist = s_list[threadIdx.x >> 5];
  int total = 0;
#pragma unroll
  for (int u = 0; u < kFilterPerThread; ++u) {
    const unsigned m = __ballot_sync(0xffffffffu, maybe[u]);
    if (maybe[u]) mylist[total + __popc(m & ((1u << lane) - 1u))] = a0 + u * 256;
    total += __popc(m);
  }
  __syncwarp();
  for (int j = 0; j < total; j += 32) {
    const bool live = j + lane < total;
    if (staged) filter_one<true, T>(A, b, live ? mylist[j + lane] : 0, live, lane, s_keys, &s_cnt);
    else filter_one<false, T>(A, b, live ? mylist[j + lane] : 0, live, lane, s_keys, &s_cnt);
  }
  if (staged) {
    __syncthreads();
    const int cnt = s_cnt;
    if (threadIdx.x == 0 && cnt > 0) s_base = atomicAdd(A.key_count + b, cnt);
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += 256) A.keys[(int64_t)b * A.n + s_base + i] = s_keys[i];
  }
}

// standalone sort_bboxes / nms_bboxes: one key per input row, nothing filtered
__global__ void __launch_bounds__(256) key_build_kernel(const float* __restrict__ scores, int64_t n, unsigned long long* __restrict__ keys,
                                                        int32_t* __restrict__ key_count) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    keys[i] = ((unsigned long long)score_to_key(scores[i]) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
  if (blockIdx.x == 0 && threadIdx.x == 0) key_count[0] = (int32_t)n;
}

DAN_D uint32_t key_index(unsigned long long key) { return 0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull); }

// sort_bboxes: tf.nn.top_k + gather + zero pad (bbox_util.py:61-72)
__global__ void __launch_bounds__(kSortThreads, 1) topk_sort_kernel(const PpArgs A, const float* __restrict__ src_scores,
                                                                 const float4* __restrict__ src_boxes) {
  extern __shared__ unsigned long long s_keys[];
  __shared__ SortScratch sc;
  const int tid = threadIdx.x;
  const int cnt = min(A.key_count[0], A.n);
  const int k = min(A.keep_topk, cnt);
  const unsigned long long* sorted = s_keys;
  if (k <= kSortCap) {
    select_and_sort(A.keys, cnt, k, s_keys, sc);
  } else {
    select_and_sort_large(A.keys, cnt, k, A.s_key, A.s_key2, s_keys, sc);
    sorted = A.s_key;
  }
  for (int r = tid; r < A.keep_topk; r += kSortThreads) {
    if (r < k) {
      const uint32_t idx = key_index(sorted[r]);
      A.s_scores[r] = src_scores[idx];
      A.s_boxes[r] = src_boxes[idx];
      if (A.s_index != nullptr) A.s_index[r] = (int32_t)idx;
    } else {
      A.s_scores[r] = 0.f;
      A.s_boxes[r] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (A.s_index != nullptr) A.s_index[r] = -1;
    }
  }
}

// ---------------------------------------------------------------------------
// pair tests of tf.image.non_max_suppression (shared by the NMS kernel below)
// ---------------------------------------------------------------------------
struct NmsBox {
  float y0, x0, y1, x1, area;
};

DAN_D NmsBox nms_norm(float4 b) {
  NmsBox r;
  r.y0 = fminf(b.x, b.z);
  r.x0 = fminf(b.y, b.w);
  r.y1 = fmaxf(b.x, b.z);
  r.x1 = fmaxf(b.y, b.w);
  r.area = fmul(fsub(r.y1, r.y0), fsub(r.x1, r.x0));
  return r;
}

// IOUGreaterThanThreshold of TF's non_max_suppression_op.cc for normalised boxes.  Kept out of line: the callers reach
// it only when a pair is within 1e-6 of the threshold (or the threshold is negative), and the chunk loop of the NMS
// kernel has to stay small enough for the instruction cache.
__device__ __noinline__ bool nms_suppresses(float4 a, float a_area, float4 b, float b_area, float thr) {
  if (a_area <= 0.f || b_area <= 0.f) return false;
  const float h = fmaxf(fsub(fminf(a.z, b.z), fmaxf(a.x, b.x)), 0.f);
  const float w = fmaxf(fsub(fminf(a.w, b.w), fmaxf(a.y, b.y)), 0.f);
  const float inter = fmul(h, w);
  if (inter == 0.f) return 0.f > thr;     // 0 / (area_a + area_b) == 0 exactly
  return fdiv(inter, fsub(fadd(a_area, b_area), inter)) > thr;
}

// same predicate; for thr >= 0 disjoint boxes are rejected first and the division is only evaluated when
// inter / union is within 1e-6 (relative) of the threshold
DAN_D bool pair_suppresses(const float4& a, float a_area, const float4& b, float b_area, float thr) {
  if (thr >= 0.f) {
    const float h = fsub(fminf(a.z, b.z), fmaxf(a.x, b.x));
    const float w = fsub(fminf(a.w, b.w), fmaxf(a.y, b.y));
    if (!(h > 0.f && w > 0.f)) return false;
    if (!(a_area > 0.f && b_area > 0.f)) return false;
    const float inter = fmul(h, w);
    const float t = fmul(thr, fsub(fadd(a_area, b_area), inter));
    if (t > 1e-30f) {
      if (inter > fmul(t, 1.000001f)) return true;
      if (inter < fmul(t, 0.999999f)) return false;
    }
  }
  return nms_suppresses(a, a_area, b, b_area, thr);
}

// two classes: softmax_1 = sigmoid(x1 - x0); an anchor whose logit difference is more than 0.05 below logit(threshold)
// cannot pass (the fp32 evaluation is accurate to ~1e-6 relative), so ~97 % of the anchors leave after one subtraction
DAN_D bool f2_maybe(const PpArgs& A, float x0, float x1) {
  return !(fsub(x1, x0) < A.reject_below) || fabsf(x0) > 1e5f || fabsf(x1) > 1e5f;
}

// ---------------------------------------------------------------------------
// K4+K5: nms_greedy_kernel, one CTA per (image, class) list, does everything after the filter.  Its steps, numbered as
// in DESIGN.md §4b:
//   0  filter_image        (FILTER) the two-class filter of the list's image, keys straight into shared memory
//   1  top_k_sort          top-k select + sort of the keys (sort.cuh)
//   2  decode_candidates   decode + clip + normalise the K best, in rank order
//      init_stripes        the 32 x 32 stripe grid over the candidates, their stripe masks, empty bitsets and hints
//   3  greedy NMS exactly as tf.image.non_max_suppression runs it, over a window of kWin candidates per round:
//      a  test_window        live candidates against the kept list: cell hints, then the stripe search
//      b  compact_survivors  the first kSurv survivors of the window, in rank order
//      c  survivor_bits      their mutual suppression bits
//      d  relax_survivors    kept / suppressed by relaxation
//      e  append_kept        the kept survivors join the kept list, its stripe bitsets and hints
//   4  write_outputs       the first nms_topk kept boxes in rank order, zero padded (bbox_util.py:80-90), peer copies
//      release_peers       (peer exchange) the last CTA raises this rank's flag in every destination
// ---------------------------------------------------------------------------
constexpr int kWin = kSortThreads;                     // candidates in the window: one per thread
constexpr int kSurv = 128;                             // survivors resolved per round
constexpr int kSurvWords = kSurv / 32;
constexpr int kMaxSweeps = 12;
constexpr int kHintCells = 32 * 32;                    // one hint pair per (y stripe, x stripe) cell of a box centre
constexpr size_t kGreedySmemMax = 186 * 1024;          // dynamic part (the kernel has ~38 KB of static shared memory)

static int next_pow2(int64_t v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// candidate slots of a list of n anchors: min(keep_topk, n), at least one.  No upper limit: the workspace holds the
// candidates of lists too long for shared memory.
static int64_t cand_slots(int64_t n, int64_t keep_topk) { return keep_topk < n ? keep_topk : (n > 0 ? n : 1); }

static GreedyPlan greedy_plan(int64_t n, int keep_topk, int nms_cap) {
  GreedyPlan g = {};
  const int sort_n = (int)(n < kSortCap ? (n > 0 ? n : 1) : kSortCap);
  g.sort_bytes = next_pow2(sort_n) * 8;
  g.slots = (int)cand_slots(n, keep_topk);
  g.wcap = (nms_cap + 31) / 32;
  const size_t cand_box = align_up((size_t)g.slots * 16, 16);
  const size_t region0 = cand_box > (size_t)g.sort_bytes ? cand_box : (size_t)g.sort_bytes;
  const size_t cand_bytes = region0 + align_up((size_t)g.slots * 4, 16) + align_up((size_t)g.slots * 8, 16);
  const size_t kept_bytes = align_up((size_t)nms_cap * 16, 16) + 2 * align_up((size_t)nms_cap * 4, 16) + (size_t)64 * g.wcap * 4;
  size_t off = g.sort_bytes;
  auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 16); return (int)at; };
  if (cand_bytes + kept_bytes <= kGreedySmemMax) {
    g.where = 0;
    off = region0;
    g.cand_area = take((size_t)g.slots * 4);
    g.cand_mask = take((size_t)g.slots * 8);
  } else {
    g.where = (size_t)g.sort_bytes + kept_bytes <= kGreedySmemMax ? 1 : 2;
  }
  if (g.where <= 1) {
    g.kept_box = take((size_t)nms_cap * 16);
    g.kept_area = take((size_t)nms_cap * 4);
    g.kept_rank = take((size_t)nms_cap * 4);
    g.stripes = take((size_t)64 * g.wcap * 4);
  }
  g.smem = (int)off;
  return g;
}

// block-wide min / max of a float over all threads (every thread gets the result)
DAN_D void block_minmax(float lo, float hi, float& out_lo, float& out_hi) {
  __shared__ int s_lo[kSortThreads / 32], s_hi[kSortThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wl = __reduce_min_sync(0xffffffffu, float_to_ordered(lo));
  const int wh = __reduce_max_sync(0xffffffffu, float_to_ordered(hi));
  if (lane == 0) { s_lo[warp] = wl; s_hi[warp] = wh; }
  __syncthreads();
  int a = (lane < kSortThreads / 32) ? s_lo[lane] : 0x7fffffff, b = (lane < kSortThreads / 32) ? s_hi[lane] : (int)0x80000000;
  a = __reduce_min_sync(0xffffffffu, a);
  b = __reduce_max_sync(0xffffffffu, b);
  out_lo = ordered_to_float(a);
  out_hi = ordered_to_float(b);
  __syncthreads();
}

// stripe masks of the broad phase (see init_stripes); monotone in the coordinate, so overlapping intervals share a bit
struct Stripes {
  float ylo, yinv, xlo, xinv;
  bool all;
  DAN_D static uint32_t axis(float v0, float v1, float lo, float inv) {
    const float f0 = (v0 - lo) * inv, f1 = (v1 - lo) * inv;
    if (!(fabsf(f0) < 1e9f) || !(fabsf(f1) < 1e9f)) return 0xffffffffu;      // non-finite or far outside: every stripe
    const int s0 = min(max((int)f0, 0), 31), s1 = min(max((int)f1, 0), 31);
    return (0xffffffffu >> (31 - s1)) & (0xffffffffu << s0);
  }
  // (x mask, y mask) of a normalised box (y0, x0, y1, x1); a box without area neither suppresses nor is suppressed
  DAN_D uint2 masks(float4 bx, float area) const {
    if (!(area > 0.f)) return make_uint2(0u, 0u);
    if (all) return make_uint2(0xffffffffu, 0xffffffffu);
    return make_uint2(axis(bx.y, bx.w, xlo, xinv), axis(bx.x, bx.z, ylo, yinv));
  }
  // cell (y stripe * 32 + x stripe) of the box centre: the key of the suppressor hints (any cell is valid for any box)
  DAN_D int cell(float4 bx) const {
    const float fy = ((bx.x + bx.z) * 0.5f - ylo) * yinv, fx = ((bx.y + bx.w) * 0.5f - xlo) * xinv;
    const int sy = (fabsf(fy) < 1e9f) ? min(max((int)fy, 0), 31) : 0;
    const int sx = (fabsf(fx) < 1e9f) ? min(max((int)fx, 0), 31) : 0;
    return sy * 32 + sx;
  }
};

// barriers among the first kSurv threads of the CTA (hardware barrier 1); the other warps wait at the next __syncthreads
DAN_D void bar_sync_chunk() { asm volatile("bar.sync 1, %0;" ::"n"(kSurv) : "memory"); }
DAN_D bool bar_or_chunk(bool pred) {
  int r;
  asm volatile(
      "{\n"
      "  .reg .pred p, q;\n"
      "  setp.ne.s32 q, %1, 0;\n"
      "  bar.red.or.pred p, 1, %2, q;\n"
      "  selp.s32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(r)
      : "r"((int)pred), "n"(kSurv)
      : "memory");
  return r != 0;
}

// A dependency chain longer than kMaxSweeps inside a chunk: one warp finishes the chunk serially (when it reaches an
// undecided survivor every earlier one is decided); lane w holds word w of the masks.  Out of line (rare).
__device__ __noinline__ void resolve_chunk_serially(const uint32_t* T, uint32_t* keptm, uint32_t* supm, int ns) {
  const int lane = threadIdx.x & 31;
  uint32_t kw = (lane < kSurvWords) ? keptm[lane] : 0u;
  uint32_t sw = (lane < kSurvWords) ? supm[lane] : 0u;
  for (int v = 0; v < ns; ++v) {
    const int w = v >> 5;
    const uint32_t bit = 1u << (v & 31);
    const uint32_t known = __shfl_sync(0xffffffffu, kw | sw, w);
    if (known & bit) continue;                 // warp-uniform
    const uint32_t t = (lane < kSurvWords && (lane << 5) < v) ? T[v * kSurvWords + lane] : 0u;
    const bool hit = __any_sync(0xffffffffu, (t & kw) != 0u);
    if (lane == w) {
      if (hit) sw |= bit;
      else kw |= bit;
    }
  }
  if (lane < kSurvWords) { keptm[lane] = kw; supm[lane] = sw; }
}

constexpr int kMaybeCap = 4096;                        // indices kept in shared memory (the rest goes to the workspace)

// A list's candidates and kept list, where the carve of the kernel put them, and the state that lives across rounds.
struct GreedyList {
  float4* cbox;            // candidates in rank order: normalised corners (y0, x0, y1, x1)
  float* carea;
  uint2* cmask;            // their stripe masks
  float4* kbox;            // kept list in the order kept
  float* karea;
  int* krank;              // rank of each kept box
  uint32_t* xs;            // [32][wcap] stripe bitsets of the kept list: kept boxes touching x stripe s
  uint32_t* ys;            // ... y stripe s
  int wcap;
  Stripes sg;
  int K;                   // candidates
  int L;                   // kept boxes so far (CTA-uniform)
  int L_prev;              // ... when the previous round tested its window
  int w_end_prev;          // end of the previous round's window: candidates below it carry state
  int c0;                  // first candidate of this round's window
};

// the kernel's static shared memory that steps a-e pass to each other
struct RoundSmem {
  unsigned char* alive;             // [kWin] ring over the window: candidate r lives in slot r % kWin
  unsigned short* list;             // [kWin] step a: window offsets of the candidates that need the full search
  int* surv;                        // [kSurv] step b: rank of survivor u, its box, area and stripe masks
  float4* sbox;
  float* sarea;
  uint2* smask;
  uint32_t (*T)[kSurvWords];        // [kSurv] step c: suppression bits of survivor v
  uint32_t* keptm;                  // step d: survivors known kept / suppressed
  uint32_t* supm;
  int (*hint)[kHintCells];          // [2] suppressor hints per cell: [0] first kept box centred there, [1] last suppressor found
  int* next;                        // [2] work counters of steps a and c
  int* nlist;                       // candidates in `list`
};

// WHERE: 0 = candidates and kept list in shared memory (the usual case), 1 = candidates in the workspace, 2 = both in the
// workspace (very long lists).  A template parameter rather than a run-time pointer choice so that the shared-memory
// accesses compile to LDS / STS / ATOMS instead of generic-address instructions.
template <int WHERE>
DAN_D GreedyList carve(const PpArgs& A, unsigned char* dyn_smem, int list) {
  const GreedyPlan& P = A.plan;
  const int64_t o = (int64_t)list * P.slots;
  GreedyList g;
  if (WHERE >= 1) {
    g.cbox = A.s_box + o;
    g.carea = A.s_area + o;
    g.cmask = A.s_mask + o;
  } else {
    g.cbox = reinterpret_cast<float4*>(dyn_smem);                                  // aliases the keys (see step 2)
    g.carea = reinterpret_cast<float*>(dyn_smem + P.cand_area);
    g.cmask = reinterpret_cast<uint2*>(dyn_smem + P.cand_mask);
  }
  uint32_t* stripes;
  if (WHERE >= 2) {
    g.kbox = A.g_kept_box + o;
    g.karea = A.g_kept_area + o;
    g.krank = A.g_kept_rank + o;
    stripes = A.g_stripes + (int64_t)list * 64 * ((P.slots + 31) / 32);
  } else {
    g.kbox = reinterpret_cast<float4*>(dyn_smem + P.kept_box);
    g.karea = reinterpret_cast<float*>(dyn_smem + P.kept_area);
    g.krank = reinterpret_cast<int*>(dyn_smem + P.kept_rank);
    stripes = reinterpret_cast<uint32_t*>(dyn_smem + P.stripes);
  }
  g.wcap = P.wcap;
  g.xs = stripes;
  g.ys = stripes + 32 * g.wcap;
  g.L = g.L_prev = g.w_end_prev = g.c0 = 0;
  return g;
}

// ---- 0. FILTER (two classes, one list per image): the CTA also runs K3 for its image - it streams the image's logits,
// keeps the indices of the few anchors the quick reject lets through, runs them through the exact path (softmax in
// tf.nn.softmax's op order, threshold, decode, clip, min-size) on dense warps, and the surviving keys land directly in
// the shared memory the sort works in: no filter launch, no key list in HBM, no global atomics.  Returns the number of
// keys; beyond the sort's shared memory they are in gkeys.
template <typename T>
DAN_D int filter_image(const PpArgs& A, int list, int b, unsigned long long* keys, unsigned long long* gkeys) {
  __shared__ int s_maybe[kMaybeCap];
  __shared__ int s_nmaybe, s_nkeys;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  int* gmaybe = A.maybe + (int64_t)list * A.n;
  const int key_cap = A.plan.sort_bytes / 8;           // keys that fit the sort's shared memory
  if (tid == 0) { s_nmaybe = 0; s_nkeys = 0; }
  __syncthreads();
  auto put = [&](int pos, int a) {
    if (pos < kMaybeCap) s_maybe[pos] = a;
    else gmaybe[pos] = a;
  };
  auto push = [&](int a) { put(atomicAdd(&s_nmaybe, 1), a); };
  // The image's logits as 16-byte vectors of kVA anchors (2 for fp32, 4 for fp16 / bf16).  The row of an image starts
  // aligned to one anchor only (8 or 4 bytes): the `head` anchors before the first 16-byte boundary and the ones behind
  // the last whole vector are read as pairs after the loop.
  constexpr int kVA = 16 / (2 * (int)sizeof(T));
  const T* x = static_cast<const T*>(A.cls) + (int64_t)b * A.n * 2;
  // (fp32 keeps the statements it had before fp16 / bf16 were added, so that it compiles to the same instructions)
  const int head = kVA == 2 ? ((reinterpret_cast<uintptr_t>(x) & 15u) ? 1 : 0)
                            : min((int)(((16u - (unsigned)(reinterpret_cast<uintptr_t>(x) & 15u)) & 15u) / (2 * sizeof(T))), A.n);
  const int nvec = kVA == 2 ? (A.n - head) >> 1 : (int)((unsigned)(A.n - head) / kVA);
  const float4* xv = reinterpret_cast<const float4*>(x + 2 * head);
  for (int v0 = 0; v0 < nvec; v0 += 4 * kSortThreads) {
    float4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int v = v0 + u * kSortThreads + tid;
      q[u] = (v < nvec) ? __ldcs(xv + v) : make_float4(0.f, 0.f, 0.f, 0.f);       // read once: streaming
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      // A warp looks at 32 * kVA consecutive anchors here.  Its survivors enter the list in ANCHOR order with one atomic
      // per warp: the exact pass below then reads neighbouring box rows from neighbouring lanes, i.e. whole sectors -
      // which matters when the rows live in host memory and every sector is a PCIe read.
      const int v = v0 + u * kSortThreads + tid;
      if constexpr (kVA == 2) {
        const bool p0 = v < nvec && f2_maybe(A, q[u].x, q[u].y);
        const bool p1 = v < nvec && f2_maybe(A, q[u].z, q[u].w);
        const unsigned m0 = __ballot_sync(0xffffffffu, p0), m1 = __ballot_sync(0xffffffffu, p1);
        if ((m0 | m1) != 0u) {
          int base = 0;
          if (lane == 0) base = atomicAdd(&s_nmaybe, __popc(m0) + __popc(m1));
          base = __shfl_sync(0xffffffffu, base, 0);
          int pos = base + __popc(m0 & lt_mask) + __popc(m1 & lt_mask);
          if (p0) put(pos++, head + 2 * v);
          if (p1) put(pos, head + 2 * v + 1);
        }
      } else {
        bool pj[kVA];
        unsigned mj[kVA], any = 0u;
#pragma unroll
        for (int j = 0; j < kVA; ++j) {
          const float2 xx = vec_pair<T>(q[u], j);
          pj[j] = v < nvec && f2_maybe(A, xx.x, xx.y);
        }
#pragma unroll
        for (int j = 0; j < kVA; ++j) {
          mj[j] = __ballot_sync(0xffffffffu, pj[j]);
          any |= mj[j];
        }
        if (any != 0u) {
          int nj = 0, below = 0;
#pragma unroll
          for (int j = 0; j < kVA; ++j) {
            nj += __popc(mj[j]);
            below += __popc(mj[j] & lt_mask);
          }
          int base = 0;
          if (lane == 0) base = atomicAdd(&s_nmaybe, nj);
          base = __shfl_sync(0xffffffffu, base, 0);
          int pos = base + below;
#pragma unroll
          for (int j = 0; j < kVA; ++j)
            if (pj[j]) put(pos++, head + kVA * v + j);
        }
      }
    }
  }
  if constexpr (kVA == 2) {                            // fp32: at most one anchor on either side
    if (tid == 0 && head == 1 && f2_maybe(A, x[0], x[1])) push(0);
    if (tid == 1 && head + 2 * nvec < A.n && f2_maybe(A, x[2 * (A.n - 1)], x[2 * (A.n - 1) + 1])) push(A.n - 1);
  } else {
    // head: threads [0, head); tail (fewer than kVA anchors behind the vectors): threads [kVA - 1, 2 kVA - 1)
    const int rest = head + kVA * nvec;
    const int t = tid - (kVA - 1);
    if (tid < head) {
      const float2 xx = make_float2(widen(x[2 * tid]), widen(x[2 * tid + 1]));
      if (f2_maybe(A, xx.x, xx.y)) push(tid);
    }
    if (t >= 0 && rest + t < A.n) {
      const float2 xx = make_float2(widen(x[2 * (rest + t)]), widen(x[2 * (rest + t) + 1]));
      if (f2_maybe(A, xx.x, xx.y)) push(rest + t);
    }
  }
  __syncthreads();
  const int nmaybe = s_nmaybe;
  for (int i0 = 0; i0 < nmaybe; i0 += kSortThreads) {
    const int i = i0 + tid;
    if (i < nmaybe) {
      const int a = (i < kMaybeCap) ? s_maybe[i] : gmaybe[i];
      const float2 xx = ld_pair(x + 2 * a);
      const float pr = softmax2_face(xx.x, xx.y);
      if (pr > A.select_thr) {                            // select_bboxes :24-36
        const float4 box = pp_box<T>(A, b, a);
        if (A.stash != nullptr) A.stash[(int64_t)b * A.n + a] = box;
        const float w = fadd(fsub(box.w, box.y), 1.f);    // filter_bboxes :50-59
        const float h = fadd(fsub(box.z, box.x), 1.f);
        if ((w > A.min_size_p1) && (h > A.min_size_p1)) {
          const unsigned long long key = ((unsigned long long)score_to_key(pr) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)a);
          const int pos = atomicAdd(&s_nkeys, 1);
          if (pos < key_cap) keys[pos] = key;
          else gkeys[pos] = key;
        }
      }
    }
  }
  __syncthreads();
  const int cnt = s_nkeys;
  if (cnt > kSortCap) {                                   // too many survivors for shared memory: the select runs on HBM
    for (int i = tid; i < min(cnt, key_cap); i += kSortThreads) gkeys[i] = keys[i];
    __syncthreads();
  }
  return cnt;
}

// ---- 1. top-k + sort of the list's cnt keys; returns K, the number of candidates, and where their sorted keys are:
// in shared memory, or at A.s_key + o for lists longer than kSortCap
template <bool FILTER>
DAN_D int top_k_sort(const PpArgs& A, int cnt, int64_t o, const unsigned long long* gkeys, unsigned long long* keys,
                     unsigned char* dyn_smem, const unsigned long long*& sorted) {
  __shared__ SortScratch sc;
  const int k_want = min(A.keep_topk, cnt);
  sorted = keys;
  if (k_want <= kSortCap) {
    // a second key buffer behind the first one when the CTA's shared memory holds it (nothing else lives there yet)
    unsigned long long* spare = ((size_t)A.plan.sort_bytes + (size_t)min(cnt, kSortCap) * 8 <= (size_t)A.plan.smem)
                                    ? reinterpret_cast<unsigned long long*>(dyn_smem + A.plan.sort_bytes) : nullptr;
    return min(select_and_sort(gkeys, cnt, k_want, keys, sc, FILTER, spare), A.keep_topk);
  }
  select_and_sort_large(gkeys, cnt, k_want, A.s_key + o, A.s_key2 + o, keys, sc);
  sorted = A.s_key + o;
  return k_want;
}

// ---- 2. decode + clip + normalise.  The candidate boxes (16 B) reuse the shared memory of the keys (8 B): the ranks
// are walked in DEscending batches of one key per thread, so a batch's boxes only overwrite key slots of ranks that
// are already done (box r covers key slots 2r and 2r+1 >= r); the barrier protects the batch's own keys.
template <bool DECODE, typename T>
DAN_D void decode_candidates(const PpArgs& A, int b, int64_t o, const unsigned long long* sorted, const float4* src_boxes,
                             GreedyList& g) {
  const int tid = threadIdx.x;
  const int K = g.K;
  for (int r0 = K > 0 ? ((K - 1) / kSortThreads) * kSortThreads : -1; r0 >= 0; r0 -= kSortThreads) {
    const int r = r0 + tid;
    const unsigned long long key = (r < K) ? sorted[r] : 0ull;
    if (r < K) A.s_key[o + r] = key;
    __syncthreads();
    if (r < K) {
      const uint32_t idx = key_index(key);
      const NmsBox nb = nms_norm(DECODE ? (A.stash != nullptr ? A.stash[(int64_t)b * A.n + idx] : pp_box<T>(A, b, (int)idx)) : src_boxes[idx]);
      g.cbox[r] = make_float4(nb.y0, nb.x0, nb.y1, nb.x1);
      g.carea[r] = nb.area;
    }
  }
  __syncthreads();
}

// Broad phase: the extent of the candidates is cut into 32 stripes per axis and every box carries the two 32-bit masks
// of the stripes it touches.  Boxes that intersect share a stripe on both axes, so a pair whose masks do not meet on
// either axis needs no exact test.  Also empties the kept list's stripe bitsets and the hints.
DAN_D void init_stripes(const PpArgs& A, GreedyList& g, RoundSmem& R) {
  const int tid = threadIdx.x;
  const int K = g.K;
  Stripes& sg = g.sg;
  {
    float ylo = 3.0e38f, yhi = -3.0e38f, xlo = 3.0e38f, xhi = -3.0e38f;
    for (int r = tid; r < K; r += kSortThreads) {
      const float4 bx = g.cbox[r];
      if (g.carea[r] > 0.f && fabsf(bx.x) < 1e30f && fabsf(bx.y) < 1e30f && fabsf(bx.z) < 1e30f && fabsf(bx.w) < 1e30f) {
        ylo = fminf(ylo, bx.x); yhi = fmaxf(yhi, bx.z);
        xlo = fminf(xlo, bx.y); xhi = fmaxf(xhi, bx.w);
      }
    }
    float ey, ex;
    block_minmax(ylo, yhi, sg.ylo, ey);
    block_minmax(xlo, xhi, sg.xlo, ex);
    sg.yinv = (ey > sg.ylo) ? 32.f / (ey - sg.ylo) : 0.f;
    sg.xinv = (ex > sg.xlo) ? 32.f / (ex - sg.xlo) : 0.f;
    sg.all = A.nms_thr < 0.f;                          // a negative threshold: disjoint boxes suppress too
  }
  for (int r = tid; r < K; r += kSortThreads) g.cmask[r] = sg.masks(g.cbox[r], g.carea[r]);
  for (int i = tid; i < 64 * g.wcap; i += kSortThreads) g.xs[i] = 0u;
  for (int i = tid; i < 2 * kHintCells; i += kSortThreads) (&R.hint[0][0])[i] = 0x7fffffff;
  if (tid < 2) R.next[tid] = 0;
  if (tid == 0) *R.nlist = 0;
  __syncthreads();
}

// ---- a. window vs kept list.  Thread t owns candidate c0 + t.  A candidate that was in the previous window has met
// the first L_prev kept boxes already; a fresh one has met none.
DAN_D void test_window(const PpArgs& A, const GreedyList& g, RoundSmem& R, int w_end) {
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  const float thr = A.nms_thr;
  const int L = g.L, L_prev = g.L_prev, w_end_prev = g.w_end_prev, c0 = g.c0;
  const int my_r = c0 + tid;
  const bool in_win = my_r < w_end;
  {
    bool alive = false, search = false;
    int upto = 0;
    if (in_win) {
      const bool fresh = my_r >= w_end_prev;
      alive = fresh ? true : (R.alive[my_r & (kWin - 1)] != 0);
      upto = fresh ? 0 : L_prev;
    }
    if (alive && L > upto) {
      const uint2 mm = g.cmask[my_r];
      if (mm.x != 0u && mm.y != 0u) {                  // (no area: no stripes, never suppressed)
        // a1. the two hinted kept boxes of the cell of its centre: a member of a cluster of near duplicates dies here,
        // after one or two exact tests by its own thread
        const float4 me = g.cbox[my_r];
        const float my_area = g.carea[my_r];
        const int cl = g.sg.cell(me);
        const int h0 = R.hint[0][cl], h1 = R.hint[1][cl];
        bool dead = false;
        if (h0 >= upto && h0 < L) dead = pair_suppresses(g.kbox[h0], g.karea[h0], me, my_area, thr);
        if (!dead && h1 != h0 && h1 >= upto && h1 < L) dead = pair_suppresses(g.kbox[h1], g.karea[h1], me, my_area, thr);
        alive = !dead;
        search = !dead;
      }
    }
    if (in_win) R.alive[my_r & (kWin - 1)] = alive ? 1 : 0;
    const unsigned sm = __ballot_sync(0xffffffffu, search);
    int base = 0;
    if (lane == 0 && sm != 0u) base = atomicAdd(R.nlist, __popc(sm));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (search) R.list[base + __popc(sm & lt_mask)] = (unsigned short)tid;
  }
  __syncthreads();
  // a2. the others against the kept list proper, which is indexed by stripe: bit j of xs[s] / ys[s] says that kept box j
  // touches x / y stripe s.  The kept boxes a candidate can intersect are (OR of xs over its x stripes) AND (OR of ys
  // over its y stripes): a group of G lanes owns one candidate, a lane one 32-bit word of the bitset, and only the set
  // bits (beyond the boxes the candidate has met already) go through the exact test; the candidate leaves at the
  // first suppressor, which becomes the cell's second hint.
  const int nlist = *R.nlist;
  if (nlist > 0) {
    const int wcap = g.wcap;
    const int W = (L + 31) >> 5;
    const int G = W <= 8 ? 8 : (W <= 16 ? 16 : 32);        // lanes per candidate
    const int cpw = 32 / G;                                // candidates per warp pass
    const int gl = lane & (G - 1), sub = lane / G;
    const unsigned gmask = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << (sub * G);
    while (true) {                                         // candidates are handed out dynamically: their cost varies a lot
      int i0 = 0;
      if (lane == 0) i0 = atomicAdd(&R.next[0], cpw);
      i0 = __shfl_sync(0xffffffffu, i0, 0);
      if (i0 >= nlist) break;
      const bool have = i0 + sub < nlist;
      const int r = c0 + (have ? (int)R.list[i0 + sub] : 0);
      const float4 me = have ? g.cbox[r] : make_float4(0.f, 0.f, 0.f, 0.f);
      const float my_area = have ? g.carea[r] : 0.f;
      const uint2 mm = have ? g.cmask[r] : make_uint2(0u, 0u);
      const int upto = (r >= w_end_prev) ? 0 : L_prev;
      bool sup = false;
      for (int wb = 0; wb < W; wb += G) {                  // one block of words unless the kept list is very long
        const int w = wb + gl;
        uint32_t poss = 0u;
        if (w < W && w >= (upto >> 5) && mm.x != 0u && mm.y != 0u) {
          // (the stripes of a box are a contiguous range: independent loads, no address chain)
          uint32_t ax = 0u, ay = 0u;
          const int xe = 31 - __clz(mm.x), ye = 31 - __clz(mm.y);
#pragma unroll 2
          for (int st = __ffs(mm.x) - 1; st <= xe; ++st) ax |= g.xs[st * wcap + w];
#pragma unroll 2
          for (int st = __ffs(mm.y) - 1; st <= ye; ++st) ay |= g.ys[st * wcap + w];
          poss = ax & ay;
          if (w == (upto >> 5)) poss &= ~((1u << (upto & 31)) - 1u);
        }
        while (__any_sync(0xffffffffu, poss != 0u && !sup)) {
          bool t = false;
          if (poss != 0u && !sup) {
            const int j = (w << 5) + __ffs(poss) - 1;
            poss &= poss - 1u;
            t = pair_suppresses(g.kbox[j], g.karea[j], me, my_area, thr);
            if (t) atomicExch(&R.hint[1][g.sg.cell(me)], j);
          }
          if ((__ballot_sync(0xffffffffu, t) & gmask) != 0u) sup = true;
        }
      }
      if (have && gl == 0 && sup) R.alive[r & (kWin - 1)] = 0;
    }
  }
  __syncthreads();
}

// ---- b. the first kSurv candidates of the window that are still alive, in rank order; returns how many (ns) and sets
// c_next, the start of the next round's window: behind the last of them
DAN_D int compact_survivors(const GreedyList& g, RoundSmem& R, int w_end, int& c_next) {
  __shared__ int s_wcnt[kSortThreads / 32];
  __shared__ int s_cnext;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const int my_r = g.c0 + tid;
  const bool in_win = my_r < w_end;
  const bool f = in_win && R.alive[my_r & (kWin - 1)] != 0;
  const unsigned fm = __ballot_sync(0xffffffffu, f);
  if (lane == 0) s_wcnt[warp] = __popc(fm);
  if (tid < kSurvWords) { R.keptm[tid] = 0u; R.supm[tid] = 0u; }
  __syncthreads();
  int total, ubase;
  {
    const int cw = (lane < kSortThreads / 32) ? s_wcnt[lane] : 0;
    int incl = cw;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int up = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += up;
    }
    total = __shfl_sync(0xffffffffu, incl, 31);
    ubase = __shfl_sync(0xffffffffu, incl - cw, warp & 31);
  }
  if (f) {
    const int u = ubase + __popc(fm & lt_mask);
    if (u < kSurv) {
      R.surv[u] = my_r;
      R.sbox[u] = g.cbox[my_r];
      R.sarea[u] = g.carea[my_r];
      R.smask[u] = g.cmask[my_r];
      if (u == kSurv - 1) s_cnext = my_r + 1;
    }
  }
  __syncthreads();
  c_next = (total >= kSurv) ? s_cnext : w_end;
  return min(total, kSurv);
}

// ---- c. suppression bits among the ns survivors: warp -> row v, lanes -> 32 earlier survivors per step
DAN_D void survivor_bits(const PpArgs& A, RoundSmem& R, int ns) {
  const int lane = threadIdx.x & 31;
  const float thr = A.nms_thr;
  while (true) {                                           // rows handed out dynamically, the longest ones first
    int vi = 0;
    if (lane == 0) vi = atomicAdd(&R.next[1], 1);
    vi = __shfl_sync(0xffffffffu, vi, 0);
    if (vi >= ns) break;
    const int v = ns - 1 - vi;
    const float4 me = R.sbox[v];
    const float my_area = R.sarea[v];
    const uint2 mm = R.smask[v];
    const int nw = (v + 31) >> 5;                    // words that hold some u < v
    for (int w = 0; w < nw; ++w) {
      const int u = (w << 5) + lane;
      const uint2 um = R.smask[u];
      const bool poss = (u < v) && (um.x & mm.x) != 0u && (um.y & mm.y) != 0u;
      unsigned bits = 0u;
      if (__any_sync(0xffffffffu, poss)) {
        const bool t = poss && pair_suppresses(R.sbox[u], R.sarea[u], me, my_area, thr);
        bits = __ballot_sync(0xffffffffu, t);
      }
      if (lane == 0) R.T[v][w] = bits;
    }
  }
  __syncthreads();
}

// ---- d. relaxation, kept(v) = no kept u in T[v]: thread v owns survivor v (the first kSurv threads).  A survivor is
// decided once one of its suppressors is known kept, or all are known suppressed; chains longer than kMaxSweeps are
// finished by resolve_chunk_serially.
DAN_D void relax_survivors(RoundSmem& R, int ns) {
  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  if (tid < kSurv) {
    uint32_t trow[kSurvWords];
    const int vw = tid >> 5;
    const uint32_t vbit = 1u << (tid & 31);
    const bool mine = tid < ns;
#pragma unroll
    for (int w = 0; w < kSurvWords; ++w) trow[w] = (mine && (w << 5) < tid) ? R.T[tid][w] : 0u;
    bool decided = !mine;
    bool open = true;
    int sweeps = 0;
    while (open && sweeps < kMaxSweeps) {
      uint32_t hitm = 0u, pendm = 0u;
      if (!decided) {
#pragma unroll
        for (int w = 0; w < kSurvWords; ++w) {
          const uint32_t kw = R.keptm[w], sw = R.supm[w];
          hitm |= trow[w] & kw;
          pendm |= trow[w] & ~(kw | sw);
        }
      }
      bar_sync_chunk();                              // every thread has read the masks of the previous sweep
      if (!decided) {
        if (hitm != 0u) { atomicOr(&R.supm[vw], vbit); decided = true; }
        else if (pendm == 0u) { atomicOr(&R.keptm[vw], vbit); decided = true; }
      }
      open = bar_or_chunk(!decided);
      ++sweeps;
    }
    if (open) {
      if (warp == 0) resolve_chunk_serially(&R.T[0][0], R.keptm, R.supm, ns);
      bar_sync_chunk();
    }
  }
  __syncthreads();
}

// ---- e. append the kept survivors in rank order; a kept box becomes the first hint of its cell unless an earlier
// (higher scoring) one is centred there.  ALL threads take part: kEntryThreads threads share one survivor, each
// enters the kept box into every kEntryThreads-th stripe of both axes (a big box touches 2 x 20 stripes: in the hands
// of the survivor's own thread alone this was the longest serial piece of a round).  Then L counts them.
DAN_D void append_kept(const PpArgs& A, GreedyList& g, RoundSmem& R, int ns) {
  const int tid = threadIdx.x;
  const int L = g.L;
  {
    constexpr int kEntryThreads = kSortThreads / kSurv;
    const int v = tid / kEntryThreads, part = tid % kEntryThreads;
    const int vw = v >> 5;
    const uint32_t vbit = 1u << (v & 31);
    if (tid < 2) R.next[tid] = 0;
    if (tid == 2) *R.nlist = 0;
    if (v < ns && (R.keptm[vw] & vbit)) {
      int before = 0;
#pragma unroll
      for (int w = 0; w < kSurvWords; ++w)
        if (w < vw) before += __popc(R.keptm[w]);
      const int pos = L + before + __popc(R.keptm[vw] & (vbit - 1u));
      if (pos < A.nms_topk) {
        const uint2 sm = R.smask[v];
        const uint32_t bit = 1u << (pos & 31);
        if (part == 0) {
          const float4 bx = R.sbox[v];
          g.kbox[pos] = bx;
          g.karea[pos] = R.sarea[v];
          g.krank[pos] = R.surv[v];
          if (sm.x != 0u) atomicMin(&R.hint[0][g.sg.cell(bx)], pos);
        }
        for (int st = part; st < 32; st += kEntryThreads) {
          if ((sm.x >> st) & 1u) atomicOr(&g.xs[st * g.wcap + (pos >> 5)], bit);
          if ((sm.y >> st) & 1u) atomicOr(&g.ys[st * g.wcap + (pos >> 5)], bit);
        }
      }
    }
  }
  __syncthreads();
  int nk = 0;
#pragma unroll
  for (int w = 0; w < kSurvWords; ++w) nk += __popc(R.keptm[w]);
  g.L_prev = L;
  g.L = min(L + nk, A.nms_topk);
}

// ---- 4. outputs, zero padded to nms_topk; with a peer exchange every slab row also goes to the other ranks
template <bool DECODE>
DAN_D void write_outputs(const PpArgs& A, int list, int64_t o, const GreedyList& g, const float* src_scores, const float4* src_boxes) {
  const int tid = threadIdx.x;
  const int kept_n = g.L;
  auto put_score = [&](int64_t oo, float v) {
    A.out_scores[oo] = v;
    for (int q = 0; q < A.npeers; ++q) *reinterpret_cast<float*>(reinterpret_cast<char*>(A.out_scores + oo) + A.peer_delta[q]) = v;
  };
  auto put_box = [&](int64_t oo, float4 v) {
    A.out_boxes[oo] = v;
    for (int q = 0; q < A.npeers; ++q) *reinterpret_cast<float4*>(reinterpret_cast<char*>(A.out_boxes + oo) + A.peer_delta[q]) = v;
  };
  for (int t = tid; t < A.nms_topk; t += kSortThreads) {
    const int64_t oo = (int64_t)list * A.nms_topk + t;
    if (t < kept_n) {
      const int pos = g.krank[t];
      const unsigned long long key = A.s_key[o + pos];
      const uint32_t idx = key_index(key);
      put_score(oo, DECODE ? key_to_score((uint32_t)(key >> 32)) : src_scores[idx]);
      put_box(oo, DECODE ? g.kbox[t] : src_boxes[idx]);     // clipped boxes are already min/max ordered
      if (A.out_index != nullptr) A.out_index[oo] = (int32_t)idx;
      if (A.out_keep != nullptr) A.out_keep[oo] = A.filler ? pos : (int32_t)idx;
    } else {
      put_score(oo, 0.f);
      put_box(oo, make_float4(0.f, 0.f, 0.f, 0.f));
      if (A.out_index != nullptr) A.out_index[oo] = -1;
      if (A.out_keep != nullptr) {
        // parse_by_class runs NMS on the zero padded top-k list: zero-area filler rows are never suppressed
        // and get selected until nms_topk is reached
        const int fpos = g.K + (t - kept_n);
        A.out_keep[oo] = (A.filler && fpos < A.keep_topk) ? fpos : -1;
      }
    }
  }
  if (tid == 0 && A.out_counts != nullptr) {
    A.out_counts[list] = kept_n;
    for (int q = 0; q < A.npeers; ++q) *reinterpret_cast<int32_t*>(reinterpret_cast<char*>(A.out_counts + list) + A.peer_delta[q]) = kept_n;
  }
}

// release (peer exchange): this CTA's rows are visible system-wide before it counts itself done; the last CTA of the
// launch bumps the rank's step number and writes it into its flag slot in every destination (dan_wait_detections polls
// those)
DAN_D void release_peers(const PpArgs& A) {
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int done = atomicAdd(A.peer_state, 1);
    if (done == (int)gridDim.x - 1) {
      A.peer_state[0] = 0;
      const int seq = A.peer_state[1] + 1;
      A.peer_state[1] = seq;
      __threadfence_system();
      for (int q = 0; q < A.npeers; ++q) *reinterpret_cast<volatile int32_t*>(A.peer_flag[q]) = seq;
    }
  }
}

// T: element type of the predictions (DECODE only; the standalone sort / NMS instantiations take fp32 scores and boxes)
template <bool DECODE, int WHERE, bool FILTER, typename T>
__global__ void __launch_bounds__(kSortThreads, 1) nms_greedy_kernel(const PpArgs A, const float* __restrict__ src_scores,
                                                                     const float4* __restrict__ src_boxes) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  // (separate arrays: one __shared__ RoundSmem-shaped struct would be padded, 16 B more static shared memory)
  __shared__ unsigned char s_alive[kWin];
  __shared__ unsigned short s_list[kWin];
  __shared__ int s_surv[kSurv];
  __shared__ float4 s_sbox[kSurv];
  __shared__ float s_sarea[kSurv];
  __shared__ uint32_t s_T[kSurv][kSurvWords];
  __shared__ uint32_t s_keptm[kSurvWords], s_supm[kSurvWords];
  __shared__ uint2 s_smask[kSurv];
  __shared__ int s_hint[2][kHintCells];
  __shared__ int s_next[2];
  __shared__ int s_nlist;
  RoundSmem R = {s_alive, s_list, s_surv, s_sbox, s_sarea, s_smask, s_T, s_keptm, s_supm, s_hint, s_next, &s_nlist};

  const int list = blockIdx.x;
  const int b = list / max(A.num_classes - 1, 1);
  const int64_t o = (int64_t)list * A.plan.slots;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(dyn_smem);
  unsigned long long* gkeys = A.keys + (int64_t)list * A.n;
  GreedyList g = carve<WHERE>(A, dyn_smem, list);

  const int cnt = FILTER ? filter_image<T>(A, list, b, keys, gkeys) : min(A.key_count[list], A.n);
  const unsigned long long* sorted;
  g.K = top_k_sort<FILTER>(A, cnt, o, gkeys, keys, dyn_smem, sorted);
  decode_candidates<DECODE, T>(A, b, o, sorted, src_boxes, g);
  init_stripes(A, g, R);
  while (g.c0 < g.K && g.L < A.nms_topk) {
    const int w_end = min(g.K, g.c0 + kWin);
    test_window(A, g, R, w_end);
    int c_next;
    const int ns = compact_survivors(g, R, w_end, c_next);
    survivor_bits(A, R, ns);
    relax_survivors(R, ns);
    append_kept(A, g, R, ns);
    g.w_end_prev = w_end;
    g.c0 = c_next;
  }
  write_outputs<DECODE>(A, list, o, g, src_scores, src_boxes);
  if (A.npeers > 0) release_peers(A);
}

// One warp polls the arrival flags of the `world` ranks in this rank's receive buffer until all have reached the step
// number this rank's own NMS kernel just produced (state[1]); it holds one warp of one SM, nothing else.
__global__ void wait_detections_kernel(const int32_t* flags, const int32_t* state, int world) {
  const int want = *reinterpret_cast<const volatile int32_t*>(state + 1);
  const int q = threadIdx.x;
  if (q < world) {
    while (*reinterpret_cast<const volatile int32_t*>(flags + q) < want) __nanosleep(100);
  }
  __syncwarp();
  __threadfence_system();
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------

struct PpLayout {
  size_t key_count, keys, maybe, stash, s_key, s_key2, s_box, s_area, kept_box, kept_area, kept_rank, s_mask, stripes, total;
};

static PpLayout pp_layout(int64_t n, int64_t lists, int64_t keep_topk, bool nms, int64_t stash_rows = 0) {
  PpLayout w;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 256); return at; };
  const int64_t ks = cand_slots(n, keep_topk);
  w.key_count = take(lists * 4);
  w.keys = take(lists * n * 8);
  w.maybe = take(nms ? lists * n * 4 : 0);
  w.stash = take(stash_rows * 16);
  w.s_key = take(lists * ks * 8);
  w.s_key2 = take(lists * ks * 8);
  w.s_box = take(nms ? lists * ks * 16 : 0);
  w.s_area = take(nms ? lists * ks * 4 : 0);
  w.kept_box = take(nms ? lists * ks * 16 : 0);
  w.kept_area = take(nms ? lists * ks * 4 : 0);
  w.kept_rank = take(nms ? lists * ks * 4 : 0);
  w.s_mask = take(nms ? lists * ks * 8 : 0);
  w.stripes = take(nms ? lists * 64 * ((ks + 31) / 32) * 4 : 0);
  w.total = off;
  return w;
}

static void pp_bind(PpArgs& A, void* ws, const PpLayout& w) {
  char* base = static_cast<char*>(ws);
  A.key_count = reinterpret_cast<int32_t*>(base + w.key_count);
  A.keys = reinterpret_cast<unsigned long long*>(base + w.keys);
  A.maybe = reinterpret_cast<int32_t*>(base + w.maybe);
  A.s_key = reinterpret_cast<unsigned long long*>(base + w.s_key);
  A.s_key2 = reinterpret_cast<unsigned long long*>(base + w.s_key2);
  A.s_box = reinterpret_cast<float4*>(base + w.s_box);
  A.s_area = reinterpret_cast<float*>(base + w.s_area);
  A.g_kept_box = reinterpret_cast<float4*>(base + w.kept_box);
  A.g_kept_area = reinterpret_cast<float*>(base + w.kept_area);
  A.g_kept_rank = reinterpret_cast<int32_t*>(base + w.kept_rank);
  A.s_mask = reinterpret_cast<uint2*>(base + w.s_mask);
  A.g_stripes = reinterpret_cast<uint32_t*>(base + w.stripes);
}

// opt-in to > 48 KB of dynamic shared memory; the attribute belongs to the (function, device) pair, so it is set on
// every call (a few hundred ns of host time) rather than cached in a process-wide flag
template <bool DECODE, int WHERE, bool FILTER, typename T>
static int launch_greedy(const PpArgs& A, int lists, const float* src_scores, const float4* src_boxes, cudaStream_t st) {
  DAN_CUDA(cudaFuncSetAttribute(nms_greedy_kernel<DECODE, WHERE, FILTER, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, A.plan.smem));
  nms_greedy_kernel<DECODE, WHERE, FILTER, T><<<lists, kSortThreads, A.plan.smem, st>>>(A, src_scores, src_boxes);
  DAN_LAUNCH_CHECK("nms_greedy_kernel");
  return DAN_OK;
}

// [filter +] sort + greedy NMS for `lists` lists
template <bool DECODE, bool FILTER, typename T>
static int run_sort_nms(const PpArgs& A_in, int lists, const float* src_scores, const float4* src_boxes, cudaStream_t st) {
  PpArgs A = A_in;
  A.plan = greedy_plan(A.n, A.keep_topk, A.nms_cap);
  if (A.plan.where == 2) return launch_greedy<DECODE, 2, FILTER, T>(A, lists, src_scores, src_boxes, st);
  if (A.plan.where == 1) return launch_greedy<DECODE, 1, FILTER, T>(A, lists, src_scores, src_boxes, st);
  return launch_greedy<DECODE, 0, FILTER, T>(A, lists, src_scores, src_boxes, st);
}

// the launches of one postprocess call: [filter kernel +] the per-list NMS kernel, with T the prediction type
template <typename T>
static int postprocess_launch(const PpArgs& A, bool fused, int lists, cudaStream_t st, cudaEvent_t* ev) {
  if (ev) DAN_CUDA(cudaEventRecord(ev[0], st));
  if (!fused) {
    DAN_CUDA(cudaMemsetAsync(A.key_count, 0, (size_t)lists * 4, st));
    if (A.n > 0) {
      pp_filter_kernel<T><<<dim3((A.n + 256 * kFilterPerThread - 1) / (256 * kFilterPerThread), A.batch), 256, 0, st>>>(A);
      DAN_LAUNCH_CHECK("pp_filter_kernel");
    }
  }
  if (ev) DAN_CUDA(cudaEventRecord(ev[1], st));
  int rc = fused ? run_sort_nms<true, true, T>(A, lists, nullptr, nullptr, st) : run_sort_nms<true, false, T>(A, lists, nullptr, nullptr, st);
  if (ev && rc == DAN_OK) DAN_CUDA(cudaEventRecord(ev[2], st));
  return rc;
}

}  // namespace dan

using namespace dan;

extern "C" {

size_t dan_postprocess_workspace_bytes(int32_t num_anchors, int32_t batch, int32_t num_classes, int32_t keep_topk) {
  if (num_anchors < 0 || batch < 0 || num_classes < 2 || keep_topk < 1) return 0;
  return pp_layout(num_anchors, (int64_t)batch * (num_classes - 1), keep_topk, true, (int64_t)batch * num_anchors).total;
}

size_t dan_sort_workspace_bytes(int64_t n, int32_t keep_topk) {
  if (n < 0 || keep_topk < 1) return 0;
  return pp_layout(n, 1, keep_topk, false).total;
}

size_t dan_nms_workspace_bytes(int64_t n, int32_t nms_topk) {
  if (n < 0 || nms_topk < 0) return 0;
  return pp_layout(n, 1, n > 0 ? n : 1, true).total;
}

// pred_dtype has been checked by the caller
static int postprocess_core(const dan_postprocess_params* p, int32_t pred_dtype, const void* cls_pred, const void* loc_pred,
                            const void* boxes_pred, const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax,
                            int32_t num_anchors, int32_t batch, float* out_boxes, float* out_scores, int32_t* out_counts,
                            int32_t* out_anchor_index, int32_t* out_keep_pos, void* workspace, size_t workspace_bytes, void* stream,
                            cudaEvent_t* ev, const dan_peer_exchange* peers) {
  const int esize = dtype_bytes(pred_dtype);
  DAN_REQUIRE(p != nullptr, DAN_ERR_INVALID_ARGUMENT, "params is NULL");
  DAN_REQUIRE(p->num_classes >= 2, DAN_ERR_INVALID_ARGUMENT, "num_classes must be >= 2 (class 0 is background), got %d", p->num_classes);
  DAN_REQUIRE(num_anchors >= 0 && batch >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  DAN_REQUIRE(batch <= 65535, DAN_ERR_UNSUPPORTED, "batch > 65535");
  DAN_REQUIRE(p->select_threshold >= 0.f, DAN_ERR_INVALID_ARGUMENT,
              "select_threshold must be >= 0 (a negative threshold would let zero-score rows carry boxes), got %g", p->select_threshold);
  DAN_REQUIRE(p->keep_topk >= 1 && p->nms_topk >= 1, DAN_ERR_INVALID_ARGUMENT, "keep_topk and nms_topk must be >= 1");
  DAN_REQUIRE((loc_pred != nullptr) != (boxes_pred != nullptr), DAN_ERR_INVALID_ARGUMENT, "exactly one of loc_pred / boxes_pred must be given");
  if (batch == 0) return DAN_OK;
  DAN_REQUIRE(cls_pred && out_boxes && out_scores, DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  DAN_REQUIRE(loc_pred == nullptr || (a_ymin && a_xmin && a_ymax && a_xmax), DAN_ERR_INVALID_ARGUMENT, "anchors needed to decode loc_pred");
  DAN_REQUIRE(aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT, "out_boxes must be 16-byte aligned");
  {
    const uintptr_t row_mask = (uintptr_t)(4 * esize - 1);      // one row of 4 values per anchor: 16 (fp32) or 8 bytes
    DAN_REQUIRE(((reinterpret_cast<uintptr_t>(loc_pred) | reinterpret_cast<uintptr_t>(boxes_pred)) & row_mask) == 0,
                DAN_ERR_INVALID_ARGUMENT, "loc_pred / boxes_pred must be %d-byte aligned", 4 * esize);
  }
  const int lists = batch * (p->num_classes - 1);
  const PpLayout w = pp_layout(num_anchors, lists, p->keep_topk, true, (int64_t)batch * num_anchors);
  DAN_REQUIRE(workspace != nullptr && workspace_bytes >= w.total, DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", w.total,
              workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  PpArgs A = {};
  A.cls = cls_pred;
  A.loc = loc_pred;
  A.boxes = boxes_pred;
  A.ay0 = a_ymin; A.ax0 = a_xmin; A.ay1 = a_ymax; A.ax1 = a_xmax;
  A.n = num_anchors;
  A.batch = batch;
  A.num_classes = p->num_classes;
  A.img_h = (float)p->image_h;
  A.img_w = (float)p->image_w;
  A.select_thr = p->select_threshold;
  A.min_size_p1 = (float)((double)p->min_size + 1.0);   // python: min_size + 1. then fp32
  {
    const double t = (double)p->select_threshold;
    A.reject_below = (p->num_classes == 2 && t > 0.0 && t <= 0.99) ? (float)(log(t / (1.0 - t)) - 0.05) : -INFINITY;
  }
  A.ps0 = p->prior_scaling[0]; A.ps1 = p->prior_scaling[1]; A.ps2 = p->prior_scaling[2]; A.ps3 = p->prior_scaling[3];
  A.keep_topk = p->keep_topk;
  A.nms_topk = p->nms_topk;
  A.nms_cap = p->nms_topk < p->keep_topk ? p->nms_topk : p->keep_topk;
  A.nms_thr = p->nms_threshold;
  A.out_boxes = reinterpret_cast<float4*>(out_boxes);
  A.out_scores = out_scores;
  A.out_counts = out_counts;
  A.out_index = out_anchor_index;
  A.out_keep = out_keep_pos;
  A.filler = 1;
  if (peers != nullptr && peers->num_destinations > 0) {
    DAN_REQUIRE(peers->num_destinations <= DAN_MAX_PEERS, DAN_ERR_UNSUPPORTED, "more than %d destinations", DAN_MAX_PEERS);
    DAN_REQUIRE(peers->state != nullptr && out_counts != nullptr, DAN_ERR_INVALID_ARGUMENT, "peer exchange needs state words and out_counts");
    A.npeers = peers->num_destinations;
    for (int q = 0; q < A.npeers; ++q) {
      DAN_REQUIRE(peers->flag[q] != nullptr && (peers->delta_bytes[q] & 15) == 0, DAN_ERR_INVALID_ARGUMENT,
                  "destination %d: NULL flag or a slab offset that is not a multiple of 16 bytes", q);
      A.peer_delta[q] = peers->delta_bytes[q];
      A.peer_flag[q] = peers->flag[q];
    }
    A.peer_state = peers->state;
  }
  pp_bind(A, workspace, w);
  // loc_pred / boxes_pred in page-locked HOST memory (cudaHostAlloc / cudaHostRegister; mapped under unified addressing):
  // the kernels read only the rows of the anchors that pass the score threshold (~3 %), straight over PCIe, and keep
  // the decoded box of such a row in the workspace so that the row is fetched once.  Pageable memory is refused.
  {
    const void* geo = loc_pred != nullptr ? loc_pred : boxes_pred;
    cudaPointerAttributes pa;
    const cudaError_t e = cudaPointerGetAttributes(&pa, geo);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
    } else if (pa.type == cudaMemoryTypeHost) {
      DAN_REQUIRE(pa.devicePointer != nullptr, DAN_ERR_INVALID_ARGUMENT, "loc_pred / boxes_pred: host memory that is not mapped for the device");
      if (loc_pred != nullptr) A.loc = pa.devicePointer;
      else A.boxes = pa.devicePointer;
      A.stash = reinterpret_cast<float4*>(static_cast<char*>(workspace) + w.stash);
    } else {
      DAN_REQUIRE(pa.type != cudaMemoryTypeUnregistered, DAN_ERR_INVALID_ARGUMENT,
                  "loc_pred / boxes_pred is pageable host memory: pass device memory or page-locked (pinned) host memory");
    }
  }
  // two classes: the NMS kernel filters its own image (one launch for the whole evaluation side) when every anchor's pair
  // of logits is aligned for one load
  const bool fused = p->num_classes == 2 && (reinterpret_cast<uintptr_t>(cls_pred) & (uintptr_t)(2 * esize - 1)) == 0;
  switch (pred_dtype) {
    case DAN_DTYPE_F16: return postprocess_launch<__half>(A, fused, lists, st, ev);
    case DAN_DTYPE_BF16: return postprocess_launch<__nv_bfloat16>(A, fused, lists, st, ev);
    default: return postprocess_launch<float>(A, fused, lists, st, ev);
  }
}

int dan_postprocess_batch_typed(const dan_postprocess_params* p, int32_t pred_dtype, const void* cls_pred, const void* loc_pred,
                                const void* boxes_pred, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                                const float* a_xmax, int32_t num_anchors, int32_t batch, float* out_boxes, float* out_scores,
                                int32_t* out_counts, int32_t* out_anchor_index, int32_t* out_keep_pos, void* workspace,
                                size_t workspace_bytes, const dan_peer_exchange* peers, void* stream, float* h_kernel_ms) {
  DAN_REQUIRE(dtype_bytes(pred_dtype) != 0, DAN_ERR_INVALID_ARGUMENT, "unknown pred_dtype %d", pred_dtype);
  DAN_REQUIRE(peers == nullptr || h_kernel_ms == nullptr, DAN_ERR_INVALID_ARGUMENT,
              "h_peers and h_kernel_ms: the profiling call does not take part in a peer exchange");
  if (h_kernel_ms == nullptr) {
    DAN_REQUIRE(batch > 0 || peers == nullptr || peers->num_destinations == 0, DAN_ERR_INVALID_ARGUMENT,
                "a rank without images cannot take part in the peer exchange (its flag would never rise)");
    return postprocess_core(p, pred_dtype, cls_pred, loc_pred, boxes_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch,
                            out_boxes, out_scores, out_counts, out_anchor_index, out_keep_pos, workspace, workspace_bytes, stream,
                            nullptr, peers);
  }
  // profiling: events around the two launches, then wait for them
  h_kernel_ms[0] = h_kernel_ms[1] = 0.f;
  cudaEvent_t ev[3];
  for (int i = 0; i < 3; ++i) DAN_CUDA(cudaEventCreate(&ev[i]));
  int rc = postprocess_core(p, pred_dtype, cls_pred, loc_pred, boxes_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors, batch,
                            out_boxes, out_scores, out_counts, out_anchor_index, out_keep_pos, workspace, workspace_bytes, stream, ev,
                            nullptr);
  if (rc == DAN_OK && batch > 0) {
    cudaError_t e = cudaEventSynchronize(ev[2]);
    if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventSynchronize");
    else for (int i = 0; i < 2; ++i) cudaEventElapsedTime(&h_kernel_ms[i], ev[i], ev[i + 1]);
  }
  for (int i = 0; i < 3; ++i) cudaEventDestroy(ev[i]);
  return rc;
}

int dan_postprocess_batch(const dan_postprocess_params* p, const float* cls_pred, const float* loc_pred, const float* boxes_pred,
                          const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax, int32_t num_anchors,
                          int32_t batch, float* out_boxes, float* out_scores, int32_t* out_counts, int32_t* out_anchor_index,
                          int32_t* out_keep_pos, void* workspace, size_t workspace_bytes, void* stream) {
  return dan_postprocess_batch_typed(p, DAN_DTYPE_F32, cls_pred, loc_pred, boxes_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors,
                                     batch, out_boxes, out_scores, out_counts, out_anchor_index, out_keep_pos, workspace,
                                     workspace_bytes, nullptr, stream, nullptr);
}

int dan_postprocess_batch_peers(const dan_postprocess_params* p, const float* cls_pred, const float* loc_pred, const float* boxes_pred,
                                const float* a_ymin, const float* a_xmin, const float* a_ymax, const float* a_xmax, int32_t num_anchors,
                                int32_t batch, float* out_boxes, float* out_scores, int32_t* out_counts, int32_t* out_anchor_index,
                                int32_t* out_keep_pos, void* workspace, size_t workspace_bytes, const dan_peer_exchange* peers,
                                void* stream) {
  return dan_postprocess_batch_typed(p, DAN_DTYPE_F32, cls_pred, loc_pred, boxes_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors,
                                     batch, out_boxes, out_scores, out_counts, out_anchor_index, out_keep_pos, workspace,
                                     workspace_bytes, peers, stream, nullptr);
}

int dan_wait_detections(const int32_t* flags, const int32_t* state, int32_t world_size, void* stream) {
  DAN_REQUIRE(flags != nullptr && state != nullptr && world_size >= 1 && world_size <= 32, DAN_ERR_INVALID_ARGUMENT, "bad arguments");
  wait_detections_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags, state, world_size);
  DAN_LAUNCH_CHECK("wait_detections_kernel");
  return DAN_OK;
}

int dan_peer_alloc(size_t bytes, void** out_ptr, void* out_handle64) {
  DAN_REQUIRE(bytes > 0 && out_ptr != nullptr && out_handle64 != nullptr, DAN_ERR_INVALID_ARGUMENT, "bad arguments");
  void* ptr = nullptr;
  DAN_CUDA(cudaMalloc(&ptr, bytes));
  cudaError_t e = cudaMemset(ptr, 0, bytes);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, ptr);
  if (e != cudaSuccess) {
    cudaFree(ptr);
    return cuda_fail(e, "cudaIpcGetMemHandle");
  }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  memcpy(out_handle64, &h, 64);
  *out_ptr = ptr;
  return DAN_OK;
}

int dan_peer_open(const void* handle64, void** out_ptr) {
  DAN_REQUIRE(handle64 != nullptr && out_ptr != nullptr, DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  DAN_CUDA(cudaIpcOpenMemHandle(out_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return DAN_OK;
}

int dan_peer_close(void* ptr) {
  if (ptr != nullptr) DAN_CUDA(cudaIpcCloseMemHandle(ptr));
  return DAN_OK;
}

int dan_peer_free(void* ptr) {
  if (ptr != nullptr) DAN_CUDA(cudaFree(ptr));
  return DAN_OK;
}

int dan_postprocess_batch_profile(const dan_postprocess_params* p, const float* cls_pred, const float* loc_pred,
                                  const float* boxes_pred, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                                  const float* a_xmax, int32_t num_anchors, int32_t batch, float* out_boxes, float* out_scores,
                                  int32_t* out_counts, int32_t* out_anchor_index, int32_t* out_keep_pos, void* workspace,
                                  size_t workspace_bytes, void* stream, float* h_kernel_ms) {
  DAN_REQUIRE(h_kernel_ms != nullptr, DAN_ERR_INVALID_ARGUMENT, "h_kernel_ms is NULL");
  return dan_postprocess_batch_typed(p, DAN_DTYPE_F32, cls_pred, loc_pred, boxes_pred, a_ymin, a_xmin, a_ymax, a_xmax, num_anchors,
                                     batch, out_boxes, out_scores, out_counts, out_anchor_index, out_keep_pos, workspace,
                                     workspace_bytes, nullptr, stream, h_kernel_ms);
}

int dan_sort_bboxes(const float* scores, const float* boxes, int64_t n, int32_t keep_topk, float* out_scores, float* out_boxes,
                    int32_t* out_index, void* workspace, size_t workspace_bytes, void* stream) {
  DAN_REQUIRE(n >= 0 && n < 0x7fffffff && keep_topk >= 1, DAN_ERR_INVALID_ARGUMENT, "bad size");
  DAN_REQUIRE(out_scores && out_boxes && aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT, "NULL / misaligned output");
  DAN_REQUIRE(n == 0 || (scores && boxes && aligned16(boxes)), DAN_ERR_INVALID_ARGUMENT, "NULL / misaligned input");
  const PpLayout w = pp_layout(n, 1, keep_topk, false);
  DAN_REQUIRE(workspace != nullptr && workspace_bytes >= w.total, DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", w.total,
              workspace_bytes);
  DAN_CUDA(cudaFuncSetAttribute(topk_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSortCap * 8)));
  cudaStream_t st = (cudaStream_t)stream;
  PpArgs A = {};
  A.n = (int)n;
  A.num_classes = 2;
  A.keep_topk = keep_topk;
  pp_bind(A, workspace, w);
  A.s_scores = out_scores;
  A.s_boxes = reinterpret_cast<float4*>(out_boxes);
  A.s_index = out_index;
  key_build_kernel<<<grid_for(n), 256, 0, st>>>(scores, n, A.keys, A.key_count);
  DAN_LAUNCH_CHECK("key_build_kernel");
  topk_sort_kernel<<<1, kSortThreads, kSortCap * 8, st>>>(A, scores, reinterpret_cast<const float4*>(boxes));
  DAN_LAUNCH_CHECK("topk_sort_kernel");
  return DAN_OK;
}

int dan_nms_bboxes(const float* scores, const float* boxes, int64_t n, int32_t nms_topk, float nms_threshold, float* out_scores,
                   float* out_boxes, int32_t* out_keep, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream) {
  DAN_REQUIRE(n >= 0 && nms_topk >= 1, DAN_ERR_INVALID_ARGUMENT, "bad size");
  DAN_REQUIRE(n < 0x7fffffff, DAN_ERR_INVALID_ARGUMENT, "bad size");
  const int n_eff = n > 0 ? (int)n : 1;
  const int cap = nms_topk < n_eff ? nms_topk : n_eff;
  DAN_REQUIRE(out_scores && out_boxes && aligned16(out_boxes), DAN_ERR_INVALID_ARGUMENT, "NULL / misaligned output");
  DAN_REQUIRE(n == 0 || (scores && boxes && aligned16(boxes)), DAN_ERR_INVALID_ARGUMENT, "NULL / misaligned input");
  const PpLayout w = pp_layout(n, 1, n_eff, true);
  DAN_REQUIRE(workspace != nullptr && workspace_bytes >= w.total, DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", w.total,
              workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  PpArgs A = {};
  A.n = (int)n;
  A.num_classes = 2;
  A.keep_topk = n_eff;
  A.nms_topk = nms_topk;
  A.nms_cap = cap;
  A.nms_thr = nms_threshold;
  A.out_boxes = reinterpret_cast<float4*>(out_boxes);
  A.out_scores = out_scores;
  A.out_counts = out_count;
  A.out_index = nullptr;
  A.out_keep = out_keep;
  A.filler = 0;
  pp_bind(A, workspace, w);
  key_build_kernel<<<grid_for(n), 256, 0, st>>>(scores, n, A.keys, A.key_count);
  DAN_LAUNCH_CHECK("key_build_kernel");
  return run_sort_nms<false, false, float>(A, 1, scores, reinterpret_cast<const float4*>(boxes), st);
}

}  // extern "C"
