// K2: anchor x GT matching and box encoding, on two paths that share the matcher rules and pass 3.
//
//   fused path  (dan_encode_batch): IoU is evaluated on the fly, tile-culled, and never written to HBM (the reference
//               materialises [N,M] fp32 and makes ~26 passes over it, anchor_manipulator.py:24-105,287).  All images
//               of the batch in each launch:
//     pass 1  enc_pass1_fused_kernel: everything that depends on ONE anchor - row maximum / argmax, stage 1 of the
//             matcher, labels, encode, ALL outputs (44 B/anchor) - plus the per-GT column maxima (atomicMax on fp32
//             bit patterns), the per-GT match counts and, mining, the stage-3 candidates in per-GT buckets
//             (pass1_task: a CTA's chunk of anchors and images; load_warp_anchors: its anchors and warp box)
//     pass 2  enc_pass2_find_kernel + enc_pass2_apply_kernel: stage 2 (mining) / the GT-side claim (dual) as a patch
//             of the few anchors whose overlap reaches a GT's column maximum (DESIGN.md §4a).  Find: summarize_columns,
//             list_reaching_warps (level 1), flag_box_hits (level 2), enqueue_flagged; apply: walk_gts twice, stage2_match
//   dense path  (dan_small_mining_match / dan_dual_max_match): the literal custom op boundary, the overlaps [N,M] of
//               one image given in HBM and read in 32 x 32 tiles transposed through shared memory (load_tile):
//     pass 1  dense_pass1_kernel: per-GT column maxima (dual with gt_max_first = 0: which GTs have an anchor-side
//             positive)
//     pass 2  dense_pass2_kernel: per anchor, stage 1 from the row maximum, stage 2 / the claim against the column
//             maxima (stage2_match), match and score; mining: the anchors still unmatched push their candidates to
//             per-GT buckets
//   pass 3  (mining only, both paths) stage 3 "hard face compensation": one CTA per image walks the GTs in ascending
//           order (the stage is order dependent, small_mining_match.cc:199-222) and patches the few affected anchors
//           (list_needy; per window window_end, load_window, resolve_window, apply_window; or rescan_overflowed)
//
// Culling (fused path): a warp owns 32 consecutive anchors; it reduces their
// bounding box with redux.sync and tests 32 GT boxes per ballot against it.  Only
// GTs that can intersect some anchor of the warp are evaluated.  A skipped pair
// has an empty intersection, for which the reference computes exactly 0, so the
// result is unchanged.  GTs whose column maximum is 0 (dual: `==` claim) or below
// FLT_EPSILON (mining: tie band) tie with zero-overlap anchors as well and are
// therefore never culled in pass 2.
//
// Precondition shared with the op's own doc string (small_mining_match.cc:42-43):
// overlaps are in [0, 1], i.e. boxes have non-negative (+1 convention) extents.
#include <float.h>
#include <stdlib.h>

#include "common.cuh"
#include "heap_order.cuh"

namespace dan {

constexpr int kEncThreads = 256;
constexpr int kBucketCap = 64;     // compensation candidates bucketed per GT before spilling

struct EncArgs {
  // anchors (fused)
  const float* ay0;
  const float* ax0;
  const float* ay1;
  const float* ax1;
  const uint8_t* mask;
  int n;
  // ground truth (fused), CSR over the batch
  const float4* gt;
  const int32_t* gt_off;
  // dense
  const float* overlaps;
  int m_dense;
  // parameters
  float low, high;       // dual: low/high thresholds; mining: negative_high / positive
  float neg_low, stop;
  int min_match;
  int ignore_between, gt_max_first;
  float ps0, ps1, ps2, ps3;
  float pa_scale;
  int debug;
  // workspace
  uint32_t* colmax;      // [G] fp32 bit patterns (>= 0)
  int32_t* cnt;          // [G] anchors matched per GT after stage 2
  int32_t* haspos;       // [G] GT has a positive anchor-side match (dual, gt_max_first=0)
  int32_t* fill;         // [G] candidates pushed per GT
  HeapItem* bucket;      // [G, kBucketCap]
  HeapItem* spill;       // [B, 2, n] (candidate list and heap of the overflow path)
  float* wbest;          // [B, ceil(n/32)] largest row maximum of each warp of fused pass 1 (read by the patch pass)
  float4* wbox;          // [ceil(n/32)] bounding box of the warp's (matching) anchors, the same for every image
  int32_t* queue_n;      // [1] warps of pass 1 that the patch pass has to re-evaluate ...
  int2* queue;           // [B * ceil(n/32)] ... as (image, warp)
  const int2* warp_map;  // [ceil(n/32)] or NULL: which anchors warp w of the fused passes owns (base, row stride): lane l
                         // holds anchor base + (l >> 3) * stride + (l & 7); NULL = 32 consecutive anchors
  // outputs
  float4* targets;
  int64_t* labels;
  float* scores;
  float4* matched;
  int32_t* match32;
  int64_t* match64;
};

// image b of the fused path owns per-GT slots [off[b] + b, off[b+1] + b + 1): one
// extra slot per image holds the dummy box of an empty image (:286).
struct ImageGt {
  int off0;     // first GT row in A.gt
  int m_real;   // GT rows given
  int m_eff;    // max(m_real, 1)
  int slot0;    // first per-GT workspace slot
};

template <bool DENSE>
DAN_D ImageGt image_gt(const EncArgs& A, int b) {
  ImageGt g;
  if (DENSE) {
    g.off0 = 0;
    g.m_real = g.m_eff = A.m_dense;
    g.slot0 = 0;
  } else {
    g.off0 = A.gt_off[b];
    g.m_real = A.gt_off[b + 1] - g.off0;
    g.m_eff = g.m_real > 0 ? g.m_real : 1;
    g.slot0 = g.off0 + b;
  }
  return g;
}

DAN_D float4 gt_box(const EncArgs& A, const ImageGt& ig, int j) {
  return (j < ig.m_real) ? __ldg(A.gt + ig.off0 + j) : make_float4(0.f, 0.f, 1.f, 1.f);
}

// The box an anchor is MATCHED with: itself (encode_anchors) or shrunk about its
// centre by pa_scale (encode_pa_anchors, anchor_manipulator.py:337-342).
struct AnchorBox {
  float y0, x0, y1, x1;  // original anchor
  float my0, mx0, my1, mx1, marea;  // matching box and its area
};

DAN_D AnchorBox load_anchor(const EncArgs& A, int a) {
  AnchorBox ab;
  ab.y0 = A.ay0[a];
  ab.x0 = A.ax0[a];
  ab.y1 = A.ay1[a];
  ab.x1 = A.ax1[a];
  if (A.pa_scale > 0.f) {
    float cy, cx, h, w;
    point2center(ab.y0, ab.x0, ab.y1, ab.x1, cy, cx, h, w);
    center2point(cy, cx, fdiv(h, A.pa_scale), fdiv(w, A.pa_scale), ab.my0, ab.mx0, ab.my1, ab.mx1);
  } else {
    ab.my0 = ab.y0;
    ab.mx0 = ab.x0;
    ab.my1 = ab.y1;
    ab.mx1 = ab.x1;
  }
  ab.marea = box_area(ab.my0, ab.mx0, ab.my1, ab.mx1);
  return ab;
}

// The original anchor box in centre form: all that the encode of a positive row and the signs of a negative row need.
struct AnchorCtr {
  float cy, cx, h, w;
};

DAN_D AnchorCtr anchor_ctr(float y0, float x0, float y1, float x1) {
  AnchorCtr c;
  point2center(y0, x0, y1, x1, c.cy, c.cx, c.h, c.w);
  return c;
}

// Encode anchor `a` of image `b` against GT box g (anchor_manipulator.py:306-326 /
// :366-387) and write every output row of a POSITIVE anchor.  raw() returns the original anchor box, which only the
// debug mode writes.
template <typename RawBox>
DAN_D void write_positive(const EncArgs& A, int64_t row, const AnchorCtr& ac, RawBox raw, float4 g, float score, int gt_index) {
  float4 t;
  if (A.debug) {
    t = raw();
  } else {
    float gcy, gcx, gh, gw;
    point2center(g.x, g.y, g.z, g.w, gcy, gcx, gh, gw);
    t.x = fdiv(fdiv(fsub(gcy, ac.cy), ac.h), A.ps0);
    t.y = fdiv(fdiv(fsub(gcx, ac.cx), ac.w), A.ps1);
    if (A.pa_scale > 0.f) {
      t.z = fdiv(cephes_logf(fdiv(fmul(gh, A.pa_scale), ac.h)), A.ps2);
      t.w = fdiv(cephes_logf(fdiv(fmul(gw, A.pa_scale), ac.w)), A.ps3);
    } else {
      t.z = fdiv(cephes_logf(fdiv(gh, ac.h)), A.ps2);
      t.w = fdiv(cephes_logf(fdiv(gw, ac.w)), A.ps3);
    }
  }
  A.targets[row] = t;
  A.labels[row] = 1;
  A.scores[row] = score;
  if (A.matched != nullptr) A.matched[row] = g;
  if (A.match32 != nullptr) A.match32[row] = gt_index;
}

// the original anchor box, for the debug mode of fused pass 1 (which keeps the centre form only): out of line, so that
// the common path does not carry its loads
__device__ __noinline__ float4 raw_anchor(const float* y0, const float* x0, const float* y1, const float* x1, int a) {
  return make_float4(y0[a], x0[a], y1[a], x1[a]);
}

DAN_D void write_positive(const EncArgs& A, int64_t row, const AnchorBox& ab, float4 g, float score, int gt_index) {
  write_positive(A, row, anchor_ctr(ab.y0, ab.x0, ab.y1, ab.x1), [&] { return make_float4(ab.y0, ab.x0, ab.y1, ab.x1); }, g,
                 score, gt_index);
}

// ---------------------------------------------------------------------------
// matcher rules shared by both paths
// ---------------------------------------------------------------------------
struct RowState {
  float best = 0.f;      // row maximum, first strictly-greatest GT wins
  int best_gt = 0;
  float ov0 = 0.f;       // overlap with GT 0
  // dual
  bool claimed = false;
  float cbest = 0.f;
  int cbest_gt = 0;
  // mining
  int owner = -1;
  float owner_ov = 0.f;
};

template <bool MINING>
DAN_D void row_update(RowState& s, int j, float ov, float cm, bool claimable) {
  if (ov > s.best) { s.best = ov; s.best_gt = j; }
  if (j == 0) s.ov0 = ov;
  if (MINING) {
    // stage 2 tie band, small_mining_match.cc:171,179; ascending j => last GT wins
    if (fabsf(fsub(ov, cm)) < FLT_EPSILON) { s.owner = j; s.owner_ov = ov; }
  } else {
    // anchor_manipulator.py:88 exact equality with the column maximum
    if (claimable && ov == cm) {
      s.claimed = true;
      if (ov > s.cbest) { s.cbest = ov; s.cbest_gt = j; }
    }
  }
}

// stage 1 of either matcher from the row maximum (small_mining_match.cc:85-93 / anchor_manipulator.py:67-76)
template <bool MINING>
DAN_D int stage1_match(const EncArgs& A, float best, int best_gt) {
  if (MINING) {
    if (best >= A.neg_low && best < A.low) return -1;
    if (best >= A.high) return best_gt;
    return -2;
  }
  const bool less = best < A.low;
  const bool between = (best < A.high) && (best >= A.low);
  const bool neg = A.ignore_between ? less : between;
  const bool ign = A.ignore_between ? between : less;
  int match = best_gt;
  if (neg) match = -1;
  if (ign) match = -2;
  return match;
}

// stage 1, then stage 2 of the mining matcher (small_mining_match.cc:178-186: the last tied GT wins) / the GT-side claim
// of the dual matcher (anchor_manipulator.py:95-104: argmax over overlap * claim mask; GT 0 if claimed only through
// zero-overlap ties) for the row in `s`: the match, and its score in `score`
template <bool MINING>
DAN_D int stage2_match(const EncArgs& A, const RowState& s, float& score) {
  int match = stage1_match<MINING>(A, s.best, s.best_gt);
  score = s.best;
  if (MINING) {
    if (s.owner >= 0) { match = s.owner; score = s.owner_ov; }
  } else if (s.claimed) {
    if (s.cbest > 0.f) { match = s.cbest_gt; score = s.cbest; }
    else { match = 0; score = s.ov0; }
  }
  return match;
}

// ---------------------------------------------------------------------------
// dense path, passes 1 and 2, on the overlaps [n, m_dense] of one image.  A warp owns 32 consecutive anchors (rows)
// and reads the matrix in 32 x 32 tiles through shared memory (row stride 33: conflict-free both ways), so that a lane
// holds a column for the column maxima and a row for the row maxima.
// ---------------------------------------------------------------------------
// the warp's tile of rows [row0, row0 + 32) and columns [j0, j0 + 32) of the [A.n, m] matrix, zero outside it: lane l
// loads column j0 + l of every row
DAN_D void load_tile(const EncArgs& A, int m, float* tile, int row0, int j0, int lane) {
  const int jc = j0 + lane;
  for (int r = 0; r < 32; ++r) {
    const int row = row0 + r;
    tile[r * 33 + lane] = (row < A.n && jc < m) ? A.overlaps[(int64_t)row * m + jc] : 0.f;
  }
  __syncwarp();
}

template <bool NEED_ROW>
__global__ void __launch_bounds__(kEncThreads) dense_pass1_kernel(const EncArgs A) {
  __shared__ float s_tile[(kEncThreads / 32) * 32 * 33];

  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int a = blockIdx.x * kEncThreads + threadIdx.x;
  const int m = A.m_dense;
  float* tile = s_tile + warp * 32 * 33;
  const int row0 = blockIdx.x * kEncThreads + warp * 32;
  if (row0 >= A.n) return;

  float best = 0.f;
  int best_gt = 0;
  for (int j0 = 0; j0 < m; j0 += 32) {
    load_tile(A, m, tile, row0, j0, lane);
    const int jc = j0 + lane;
    // column maximum of the 32x32 tile: lane == column
    float cmx = 0.f;
    for (int r = 0; r < 32; ++r) cmx = fmaxf(cmx, tile[r * 33 + lane]);
    if (jc < m && cmx > 0.f) atomicMax(A.colmax + jc, __float_as_uint(cmx));
    if (NEED_ROW) {
      const int lim = min(32, m - j0);
      for (int jj = 0; jj < lim; ++jj) {
        const float ov = tile[lane * 33 + jj];
        if (ov > best) { best = ov; best_gt = j0 + jj; }
      }
    }
    __syncwarp();
  }

  if (NEED_ROW && a < A.n) {
    // anchor-side positive (match_indices >= 0 in anchor_manipulator.py:67-76)
    const bool less = best < A.low;
    const bool between = (best < A.high) && (best >= A.low);
    if (!less && !between) A.haspos[best_gt] = 1;
  }
}

template <bool MINING>
__global__ void __launch_bounds__(kEncThreads) dense_pass2_kernel(const EncArgs A) {
  __shared__ float s_tile[(kEncThreads / 32) * 32 * 33];

  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int a = blockIdx.x * kEncThreads + threadIdx.x;
  const bool valid = a < A.n;
  const int m = A.m_dense;
  const bool need_haspos = !MINING && !A.gt_max_first;
  float* tile = s_tile + warp * 32 * 33;
  const int row0 = blockIdx.x * kEncThreads + warp * 32;

  RowState s;
  // ---- sweep the GTs: two rounds only when compensation candidates must be pushed
  bool push_round = false;
  bool warp_push = false;
  int match = -1;
  float score = 0.f;
  for (int round = 0; round < 2; ++round) {
    if (row0 < A.n && (round == 0 || warp_push)) {
      for (int j0 = 0; j0 < m; j0 += 32) {
        load_tile(A, m, tile, row0, j0, lane);
        const int lim = min(32, m - j0);
        for (int jj = 0; jj < lim; ++jj) {
          const int j = j0 + jj;
          const float ov = tile[lane * 33 + jj];
          if (round == 0) {
            const float cm = __uint_as_float(A.colmax[j]);
            const bool claimable = !need_haspos || A.haspos[j] == 0;
            row_update<MINING>(s, j, ov, cm, claimable);
          } else if (MINING && push_round && ov > A.stop) {
            const int pos = atomicAdd(A.fill + j, 1);
            if (pos < kBucketCap) A.bucket[(int64_t)j * kBucketCap + pos] = HeapItem{ov, a};
          }
        }
        __syncwarp();
      }
    }

    if (round == 1) break;

    // ---- resolve this anchor (end of round 0)
    match = stage2_match<MINING>(A, s, score);
    if (MINING) {
      if (valid && match >= 0) atomicAdd(A.cnt + match, 1);
      push_round = valid && match < 0 && s.best > A.stop;
    }
    // round 1 runs only in CTAs with a pushing anchor, and there only in the warps that hold one
    if (!MINING || !__syncthreads_or(push_round ? 1 : 0)) break;
    warp_push = __any_sync(0xffffffffu, push_round);
  }

  if (!valid) return;
  if (A.match32 != nullptr) A.match32[a] = match;
  if (A.match64 != nullptr) A.match64[a] = match;
  A.scores[a] = score;
}

// ---------------------------------------------------------------------------
// per-warp GT iteration of the FUSED path
// ---------------------------------------------------------------------------
struct WarpBox {
  float y0, x0, y1, x1;
};

DAN_D WarpBox warp_bbox(bool active, const AnchorBox& ab) {
  const float inf = __int_as_float(0x7f800000);
  WarpBox wb;
  wb.y0 = warp_min_f(active ? ab.my0 : inf);
  wb.x0 = warp_min_f(active ? ab.mx0 : inf);
  wb.y1 = warp_max_f(active ? ab.my1 : -inf);
  wb.x1 = warp_max_f(active ? ab.mx1 : -inf);
  return wb;
}

// conservative "may intersect some anchor of the warp" test (see file header):
// a pair intersects only if fl(min(ymax) - max(ymin)) > -1, and the warp box
// dominates every anchor of the warp, so >= -1 on the warp box never misses.
DAN_D bool may_hit(const WarpBox& wb, float4 g) {
  const float dy = fsub(fminf(wb.y1, g.z), fmaxf(wb.y0, g.x));
  const float dx = fsub(fminf(wb.x1, g.w), fmaxf(wb.x0, g.y));
  return (dy >= -1.f) && (dx >= -1.f);
}

// ---------------------------------------------------------------------------
// FUSED path.  Pass 1 is a warp-autonomous kernel:
//   * a CTA of pass 1 owns a chunk of kFusedThreads anchors (a warp: 32 of them) and walks one image or, on the fine
//     pyramid levels, a group of images with them: the anchor loads, the mask, the warp -> anchors table,
//     the PA transform, the warp bounding box and the anchors' centre form are paid once per CTA;
//   * no shared memory and no CTA barrier: the ground truth of an image is a few hundred bytes, read through the
//     read-only path (32 boxes per coalesced load for the cull test, broadcast loads for the hits);
//   * per-GT column maxima of pass 1 are reduced in the warp (redux.sync) and the lane that loaded GT k issues one
//     atomicMax for it, so the atomics of a warp go to 32 different addresses.
// ---------------------------------------------------------------------------
constexpr int kFusedThreads = 128;

// Images per CTA of pass 1 on the fine levels.  A warp there meets ~2 GTs per image (~150 warp instructions) against
// ~350 instructions of per-(warp, image) bookkeeping, so it walks several images; a warp of a coarse level meets every
// GT of the image and keeps one, so that it does not become the tail of the launch (profiles/r03_pass1_breakdown.md).
// Measured on B200 at batch 32: 2 images give back 3.5 % of the rate with steps in flight, 8 add 1 % to it but make a
// lone pass 1 30 % longer.
constexpr int kFineImages = 4;
// a hinted level of at least this many cells (32 warps) counts as fine: at 640^2 the 160^2 / 80^2 / 40^2 levels
// (2.1 / 2.7 / 4.4 culled GTs per warp and image), not the 20^2 one (11.8)
constexpr int kFineMinCells = 1024;

// Which anchor lane `lane` of warp `wid` owns.  Without a layout hint a warp holds 32 consecutive anchors: on a pyramid
// level that is a 32 x 1 strip of cells, whose bounding box meets far more ground-truth boxes than its anchors do.
// With the hint (dan_encode_params.num_grids) the warps of a one-anchor-per-cell level hold 8 x 4 TILES of cells
// instead (the table is built by enc_warp_map_kernel): ~28 % fewer (warp, GT) pairs to evaluate at 640^2, the same
// anchors, the same per-anchor arithmetic - the results do not depend on it.  The index grows with the lane either way.
DAN_D int warp_anchor(const EncArgs& A, int wid, int lane) {
  if (A.warp_map == nullptr) return wid * 32 + lane;
  const int2 m = __ldg(A.warp_map + wid);
  return m.x + (lane >> 3) * m.y + (lane & 7);
}

// Non-positive anchors.  The reference multiplies the encoded targets of EVERY anchor by float(positive)
// (anchor_manipulator.py:324) and gathers GT clip(match, 0) = GT 0 for the non-positive ones (:297,306), so their
// targets are 0 * t = a zero with the SIGN of t, and their matched box is 0 * GT 0.  NegCtx holds what is needed to
// reproduce those signs without evaluating t: per image GT 0 in centre form (uniform over the warp).
struct NegCtx {
  float gcy, gcx, gh, gw;     // GT 0 (gh, gw already multiplied by pa_scale for encode_pa_anchors)
  float4 mzero;               // 0 * GT 0
  uint32_t ps_sign[4];        // sign bits of the prior scaling
};

DAN_D uint32_t sign_of(float v) { return __float_as_uint(v) & 0x80000000u; }

DAN_D NegCtx neg_ctx(const EncArgs& A, const ImageGt& ig) {
  NegCtx c;
  const float4 g = gt_box(A, ig, 0);
  point2center(g.x, g.y, g.z, g.w, c.gcy, c.gcx, c.gh, c.gw);
  if (A.pa_scale > 0.f) { c.gh = fmul(c.gh, A.pa_scale); c.gw = fmul(c.gw, A.pa_scale); }
  c.mzero = make_float4(__uint_as_float(sign_of(g.x)), __uint_as_float(sign_of(g.y)), __uint_as_float(sign_of(g.z)),
                        __uint_as_float(sign_of(g.w)));
  c.ps_sign[0] = sign_of(A.ps0); c.ps_sign[1] = sign_of(A.ps1); c.ps_sign[2] = sign_of(A.ps2); c.ps_sign[3] = sign_of(A.ps3);
  return c;
}

// sign bit of log(num / den) for num >= 0: negative iff the quotient is below 1 (for den > 0 the correctly rounded quotient
// is below 1 exactly when num < den)
DAN_D uint32_t log_ratio_sign(float num, float den) {
  const bool below = (den > 0.f) ? (num < den) : (fdiv(num, den) < 1.f);
  return below ? 0x80000000u : 0u;
}

// every output row of a NON-positive anchor; the 44 B/anchor of a step are written once and not read again by the
// encode kernels: streaming stores
template <typename RawBox>
DAN_D void write_negative(const EncArgs& A, int64_t row, const AnchorCtr& ac, RawBox raw, const NegCtx& c, float score, int match) {
  float4 t;
  if (A.debug) {
    const float4 r = raw();
    t = make_float4(__uint_as_float(sign_of(r.x)), __uint_as_float(sign_of(r.y)), __uint_as_float(sign_of(r.z)),
                    __uint_as_float(sign_of(r.w)));
  } else {
    t.x = __uint_as_float(sign_of(fsub(c.gcy, ac.cy)) ^ sign_of(ac.h) ^ c.ps_sign[0]);
    t.y = __uint_as_float(sign_of(fsub(c.gcx, ac.cx)) ^ sign_of(ac.w) ^ c.ps_sign[1]);
    t.z = __uint_as_float(log_ratio_sign(c.gh, ac.h) ^ c.ps_sign[2]);
    t.w = __uint_as_float(log_ratio_sign(c.gw, ac.w) ^ c.ps_sign[3]);
  }
  __stcs(A.targets + row, t);
  __stcs(reinterpret_cast<long long*>(A.labels) + row, (long long)((match < -1) ? -1 : 0));   // anchor_manipulator.py:300-302
  __stcs(A.scores + row, score);
  if (A.matched != nullptr) __stcs(A.matched + row, c.mzero);
  if (A.match32 != nullptr) __stcs(A.match32 + row, match);
}

// CTA -> (anchor chunk, images [b0, b_end)) of pass 1.  The chunks are walked from the END of the anchor array: the
// coarse pyramid levels live there, their warps see every GT and run the longest, so they must not be the tail of the
// launch.  The last `coarse_chunks` chunks come first, one CTA per image, all images of a chunk next to each other; then
// the fine chunks, one CTA per group of kFineImages images.  Fine chunks exist only with the layout hint, i.e. in the
// TILED instantiation.  pass1_grid() is the host's count of these CTAs.
struct Pass1Task {
  int from_end, b0, b_end;    // the anchor chunk, counted from the end of the anchor array; the images of the CTA
};

template <bool TILED>
DAN_D Pass1Task pass1_task(int batch, int coarse_chunks) {
  int from_end, b0, b_end;
  const int coarse_ctas = coarse_chunks * batch;
  if (!TILED || (int)blockIdx.x < coarse_ctas) {
    from_end = blockIdx.x / batch;
    b0 = blockIdx.x - from_end * batch;
    b_end = b0 + 1;
  } else {
    const int groups = (batch + kFineImages - 1) / kFineImages;
    const int j = blockIdx.x - coarse_ctas;
    const int c = j / groups;
    from_end = coarse_chunks + c;
    b0 = (j - c * groups) * kFineImages;
    b_end = min(batch, b0 + kFineImages);
  }
  return {from_end, b0, b_end};
}

static int pass1_grid(int batch, int coarse_chunks, int fine_chunks) {
  return coarse_chunks * batch + fine_chunks * ((batch + kFineImages - 1) / kFineImages);
}

// The anchor a of this lane of pass 1 (valid: a < A.n) in its matching and centre forms and whether the mask keeps it,
// loaded once for all the images of the CTA, and the bounding box of the warp's active anchors, which the CTA of image 0
// stores for pass 2
DAN_D void load_warp_anchors(const EncArgs& A, int a, bool valid, int wid, int nwarps, int b0, int lane, AnchorBox& ab,
                             AnchorCtr& ac, bool& active, WarpBox& wb) {
  ab = {};
  ac = {};
  active = false;
  if (valid) {
    ab = load_anchor(A, a);
    ac = anchor_ctr(ab.y0, ab.x0, ab.y1, ab.x1);
    active = (A.mask == nullptr) || (A.mask[a] != 0);
  }
  wb = warp_bbox(active, ab);
  if (b0 == 0 && lane == 0 && wid < nwarps) A.wbox[wid] = make_float4(wb.y0, wb.x0, wb.y1, wb.x1);
}

// pass 1 (fused path): everything that depends on ONE anchor only - row maximum / argmax, stage 1 of the matcher,
// labels, encode, ALL outputs - plus the two cross-anchor quantities the later passes need: the per-GT column maxima
// (atomicMax) and, for the mining matcher, the stage-3 candidates (overlap > stop_positive_thres) and the per-GT
// match counts.  What stage 2 / the GT-side claim of the dual matcher changes afterwards is a handful of anchors per
// GT; pass 2 finds and patches them.
// TILED: the warps hold the tiles of the layout hint (A.warp_map != NULL); a separate instantiation because the kernel
// sits on its register cap and the strip version can derive everything from threadIdx.  The cap is 40 registers: every
// instantiation uses all 40 without spilling, and on B200 this build was 1 % faster than one capped at 32.  The culled
// GT walk of an image and the row's end stay inline: as functions they reorder the front end's output, and ptxas then
// allocates this register-capped kernel differently.
template <bool NEED_ROW, bool MINING, bool TILED>
__global__ void __maxnreg__(40) enc_pass1_fused_kernel(const EncArgs A, int batch, int coarse_chunks) {
  const int lane = threadIdx.x & 31;
  const int nwarps = (A.n + 31) >> 5;
  const int nchunks = (A.n + kFusedThreads - 1) / kFusedThreads;
  const Pass1Task t = pass1_task<TILED>(batch, coarse_chunks);
  const int b0 = t.b0, b_end = t.b_end;
  // the warp's index (wbest / wbox / queue entries are per warp) and its anchors
  const int wid = (nchunks - 1 - t.from_end) * (kFusedThreads / 32) + (threadIdx.x >> 5);
  const int a = TILED ? ((wid < nwarps) ? warp_anchor(A, wid, lane) : A.n) : wid * 32 + lane;
  const bool valid = a < A.n;
  AnchorBox ab;
  AnchorCtr ac;
  bool active;
  WarpBox wb;
  load_warp_anchors(A, a, valid, wid, nwarps, b0, lane, ab, ac, active, wb);
  const auto raw = [&] { return raw_anchor(A.ay0, A.ax0, A.ay1, A.ax1, a); };
  for (int b = b0; b < b_end; ++b) {
    const ImageGt ig = image_gt<false>(A, b);
    float best = 0.f;
    int best_gt = 0;
    for (int k0 = 0; k0 < ig.m_eff; k0 += 32) {
      const int k = k0 + lane;
      // (gt_box(A, ig, k) for k < m_eff; the lanes beyond m_eff stay out of the ballot and are never broadcast)
      float4 gk = make_float4(0.f, 0.f, 1.f, 1.f);
      if (k < ig.m_real) gk = __ldg(A.gt + ig.off0 + k);
      unsigned hits = __ballot_sync(0xffffffffu, (k < ig.m_eff) && may_hit(wb, gk));
      const float gk_area = box_area(gk.x, gk.y, gk.z, gk.w);      // once per GT, broadcast with the box below
      uint32_t my_colmax = 0u;            // column maximum of GT k over this warp's anchors
      while (hits) {
        const int kl = __ffs(hits) - 1;
        hits &= hits - 1;
        // lane kl loaded this GT for the cull test above: broadcast it instead of fetching it again
        const float4 g = make_float4(__shfl_sync(0xffffffffu, gk.x, kl), __shfl_sync(0xffffffffu, gk.y, kl),
                                     __shfl_sync(0xffffffffu, gk.z, kl), __shfl_sync(0xffffffffu, gk.w, kl));
        const float g_area = __shfl_sync(0xffffffffu, gk_area, kl);
        bool hit = false;
        float ov = 0.f;
        if (active) ov = pair_iou(ab.my0, ab.mx0, ab.my1, ab.mx1, ab.marea, g.x, g.y, g.z, g.w, g_area, hit);
        const uint32_t wmax = __reduce_max_sync(0xffffffffu, (ov > 0.f) ? __float_as_uint(ov) : 0u);
        if (lane == kl) my_colmax = wmax;
        if (ov > best) { best = ov; best_gt = k0 + kl; }      // first strictly-greatest GT wins (tf.argmax / :76-83)
        if (MINING && ov > A.stop) {
          // possible stage-3 compensation candidate (small_mining_match.cc:206); whether the anchor is still
          // unmatched is only known after stage 2, pass 3 filters on that
          const int pos = atomicAdd(A.fill + ig.slot0 + k0 + kl, 1);
          if (pos < kBucketCap)
            A.bucket[(int64_t)(ig.slot0 + k0 + kl) * kBucketCap + pos] = HeapItem{ov, a};
        }
      }
      if (my_colmax != 0u) atomicMax(A.colmax + ig.slot0 + k, my_colmax);
    }
    // no overlap of this warp exceeds the largest row maximum of its lanes: pass 2 uses it to skip the warp
    const uint32_t wbest = __reduce_max_sync(0xffffffffu, __float_as_uint(best));
    if (lane == 0 && wid < nwarps) A.wbest[(int64_t)b * nwarps + wid] = __uint_as_float(wbest);   // (the last CTA may hold a warp beyond the anchors)
    if (valid) {
      const int match = stage1_match<MINING>(A, best, best_gt);
      const int64_t row = (int64_t)b * A.n + a;
      if (match >= 0) {
        if (MINING) atomicAdd(A.cnt + ig.slot0 + match, 1);
        if (NEED_ROW) A.haspos[ig.slot0 + match] = 1;          // anchor-side positive (anchor_manipulator.py:67-76)
        write_positive(A, row, ac, raw, gt_box(A, ig, match), best, match);
      } else {
        write_negative(A, row, ac, raw, neg_ctx(A, ig), best, match);
      }
    }
  }
}

// pass 2 (fused path): stage 2 of the mining matcher (small_mining_match.cc:160-197) / the GT-side claim of the dual
// matcher (anchor_manipulator.py:84-104) as a PATCH.  An anchor is affected only if its overlap with some GT k reaches
// that GT's column maximum cm[k] (to within FLT_EPSILON for the mining matcher).  One thread per warp of pass 1 first
// compares the warp's largest row maximum with the image's column maxima; the few warps that can reach one (and all
// warps when a GT has no overlap at all: its "maximum" 0 ties with every zero-overlap anchor, tie T7) are collected
// and re-evaluated by full warps: row maximum again, tie / claim test, and the outputs of the anchors whose match
// changed are rewritten (a patched anchor is always positive).
constexpr int kPatchThreads = 128;
constexpr int kPatchGt = 1024;        // GT boxes staged in shared memory at a time

// A warp's walk over the GTs of image `ig`, 32 per ballot: each GT k for which test(wide, column maximum, box) holds on
// its lane (wide: see the file header) is broadcast, and every lane runs visit(k, its overlap (0 if inactive), col. max)
template <bool MINING, typename Test, typename Visit>
DAN_D void walk_gts(const EncArgs& A, const ImageGt& ig, int lane, bool active, const AnchorBox& ab, Test test,
                    Visit visit) {
  for (int k0 = 0; k0 < ig.m_eff; k0 += 32) {
    const int k = k0 + lane;
    bool t = false;
    float cmk = 0.f;                                   // GT k's column maximum and box
    float4 gk = make_float4(0.f, 0.f, 0.f, 0.f);
    if (k < ig.m_eff) {
      cmk = __uint_as_float(__ldg(A.colmax + ig.slot0 + k));
      gk = gt_box(A, ig, k);
      t = test(MINING ? (cmk < FLT_EPSILON) : (cmk == 0.f), cmk, gk);
    }
    unsigned hits = __ballot_sync(0xffffffffu, t);
    while (hits) {
      const int kl = __ffs(hits) - 1;
      hits &= hits - 1;
      const float4 g = make_float4(__shfl_sync(0xffffffffu, gk.x, kl), __shfl_sync(0xffffffffu, gk.y, kl),
                                   __shfl_sync(0xffffffffu, gk.z, kl), __shfl_sync(0xffffffffu, gk.w, kl));
      const float cm = __shfl_sync(0xffffffffu, cmk, kl);
      bool hit = false;
      float ov = 0.f;
      if (active) ov = pair_iou(ab.my0, ab.mx0, ab.my1, ab.mx1, ab.marea, g.x, g.y, g.z, g.w, box_area(g.x, g.y, g.z, g.w), hit);
      visit(k0 + kl, ov, cm);
    }
  }
}

// Shared arrays of enc_pass2_find_kernel: staged GT boxes and column maxima, the warps level 1 lists (reach, box, flag).
// Separate __shared__ arrays behind pointers: as one __shared__ struct they cost the kernel two more registers.
struct FindSmem {
  int* list;        // [kPatchThreads]: the listed warps of pass 1 ...
  float* reach;     //   ... their reach (wbest, widened by the mining tie band) ...
  float4* wbox;     //   ... their bounding box ...
  int* flag;        //   ... and whether they go to the queue
  float4* box;      // [kPatchGt]: staged GT boxes ...
  float* cm;        //   ... and column maxima
  int& n;           // listed warps
  float* cmin;      // [kPatchThreads / 32]: per-warp partial minimum column maximum ...
  int* wide;        //   ... and "wide" flag
};

// The smallest column maximum of image `ig` and whether a GT ties with zero-overlap anchors (wide), over the CTA; with
// `staged` the GT boxes and column maxima are staged in S on the way.  Ends with a barrier.
template <bool MINING>
DAN_D void summarize_columns(const EncArgs& A, const ImageGt& ig, bool staged, const FindSmem& S, float& cmin,
                             bool& wide) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  cmin = 3.0e38f;
  wide = false;
  for (int k = tid; k < ig.m_eff; k += kPatchThreads) {
    const float cm = __uint_as_float(A.colmax[ig.slot0 + k]);
    if (staged) {
      S.cm[k] = cm;
      S.box[k] = gt_box(A, ig, k);
    }
    wide |= MINING ? (cm < FLT_EPSILON) : (cm == 0.f);
    cmin = fminf(cmin, cm);
  }
  cmin = warp_min_f(cmin);
  wide = __any_sync(0xffffffffu, wide);
  if (lane == 0) { S.cmin[warp] = cmin; S.wide[warp] = wide ? 1 : 0; }
  if (tid == 0) S.n = 0;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < kPatchThreads / 32; ++w) { cmin = fminf(cmin, S.cmin[w]); wide |= S.wide[w] != 0; }
}

// Level 1, a thread per warp of pass 1: can the warp reach the smallest column maximum at all?  Lists those that can in
// S (flagged at once when the image is wide) and returns their number, after a barrier.
template <bool MINING>
DAN_D int list_reaching_warps(const EncArgs& A, int b, float cmin, bool wide, const FindSmem& S) {
  const int nwarps = (A.n + 31) >> 5;
  const int wr = blockIdx.y * kPatchThreads + threadIdx.x;
  bool cand = false;
  float my_reach = 0.f;
  if (wr < nwarps) {
    const float wb = A.wbest[(int64_t)b * nwarps + wr];
    my_reach = MINING ? fadd(wb, 2.f * FLT_EPSILON) : wb;
    cand = wide || (my_reach >= cmin);
  }
  if (cand) {
    const int pos = atomicAdd(&S.n, 1);
    S.list[pos] = wr;
    S.reach[pos] = my_reach;
    S.wbox[pos] = A.wbox[wr];                                 // (all candidates of the CTA in one round trip)
    S.flag[pos] = wide ? 1 : 0;
  }
  __syncthreads();
  return S.n;
}

// Level 2, still without touching the anchors: flag a listed warp if some GT's column maximum is within its reach AND the
// GT's box meets its bounding box; a warp tests 32 GTs per step for each of its list entries.  Ends with a barrier.
DAN_D void flag_box_hits(const EncArgs& A, const ImageGt& ig, bool staged, int n_list, const FindSmem& S) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int c0 = 0; c0 < ig.m_eff; c0 += kPatchGt) {
    const int mc = min(kPatchGt, ig.m_eff - c0);
    if (!staged) {
      __syncthreads();
      for (int k = tid; k < mc; k += kPatchThreads) {
        S.box[k] = gt_box(A, ig, c0 + k);
        S.cm[k] = __uint_as_float(A.colmax[ig.slot0 + c0 + k]);
      }
      __syncthreads();
    }
    for (int i = warp; i < n_list; i += kPatchThreads / 32) {
      if (S.flag[i]) continue;                               // (warp-uniform)
      const float reach_w = S.reach[i];
      const float4 wq = S.wbox[i];
      const WarpBox wrec = {wq.x, wq.y, wq.z, wq.w};
      bool any = false;
      for (int k0 = 0; k0 < mc && !any; k0 += 32) {
        const int k = k0 + lane;
        any = __any_sync(0xffffffffu, (k < mc) && (S.cm[k] <= reach_w) && may_hit(wrec, S.box[k]));
      }
      if (any && lane == 0) S.flag[i] = 1;
      __syncwarp();
    }
  }
  __syncthreads();
}

// The flagged warps go to the batch-wide queue of enc_pass2_apply_kernel: they cluster in a few CTAs (the coarse levels
// meet every GT), and each costs a chain of dependent loads, so they are spread over the whole GPU
DAN_D void enqueue_flagged(const EncArgs& A, int b, int n_list, const FindSmem& S) {
  const int tid = threadIdx.x, lane = tid & 31;
  const bool flagged = tid < n_list && S.flag[tid] != 0;
  const unsigned fm = __ballot_sync(0xffffffffu, flagged);
  if (fm != 0u) {
    int base = 0;
    if (lane == 0) base = atomicAdd(A.queue_n, __popc(fm));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (flagged) A.queue[base + __popc(fm & ((1u << lane) - 1u))] = make_int2(b, S.list[tid]);
  }
}

// first and second level of pass 2, one CTA per (image, 128 warps of pass 1)
template <bool MINING>
__global__ void __launch_bounds__(kPatchThreads) enc_pass2_find_kernel(const EncArgs A) {
  __shared__ int s_list[kPatchThreads];
  __shared__ float s_reach[kPatchThreads];
  __shared__ float4 s_wbox[kPatchThreads];
  __shared__ int s_flag[kPatchThreads];
  __shared__ float4 s_box[kPatchGt];
  __shared__ float s_cm[kPatchGt];
  __shared__ int s_n;
  __shared__ float s_cmin[kPatchThreads / 32];
  __shared__ int s_wide[kPatchThreads / 32];
  const FindSmem S = {s_list, s_reach, s_wbox, s_flag, s_box, s_cm, s_n, s_cmin, s_wide};
  const int b = blockIdx.x;
  const ImageGt ig = image_gt<false>(A, b);
  // the usual case: all GT boxes and column maxima of the image fit the staging arrays and stay there
  const bool staged = ig.m_eff <= kPatchGt;
  float cmin;
  bool wide;
  summarize_columns<MINING>(A, ig, staged, S, cmin, wide);
  const int n_list = list_reaching_warps<MINING>(A, b, cmin, wide, S);
  if (n_list == 0) return;                                   // (CTA-uniform)
  if (!wide) flag_box_hits(A, ig, staged, n_list, S);
  enqueue_flagged(A, b, n_list, S);
}

// third level of pass 2: one warp per queued (image, warp of pass 1): load the anchors, evaluate the GTs the warp can
// reach, and if an anchor really ties with (mining) / is claimed by (dual) a GT, evaluate the full row again - the row
// maximum decides what stage 1 had written - and rewrite the outputs of the anchors whose match changed.
template <bool MINING>
__global__ void __launch_bounds__(kPatchThreads) enc_pass2_apply_kernel(const EncArgs A) {
  const int lane = threadIdx.x & 31;
  const int nwarps = (A.n + 31) >> 5;
  const bool need_haspos = !MINING && !A.gt_max_first;
  const int total = *A.queue_n;
  const int wstride = gridDim.x * (kPatchThreads / 32);
  for (int e = blockIdx.x * (kPatchThreads / 32) + (threadIdx.x >> 5); e < total; e += wstride) {
    const int2 q = A.queue[e];
    const int b = q.x;
    const ImageGt ig = image_gt<false>(A, b);
    const int a = warp_anchor(A, q.y, lane);
    const bool valid = a < A.n;
    const float wb = A.wbest[(int64_t)b * nwarps + q.y];
    const float reach_w = MINING ? fadd(wb, 2.f * FLT_EPSILON) : wb;
    AnchorBox ab = {};
    bool active = false;
    if (valid) {
      ab = load_anchor(A, a);
      active = (A.mask == nullptr) || (A.mask[a] != 0);
    }
    const WarpBox wbx = warp_bbox(active, ab);
    // the GTs the warp can reach: does any anchor really tie with / get claimed by one?
    bool tie = false;
    walk_gts<MINING>(A, ig, lane, active, ab,
                     [&](bool widek, float cmk, float4 gk) { return widek || (cmk <= reach_w && may_hit(wbx, gk)); },
                     [&](int kk, float ov, float cm) {
                       if (MINING) tie |= fabsf(fsub(ov, cm)) < FLT_EPSILON;
                       else tie |= (ov == cm) && (!need_haspos || A.haspos[ig.slot0 + kk] == 0);
                     });
    if (!__any_sync(0xffffffffu, tie && valid)) continue;
    // the full row again, then the patch
    RowState s;
    walk_gts<MINING>(A, ig, lane, active, ab, [&](bool widek, float, float4 gk) { return may_hit(wbx, gk) || widek; },
                     [&](int kk, float ov, float cm) {
                       row_update<MINING>(s, kk, ov, cm, !need_haspos || A.haspos[ig.slot0 + kk] == 0);
                     });
    if (!valid) continue;
    const int match1 = stage1_match<MINING>(A, s.best, s.best_gt);
    float score;
    const int match = stage2_match<MINING>(A, s, score);
    if (MINING && match != match1) {
      if (match1 >= 0) atomicSub(A.cnt + ig.slot0 + match1, 1);
      atomicAdd(A.cnt + ig.slot0 + match, 1);
    }
    if (match != match1 || score != s.best)
      write_positive(A, (int64_t)b * A.n + a, ab, gt_box(A, ig, match), score, match);
  }
}

// ---------------------------------------------------------------------------
// pass 3: stage 3 "hard face compensation", small_mining_match.cc:199-222.
//
// The reference walks the GTs in ascending order; a GT j that is short of min_match takes its best still-unmatched
// anchors with overlap > stop_positive_thres, so GT j sees what the GTs before it took.  That order dependence only
// exists between GTs that share a candidate anchor.  One CTA per image; the needy GTs are handled in WINDOWS of up to
// kP3Window consecutive needy GTs, a warp per GT:
//     sel_j = the `need_j` best candidates of j that are not selected by a needy GT before j
// is iterated from "nothing is blocked" until no GT's blocked set changes.  The lowest GT of the window is never
// blocked, so it is final after the first round, the next one after the second, ...: the fixed point is unique and is
// the reference's sequential result; the number of rounds is the longest chain of GTs that actually compete for an
// anchor (faces are mostly disjoint: two rounds, the second only confirms).  The selections of a window are then
// written to the outputs (by all warps) before the next window loads its candidates, which see them as matched.
// A GT whose candidate bucket overflowed (more than kBucketCap anchors above the stop threshold) is handled alone,
// by a rescan of all anchors of the image in index order, exactly like the reference's loop.
// Equal overlaps: pop order of a max-heap == descending key; only a tie that straddles the min_match cut depends
// on libstdc++'s heap layout, which is then reproduced exactly (heap_order.cuh).
// ---------------------------------------------------------------------------
template <bool DENSE>
DAN_D bool still_unmatched(const EncArgs& A, int64_t row) {
  if (DENSE) return reinterpret_cast<const volatile int32_t*>(A.match32)[row] < 0;
  return reinterpret_cast<const volatile int64_t*>(A.labels)[row] < 1;
}

template <bool DENSE>
DAN_D void apply_compensation(const EncArgs& A, const ImageGt& ig, int b, int a, int j, float ov) {
  const int64_t row = (int64_t)b * A.n + a;
  if (DENSE) {
    A.match32[row] = j;
    A.scores[row] = ov;
  } else {
    write_positive(A, row, load_anchor(A, a), gt_box(A, ig, j), ov, j);
  }
}

constexpr int kP3Threads = 512;
constexpr int kP3Warps = kP3Threads / 32;
constexpr int kP3Range = 1024;      // GTs scanned for neediness at a time
constexpr int kP3Window = 64;       // needy GTs resolved together
constexpr int kP3SelCap = 1024;     // selections of a window (half the hash table)
constexpr int kP3Hash = 2048;       // anchors selected in the current round -> lowest selecting GT (open addressing)

struct P3Hash {
  int* key;        // [kP3Hash], -1 = empty
  int* val;        // [kP3Hash]
};

DAN_D void p3_hash_put(const P3Hash& h, int a, int q) {
  unsigned i = ((unsigned)a * 2654435761u) & (kP3Hash - 1);
  while (true) {
    const int old = atomicCAS(&h.key[i], -1, a);
    if (old < 0 || old == a) {
      atomicMin(&h.val[i], q);
      return;
    }
    i = (i + 1) & (kP3Hash - 1);
  }
}

// lowest needy GT (window position) that selected anchor a in the last round, INT_MAX if none
DAN_D int p3_hash_get(const P3Hash& h, int a) {
  unsigned i = ((unsigned)a * 2654435761u) & (kP3Hash - 1);
  while (true) {
    const int k = h.key[i];
    if (k == a) return h.val[i];
    if (k < 0) return 0x7fffffff;
    i = (i + 1) & (kP3Hash - 1);
  }
}

// The `need` best of the c <= kBucketCap entries of `list` whose bit is set in `live`, as a bit mask over the entries.
// Executed by one full warp; sort_buf / heap: kBucketCap entries of scratch each (only used when a tie straddles the cut).
DAN_D unsigned long long select_from_bucket(const HeapItem* list, int c, unsigned long long live, int need, HeapItem* sort_buf,
                                            HeapItem* heap, unsigned char* sort_slot) {
  const int lane = threadIdx.x & 31;
  if (__popcll(live) <= need) return live;
  // one ranking pass: entry e is popped before the cut iff its whole tie group fits (ge <= need), after the cut iff
  // g >= need; a tie group with g < need < ge straddles the cut
  const bool l0 = (live >> lane) & 1ull, l1 = (live >> (lane + 32)) & 1ull;
  const float k0 = l0 ? list[lane].key : 0.f;
  const float k1 = l1 ? list[lane + 32].key : 0.f;
  int g0 = 0, ge0 = 0, g1 = 0, ge1 = 0;
  for (int e = 0; e < c; ++e) {
    if ((live >> e) & 1ull) {                              // warp-uniform
      const float v = list[e].key;
      g0 += (v > k0) ? 1 : 0;
      ge0 += (v >= k0) ? 1 : 0;
      g1 += (v > k1) ? 1 : 0;
      ge1 += (v >= k1) ? 1 : 0;
    }
  }
  const bool st = (l0 && g0 < need && ge0 > need) || (l1 && g1 < need && ge1 > need);
  if (!__any_sync(0xffffffffu, st)) {
    const unsigned lo = __ballot_sync(0xffffffffu, l0 && ge0 <= need);
    const unsigned hi = __ballot_sync(0xffffffffu, l1 && ge1 <= need);
    return ((unsigned long long)hi << 32) | lo;
  }
  // The exact path: every live entry is a member of the reference's heap, pushed in ascending anchor order
  // (small_mining_match.cc:204-209).  The bucket is unordered: each lane ranks its two entries by anchor index.
  const int id0 = l0 ? list[lane].id : 0x7fffffff, id1 = l1 ? list[lane + 32].id : 0x7fffffff;
  int r0 = 0, r1 = 0;
  for (int f = 0; f < c; ++f) {
    if ((live >> f) & 1ull) {
      const int idf = list[f].id;
      r0 += (idf < id0) ? 1 : 0;
      r1 += (idf < id1) ? 1 : 0;
    }
  }
  if (l0) { sort_buf[r0] = HeapItem{k0, id0}; sort_slot[r0] = (unsigned char)lane; }
  if (l1) { sort_buf[r1] = HeapItem{k1, id1}; sort_slot[r1] = (unsigned char)(lane + 32); }
  __syncwarp();
  unsigned long long sel = 0ull;
  if (lane == 0) {
    // HeapItem.id carries the position in sort_buf so that the popped items can be mapped back to bucket entries
    const int n = __popcll(live);
    int len = 0;
    for (int e = 0; e < n; ++e) heap_push(heap, len, HeapItem{sort_buf[e].key, e});
    for (int p = 0; p < need && len > 0; ++p) sel |= 1ull << sort_slot[heap_pop(heap, len).id];
  }
  __syncwarp();
  const unsigned lo = __shfl_sync(0xffffffffu, (unsigned)sel, 0), hi = __shfl_sync(0xffffffffu, (unsigned)(sel >> 32), 0);
  return ((unsigned long long)hi << 32) | lo;
}

// Overflowed bucket: all candidates of GT j in anchor order are in `list` (c entries, HBM); take the `need` best and
// apply them at once.  Executed by one full warp; sort_buf / heap: c entries of HBM scratch each.
template <bool DENSE>
DAN_D void compensate_from_spill(const EncArgs& A, const ImageGt& ig, int b, int j, int need, HeapItem* list, int c, HeapItem* heap) {
  const int lane = threadIdx.x & 31;
  if (c <= need) {
    for (int e = lane; e < c; e += 32) apply_compensation<DENSE>(A, ig, b, list[e].id, j, list[e].key);
    return;
  }
  int got = 0;
  bool straddle = false;
  while (got < need) {
    float lmax = 0.f;
    for (int e = lane; e < c; e += 32) lmax = fmaxf(lmax, list[e].key);
    const uint32_t wbits = __reduce_max_sync(0xffffffffu, __float_as_uint(lmax));
    if (wbits == 0u) break;
    const float wmax = __uint_as_float(wbits);
    int eq = 0;
    for (int e = lane; e < c; e += 32) eq += (list[e].key == wmax) ? 1 : 0;
    const int total = __reduce_add_sync(0xffffffffu, eq);
    if (got + total > need) { straddle = true; break; }
    for (int e = lane; e < c; e += 32) {
      if (list[e].key == wmax) {
        apply_compensation<DENSE>(A, ig, b, list[e].id, j, wmax);
        list[e].key = -wmax;     // taken; the value is kept for the exact path
      }
    }
    got += total;
    __syncwarp();
  }
  if (straddle) {
    __syncwarp();
    // every live or already taken entry was a member of the reference's heap, pushed in ascending anchor order (the
    // spill list is in that order)
    if (lane == 0) {
      int len = 0;
      for (int e = 0; e < c; ++e) heap_push(heap, len, HeapItem{fabsf(list[e].key), list[e].id});
      for (int p = 0; p < need && len > 0; ++p) {
        const HeapItem it = heap_pop(heap, len);
        apply_compensation<DENSE>(A, ig, b, it.id, j, it.key);     // re-applying an entry taken above is idempotent
      }
    }
  }
  __syncwarp();
}

struct P3Smem {
  HeapItem cand[kP3Window][kBucketCap];        // candidate buckets of the window (32 KB)
  HeapItem sort_buf[kP3Warps][kBucketCap];     // per-warp scratch of the exact tie path
  HeapItem heap[kP3Warps][kBucketCap];
  unsigned char sort_slot[kP3Warps][kBucketCap];
  int hash_key[kP3Hash];
  int hash_val[kP3Hash];
  unsigned long long alive[kP3Window];         // candidate still unmatched after stage 2 and the earlier windows
  unsigned long long blocked[kP3Window];       // ... but selected by an earlier GT of the window in the last round
  unsigned long long sel[kP3Window];
  int dirty[kP3Window];                        // blocked set changed in the last round: select again
  int needy_j[kP3Range], needy_need[kP3Range], needy_fill[kP3Range];
  int warp_cnt[kP3Warps];
};

// The GTs of [j0, j0 + kP3Range) short of min_match, ascending, with need and bucket fill into S.needy_*; their number
DAN_D int list_needy(const EncArgs& A, const ImageGt& ig, int j0, P3Smem& S) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int nneedy = 0;
  for (int jb = 0; jb < kP3Range && j0 + jb < ig.m_eff; jb += kP3Threads) {
    const int j = j0 + jb + tid;
    int need = 0, fill = 0;
    if (j < ig.m_eff) {
      need = A.min_match - A.cnt[ig.slot0 + j];
      fill = A.fill[ig.slot0 + j];
    }
    const unsigned m = __ballot_sync(0xffffffffu, need > 0);
    if (lane == 0) S.warp_cnt[warp] = __popc(m);
    __syncthreads();
    int before = nneedy;
    for (int w = 0; w < kP3Warps; ++w) {
      if (w < warp) before += S.warp_cnt[w];
      nneedy += S.warp_cnt[w];
    }
    if (need > 0) {
      const int pos = before + __popc(m & ((1u << lane) - 1u));
      S.needy_j[pos] = j;
      S.needy_need[pos] = need;
      S.needy_fill[pos] = fill;
    }
    __syncthreads();
  }
  return nneedy;
}

// Needy GT q, whose bucket overflowed, by one warp: rescan every anchor of the image in index order; everything before
// this GT is already in the outputs, the GT is alone in its "window", and its patches are applied at once
template <bool DENSE>
DAN_D void rescan_overflowed(const EncArgs& A, const ImageGt& ig, int b, int q, const P3Smem& S) {
  const int lane = threadIdx.x & 31;
  const int gj = S.needy_j[q];
  HeapItem* list = A.spill + (int64_t)b * 2 * A.n;   // then the heap of compensate_from_spill
  int c = 0;
  const float4 gb = DENSE ? make_float4(0.f, 0.f, 0.f, 0.f) : gt_box(A, ig, gj);
  const float garea = box_area(gb.x, gb.y, gb.z, gb.w);
  for (int a0 = 0; a0 < A.n; a0 += 32) {
    const int a = a0 + lane;
    bool ok = false;
    float ov = 0.f;
    if (a < A.n) {
      if (DENSE) {
        ov = A.overlaps[(int64_t)a * ig.m_eff + gj];
      } else if (A.mask == nullptr || A.mask[a] != 0) {
        const AnchorBox ab = load_anchor(A, a);
        bool hit;
        ov = pair_iou(ab.my0, ab.mx0, ab.my1, ab.mx1, ab.marea, gb.x, gb.y, gb.z, gb.w, garea, hit);
      }
      ok = (ov > A.stop) && still_unmatched<DENSE>(A, (int64_t)b * A.n + a);
    }
    const unsigned mm = __ballot_sync(0xffffffffu, ok);
    if (ok) list[c + __popc(mm & ((1u << lane) - 1u))] = HeapItem{ov, a};
    c += __popc(mm);
  }
  __threadfence_block();
  __syncwarp();
  compensate_from_spill<DENSE>(A, ig, b, gj, S.needy_need[q], list, c, list + A.n);
}

// the end q1 of the window [q0, q1): consecutive needy GTs with intact buckets, at most kP3Window, kP3SelCap selections
DAN_D int window_end(const P3Smem& S, int q0, int nneedy) {
  int q1 = q0, budget = 0;
  while (q1 < nneedy && q1 - q0 < kP3Window && S.needy_fill[q1] <= kBucketCap) {
    const int take = min(S.needy_need[q1], S.needy_fill[q1]);
    if (q1 > q0 && budget + take > kP3SelCap) break;
    budget += take;
    ++q1;
  }
  return q1;
}

// The candidates of the window's nq GTs, and which of them are still unmatched after stage 2 and after the windows
// before this one (already in HBM).  Ends with a barrier.
template <bool DENSE>
DAN_D void load_window(const EncArgs& A, const ImageGt& ig, int b, int q0, int nq, P3Smem& S) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int g = warp; g < nq; g += kP3Warps) {
    const int gj = S.needy_j[q0 + g], gfill = S.needy_fill[q0 + g];
    bool a0 = false, a1 = false;
    if (lane < gfill) {
      const HeapItem it = A.bucket[(int64_t)(ig.slot0 + gj) * kBucketCap + lane];
      S.cand[g][lane] = it;
      a0 = still_unmatched<DENSE>(A, (int64_t)b * A.n + it.id);
    }
    if (lane + 32 < gfill) {
      const HeapItem it = A.bucket[(int64_t)(ig.slot0 + gj) * kBucketCap + lane + 32];
      S.cand[g][lane + 32] = it;
      a1 = still_unmatched<DENSE>(A, (int64_t)b * A.n + it.id);
    }
    const unsigned lo = __ballot_sync(0xffffffffu, a0), hi = __ballot_sync(0xffffffffu, a1);
    if (lane == 0) {
      S.alive[g] = ((unsigned long long)hi << 32) | lo;
      S.blocked[g] = 0ull;
      S.dirty[g] = 1;
    }
  }
  __syncthreads();
}

// The fixed-point rounds of the window, until no blocked set changes; the selections are left in S.sel (CTA-uniform)
DAN_D void resolve_window(int q0, int nq, P3Smem& S) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const P3Hash hash{S.hash_key, S.hash_val};
  while (true) {
    for (int g = warp; g < nq; g += kP3Warps) {
      if (S.dirty[g] == 0) continue;                        // (warp-uniform: written by this warp in the last round)
      const unsigned long long live = S.alive[g] & ~S.blocked[g];
      const unsigned long long sel = select_from_bucket(S.cand[g], S.needy_fill[q0 + g], live, S.needy_need[q0 + g],
                                                        S.sort_buf[warp], S.heap[warp], S.sort_slot[warp]);
      if (lane == 0) S.sel[g] = sel;
    }
    for (int i = tid; i < kP3Hash; i += kP3Threads) { S.hash_key[i] = -1; S.hash_val[i] = 0x7fffffff; }
    __syncthreads();
    if (nq == 1) break;                                     // a lone GT has nobody to compete with
    for (int g = warp; g < nq; g += kP3Warps) {
      const unsigned long long sel = S.sel[g];
      if ((sel >> lane) & 1ull) p3_hash_put(hash, S.cand[g][lane].id, g);
      if ((sel >> (lane + 32)) & 1ull) p3_hash_put(hash, S.cand[g][lane + 32].id, g);
    }
    __syncthreads();
    bool changed = false;
    for (int g = warp; g < nq; g += kP3Warps) {
      const unsigned long long alive = S.alive[g];
      const bool b0 = ((alive >> lane) & 1ull) && p3_hash_get(hash, S.cand[g][lane].id) < g;
      const bool b1 = ((alive >> (lane + 32)) & 1ull) && p3_hash_get(hash, S.cand[g][lane + 32].id) < g;
      const unsigned lo = __ballot_sync(0xffffffffu, b0), hi = __ballot_sync(0xffffffffu, b1);
      const unsigned long long blocked = ((unsigned long long)hi << 32) | lo;
      const bool diff = blocked != S.blocked[g];
      changed |= diff;
      __syncwarp();
      if (lane == 0) {
        S.blocked[g] = blocked;
        S.dirty[g] = diff ? 1 : 0;
      }
    }
    if (!__syncthreads_or(changed ? 1 : 0)) break;
  }
}

// the window's selections go to the outputs (by all warps); ends with a barrier
template <bool DENSE>
DAN_D void apply_window(const EncArgs& A, const ImageGt& ig, int b, int q0, int nq, const P3Smem& S) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int g = warp; g < nq; g += kP3Warps) {
    const unsigned long long sel = S.sel[g];
    const int gj = S.needy_j[q0 + g];
    if ((sel >> lane) & 1ull) apply_compensation<DENSE>(A, ig, b, S.cand[g][lane].id, gj, S.cand[g][lane].key);
    if ((sel >> (lane + 32)) & 1ull) apply_compensation<DENSE>(A, ig, b, S.cand[g][lane + 32].id, gj, S.cand[g][lane + 32].key);
  }
  __syncthreads();
}

template <bool DENSE>
__global__ void __launch_bounds__(kP3Threads) enc_pass3_kernel(const EncArgs A) {
  extern __shared__ __align__(16) unsigned char p3_raw[];
  P3Smem& S = *reinterpret_cast<P3Smem*>(p3_raw);
  const int b = blockIdx.x;
  const ImageGt ig = image_gt<DENSE>(A, b);
  for (int j0 = 0; j0 < ig.m_eff; j0 += kP3Range) {
    const int nneedy = list_needy(A, ig, j0, S);
    int q0 = 0;
    while (q0 < nneedy) {                                    // (all decisions below are CTA-uniform)
      if (S.needy_fill[q0] > kBucketCap) {
        if ((threadIdx.x >> 5) == 0) rescan_overflowed<DENSE>(A, ig, b, q0, S);
        __syncthreads();
        q0 += 1;
        continue;
      }
      const int q1 = window_end(S, q0, nneedy);
      load_window<DENSE>(A, ig, b, q0, q1 - q0, S);
      resolve_window(q0, q1 - q0, S);
      apply_window<DENSE>(A, ig, b, q0, q1 - q0, S);
      q0 = q1;
    }
    __syncthreads();
  }
}

// M == 0 on the dense mining op: stage 1 leaves every anchor at (-2, lowest())
__global__ void fill_empty_match_kernel(int32_t* match, float* scores, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    match[i] = -2;
    scores[i] = -FLT_MAX;
  }
}

// the warp -> anchors table of the layout hint (warp_anchor): warps inside a hinted grid hold 8 x 4 tiles of cells
struct GridHint {
  int n;
  int start[DAN_MAX_GRIDS], w[DAN_MAX_GRIDS], h[DAN_MAX_GRIDS];
};

__global__ void __launch_bounds__(256) enc_warp_map_kernel(int2* map, int nwarps, const GridHint H) {
  const int wid = blockIdx.x * blockDim.x + threadIdx.x;
  if (wid >= nwarps) return;
  int2 m = make_int2(wid * 32, 8);
#pragma unroll
  for (int g = 0; g < DAN_MAX_GRIDS; ++g) {
    if (g < H.n) {
      const int wbeg = H.start[g] >> 5, wcnt = (H.w[g] * H.h[g]) >> 5;
      if (wid >= wbeg && wid < wbeg + wcnt) {
        const int j = wid - wbeg, tiles_per_band = H.w[g] >> 3;
        const int band = j / tiles_per_band, tcol = j - band * tiles_per_band;
        m = make_int2(H.start[g] + band * 4 * H.w[g] + tcol * 8, H.w[g]);
      }
    }
  }
  map[wid] = m;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct WsLayout {
  size_t colmax, cnt, haspos, fill, queue_n, zero_bytes, bucket, spill, wbest, wbox, queue, warp_map, total;
};

static WsLayout ws_layout(int64_t n, int64_t batch, int64_t slots) {
  WsLayout w;
  size_t off = 0;
  w.colmax = off; off += align_up(slots * 4, 256);
  w.cnt = off;    off += align_up(slots * 4, 256);
  w.haspos = off; off += align_up(slots * 4, 256);
  w.fill = off;   off += align_up(slots * 4, 256);
  w.queue_n = off; off += 256;
  w.zero_bytes = off;
  w.bucket = off; off += align_up(slots * kBucketCap * sizeof(HeapItem), 256);
  w.spill = off;  off += align_up(batch * 2 * n * sizeof(HeapItem), 256);
  w.wbest = off;  off += align_up(batch * ((n + 31) / 32) * 4, 256);
  w.wbox = off;   off += align_up(((n + 31) / 32) * 16, 256);
  w.queue = off;  off += align_up(batch * ((n + 31) / 32) * 8, 256);
  w.warp_map = off; off += align_up(((n + 31) / 32) * 8, 256);
  w.total = off;
  return w;
}

static int check_mining_attrs(float neg_low, float neg_high, float pos, int min_match, float stop) {
  // small_mining_match.cc:292-305
  DAN_REQUIRE(neg_low >= 0.f && neg_low < 1.f, DAN_ERR_INVALID_ARGUMENT, "Need Attr 1 > negative_low_thres >= 0, got %g", neg_low);
  DAN_REQUIRE(neg_high > neg_low && neg_high < 1.f, DAN_ERR_INVALID_ARGUMENT,
              "Need Attr 1 > negative_high_thres > negative_low_thres, got %g", neg_high);
  DAN_REQUIRE(pos >= neg_high && pos < 1.f, DAN_ERR_INVALID_ARGUMENT, "Need Attr 1 > positive_thres >= negative_high_thres, got %g", pos);
  DAN_REQUIRE(stop >= 0.f && stop < 1.f, DAN_ERR_INVALID_ARGUMENT, "Need Attr 1 > stop_positive_thres >= 0., got %g", stop);
  DAN_REQUIRE(min_match >= 1, DAN_ERR_INVALID_ARGUMENT, "Need Attr min_match >= 1, got %d", min_match);
  return DAN_OK;
}

static void bind_workspace(EncArgs& A, void* workspace, const WsLayout& w) {
  char* base = static_cast<char*>(workspace);
  A.colmax = reinterpret_cast<uint32_t*>(base + w.colmax);
  A.cnt = reinterpret_cast<int32_t*>(base + w.cnt);
  A.haspos = reinterpret_cast<int32_t*>(base + w.haspos);
  A.fill = reinterpret_cast<int32_t*>(base + w.fill);
  A.bucket = reinterpret_cast<HeapItem*>(base + w.bucket);
  A.spill = reinterpret_cast<HeapItem*>(base + w.spill);
  A.wbest = reinterpret_cast<float*>(base + w.wbest);
  A.wbox = reinterpret_cast<float4*>(base + w.wbox);
  A.queue_n = reinterpret_cast<int32_t*>(base + w.queue_n);
  A.queue = reinterpret_cast<int2*>(base + w.queue);
}

// Fused pass 1.  fine_chunks: the leading chunks of kFusedThreads anchors that lie on fine pyramid levels; their CTAs
// walk kFineImages images each.
template <bool NEED_ROW, bool MINING, bool TILED>
static void launch_pass1(const EncArgs& A, int batch, int fine_chunks, cudaStream_t st) {
  const int coarse_chunks = (A.n + kFusedThreads - 1) / kFusedThreads - fine_chunks;
  const int grid = pass1_grid(batch, coarse_chunks, fine_chunks);
  enc_pass1_fused_kernel<NEED_ROW, MINING, TILED><<<grid, kFusedThreads, 0, st>>>(A, batch, coarse_chunks);
}

// Pass 3 (mining only) of either path, one CTA per image.
template <bool DENSE>
static int launch_pass3(const EncArgs& A, int batch, cudaStream_t st) {
  // (the attribute belongs to the (function, device) pair: set on every call, like the other big-smem kernels)
  DAN_CUDA(cudaFuncSetAttribute(enc_pass3_kernel<DENSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(P3Smem)));
  enc_pass3_kernel<DENSE><<<batch, kP3Threads, sizeof(P3Smem), st>>>(A);
  DAN_LAUNCH_CHECK("enc_pass3_kernel");
  return DAN_OK;
}

// The fused path.  ev (optional, 4 events): recorded before pass 1 and after each pass, for the profile entry point
static int run_fused(const EncArgs& A, bool mining, bool need_row, int batch, int fine_chunks, cudaStream_t st, cudaEvent_t* ev) {
  if (ev) DAN_CUDA(cudaEventRecord(ev[0], st));
  if (A.warp_map != nullptr) {
    if (mining) launch_pass1<false, true, true>(A, batch, fine_chunks, st);
    else if (need_row) launch_pass1<true, false, true>(A, batch, fine_chunks, st);
    else launch_pass1<false, false, true>(A, batch, fine_chunks, st);
  } else {
    if (mining) launch_pass1<false, true, false>(A, batch, fine_chunks, st);
    else if (need_row) launch_pass1<true, false, false>(A, batch, fine_chunks, st);
    else launch_pass1<false, false, false>(A, batch, fine_chunks, st);
  }
  DAN_LAUNCH_CHECK("enc_pass1_kernel");
  if (ev) DAN_CUDA(cudaEventRecord(ev[1], st));
  const dim3 pgrid(batch, ((A.n + 31) / 32 + kPatchThreads - 1) / kPatchThreads);
  const int agrid = 148 * 4;                           // the queue is walked by a fixed grid (its length is only known on the device)
  if (mining) {
    enc_pass2_find_kernel<true><<<pgrid, kPatchThreads, 0, st>>>(A);
    enc_pass2_apply_kernel<true><<<agrid, kPatchThreads, 0, st>>>(A);
  } else {
    enc_pass2_find_kernel<false><<<pgrid, kPatchThreads, 0, st>>>(A);
    enc_pass2_apply_kernel<false><<<agrid, kPatchThreads, 0, st>>>(A);
  }
  DAN_LAUNCH_CHECK("enc_pass2_kernel");
  if (ev) DAN_CUDA(cudaEventRecord(ev[2], st));
  if (mining) {
    const int rc = launch_pass3<false>(A, batch, st);
    if (rc != DAN_OK) return rc;
  }
  if (ev) DAN_CUDA(cudaEventRecord(ev[3], st));
  return DAN_OK;
}

// The dense path, for both dense entry points: A holds the matrix, the matcher's parameters and the outputs; this binds
// the workspace and launches the passes on the one image.
static int run_dense(EncArgs A, bool mining, bool need_row, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const WsLayout w = ws_layout(A.n, 1, (int64_t)A.m_dense + 1);
  DAN_REQUIRE(workspace != nullptr && workspace_bytes >= w.total, DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu",
              w.total, workspace_bytes);
  bind_workspace(A, workspace, w);
  DAN_CUDA(cudaMemsetAsync(workspace, 0, w.zero_bytes, st));
  const int grid = (A.n + kEncThreads - 1) / kEncThreads;
  if (need_row) dense_pass1_kernel<true><<<grid, kEncThreads, 0, st>>>(A);
  else dense_pass1_kernel<false><<<grid, kEncThreads, 0, st>>>(A);
  DAN_LAUNCH_CHECK("dense_pass1_kernel");
  if (mining) dense_pass2_kernel<true><<<grid, kEncThreads, 0, st>>>(A);
  else dense_pass2_kernel<false><<<grid, kEncThreads, 0, st>>>(A);
  DAN_LAUNCH_CHECK("dense_pass2_kernel");
  return mining ? launch_pass3<true>(A, 1, st) : DAN_OK;
}

// CUDA-event timing of a launch sequence (profile entry points only): creates n events, runs fn(ev), synchronises
// on the last one and writes the n-1 intervals in milliseconds.
template <typename Fn>
static int timed_sequence(int n_events, float* h_ms, Fn fn) {
  cudaEvent_t ev[8];
  for (int i = 0; i < n_events; ++i) DAN_CUDA(cudaEventCreate(&ev[i]));
  int rc = fn(ev);
  if (rc == DAN_OK) {
    cudaError_t e = cudaEventSynchronize(ev[n_events - 1]);
    if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventSynchronize");
  }
  if (rc == DAN_OK)
    for (int i = 0; i + 1 < n_events; ++i) cudaEventElapsedTime(&h_ms[i], ev[i], ev[i + 1]);
  for (int i = 0; i < n_events; ++i) cudaEventDestroy(ev[i]);
  return rc;
}

}  // namespace dan

using namespace dan;

extern "C" {

size_t dan_match_workspace_bytes(int32_t num_anchors, int32_t num_gt) {
  if (num_anchors < 0 || num_gt < 0) return 0;
  return ws_layout(num_anchors, 1, (int64_t)num_gt + 1).total;
}

size_t dan_encode_workspace_bytes(int32_t num_anchors, int32_t batch, int32_t total_gt) {
  if (num_anchors < 0 || batch < 0 || total_gt < 0) return 0;
  return ws_layout(num_anchors, batch, (int64_t)total_gt + batch).total;
}

int dan_small_mining_match(const float* overlaps, int32_t num_anchors, int32_t num_gt, float negative_low_thres,
                           float negative_high_thres, float positive_thres, int32_t min_match, float stop_positive_thres,
                           int32_t* out_match_indices, float* out_match_scores, void* workspace, size_t workspace_bytes,
                           void* stream) {
  int rc = check_mining_attrs(negative_low_thres, negative_high_thres, positive_thres, min_match, stop_positive_thres);
  if (rc != DAN_OK) return rc;
  DAN_REQUIRE(num_anchors >= 0 && num_gt >= 0, DAN_ERR_INVALID_ARGUMENT, "inputs must be in 'num_anchors x num_ground_truth' format.");
  if (num_anchors == 0) return DAN_OK;
  DAN_REQUIRE(out_match_indices && out_match_scores, DAN_ERR_INVALID_ARGUMENT, "NULL output");
  cudaStream_t st = (cudaStream_t)stream;
  if (num_gt == 0) {
    fill_empty_match_kernel<<<(num_anchors + 255) / 256, 256, 0, st>>>(out_match_indices, out_match_scores, num_anchors);
    DAN_LAUNCH_CHECK("fill_empty_match_kernel");
    return DAN_OK;
  }
  DAN_REQUIRE(overlaps != nullptr, DAN_ERR_INVALID_ARGUMENT, "NULL overlaps");
  EncArgs A = {};
  A.n = num_anchors;
  A.overlaps = overlaps;
  A.m_dense = num_gt;
  A.low = negative_high_thres;
  A.high = positive_thres;
  A.neg_low = negative_low_thres;
  A.stop = stop_positive_thres;
  A.min_match = min_match;
  A.gt_max_first = 1;
  A.ignore_between = 1;
  A.match32 = out_match_indices;
  A.scores = out_match_scores;
  return run_dense(A, true, false, workspace, workspace_bytes, st);
}

int dan_dual_max_match(const float* overlaps, int32_t num_anchors, int32_t num_gt, float low_thres, float high_thres,
                       int32_t ignore_between, int32_t gt_max_first, int64_t* out_match_indices, float* out_match_scores,
                       void* workspace, size_t workspace_bytes, void* stream) {
  DAN_REQUIRE(num_anchors >= 0 && num_gt >= 1, DAN_ERR_INVALID_ARGUMENT,
              "do_dual_max_match needs overlap_matrix [num_anchors, num_gt>=1] (tf.argmax over an empty axis is an error)");
  if (num_anchors == 0) return DAN_OK;
  DAN_REQUIRE(overlaps && out_match_indices && out_match_scores, DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  EncArgs A = {};
  A.n = num_anchors;
  A.overlaps = overlaps;
  A.m_dense = num_gt;
  A.low = low_thres;
  A.high = high_thres;
  A.ignore_between = ignore_between ? 1 : 0;
  A.gt_max_first = gt_max_first ? 1 : 0;
  A.match64 = out_match_indices;
  A.scores = out_match_scores;
  return run_dense(A, false, !gt_max_first, workspace, workspace_bytes, (cudaStream_t)stream);
}

static int encode_core(const dan_encode_params* p, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                       const float* a_xmax, const uint8_t* inside_mask, int32_t num_anchors, const float* gt_boxes,
                       const int32_t* gt_offsets, int32_t batch, int32_t total_gt, float* out_targets, int64_t* out_labels,
                       float* out_scores, float* out_matched_gt, int32_t* out_match, void* workspace, size_t workspace_bytes,
                       void* stream, cudaEvent_t* ev) {
  DAN_REQUIRE(p != nullptr, DAN_ERR_INVALID_ARGUMENT, "params is NULL");
  DAN_REQUIRE(p->matcher == DAN_MATCH_DUAL || p->matcher == DAN_MATCH_MINING, DAN_ERR_INVALID_ARGUMENT, "unknown matcher %d", p->matcher);
  DAN_REQUIRE(num_anchors >= 0 && batch >= 0 && total_gt >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  DAN_REQUIRE(batch <= 65535, DAN_ERR_UNSUPPORTED, "batch > 65535");
  DAN_REQUIRE(num_anchors <= 4000000, DAN_ERR_UNSUPPORTED, "more than 4,000,000 anchors per image");
  const bool mining = p->matcher == DAN_MATCH_MINING;
  if (mining) {
    int rc = check_mining_attrs(p->negative_low_thres, p->ignore_threshold, p->positive_threshold, p->min_match, p->stop_positive_thres);
    if (rc != DAN_OK) return rc;
  }
  DAN_REQUIRE(p->pa_scale >= 0.f, DAN_ERR_INVALID_ARGUMENT, "pa_scale must be >= 0");
  if (num_anchors == 0 || batch == 0) return DAN_OK;
  DAN_REQUIRE(a_ymin && a_xmin && a_ymax && a_xmax && gt_offsets && out_targets && out_labels && out_scores, DAN_ERR_INVALID_ARGUMENT,
              "NULL pointer");
  DAN_REQUIRE(total_gt == 0 || gt_boxes != nullptr, DAN_ERR_INVALID_ARGUMENT, "gt_boxes is NULL");
  DAN_REQUIRE(aligned16(gt_boxes) && aligned16(out_targets) && aligned16(out_matched_gt), DAN_ERR_INVALID_ARGUMENT,
              "gt_boxes / out_targets / out_matched_gt must be 16-byte aligned");
  const WsLayout w = ws_layout(num_anchors, batch, (int64_t)total_gt + batch);
  DAN_REQUIRE(workspace != nullptr && workspace_bytes >= w.total, DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu",
              w.total, workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  EncArgs A = {};
  A.ay0 = a_ymin; A.ax0 = a_xmin; A.ay1 = a_ymax; A.ax1 = a_xmax;
  A.mask = inside_mask;
  A.n = num_anchors;
  A.gt = reinterpret_cast<const float4*>(gt_boxes);
  A.gt_off = gt_offsets;
  A.low = p->ignore_threshold;
  A.high = p->positive_threshold;
  A.neg_low = p->negative_low_thres;
  A.stop = p->stop_positive_thres;
  A.min_match = p->min_match;
  A.ignore_between = mining ? 1 : (p->ignore_between ? 1 : 0);
  A.gt_max_first = mining ? 1 : (p->gt_max_first ? 1 : 0);
  A.ps0 = p->prior_scaling[0]; A.ps1 = p->prior_scaling[1]; A.ps2 = p->prior_scaling[2]; A.ps3 = p->prior_scaling[3];
  A.pa_scale = p->pa_scale;
  A.debug = p->debug;
  A.targets = reinterpret_cast<float4*>(out_targets);
  A.labels = out_labels;
  A.scores = out_scores;
  A.matched = reinterpret_cast<float4*>(out_matched_gt);
  A.match32 = out_match;
  bind_workspace(A, workspace, w);
  DAN_CUDA(cudaMemsetAsync(workspace, 0, w.zero_bytes, st));
  int fine_end = 0;
  if (p->num_grids > 0) {
    // layout hint: levels of one anchor per cell, row major.  The tiles need whole warps and whole 8 x 4 blocks.
    DAN_REQUIRE(p->num_grids <= DAN_MAX_GRIDS, DAN_ERR_INVALID_ARGUMENT, "num_grids must be in [0, %d], got %d", DAN_MAX_GRIDS, p->num_grids);
    GridHint H = {};
    H.n = p->num_grids;
    int64_t prev_end = 0;
    for (int g = 0; g < H.n; ++g) {
      const int64_t gs = p->grid_start[g], gw = p->grid_w[g], gh = p->grid_h[g];
      DAN_REQUIRE(gs >= prev_end && (gs & 31) == 0 && gw > 0 && gh > 0 && (gw & 7) == 0 && (gh & 3) == 0 && gs + gw * gh <= num_anchors,
                  DAN_ERR_INVALID_ARGUMENT,
                  "grid %d (start %lld, %lld x %lld): needs start %% 32 == 0, width %% 8 == 0, height %% 4 == 0, ascending, inside the anchors",
                  g, (long long)gs, (long long)gw, (long long)gh);
      H.start[g] = (int)gs; H.w[g] = (int)gw; H.h[g] = (int)gh;
      prev_end = gs + gw * gh;
    }
    // the fine levels of pass 1: the hinted grids of at least kFineMinCells cells from anchor 0 on
    for (int g = 0; g < H.n && H.start[g] == fine_end && H.w[g] * H.h[g] >= kFineMinCells; ++g) fine_end += H.w[g] * H.h[g];
    int2* map = reinterpret_cast<int2*>(static_cast<char*>(workspace) + w.warp_map);
    const int nwarps = (num_anchors + 31) / 32;
    enc_warp_map_kernel<<<(nwarps + 255) / 256, 256, 0, st>>>(map, nwarps, H);
    DAN_LAUNCH_CHECK("enc_warp_map_kernel");
    A.warp_map = map;
  }
  return run_fused(A, mining, !mining && !A.gt_max_first, batch, fine_end / kFusedThreads, st, ev);
}

int dan_encode_batch(const dan_encode_params* p, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                     const float* a_xmax, const uint8_t* inside_mask, int32_t num_anchors, const float* gt_boxes,
                     const int32_t* gt_offsets, int32_t batch, int32_t total_gt, float* out_targets, int64_t* out_labels,
                     float* out_scores, float* out_matched_gt, int32_t* out_match, void* workspace, size_t workspace_bytes,
                     void* stream) {
  return encode_core(p, a_ymin, a_xmin, a_ymax, a_xmax, inside_mask, num_anchors, gt_boxes, gt_offsets, batch, total_gt, out_targets,
                     out_labels, out_scores, out_matched_gt, out_match, workspace, workspace_bytes, stream, nullptr);
}

int dan_encode_batch_profile(const dan_encode_params* p, const float* a_ymin, const float* a_xmin, const float* a_ymax,
                             const float* a_xmax, const uint8_t* inside_mask, int32_t num_anchors, const float* gt_boxes,
                             const int32_t* gt_offsets, int32_t batch, int32_t total_gt, float* out_targets, int64_t* out_labels,
                             float* out_scores, float* out_matched_gt, int32_t* out_match, void* workspace, size_t workspace_bytes,
                             void* stream, float* h_pass_ms) {
  DAN_REQUIRE(h_pass_ms != nullptr, DAN_ERR_INVALID_ARGUMENT, "h_pass_ms is NULL");
  h_pass_ms[0] = h_pass_ms[1] = h_pass_ms[2] = 0.f;
  return timed_sequence(4, h_pass_ms, [&](cudaEvent_t* ev) {
    return encode_core(p, a_ymin, a_xmin, a_ymax, a_xmax, inside_mask, num_anchors, gt_boxes, gt_offsets, batch, total_gt, out_targets,
                       out_labels, out_scores, out_matched_gt, out_match, workspace, workspace_bytes, stream, ev);
  });
}

}  // extern "C"
