// SURVEY.md 8(f2): the evaluation merge the reference's scripts actually use.
//
//   detect_face (eval_sfd.py:95-114, after net.run): boxes / shrink, columns (xmin, ymin, xmax, ymax, score), keep the
//       top min(N - 1, 1.5 * max_per_image) detections by descending score.
//   bbox_vote   (eval_sfd.py:170-210 = eval_dan.py:201-241): a numpy while-loop that repeatedly takes the best remaining
//       detection, removes everything with IoU >= thr to it (+1 pixel convention) and replaces the group by its
//       score-weighted mean; groups of one are dropped; the first max_per_image groups are returned.
//
// bbox_vote without the shrinking array: in descending score order, a detection that no earlier HEAD overlaps with
// IoU >= thr is a head, every other one joins the FIRST head that overlaps it (pinned against the reference's own
// function, tests/golden/vote_reference.npz).  One 1024-thread CTA per image keeps the sorted detections in shared
// memory (vote_plan); bbox_vote_kernel runs these steps (DESIGN.md §4e):
//   1.  sort_and_gather  64-bit keys (score bits << 32 | index), bitonic sort (sort.cuh); equal scores: higher index
//                        first, i.e. numpy's argsort(kind="stable")[::-1] (the reference's default quicksort leaves ties
//                        unspecified).  Thread t keeps the score ranks t, t + 1024, ... in registers (VoteRegs).
//       init_stripes     broad phase of step 2: a stripe grid over the detections' extent, each detection's stripes
//   2.  heads in score order, 32 candidates per round (five barriers each):
//   2a. list_candidates  warp 0 lists the next (up to) 32 unassigned positions = the round's candidates
//   2b. candidate_masks  the candidates against each other: 32x32 pair tests -> one bit mask per candidate
//   2c. resolve_heads    which candidates are heads, which join an earlier head of the round; the heads' stripes
//   2d. join_heads       every thread tests its own live detections against the round's heads
//   3.  number_groups    the groups with >= 2 members are numbered in head order (block scan)
//       write_groups     one warp walks the members of a group in score order: box sums accumulate sequentially like
//                        np.sum(axis=0), the score sum reproduces numpy's pairwise summation (8 interleaved accumulators
//                        up to 128 elements, recursive halving beyond), all in fp32 without FMA
//       write_assign     the head of every detection (optional output)
// bbox_vote_large_kernel runs the same steps for images of more than kSortCap detections (up to kVoteLargeCap): the
// detections live in the workspace (vote_large_plan), the alive set is a bitmap in shared memory, and positions and counts
// are int32.  The steps that both kernels share are templated on the image's layout (VoteImage, VoteImageLarge).
#include "common.cuh"

namespace dan {

#include "sort.cuh"

namespace {

constexpr uint16_t kFree = 0xFFFFu;      // not assigned yet
constexpr uint16_t kGone = 0xFFFEu;      // a head that does not even match itself (NaN IoU): deleted alone
constexpr int kVoteLargeCap = 1 << 20;   // detections per image of bbox_vote_large_kernel (its alive bitmap: 128 KB)

// Dynamic shared memory of one bbox_vote_kernel launch (vote_plan).  Offsets are in bytes from the start of the dynamic
// shared memory, where the sort keys start; the boxes overwrite the keys once they are consumed.
struct VotePlan {
  int score;                  // [cap] float, after max(keys, boxes)
  int assign;                 // [cap] uint16: head position of each detection (kFree, kGone)
  int count;                  // [cap] uint16: members of the group headed there (4-byte aligned: two per atomic word)
  int qlist;                  // [cap] uint16: head position of group q
  int smem;                   // dynamic shared memory of the launch
};

constexpr int kVoteSmemMax = 221 * 1024;  // dynamic part (the kernel has ~1 KB of static shared memory)

static VotePlan vote_plan(int cap) {
  int pad = 256;                          // the sort pads the keys to a power of two (here at least 256)
  while (pad < cap) pad <<= 1;
  const int u16 = (int)align_up((size_t)cap * 2, 16);
  VotePlan p;
  p.score = pad * 8 > cap * 16 ? pad * 8 : cap * 16;
  p.assign = p.score + cap * 4;
  p.count = p.assign + u16;
  p.qlist = p.count + u16;
  p.smem = p.qlist + u16;
  return p;
}

struct VoteArgs {
  const float* det;           // [B, cap, 5] (xmin, ymin, xmax, ymax, score)
  const int32_t* counts;      // [B] valid rows of each image (NULL: all cap rows)
  int cap;
  float thr;
  int max_out;
  VotePlan plan;              // shared-memory plan of the launch
  float* out;                 // [B, max_out, 5] zero padded
  int32_t* out_count;         // [B]
  int32_t* out_order;         // [B, cap] optional: sorted position -> input row
  int32_t* out_assign;        // [B, cap] optional: sorted position -> head position (-2: deleted head)
};

// +1 pixel convention, float32, the operation order of eval_sfd.py:176-185
DAN_D float vote_area(const float4& b) { return fmul(fadd(fsub(b.z, b.x), 1.f), fadd(fsub(b.w, b.y), 1.f)); }

DAN_D bool vote_overlaps(const float4& h, float area_h, const float4& b, float thr) {
  const float xx1 = fmaxf(h.x, b.x), yy1 = fmaxf(h.y, b.y), xx2 = fminf(h.z, b.z), yy2 = fminf(h.w, b.w);
  const float w = fmaxf(0.f, fadd(fsub(xx2, xx1), 1.f)), hh = fmaxf(0.f, fadd(fsub(yy2, yy1), 1.f));
  const float inter = fmul(w, hh);
  const float o = fdiv(inter, fsub(fadd(area_h, vote_area(b)), inter));
  return o >= thr;                      // false for NaN, like numpy
}

// Broad phase of the head search: the extent of the detections (+1 pixel on the far sides, the overlap convention above)
// is cut into 32 stripes per axis.  A detection touches a contiguous range of stripes per axis, packed into 20 bits
// (xlo | xhi << 5 | ylo << 10 | yhi << 15); kEverywhere marks a box that must meet every head in the exact test
// (non-finite coordinates, a threshold <= 0 for which disjoint boxes "overlap" too).  vote_overlaps() can only be true
// for thr > 0 when the intersection has positive width and height, i.e. when [x1, x2 + 1] and [y1, y2 + 1] of the two
// boxes intersect - and intervals that intersect share a stripe, because the stripe of a coordinate is a monotone
// function of it.
constexpr uint32_t kEverywhere = 1u << 20;

struct VoteStripes {
  float xlo, xinv, ylo, yinv;
  bool all;
  DAN_D int stripe(float v, float lo, float inv) const { return min(max((int)fmul(fsub(v, lo), inv), 0), 31); }
  DAN_D uint32_t range(const float4& b) const {
    if (all || !(fabsf(b.x) < 1e30f && fabsf(b.y) < 1e30f && fabsf(b.z) < 1e30f && fabsf(b.w) < 1e30f)) return kEverywhere;
    return (uint32_t)stripe(b.x, xlo, xinv) | ((uint32_t)stripe(fadd(b.z, 1.f), xlo, xinv) << 5) |
           ((uint32_t)stripe(b.y, ylo, yinv) << 10) | ((uint32_t)stripe(fadd(b.w, 1.f), ylo, yinv) << 15);
  }
};

// bit s set for every stripe s in [lo, hi]
DAN_D uint32_t stripe_span(uint32_t lo, uint32_t hi) { return ((2u << hi) - 1u) & ~((1u << lo) - 1u); }

// walks the members of one group in score order.  One WARP walks one group, all lanes in lock step (every lane holds
// the same sums): the search for the next member looks at 32 positions at a time (one ballot) instead of one.
template <class Pos> struct MemberIterT {
  const Pos* assign;
  const float4* box;
  const float* score;
  int n;
  Pos head;
  int pos;                              // next window of 32 positions to look at
  int base = 0;                         // first position of the window `pending` describes
  unsigned pending = 0u;                // members of the current window that have not been consumed
  float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;            // sequential sums of box * score (np.sum(axis=0))
  float mx = -INFINITY;                                     // running max score
  // the head is the first member of its own group (a deleted head has count 0)
  DAN_D MemberIterT(const Pos* assign_, const float4* box_, const float* score_, int n_, Pos head_)
      : assign(assign_), box(box_), score(score_), n(n_), head(head_), pos(head_) {}
  DAN_D float next() {                  // score of the next member; accumulates its weighted box (warp-uniform)
    const int lane = threadIdx.x & 31;
    while (pending == 0u) {             // (the caller asks for exactly count[head] members, so one more always exists)
      const int p = pos + lane;
      pending = __ballot_sync(0xffffffffu, p < n && assign[p] == head);
      base = pos;
      pos += 32;
    }
    const int i = base + __ffs(pending) - 1;
    pending &= pending - 1u;
    const float4 b = box[i];
    const float s = score[i];
    sx = fadd(sx, fmul(b.x, s));
    sy = fadd(sy, fmul(b.y, s));
    sz = fadd(sz, fmul(b.z, s));
    sw = fadd(sw, fmul(b.w, s));
    mx = fmaxf(mx, s);
    return s;
  }
};

// numpy's pairwise_sum (float32 add-reduce) over the next m member scores.  The leaf (<= 128 elements) is inlined so
// that the iterator stays in registers; the recursive halving above 128 elements runs on a small explicit stack of
// DEPTH levels, pairwise_depth(largest m).
template <class It> DAN_D float numpy_pairwise_leaf(It& it, int m) {
  if (m < 8) {
    float res = 0.f;
    for (int i = 0; i < m; ++i) res = fadd(res, it.next());
    return res;
  }
  float r[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = it.next();
  int i = 8;
  for (; i < m - (m % 8); i += 8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = fadd(r[k], it.next());
  }
  float res = fadd(fadd(fadd(r[0], r[1]), fadd(r[2], r[3])), fadd(fadd(r[4], r[5]), fadd(r[6], r[7])));
  for (; i < m; ++i) res = fadd(res, it.next());
  return res;
}

// levels of the stack for every m <= max_m: a block of m splits into m / 2 rounded down to a multiple of 8 and the
// rest, which is at most max_m / 2 + 8
constexpr int pairwise_depth(int max_m) { return max_m <= 128 ? 1 : 1 + pairwise_depth(max_m / 2 + 8); }
static_assert(pairwise_depth(kSortCap) == 8 && pairwise_depth(kVoteLargeCap) == 15, "numpy_pairwise stack depths");

template <int DEPTH, class It> DAN_D float numpy_pairwise(It& it, int m) {
  int fm[DEPTH], stage[DEPTH];
  float left[DEPTH];
  int sp = 0;
  fm[0] = m; stage[0] = 0; left[0] = 0.f;
  float ret = 0.f;
  while (sp >= 0) {
    const int cm = fm[sp];
    if (cm <= 128) {
      ret = numpy_pairwise_leaf(it, cm);
      --sp;
      continue;
    }
    int m2 = cm / 2;
    m2 -= m2 % 8;
    if (stage[sp] == 0) {
      stage[sp] = 1;
      ++sp; fm[sp] = m2; stage[sp] = 0;
    } else if (stage[sp] == 1) {
      left[sp] = ret;
      stage[sp] = 2;
      ++sp; fm[sp] = cm - m2; stage[sp] = 0;
    } else {
      ret = fadd(left[sp], ret);
      --sp;
    }
  }
  return ret;
}

// count[head] += 1.  Two uint16 counts share one 32-bit word (VotePlan::count is 4-byte aligned), and no count exceeds
// the 8192 detections of an image, so the low half never carries into the high one.
DAN_D void count_member(uint16_t* count, int head) {
  atomicAdd(reinterpret_cast<unsigned int*>(count) + (head >> 1), 1u << ((head & 1) * 16));
}
DAN_D void count_member(int32_t* count, int head) { atomicAdd(count + head, 1); }

constexpr int kPer = kSortCap / kSortThreads;    // score ranks per thread: t, t + 1024, ...

// An image's detections in the launch's dynamic shared memory (vote_plan), indexed by score rank.
struct VoteImage {
  using Pos = uint16_t;       // a position (score rank), as stored in assign and qlist
  static constexpr Pos kGonePos = kGone;
  static constexpr int kDepth = pairwise_depth(kSortCap);
  int b, n;                   // image, detections
  unsigned long long* keys;   // step 1: the sort keys, ...
  float4* box;                // ... which the boxes overwrite
  float* score;
  uint16_t* assign;
  uint16_t* count;
  uint16_t* qlist;
};

// The thread's detections (score ranks tid + e * kSortThreads), in registers: every index into the arrays is a
// compile-time constant.
struct VoteRegs {
  float4 box[kPer];
  int rank[kPer];             // -1: none
  uint32_t range[kPer];       // packed stripe ranges (VoteStripes::range)
  unsigned alive;             // bit e: rank[e] is not assigned yet
};

// the kernel's static shared memory that the steps of a round pass to each other
struct VoteRound {
  int* cand;                  // [32] step a: positions of the round's candidates
  int* ncand;
  unsigned* mask;             // [32] step b: bit m of mask[k] = candidate k overlaps the earlier candidate m
  unsigned* selfok;           // step b: bit k = candidate k overlaps itself (not NaN)
  unsigned* xs;               // [32] step c: bit m of xs[s] = the round's head m touches x stripe s
  unsigned* ys;               // ... y stripe s
};

DAN_D VoteImage carve(const VoteArgs& A, unsigned char* dyn_smem) {
  VoteImage im;
  im.b = blockIdx.x;
  im.n = A.counts ? min(max(A.counts[im.b], 0), A.cap) : A.cap;
  im.keys = reinterpret_cast<unsigned long long*>(dyn_smem);
  im.box = reinterpret_cast<float4*>(dyn_smem);
  im.score = reinterpret_cast<float*>(dyn_smem + A.plan.score);
  im.assign = reinterpret_cast<uint16_t*>(dyn_smem + A.plan.assign);
  im.count = reinterpret_cast<uint16_t*>(dyn_smem + A.plan.count);
  im.qlist = reinterpret_cast<uint16_t*>(dyn_smem + A.plan.qlist);
  return im;
}

// ---- 1. sort by descending score (:171-172), then gather through registers (the boxes overwrite the key storage)
DAN_D void sort_and_gather(const VoteArgs& A, const VoteImage& im, VoteRegs& R) {
  const int tid = threadIdx.x;
  const float* det = A.det + (int64_t)im.b * A.cap * 5;
  for (int i = tid; i < im.n; i += kSortThreads)
    im.keys[i] = ((unsigned long long)score_to_key(det[i * 5 + 4]) << 32) | (unsigned long long)(uint32_t)i;
  __syncthreads();
  sort_smem_keys(im.keys, im.n);
  float rs[kPer];
#pragma unroll
  for (int e = 0; e < kPer; ++e) {
    const int r = tid + e * kSortThreads;
    R.rank[e] = -1;
    if (r < im.n) {
      const int i = (int)(uint32_t)(im.keys[r] & 0xFFFFFFFFull);
      R.rank[e] = r;
      R.box[e] = make_float4(det[i * 5], det[i * 5 + 1], det[i * 5 + 2], det[i * 5 + 3]);
      rs[e] = det[i * 5 + 4];
      if (A.out_order) A.out_order[(int64_t)im.b * A.cap + r] = i;
    }
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < kPer; ++e) {
    if (R.rank[e] >= 0) {
      im.box[R.rank[e]] = R.box[e];
      im.score[R.rank[e]] = rs[e];
      im.assign[R.rank[e]] = kFree;
      im.count[R.rank[e]] = 0;
    }
  }
  __syncthreads();
}

// The stripe grid over the extent of the detections with finite coordinates below 1e30, and the stripe range of each
// of the thread's detections; all of them are alive.
DAN_D VoteStripes init_stripes(const VoteArgs& A, VoteRegs& R) {
  float x0 = 3.0e38f, x1 = -3.0e38f, y0 = 3.0e38f, y1 = -3.0e38f;
#pragma unroll
  for (int e = 0; e < kPer; ++e) {
    const float4 bx = R.box[e];
    if (R.rank[e] >= 0 && fabsf(bx.x) < 1e30f && fabsf(bx.y) < 1e30f && fabsf(bx.z) < 1e30f && fabsf(bx.w) < 1e30f) {
      x0 = fminf(x0, bx.x); x1 = fmaxf(x1, fadd(bx.z, 1.f));
      y0 = fminf(y0, bx.y); y1 = fmaxf(y1, fadd(bx.w, 1.f));
    }
  }
  VoteStripes sg;
  float ex, ey;
  block_minmax(x0, x1, sg.xlo, ex);
  block_minmax(y0, y1, sg.ylo, ey);
  sg.xinv = (ex > sg.xlo) ? fdiv(32.f, fsub(ex, sg.xlo)) : 0.f;
  sg.yinv = (ey > sg.ylo) ? fdiv(32.f, fsub(ey, sg.ylo)) : 0.f;
  sg.all = !(A.thr > 0.f);
  R.alive = 0u;
#pragma unroll
  for (int e = 0; e < kPer; ++e) {
    R.alive |= (R.rank[e] >= 0) ? (1u << e) : 0u;
    R.range[e] = (R.rank[e] >= 0) ? sg.range(R.box[e]) : 0u;
  }
  return sg;
}

// ---- 2. heads in score order (:173-190), 32 candidate heads per round.
// a. warp 0 lists the next (up to) 32 unassigned positions from `cur` on; returns their number (CTA-uniform)
DAN_D int list_candidates(const VoteImage& im, const VoteRound& S, int cur) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    int have = 0, p = cur;
    while (p < im.n && have < 32) {
      const bool un = (p + lane < im.n) && im.assign[p + lane] == kFree;
      const unsigned m = __ballot_sync(0xffffffffu, un);
      const int rank = have + __popc(m & ((1u << lane) - 1u));
      if (un && rank < 32) S.cand[rank] = p + lane;
      have += __popc(m);
      p += 32;
    }
    if (lane == 0) *S.ncand = min(have, 32);
  }
  __syncthreads();
  return *S.ncand;
}

// b. thread (k = warp, m = lane) tests candidate k against the earlier candidate m -> 32 row masks, and candidate k
// against itself
template <class Image> DAN_D void candidate_masks(const VoteArgs& A, const Image& im, const VoteRound& S, int ncand) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = warp, m = lane;
  bool ov = false, self_ok = false;
  if (k < ncand && m <= k && m < ncand) {
    const float4 bm = im.box[S.cand[m]];
    const bool hit = vote_overlaps(bm, vote_area(bm), im.box[S.cand[k]], A.thr);
    ov = hit && m < k;
    self_ok = hit && m == k;
  }
  const unsigned row = __ballot_sync(0xffffffffu, ov);
  const unsigned so = __ballot_sync(0xffffffffu, self_ok);
  if (lane == 0) S.mask[k] = row;
  if (lane == 0 && k == 0) *S.selfok = 0u;
  __syncthreads();
  if (lane == 0 && so) atomicOr(S.selfok, 1u << k);
  __syncthreads();
}

// c. every thread resolves the candidates from the masks (bit operations): candidate k is a head unless an earlier HEAD
// of the round overlaps it, then it joins the first such head; lane k of warp 0 writes candidate k's assign and count.
// Warp s publishes which of the round's heads touch x / y stripe s (two ballots).  Returns the heads (bit k: candidate k).
template <class Image> DAN_D unsigned resolve_heads(const Image& im, const VoteRound& S, const VoteStripes& sg, int ncand) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned heads = 0u;
  int joined = -1;
  for (int k = 0; k < ncand; ++k) {
    const unsigned mk = S.mask[k] & heads;
    if (mk == 0u) heads |= 1u << k;
    if (warp == 0 && lane == k) joined = mk ? __ffs(mk) - 1 : -1;
  }
  if (warp == 0 && lane < ncand) {
    const int pos = S.cand[lane];
    if (joined >= 0) {
      im.assign[pos] = (typename Image::Pos)S.cand[joined];
      count_member(im.count, S.cand[joined]);
    } else if ((*S.selfok >> lane) & 1u) {
      im.assign[pos] = (typename Image::Pos)pos;
      count_member(im.count, pos);
    } else {
      im.assign[pos] = Image::kGonePos;                    // NaN self IoU: deleted alone (:189-190)
    }
  }
  uint32_t q = 0u;
  const bool is_head = lane < ncand && ((heads >> lane) & 1u);
  if (is_head) q = sg.range(im.box[S.cand[lane]]);
  const bool every = (q & kEverywhere) != 0u;
  const unsigned hx = __ballot_sync(0xffffffffu, is_head && (every || ((stripe_span(q & 31u, (q >> 5) & 31u) >> warp) & 1u)));
  const unsigned hy = __ballot_sync(0xffffffffu, is_head && (every || ((stripe_span((q >> 10) & 31u, (q >> 15) & 31u) >> warp) & 1u)));
  if (lane == 0) { S.xs[warp] = hx; S.ys[warp] = hy; }
  __syncthreads();
  return heads;
}

// the round's heads that a detection of stripe range q can overlap: (OR over its x stripes) AND (OR over its y stripes)
DAN_D unsigned possible_heads(const VoteRound& S, uint32_t q, unsigned heads) {
  if (q & kEverywhere) return heads;
  unsigned ax = 0u, ay = 0u;
  for (uint32_t st = q & 31u; st <= ((q >> 5) & 31u); ++st) ax |= S.xs[st];
  for (uint32_t st = (q >> 10) & 31u; st <= ((q >> 15) & 31u); ++st) ay |= S.ys[st];
  return ax & ay;
}

// d. every thread looks its own alive detections behind the round's last candidate up in the stripe index - (OR over
// the detection's x stripes) AND (OR over its y stripes) = the round's heads it can overlap - and runs the exact test on
// those only, in head order: the first hit is the head it joins
DAN_D void join_heads(const VoteArgs& A, const VoteImage& im, const VoteRound& S, VoteRegs& R, unsigned heads, int last) {
  const int tid = threadIdx.x;
#pragma unroll
  for (int e = 0; e < kPer; ++e)                           // the candidates themselves are settled
    if (tid + e * kSortThreads <= last) R.alive &= ~(1u << e);
#pragma unroll
  for (int e = 0; e < kPer; ++e) {
    if ((R.alive >> e) & 1u) {
      unsigned poss = possible_heads(S, R.range[e], heads);
      const int r = tid + e * kSortThreads;                // (the box itself stays in shared memory: it is needed rarely)
      const float4 me = poss ? im.box[r] : make_float4(0.f, 0.f, 0.f, 0.f);
      while (poss) {                                       // ascending = head order: the first hit is the head it joins
        const int m = __ffs(poss) - 1;
        poss &= poss - 1u;
        const int hp = S.cand[m];
        const float4 h = im.box[hp];
        if (vote_overlaps(h, vote_area(h), me, A.thr)) {
          im.assign[r] = (uint16_t)hp;
          R.alive &= ~(1u << e);
          count_member(im.count, hp);
          poss = 0u;                                       // (no `break`: the lanes of the warp leave the loop together,
                                                           // racecheck saw them reach the barrier apart otherwise)
        }
      }
    }
  }
  __syncthreads();
}

// ---- 3. groups with at least two members, numbered in head order (:191-197, :205): qlist[q] = head of group q.
// Returns the number of groups written (at most max_out).  s_scan [32] and s_total: the block scan's shared memory.
template <class Image> DAN_D int number_groups(const VoteArgs& A, const Image& im, int* s_scan, int& s_total) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int E = (im.n + kSortThreads - 1) / kSortThreads;
  int mine_cnt = 0;
  for (int e = 0; e < E; ++e) {
    const int r = tid * E + e;
    if (r < im.n && im.count[r] >= 2) ++mine_cnt;
  }
  int incl = mine_cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += v;
  }
  if (lane == 31) s_scan[warp] = incl;
  __syncthreads();
  int before = 0, total = 0;
  for (int w = 0; w < kSortThreads / 32; ++w) {
    if (w < warp) before += s_scan[w];
    total += s_scan[w];
  }
  int q = before + incl - mine_cnt;
  for (int e = 0; e < E; ++e) {
    const int r = tid * E + e;
    if (r < im.n && im.count[r] >= 2) {
      if (q < A.max_out) im.qlist[q] = (typename Image::Pos)r;
      ++q;
    }
  }
  if (tid == 0) s_total = min(total, A.max_out);
  __syncthreads();
  return s_total;
}

DAN_D int number_groups(const VoteArgs& A, const VoteImage& im) {
  __shared__ int s_scan[kSortThreads / 32];
  __shared__ int s_total;
  return number_groups(A, im, s_scan, s_total);
}

// one warp per group (warp-uniform control flow): the score-weighted mean box and the max score (:198-203)
template <class Image> DAN_D void write_groups(const VoteArgs& A, const Image& im, int groups) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* out = A.out + (int64_t)im.b * A.max_out * 5;
  for (int g = warp; g < A.max_out; g += kSortThreads / 32) {
    float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f, o4 = 0.f;
    if (g < groups) {
      MemberIterT<typename Image::Pos> it(im.assign, im.box, im.score, im.n, im.qlist[g]);
      const float ssum = numpy_pairwise<Image::kDepth>(it, (int)im.count[it.head]);    // :199-201
      o0 = fdiv(it.sx, ssum); o1 = fdiv(it.sy, ssum); o2 = fdiv(it.sz, ssum); o3 = fdiv(it.sw, ssum);
      o4 = it.mx;                                                       // :200,202
    }
    if (lane == 0) { out[g * 5] = o0; out[g * 5 + 1] = o1; out[g * 5 + 2] = o2; out[g * 5 + 3] = o3; out[g * 5 + 4] = o4; }
  }
  if (tid == 0) A.out_count[im.b] = groups;
}

template <class Image> DAN_D void write_assign(const VoteArgs& A, const Image& im) {
  for (int r = threadIdx.x; r < im.n; r += kSortThreads)
    A.out_assign[(int64_t)im.b * A.cap + r] = im.assign[r] == Image::kGonePos ? -2 : (int)im.assign[r];
}

__global__ void __launch_bounds__(kSortThreads, 1) bbox_vote_kernel(const VoteArgs A) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ int s_cand[32];
  __shared__ int s_ncand;
  __shared__ unsigned s_mask[32], s_selfok, s_xs[32], s_ys[32];
  const VoteRound S = {s_cand, &s_ncand, s_mask, &s_selfok, s_xs, s_ys};
  const VoteImage im = carve(A, dyn_smem);
  VoteRegs R;
  sort_and_gather(A, im, R);
  const VoteStripes sg = init_stripes(A, R);
  int cur = 0;
  while (true) {
    const int ncand = list_candidates(im, S, cur);
    if (ncand == 0) break;
    const int last = S.cand[ncand - 1];
    candidate_masks(A, im, S, ncand);
    const unsigned heads = resolve_heads(im, S, sg, ncand);
    join_heads(A, im, S, R, heads, last);
    cur = last + 1;
  }
  __syncthreads();
  write_groups(A, im, number_groups(A, im));
  if (A.out_assign) write_assign(A, im);
}

// ---- bbox_vote_large_kernel: the same steps for images of more than kSortCap detections.  The detections live in the
// workspace (vote_large_plan) instead of registers and shared memory; shared memory holds the alive set, one bit per
// position, so that a round reads only the words behind its last candidate and the rows still alive there.

// Workspace and dynamic shared memory of one bbox_vote_large_kernel launch.  Workspace offsets are in bytes from the
// start of an image's slice (image * `image`); every array is 256-byte aligned.
struct VoteLargePlan {
  size_t image;               // workspace bytes per image
  size_t keys;                // [cap] u64 sort keys (score bits << 32 | row), then [cap] u64 the sort's merge buffer
  size_t merge;               //   (= keys + 8 * cap); the boxes overwrite both once the keys are sorted:
  size_t box;                 // [cap] float4 (= keys)
  size_t sorted;              // [cap] u64 the sorted keys
  size_t score;               // [cap] float
  size_t assign;              // [cap] int32: head position of each detection (-1 free, -2 a deleted head)
  size_t count;               // [cap] int32: members of the group headed there
  size_t qlist;               // [cap] int32: head position of group q
  size_t range;               // [cap] uint32: stripe ranges (VoteStripes::range)
  int smem;                   // dynamic shared memory: the alive bitmap, after the sort's kSortCap keys there
};

static VoteLargePlan vote_large_plan(int cap) {
  VoteLargePlan p = {};
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 256); return at; };
  p.keys = p.box = take((size_t)cap * 16);
  p.merge = p.keys + (size_t)cap * 8;
  p.sorted = take((size_t)cap * 8);
  p.score = take((size_t)cap * 4);
  p.assign = take((size_t)cap * 4);
  p.count = take((size_t)cap * 4);
  p.qlist = take((size_t)cap * 4);
  p.range = take((size_t)cap * 4);
  p.image = off;
  const int bitmap = (int)align_up((size_t)(cap + 31) / 32 * 4, 16), sort = kSortCap * 8;
  p.smem = bitmap > sort ? bitmap : sort;
  return p;
}
static_assert(kVoteLargeCap / 8 <= kVoteSmemMax, "the alive bitmap of kVoteLargeCap detections fits shared memory");

struct VoteLargeArgs {
  VoteArgs v;                 // inputs and outputs (v.plan is not used)
  VoteLargePlan plan;
  unsigned char* ws;          // [B, plan.image] workspace
};

// An image's detections in the workspace, indexed by score rank, and its alive set in shared memory.
struct VoteImageLarge {
  using Pos = int32_t;
  static constexpr Pos kFreePos = -1, kGonePos = -2;
  static constexpr int kDepth = pairwise_depth(kVoteLargeCap);
  int b, n;                   // image, detections
  int words;                  // words of the alive bitmap: ceil(n / 32)
  unsigned long long *keys, *merge, *sorted;
  float4* box;
  float* score;
  int32_t* assign;
  int32_t* count;
  int32_t* qlist;
  uint32_t* range;
  unsigned* alive;            // shared: bit (r & 31) of word (r >> 5) = position r is not assigned yet
  unsigned long long* s_keys; // shared: the sort's keys (step 1, before the bitmap exists)
};

DAN_D VoteImageLarge carve_large(const VoteLargeArgs& L, unsigned char* dyn_smem) {
  VoteImageLarge im;
  im.b = blockIdx.x;
  im.n = L.v.counts ? min(max(L.v.counts[im.b], 0), L.v.cap) : L.v.cap;
  im.words = (im.n + 31) >> 5;
  unsigned char* ws = L.ws + (size_t)im.b * L.plan.image;
  im.keys = reinterpret_cast<unsigned long long*>(ws + L.plan.keys);
  im.merge = reinterpret_cast<unsigned long long*>(ws + L.plan.merge);
  im.sorted = reinterpret_cast<unsigned long long*>(ws + L.plan.sorted);
  im.box = reinterpret_cast<float4*>(ws + L.plan.box);
  im.score = reinterpret_cast<float*>(ws + L.plan.score);
  im.assign = reinterpret_cast<int32_t*>(ws + L.plan.assign);
  im.count = reinterpret_cast<int32_t*>(ws + L.plan.count);
  im.qlist = reinterpret_cast<int32_t*>(ws + L.plan.qlist);
  im.range = reinterpret_cast<uint32_t*>(ws + L.plan.range);
  im.alive = reinterpret_cast<unsigned*>(dyn_smem);
  im.s_keys = reinterpret_cast<unsigned long long*>(dyn_smem);
  return im;
}

// 1. the keys of all n rows sorted in the workspace (runs of kSortCap in shared memory, then merged), then the boxes,
// scores and out_order gathered into score order
DAN_D void sort_and_gather_large(const VoteArgs& A, const VoteImageLarge& im, SortScratch& sc) {
  const int tid = threadIdx.x;
  const float* det = A.det + (int64_t)im.b * A.cap * 5;
  for (int i = tid; i < im.n; i += kSortThreads)
    im.keys[i] = ((unsigned long long)score_to_key(det[i * 5 + 4]) << 32) | (unsigned long long)(uint32_t)i;
  __syncthreads();
  select_and_sort_large(im.keys, im.n, im.n, im.sorted, im.merge, im.s_keys, sc);
  for (int r = tid; r < im.n; r += kSortThreads) {
    const int i = (int)(uint32_t)(im.sorted[r] & 0xFFFFFFFFull);
    im.box[r] = make_float4(det[i * 5], det[i * 5 + 1], det[i * 5 + 2], det[i * 5 + 3]);
    im.score[r] = det[i * 5 + 4];
    im.assign[r] = VoteImageLarge::kFreePos;
    im.count[r] = 0;
    if (A.out_order) A.out_order[(int64_t)im.b * A.cap + r] = i;
  }
  __syncthreads();
}

// the stripe grid, every detection's stripe range, and all n positions alive (the bitmap overwrites the sort's keys)
DAN_D VoteStripes init_stripes_large(const VoteArgs& A, const VoteImageLarge& im) {
  const int tid = threadIdx.x;
  float x0 = 3.0e38f, x1 = -3.0e38f, y0 = 3.0e38f, y1 = -3.0e38f;
  for (int r = tid; r < im.n; r += kSortThreads) {
    const float4 bx = im.box[r];
    if (fabsf(bx.x) < 1e30f && fabsf(bx.y) < 1e30f && fabsf(bx.z) < 1e30f && fabsf(bx.w) < 1e30f) {
      x0 = fminf(x0, bx.x); x1 = fmaxf(x1, fadd(bx.z, 1.f));
      y0 = fminf(y0, bx.y); y1 = fmaxf(y1, fadd(bx.w, 1.f));
    }
  }
  VoteStripes sg;                                          // (init_stripes, over the workspace)
  float ex, ey;
  block_minmax(x0, x1, sg.xlo, ex);
  block_minmax(y0, y1, sg.ylo, ey);
  sg.xinv = (ex > sg.xlo) ? fdiv(32.f, fsub(ex, sg.xlo)) : 0.f;
  sg.yinv = (ey > sg.ylo) ? fdiv(32.f, fsub(ey, sg.ylo)) : 0.f;
  sg.all = !(A.thr > 0.f);
  for (int r = tid; r < im.n; r += kSortThreads) im.range[r] = sg.range(im.box[r]);
  for (int w = tid; w < im.words; w += kSortThreads) im.alive[w] = w < (im.n >> 5) ? 0xffffffffu : (1u << (im.n & 31)) - 1u;
  __syncthreads();
  return sg;
}

// a. warp 0 lists the next (up to) 32 alive positions from `cur` on, 32 positions per bitmap word, and clears their
// bits: every position before the round's last candidate is then settled.  Returns their number (CTA-uniform).
DAN_D int list_candidates_large(const VoteImageLarge& im, const VoteRound& S, int cur) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    int have = 0;
    for (int w = cur >> 5; w < im.words && have < 32; ++w) {
      const unsigned word = im.alive[w];
      const int rank = have + __popc(word & ((1u << lane) - 1u));
      const bool take = ((word >> lane) & 1u) && rank < 32;
      if (take) S.cand[rank] = w * 32 + lane;
      const unsigned taken = __ballot_sync(0xffffffffu, take);
      if (lane == 0 && taken) im.alive[w] = word & ~taken;
      have += __popc(word);
    }
    if (lane == 0) *S.ncand = min(have, 32);
  }
  __syncthreads();
  return *S.ncand;
}

// d. the alive detections behind the round's last candidate, one bitmap word per thread at a time, test the round's
// heads they can overlap in head order: the first hit is the head they join.  A warp takes 32 consecutive words per
// iteration and its lanes meet after each (they hold different numbers of alive rows), so that the lanes of a warp leave
// the loop together and reach the barrier together, as in join_heads.
DAN_D void join_heads_large(const VoteArgs& A, const VoteImageLarge& im, const VoteRound& S, unsigned heads, int last) {
  const int lane = threadIdx.x & 31;
  for (int w0 = ((last + 1) >> 5) + (int)(threadIdx.x & ~31u); w0 < im.words; w0 += kSortThreads) {   // warp-uniform
    const int w = w0 + lane;
    const unsigned word = w < im.words ? im.alive[w] : 0u;
    unsigned left = word;
    for (unsigned todo = word; todo != 0u; todo &= todo - 1u) {
      const int r = w * 32 + __ffs(todo) - 1;
      unsigned poss = possible_heads(S, im.range[r], heads);
      const float4 me = poss ? im.box[r] : make_float4(0.f, 0.f, 0.f, 0.f);
      while (poss) {
        const int m = __ffs(poss) - 1;
        poss &= poss - 1u;
        const int hp = S.cand[m];
        const float4 h = im.box[hp];
        if (vote_overlaps(h, vote_area(h), me, A.thr)) {
          im.assign[r] = hp;
          left &= ~(1u << (r & 31));
          count_member(im.count, hp);
          poss = 0u;
        }
      }
    }
    if (left != word) im.alive[w] = left;
    __syncwarp();
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kSortThreads, 1) bbox_vote_large_kernel(const VoteLargeArgs L) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ SortScratch sc;
  __shared__ int s_scan[kSortThreads / 32], s_total;
  __shared__ int s_cand[32];
  __shared__ int s_ncand;
  __shared__ unsigned s_mask[32], s_selfok, s_xs[32], s_ys[32];
  const VoteRound S = {s_cand, &s_ncand, s_mask, &s_selfok, s_xs, s_ys};
  const VoteArgs A = L.v;
  const VoteImageLarge im = carve_large(L, dyn_smem);
  sort_and_gather_large(A, im, sc);
  const VoteStripes sg = init_stripes_large(A, im);
  int cur = 0;
  while (true) {
    const int ncand = list_candidates_large(im, S, cur);
    if (ncand == 0) break;
    const int last = S.cand[ncand - 1];
    candidate_masks(A, im, S, ncand);
    const unsigned heads = resolve_heads(im, S, sg, ncand);
    join_heads_large(A, im, S, heads, last);
    cur = last + 1;
  }
  __syncthreads();
  write_groups(A, im, number_groups(A, im, s_scan, s_total));
  if (A.out_assign) write_assign(A, im);
}

// detect_face (eval_sfd.py:95-114) for B images of N anchors, in two kernels:
//   face_key_kernel     grid-wide over B x N: key = score bits << 32 | anchor (equal scores: higher anchor first), and a
//                       per-image histogram of the keys' face_bin() (shared-memory histogram per CTA, flushed with one
//                       global atomic per non-empty bin)
//   face_select_kernel  one CTA per image: the histogram gives the bin that holds the k-th key; one pass over the image's
//                       keys compacts those in that bin or above into shared memory, where they are sorted.  Only the k
//                       rows are read (or decoded from the offsets), divided by shrink and written.
// The score comes from the scores of decoded boxes (dan_detect_face_select) or from the two logits (the softmax in
// tf.nn.softmax's op order, dan_detect_face_batch); the box from a decoded row or from a decode of the offset row.
constexpr int kFaceBins = 4096;             // histogram bins per image
constexpr int kFaceKeyThreads = 512;
constexpr int kFaceChunk = 8 * kFaceKeyThreads;   // anchors per CTA of the key kernel

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

// eval_sfd.py:101-112, one CTA per image
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
    // the bin t of the k-th largest key: thread i holds bins 4i .. 4i + 3, `above` counts the keys in higher bins
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
    if (above < k && above + c >= k) {                     // exactly one thread: the bins hold all n > k keys
      int cum = above, t = kPer * tid;
      for (int j = kPer - 1; j >= 0; --j) {
        cum += hb[j];
        if (cum >= k) { t = kPer * tid + j; break; }
      }
      s_bin = t;
      s_ge = cum;
    }
    __syncthreads();
    const int t = s_bin, ge = s_ge;
    if (ge <= kSortCap) {
      // one pass: the ge keys in bin t or above (a superset of the top k) into shared memory, one atomic per warp
      for (int i0 = 0; i0 < A.n; i0 += 4 * kSortThreads) {
        unsigned long long q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * kSortThreads + tid;
          q[u] = i < A.n ? __ldcs(keys + i) : 0ull;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool keep = i0 + u * kSortThreads + tid < A.n && face_bin(q[u]) >= t;
          const unsigned m = __ballot_sync(0xffffffffu, keep);
          if (m != 0u) {
            int base = 0;
            if (lane == 0) base = atomicAdd(&sc.fill, __popc(m));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (keep) s_keys[base + __popc(m & ((1u << lane) - 1u))] = q[u];
          }
        }
      }
      __syncthreads();
      select_and_sort(keys, ge, k, s_keys, sc, true, s_keys + kSortCap);
    } else {
      // more keys share the k-th key's bin than shared memory holds: radix select over all of the image's keys
      select_and_sort(keys, A.n, k, s_keys, sc, false, s_keys + kSortCap);
    }
  }
  float* out = A.out + (int64_t)b * A.top * 5;
  for (int r = tid; r < A.top; r += kSortThreads) {
    float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f, o4 = 0.f;
    int idx = -1;
    if (r < k) {
      const unsigned long long key = s_keys[r];
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

constexpr size_t kFaceSelectSmem = 2 * kSortCap * sizeof(unsigned long long);

static size_t face_hist_bytes(int32_t batch) { return align_up((size_t)batch * kFaceBins * sizeof(int), 256); }

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

}  // namespace

}  // namespace dan

using namespace dan;

extern "C" {

size_t dan_detect_face_batch_workspace_bytes(int64_t num_anchors, int32_t batch) {
  if (num_anchors < 0 || batch < 0) return 0;
  return face_hist_bytes(batch) + align_up((size_t)num_anchors * (size_t)batch * 8, 256);
}

size_t dan_detect_face_workspace_bytes(int64_t n) { return dan_detect_face_batch_workspace_bytes(n, 1); }

int dan_detect_face_select(const float* bboxes, const float* scores, int64_t n, float shrink, int32_t top, float* out_det,
                           int32_t* out_index, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream) {
  DAN_REQUIRE(n >= 0 && n < ((int64_t)1 << 31), DAN_ERR_INVALID_ARGUMENT, "bad n");
  DAN_REQUIRE(top >= 1 && top <= kSortCap, DAN_ERR_UNSUPPORTED, "top must be in [1, %d]", kSortCap);
  DAN_REQUIRE(out_det && out_count, DAN_ERR_INVALID_ARGUMENT, "NULL output");
  DAN_REQUIRE(n == 0 || (bboxes && scores && aligned16(bboxes)), DAN_ERR_INVALID_ARGUMENT, "NULL / misaligned input");
  const size_t need = dan_detect_face_workspace_bytes(n);
  DAN_REQUIRE(n == 0 || (workspace != nullptr && workspace_bytes >= need), DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu",
              need, workspace_bytes);
  FaceScores score = {scores};
  FaceBoxes box = {reinterpret_cast<const float4*>(bboxes)};
  return face_launch(score, box, n, 1, shrink, top, out_det, out_index, out_count, workspace, (cudaStream_t)stream);
}

int dan_detect_face_batch(int32_t pred_dtype, const void* cls_pred, const void* loc_pred, const float* a_ymin, const float* a_xmin,
                          const float* a_ymax, const float* a_xmax, int64_t num_anchors, int32_t batch, const float* h_prior_scaling,
                          float shrink, int32_t top, float* out_det, int32_t* out_index, void* workspace, size_t workspace_bytes,
                          void* stream) {
  const int esize = dtype_bytes(pred_dtype);
  DAN_REQUIRE(esize != 0, DAN_ERR_INVALID_ARGUMENT, "unknown pred_dtype %d", pred_dtype);
  DAN_REQUIRE(num_anchors >= 0 && num_anchors < ((int64_t)1 << 31) && batch >= 0, DAN_ERR_INVALID_ARGUMENT, "bad num_anchors / batch");
  DAN_REQUIRE(top >= 1 && top <= kSortCap, DAN_ERR_UNSUPPORTED, "top must be in [1, %d]", kSortCap);
  if (batch == 0) return DAN_OK;
  DAN_REQUIRE(cls_pred && loc_pred && a_ymin && a_xmin && a_ymax && a_xmax && h_prior_scaling && out_det, DAN_ERR_INVALID_ARGUMENT,
              "NULL pointer");
  DAN_REQUIRE((reinterpret_cast<uintptr_t>(loc_pred) & (uintptr_t)(4 * esize - 1)) == 0, DAN_ERR_INVALID_ARGUMENT,
              "loc_pred must be %d-byte aligned", 4 * esize);
  const int64_t chunks = (num_anchors + kFaceChunk - 1) / kFaceChunk;
  DAN_REQUIRE(chunks * batch < ((int64_t)1 << 31), DAN_ERR_UNSUPPORTED, "batch x num_anchors too large");
  const size_t need = dan_detect_face_batch_workspace_bytes(num_anchors, batch);
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

size_t dan_bbox_vote_workspace_bytes(int32_t batch, int32_t capacity) {
  if (batch < 0 || capacity <= kSortCap || capacity > kVoteLargeCap) return 0;
  return (size_t)batch * vote_large_plan(capacity).image;
}

int dan_bbox_vote_ws(const float* det, const int32_t* counts, int32_t batch, int32_t capacity, float nms_threshold,
                     int32_t max_per_image, float* out_det, int32_t* out_count, int32_t* out_order, int32_t* out_assign,
                     void* workspace, size_t workspace_bytes, void* stream) {
  DAN_REQUIRE(batch >= 0 && capacity >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  DAN_REQUIRE(capacity <= kVoteLargeCap, DAN_ERR_UNSUPPORTED, "more than %d detections per image", kVoteLargeCap);
  DAN_REQUIRE(max_per_image >= 1 && max_per_image <= 65535, DAN_ERR_INVALID_ARGUMENT, "max_per_image must be in [1, 65535]");
  if (batch == 0) return DAN_OK;
  DAN_REQUIRE(out_det && out_count && (capacity == 0 || det), DAN_ERR_INVALID_ARGUMENT, "NULL pointer");
  VoteArgs A = {};
  A.det = det;
  A.counts = counts;
  A.cap = capacity;
  A.thr = nms_threshold;
  A.max_out = max_per_image;
  A.out = out_det;
  A.out_count = out_count;
  A.out_order = out_order;
  A.out_assign = out_assign;
  cudaStream_t st = (cudaStream_t)stream;
  if (capacity > kSortCap) {
    const size_t need = dan_bbox_vote_workspace_bytes(batch, capacity);
    DAN_REQUIRE(workspace != nullptr && workspace_bytes >= need, DAN_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu",
                need, workspace_bytes);
    DAN_REQUIRE(aligned16(workspace), DAN_ERR_INVALID_ARGUMENT, "workspace must be 16-byte aligned");
    VoteLargeArgs L = {};
    L.v = A;
    L.plan = vote_large_plan(capacity);
    L.ws = static_cast<unsigned char*>(workspace);
    DAN_CUDA(cudaFuncSetAttribute(bbox_vote_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kVoteSmemMax));
    bbox_vote_large_kernel<<<batch, kSortThreads, L.plan.smem, st>>>(L);
    DAN_LAUNCH_CHECK("bbox_vote_large_kernel");
    return DAN_OK;
  }
  A.plan = vote_plan(capacity);
  DAN_REQUIRE(A.plan.smem <= kVoteSmemMax, DAN_ERR_UNSUPPORTED, "capacity %d needs %d bytes of shared memory", capacity, A.plan.smem);
  DAN_CUDA(cudaFuncSetAttribute(bbox_vote_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kVoteSmemMax));
  bbox_vote_kernel<<<batch, kSortThreads, A.plan.smem, st>>>(A);
  DAN_LAUNCH_CHECK("bbox_vote_kernel");
  return DAN_OK;
}

int dan_bbox_vote(const float* det, const int32_t* counts, int32_t batch, int32_t capacity, float nms_threshold,
                  int32_t max_per_image, float* out_det, int32_t* out_count, int32_t* out_order, int32_t* out_assign,
                  void* stream) {
  DAN_REQUIRE(batch >= 0 && capacity >= 0, DAN_ERR_INVALID_ARGUMENT, "negative size");
  DAN_REQUIRE(capacity <= kSortCap, DAN_ERR_UNSUPPORTED, "more than %d detections per image", kSortCap);
  return dan_bbox_vote_ws(det, counts, batch, capacity, nms_threshold, max_per_image, out_det, out_count, out_order, out_assign,
                          nullptr, 0, stream);
}

}  // extern "C"
