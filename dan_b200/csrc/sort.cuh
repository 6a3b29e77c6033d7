// Block-wide top-k + sort of 64-bit keys in shared memory (1024-thread CTAs), shared by the postprocess and the
// evaluation-merge kernels.  Include it INSIDE `namespace dan { ... }` of a .cu file, after common.cuh.
#pragma once

constexpr int kSortCap = 8192;      // keys sorted in shared memory (64 KB)
constexpr int kSortThreads = 1024;  // threads per CTA of the sort kernels

// order-preserving float <-> uint32 (descending key order = descending score)
DAN_D uint32_t score_to_key(float s) { return (uint32_t)float_to_ordered(s) ^ 0x80000000u; }
DAN_D float key_to_score(uint32_t k) { return ordered_to_float((int)(k ^ 0x80000000u)); }

// ---------------------------------------------------------------------------
// K4: per-list top-k (radix select when needed) + bitonic sort, all in shared memory.
// Every thread of the CTA calls it; returns the number of sorted keys m (descending in s_keys[0, m)).
// ---------------------------------------------------------------------------
struct SortScratch {
  int hist[256];
  unsigned long long prefix;
  int remaining;
  int fill;
};

// compare-exchange stage at distance ST (a power of two < KPT) inside a thread's KPT keys; all register indices
// are static
template <int KPT, int ST>
DAN_D void reg_stage(unsigned long long (&r)[KPT], int lsize, bool desc_t) {
  constexpr int LK = KPT == 32 ? 5 : KPT == 16 ? 4 : KPT == 8 ? 3 : KPT == 4 ? 2 : KPT == 2 ? 1 : 0;
#pragma unroll
  for (int e = 0; e < KPT; ++e) {
    if ((e & ST) == 0) {
      const bool desc = (lsize >= LK) ? desc_t : (((e >> lsize) & 1) == 0);
      const unsigned long long x = r[e], y = r[e | ST];
      if ((x < y) == desc) { r[e] = y; r[e | ST] = x; }
    }
  }
}

// Bitonic sort (descending) of P = 2^lp2 64-bit keys with the keys held in REGISTERS, KPT per thread: thread t owns
// the consecutive keys KPT*t .. KPT*t + KPT-1 and T = P / KPT threads take part (KPT is chosen so that as many of the
// CTA's 1024 threads as possible work: the sort is a chain of ~lp2^2/2 dependent stages, so the time is stages x
// per-stage latency, and the per-stage latency grows with the keys a thread has to move).  Compare-exchange partners at a
// distance below KPT are in the same thread, up to 16*KPT in another lane of the same warp (shfl.xor), and only the
// larger distances go through shared memory, written transposed ([e][thread]) so that both the store and the
// partner's load are conflict free.
template <int KPT>
DAN_D void bitonic_sort_regs(unsigned long long* s_keys, int lp2) {
  constexpr int LK = KPT == 32 ? 5 : KPT == 16 ? 4 : KPT == 8 ? 3 : KPT == 4 ? 2 : KPT == 2 ? 1 : 0;
  const int tid = threadIdx.x;
  const int T = 1 << (lp2 - LK);                // threads that own keys
  const bool active = tid < T;
  unsigned long long r[KPT];
  if (active) {
#pragma unroll
    for (int e = 0; e < KPT; ++e) r[e] = s_keys[KPT * tid + e];
  }
  for (int lsize = 1; lsize <= lp2; ++lsize) {
    // direction of the merge this key takes part in: descending iff bit `lsize` of its index is 0
    const bool desc_t = ((tid >> (lsize >= LK ? lsize - LK : 0)) & 1) == 0;
    for (int ls = lsize - 1; ls >= 0; --ls) {
      if (ls >= LK + 5) {
        __syncthreads();
        if (active) {
#pragma unroll
          for (int e = 0; e < KPT; ++e) s_keys[e * T + tid] = r[e];
        }
        __syncthreads();
        if (active) {
          const int partner = tid ^ (1 << (ls - LK));
          const bool keep_max = ((tid & (1 << (ls - LK))) == 0) == desc_t;
#pragma unroll
          for (int e = 0; e < KPT; ++e) {
            const unsigned long long o = s_keys[e * T + partner];
            r[e] = ((r[e] < o) == keep_max) ? o : r[e];      // keys are unique: max takes o iff r < o, min iff r > o
          }
        }
      } else if (!active) {
        // warps that own no keys only take part in the barriers above (T is a multiple of 32: warp-uniform)
      } else if (ls >= LK) {
        const int lmask = 1 << (ls - LK);
        const bool keep_max = ((tid & lmask) == 0) == desc_t;
#pragma unroll
        for (int e = 0; e < KPT; ++e) {
          const unsigned long long o = __shfl_xor_sync(0xffffffffu, r[e], lmask);
          r[e] = ((r[e] < o) == keep_max) ? o : r[e];
        }
      } else {
        if constexpr (KPT > 16) { if (ls == 4) reg_stage<KPT, 16>(r, lsize, desc_t); }
        if constexpr (KPT > 8) { if (ls == 3) reg_stage<KPT, 8>(r, lsize, desc_t); }
        if constexpr (KPT > 4) { if (ls == 2) reg_stage<KPT, 4>(r, lsize, desc_t); }
        if constexpr (KPT > 2) { if (ls == 1) reg_stage<KPT, 2>(r, lsize, desc_t); }
        if constexpr (KPT > 1) { if (ls == 0) reg_stage<KPT, 1>(r, lsize, desc_t); }
      }
    }
  }
  __syncthreads();
  if (active) {
#pragma unroll
    for (int e = 0; e < KPT; ++e) s_keys[KPT * tid + e] = r[e];
  }
  __syncthreads();
}

// Sorts the m <= kSortCap keys in s_keys[0, m) in place, descending (all threads of the CTA call it; the slots up to
// the next power of two are overwritten with 0).
DAN_D void sort_smem_keys(unsigned long long* s_keys, int m) {
  const int tid = threadIdx.x;
  // pad to a power of two with 0 (smaller than any real key: the low word of a real key is ~index != 0)
  int lp2 = 0;
  while ((1 << lp2) < m) ++lp2;
  const int p2 = 1 << lp2;
  for (int i = m + tid; i < p2; i += kSortThreads) s_keys[i] = 0ull;
  __syncthreads();
  if (lp2 >= 5) {            // (at least one full warp of owners)
    // keys per thread: the smallest power of two that lets the 1024 threads own all 2^lp2 <= kSortCap keys
    const int lk = lp2 > 10 ? lp2 - 10 : 0;
    if (lk == 0) bitonic_sort_regs<1>(s_keys, lp2);
    else if (lk == 1) bitonic_sort_regs<2>(s_keys, lp2);
    else if (lk == 2) bitonic_sort_regs<4>(s_keys, lp2);
    else if (lk == 3) bitonic_sort_regs<8>(s_keys, lp2);
    return;
  }
  // small lists: plain bitonic sort in shared memory, descending; strides are powers of two -> shifts only
  for (int lsize = 1; lsize <= lp2; ++lsize) {
    for (int ls = lsize - 1; ls >= 0; --ls) {
      const int stride = 1 << ls;
      for (int t = tid; t < (p2 >> 1); t += kSortThreads) {
        const int lo = ((t >> ls) << (ls + 1)) | (t & (stride - 1));
        const int hi = lo | stride;
        const bool desc = ((lo >> lsize) & 1) == 0;
        const unsigned long long x = s_keys[lo], y = s_keys[hi];
        if ((x < y) == desc) { s_keys[lo] = y; s_keys[hi] = x; }
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------------------
// Merge sort of m <= kSortCap unique keys in shared memory, descending, with a second buffer of m keys: every warp sorts
// tiles of 128 keys in registers (bitonic network on shuffles, no CTA barrier), then the sorted runs are merged
// pairwise log2(m / 128) times - each key finds its place in the merged run by a binary search in the sibling run.
// ~2 us for 2048 keys instead of ~12 us for the register bitonic sort of the whole array (which moves every 64-bit key
// through log^2 stages).  The result ends in s_a.  All threads of the CTA call it.
// ---------------------------------------------------------------------------
DAN_D void warp_sort_tile128(unsigned long long (&r)[4], int lane) {
  // key index inside the tile: 4 * lane + e; stage (lsize, ls): partner at distance 2^ls, direction from bit lsize
  for (int lsize = 1; lsize <= 7; ++lsize) {
    const bool desc_t = ((lane >> (lsize >= 2 ? lsize - 2 : 0)) & 1) == 0;
    for (int ls = lsize - 1; ls >= 0; --ls) {
      if (ls >= 2) {
        const int lmask = 1 << (ls - 2);
        const bool keep_max = ((lane & lmask) == 0) == desc_t;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const unsigned long long o = __shfl_xor_sync(0xffffffffu, r[e], lmask);
          r[e] = ((r[e] < o) == keep_max) ? o : r[e];
        }
      } else if (ls == 1) {
        reg_stage<4, 2>(r, lsize, desc_t);
      } else {
        reg_stage<4, 1>(r, lsize, desc_t);
      }
    }
  }
}

DAN_D void merge_sort_smem_keys(unsigned long long* s_a, unsigned long long* s_b, int m) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int rounds = 0;
  for (int run = 128; run < m; run <<= 1) ++rounds;
  unsigned long long* src = (rounds & 1) ? s_b : s_a;        // the tiles start where an even number of hops ends in s_a
  unsigned long long* dst = (rounds & 1) ? s_a : s_b;
  // tiles: read from s_a, write to src (the same tile's slots: no other warp touches them)
  for (int t0 = warp * 128; t0 < m; t0 += (kSortThreads / 32) * 128) {
    unsigned long long r[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = t0 + 4 * lane + e;
      r[e] = (i < m) ? s_a[i] : 0ull;                        // (0 sorts behind every real key and is not written back)
    }
    warp_sort_tile128(r, lane);
    __syncwarp();
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = t0 + 4 * lane + e;
      if (i < m) src[i] = r[e];
    }
  }
  __syncthreads();
  for (int run = 128; run < m; run <<= 1) {
    for (int i = tid; i < m; i += kSortThreads) {
      const int base = (i / (2 * run)) * (2 * run);
      const bool second = i - base >= run;
      const int x_lo = base + (second ? run : 0), y_lo = base + (second ? 0 : run);
      const int y_len = max(0, min(run, m - y_lo));
      const unsigned long long key = src[i];
      int lo = 0, hi = y_len;                                // keys of the sibling run that precede `key` (keys are unique)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (src[y_lo + mid] > key) lo = mid + 1;
        else hi = mid;
      }
      dst[base + (i - x_lo) + lo] = key;
    }
    __syncthreads();
    unsigned long long* t = src; src = dst; dst = t;
  }
}

// k-th largest of the cnt keys in `keys` (HBM): block radix select, MSB first, 8 bits per pass
DAN_D unsigned long long radix_select_kth(const unsigned long long* __restrict__ keys, int cnt, int k, SortScratch& sc) {
  const int tid = threadIdx.x;
  if (tid == 0) { sc.prefix = 0ull; sc.remaining = k; }
  unsigned long long prefix_mask = 0ull;
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256; i += kSortThreads) sc.hist[i] = 0;
    __syncthreads();
    const unsigned long long prefix = sc.prefix;
    for (int i = tid; i < cnt; i += kSortThreads) {
      const unsigned long long key = keys[i];
      if ((key & prefix_mask) == prefix) atomicAdd(&sc.hist[(int)((key >> shift) & 255ull)], 1);
    }
    __syncthreads();
    if (tid == 0) {
      int cum = 0, bin = 255;
      for (; bin > 0; --bin) {
        if (cum + sc.hist[bin] >= sc.remaining) break;
        cum += sc.hist[bin];
      }
      sc.remaining -= cum;
      sc.prefix = prefix | ((unsigned long long)bin << shift);
    }
    prefix_mask |= 255ull << shift;
    __syncthreads();
  }
  return sc.prefix;
}

// staged = true: when cnt <= kSortCap the keys are already in s_keys[0, cnt) (the caller produced them there)
// s_spare: optional second shared-memory buffer of >= min(cnt, k, kSortCap) keys -> merge sort instead of the bitonic one
DAN_D int select_and_sort(const unsigned long long* __restrict__ keys, int cnt, int k, unsigned long long* s_keys, SortScratch& sc,
                          bool staged = false, unsigned long long* s_spare = nullptr) {
  const int tid = threadIdx.x;
  int m = cnt;
  if (cnt <= kSortCap) {
    if (!staged)
      for (int i = tid; i < cnt; i += kSortThreads) s_keys[i] = keys[i];
  } else {
    const unsigned long long kth = radix_select_kth(keys, cnt, k, sc);
    if (tid == 0) sc.fill = 0;
    __syncthreads();
    for (int i = tid; i < cnt; i += kSortThreads) {
      const unsigned long long key = keys[i];
      if (key >= kth) s_keys[atomicAdd(&sc.fill, 1)] = key;   // exactly k keys (keys are unique)
    }
    m = k;
  }
  if (s_spare != nullptr && m > 128) {
    __syncthreads();
    merge_sort_smem_keys(s_keys, s_spare, m);
  } else {
    sort_smem_keys(s_keys, m);
  }
  return m;
}

// More than kSortCap keys to keep (no upper limit): the k largest of `keys` are compacted into buf_a (HBM), sorted in
// runs of kSortCap in shared memory, and the runs are merged pairwise between buf_a and buf_b - every key finds its place
// in the merged run by a binary search in the other run (keys are unique).  The sorted keys end in buf_a.  One CTA; meant
// for the rare long lists (tf.nn.top_k / tf.image.non_max_suppression have no size limit, so neither does this path).
DAN_D void select_and_sort_large(const unsigned long long* __restrict__ keys, int cnt, int k, unsigned long long* buf_a,
                                 unsigned long long* buf_b, unsigned long long* s_keys, SortScratch& sc) {
  const int tid = threadIdx.x;
  if (cnt > k) {
    const unsigned long long kth = radix_select_kth(keys, cnt, k, sc);
    if (tid == 0) sc.fill = 0;
    __syncthreads();
    for (int i = tid; i < cnt; i += kSortThreads) {
      const unsigned long long key = keys[i];
      if (key >= kth) buf_a[atomicAdd(&sc.fill, 1)] = key;
    }
  } else {
    for (int i = tid; i < k; i += kSortThreads) buf_a[i] = keys[i];
  }
  __syncthreads();
  for (int r0 = 0; r0 < k; r0 += kSortCap) {
    const int m = min(kSortCap, k - r0);
    for (int i = tid; i < m; i += kSortThreads) s_keys[i] = buf_a[r0 + i];
    __syncthreads();
    sort_smem_keys(s_keys, m);
    for (int i = tid; i < m; i += kSortThreads) buf_a[r0 + i] = s_keys[i];
    __syncthreads();
  }
  unsigned long long* src = buf_a;
  unsigned long long* dst = buf_b;
  for (long long run = kSortCap; run < k; run *= 2) {
    for (int i = tid; i < k; i += kSortThreads) {
      const long long base = (i / (2 * run)) * (2 * run);
      const bool second = i - base >= run;
      const long long x_lo = base + (second ? run : 0), y_lo = base + (second ? 0 : run);
      const long long y_len = max(0ll, min(run, (long long)k - y_lo));
      const unsigned long long key = src[i];
      long long lo = 0, hi = y_len;                       // number of keys of the other run that precede `key`
      while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (src[y_lo + mid] > key) lo = mid + 1;
        else hi = mid;
      }
      dst[base + (i - x_lo) + lo] = key;
    }
    __syncthreads();
    unsigned long long* t = src; src = dst; dst = t;
  }
  if (src != buf_a) {
    for (int i = tid; i < k; i += kSortThreads) buf_a[i] = src[i];
    __syncthreads();
  }
}
