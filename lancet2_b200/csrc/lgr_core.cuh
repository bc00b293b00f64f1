// lgr_core.cuh — scalar (one lane = one (read, haplotype) pair) device logic of the
// realignment path.  Everything here is `__host__ __device__` so that the very same
// code is (a) what the sm_100a kernels in lgr_kernels.cu execute per lane and (b)
// compiled by g++ into tests/hostemu (test infrastructure) to check the control
// flow against the oracle without a GPU.  It is NOT a CPU fallback: the product
// library never calls it on the host.
//
// What it implements (reference call sites → minimap2 2.30 stage, see DESIGN.md):
//   genotyper.cpp:250  mm_idx_str     → sketch() + sorted minimizer table
//   genotyper.cpp:387  mm_map         → map_chain_phase(): seeds, anchors, chain DP,
//                                        backtrack, regs, parent/sub selection,
//                                        SR max-stretch + extension windows
//                                      ext_dp_scalar(): ksw2 extz (pruned, exact)
//                                      finish_pair(): cigar assembly, mm_fix_cigar,
//                                        mm_update_extra, filter, hit sort, NM
//   genotyper.cpp:269-321 / combined_scorer.cpp:60-108 / local_scorer.cpp:166-305
//                                    → score_read_variant()
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define LGR_HD __host__ __device__ __forceinline__
#define LGR_HDN __host__ __device__ __noinline__
#else
#include <cmath>
#include <cstring>
#define LGR_HD inline
#define LGR_HDN inline
#endif

namespace lgr {

// ------------------------------------------------------------------------------------
// parameters as the device sees them
// ------------------------------------------------------------------------------------
struct DevParams {
  int32_t k, w, a, b, q, e, sc_ambi, bw, end_bonus;
  int32_t max_gap, max_gap_ref, max_skip, max_iter, min_cnt, min_sc, min_dp_max;
  int32_t max_max_occ, occ_dist, best_n, seed, mask_len;
  float pen_gap, pen_skip, mask_level, pri_ratio, max_clip_ratio, q_occ_frac;
  int32_t min_strand_sc;  // (int)(max_gap * 0.8)
};

constexpr int kSmallCells = 512;            // extension tails with at most this many (pruned) DP cells run inline
constexpr int kSmallDim = 22;               // floor(sqrt(kSmallCells)): bound of min(m, T) for such a tail
constexpr int kSmallCig = 96;               // cigar runs of such a tail (<= 4*min(m,T)+1; overflow is flagged)
constexpr int kInlineCig = 6;               // cigar ops kept inline in an ExtRec
constexpr int kMaxWindow = 32;              // minimizer window cap (reference uses w = 5)
constexpr int32_t kNegInf = -0x40000000;
#ifdef LGR_CORE_SELFCHECK
// host emulation only (tests/hostemu): closed forms of the warp kernels checked against the scalar paths
static long long lgr_selfcheck_failures = 0, lgr_selfcheck_colinear_seen = 0, lgr_selfcheck_ext_seen = 0, lgr_selfcheck_tail_seen = 0, lgr_selfcheck_sorted_seen = 0;
#endif

// strided view: element i of a per-lane array interleaved over S lanes
template <typename T, int S>
struct Strided {
  T* p;
  LGR_HD T& operator[](int i) const { return p[(size_t)i * S]; }
};

// code byte per base: low nibble = minimap2 nt4 code (0..3, 4 = ambiguous),
// high nibble = Lancet ENCODE_TABLE code (scoring_constants.h:48-74; U is 4 there)
LGR_HD uint8_t encode_base(uint8_t c) {
  uint8_t mm = 4, ln = 4;
  switch (c) {
    case 'A': case 'a': mm = 0; ln = 0; break;
    case 'C': case 'c': mm = 1; ln = 1; break;
    case 'G': case 'g': mm = 2; ln = 2; break;
    case 'T': case 't': mm = 3; ln = 3; break;
    case 'U': case 'u': mm = 3; ln = 4; break;
    default: break;
  }
  return (uint8_t)(mm | (ln << 4));
}

// ------------------------------------------------------------------------------------
// hashes (minimap2 sketch.c hash64 with mask; hit.c hash64; khash.h Wang / X31)
// ------------------------------------------------------------------------------------
LGR_HD uint64_t hash64_mask(uint64_t key, uint64_t mask) {
  key = (~key + (key << 21)) & mask;
  key = key ^ key >> 24;
  key = ((key + (key << 3)) + (key << 8)) & mask;
  key = key ^ key >> 14;
  key = ((key + (key << 2)) + (key << 4)) & mask;
  key = key ^ key >> 28;
  key = (key + (key << 31)) & mask;
  return key;
}
// the same function in 32-bit arithmetic, exact whenever the mask has at most 32 bits (k <= 16):
// adds and left shifts commute with reduction mod 2^32 and every right shift acts on a value
// already reduced by the mask
LGR_HD uint32_t hash64_mask_narrow(uint32_t key, uint32_t mask) {
  key = (~key + (key << 21)) & mask;
  key = key ^ key >> 24;
  key = ((key + (key << 3)) + (key << 8)) & mask;
  key = key ^ key >> 14;
  key = ((key + (key << 2)) + (key << 4)) & mask;
  key = key ^ key >> 28;
  key = (key + (key << 31)) & mask;
  return key;
}
LGR_HD uint64_t hash64_full(uint64_t key) {
  key = ~key + (key << 21);
  key = key ^ key >> 24;
  key = ((key + (key << 3)) + (key << 8));
  key = key ^ key >> 14;
  key = ((key + (key << 2)) + (key << 4));
  key = key ^ key >> 28;
  key = key + (key << 31);
  return key;
}
LGR_HD uint32_t wang_hash(uint32_t key) {
  key += ~(key << 15);
  key ^= (key >> 10);
  key += (key << 3);
  key ^= (key >> 6);
  key += ~(key << 11);
  key ^= (key >> 16);
  return key;
}

// ------------------------------------------------------------------------------------
// minimizer sketch (minimap2 sketch.c: mm_sketch, non-HPC).  codes: nt4 in low nibble.
// Emits (x = hash<<8 | span, y = pos<<1 | strand) in upstream order.  Returns the count;
// entries beyond `cap` are counted but not stored.
// ------------------------------------------------------------------------------------
template <typename OutX, typename OutY>
LGR_HD int sketch(const uint8_t* codes, int len, int w, int k, OutX out_x, OutY out_y, int cap) {
  const uint64_t shift1 = 2 * (k - 1), mask = (1ULL << 2 * k) - 1;
  uint64_t kmer0 = 0, kmer1 = 0;
  uint64_t bx[kMaxWindow];
  uint32_t by[kMaxWindow];
  for (int j = 0; j < w; ++j) bx[j] = UINT64_MAX, by[j] = UINT32_MAX;
  uint64_t min_x = UINT64_MAX;
  uint32_t min_y = UINT32_MAX;
  int l = 0, buf_pos = 0, min_pos = 0, kmer_span = 0, n = 0;
#define LGR_EMIT(X, Y)                       \
  do {                                       \
    if (n < cap) out_x[n] = (X), out_y[n] = (Y); \
    ++n;                                     \
  } while (0)
  for (int i = 0; i < len; ++i) {
    const int c = codes[i] & 0xf;
    uint64_t ix = UINT64_MAX;
    uint32_t iy = UINT32_MAX;
    if (c < 4) {
      kmer_span = l + 1 < k ? l + 1 : k;
      kmer0 = (kmer0 << 2 | (uint64_t)c) & mask;
      kmer1 = (kmer1 >> 2) | (3ULL ^ (uint64_t)c) << shift1;
      if (kmer0 == kmer1) continue;
      const int z = kmer0 < kmer1 ? 0 : 1;
      ++l;
      if (l >= k && kmer_span < 256) {
        ix = hash64_mask(z ? kmer1 : kmer0, mask) << 8 | (uint64_t)kmer_span;
        iy = (uint32_t)i << 1 | (uint32_t)z;
      }
    } else {
      l = 0;
      kmer_span = 0;
    }
    bx[buf_pos] = ix, by[buf_pos] = iy;
    if (l == w + k - 1 && min_x != UINT64_MAX) {
      for (int j = buf_pos + 1; j < w; ++j)
        if (min_x == bx[j] && by[j] != min_y) LGR_EMIT(bx[j], by[j]);
      for (int j = 0; j < buf_pos; ++j)
        if (min_x == bx[j] && by[j] != min_y) LGR_EMIT(bx[j], by[j]);
    }
    if (ix <= min_x) {
      if (l >= w + k && min_x != UINT64_MAX) LGR_EMIT(min_x, min_y);
      min_x = ix, min_y = iy, min_pos = buf_pos;
    } else if (buf_pos == min_pos) {
      if (l >= w + k - 1 && min_x != UINT64_MAX) LGR_EMIT(min_x, min_y);
      min_x = UINT64_MAX;
      for (int j = buf_pos + 1; j < w; ++j)
        if (min_x >= bx[j]) min_x = bx[j], min_y = by[j], min_pos = j;
      for (int j = 0; j <= buf_pos; ++j)
        if (min_x >= bx[j]) min_x = bx[j], min_y = by[j], min_pos = j;
      if (l >= w + k - 1 && min_x != UINT64_MAX) {
        for (int j = buf_pos + 1; j < w; ++j)
          if (min_x == bx[j] && min_y != by[j]) LGR_EMIT(bx[j], by[j]);
        for (int j = 0; j <= buf_pos; ++j)
          if (min_x == bx[j] && min_y != by[j]) LGR_EMIT(bx[j], by[j]);
      }
    }
    if (++buf_pos == w) buf_pos = 0;
  }
  if (min_x != UINT64_MAX) LGR_EMIT(min_x, min_y);
#undef LGR_EMIT
  return n;
}

// ------------------------------------------------------------------------------------
// sketch_sr<W>: the same mm_sketch state machine with the w-slot ring buffer unrolled into
// a shift register of compile-time width, so that every slot lives in a register (the ring
// buffer version indexes its slots dynamically, which puts them in local memory and the
// per-base latency of the one-lane-per-sequence sketch kernels is exactly that).
// Ring → shift register: after the write, slots read oldest → newest are win[0..W-1]; the
// minimum's slot index drops by one per write and "buf_pos == min_pos" is "index fell below 0".
// emit(x, y) receives the minimizers in upstream order; returns their count.
// ------------------------------------------------------------------------------------
// The window state machine of mm_sketch on its own: step(ix, iy, l) consumes the k-mer record of
// one base (ix = UINT64_MAX when the base has no valid k-mer; l = number of consecutive
// unambiguous bases ending here, 0 for an ambiguous base) — shared by the sequential sketch
// below and by the warp kernel that computes the records 32 at a time.
template <int W, typename XT = uint64_t>
struct MinimizerWindow {
  static constexpr XT kMax = (XT)~(XT)0;
  XT wx[W];
  uint32_t wy[W];
  XT min_x;
  uint32_t min_y;
  int min_idx, k;
  LGR_HD void init(int k_) {
#pragma unroll
    for (int j = 0; j < W; ++j) wx[j] = kMax, wy[j] = UINT32_MAX;
    min_x = kMax, min_y = UINT32_MAX, min_idx = W - 1, k = k_;
  }
  // One position of mm_sketch's window loop.  Written so that the common emission (the old
  // minimum, when a new record takes over or the minimum leaves the window) has ONE call site
  // and the rescan is a select chain: lanes of a warp that sketch different sequences then
  // diverge only on that one short predicated block, not on four copies of it.  The two
  // "identical k-mer" emission loops stay as (rare) branches.
  template <typename Emit>
  LGR_HD void step(XT ix, uint32_t iy, int l, Emit& emit) {
#pragma unroll
    for (int j = 0; j + 1 < W; ++j) wx[j] = wx[j + 1], wy[j] = wy[j + 1];
    wx[W - 1] = ix, wy[W - 1] = iy;
    --min_idx;
    const bool have_min = min_x != kMax;
    if (l == W + k - 1 && have_min) {  // first full window of a run: identical k-mers not stored yet
#pragma unroll
      for (int j = 0; j + 1 < W; ++j)
        if (min_x == wx[j] && wy[j] != min_y) emit(min_x, wy[j]);
    }
    const bool takes_over = ix <= min_x;
    const bool fell_out = !takes_over && min_idx < 0;
    if (have_min && ((takes_over && l >= W + k) || (fell_out && l >= W + k - 1))) emit(min_x, min_y);
    // right-most minimum of the window (what the rescan finds); only used when the old one fell out
    XT rx = kMax;
    uint32_t ry = UINT32_MAX;
    int ri = W - 1;
#pragma unroll
    for (int j = 0; j < W; ++j) {
      const bool le = rx >= wx[j];
      rx = le ? wx[j] : rx, ry = le ? wy[j] : ry, ri = le ? j : ri;
    }
    if (takes_over) {
      min_x = ix, min_y = iy, min_idx = W - 1;
    } else if (fell_out) {
      min_x = rx, min_y = ry, min_idx = ri;
      if (l >= W + k - 1 && rx != kMax) {
        bool any = false;
#pragma unroll
        for (int j = 0; j < W; ++j) any |= rx == wx[j] && ry != wy[j];
        if (any) {
#pragma unroll
          for (int j = 0; j < W; ++j)
            if (rx == wx[j] && ry != wy[j]) emit(rx, wy[j]);
        }
      }
    }
  }
  template <typename Emit>
  LGR_HD void finish(Emit& emit) {
    if (min_x != kMax) emit(min_x, min_y);
  }
};

// XT = uint32_t is exact for 2k + 8 <= 32 (hash << 8 | span fits, and never equals the all-ones
// "no k-mer" marker); Emit always receives the 64-bit record value.
template <int W, typename XT, typename Emit>
LGR_HD int sketch_sr_impl(const uint8_t* codes, int len, int k, Emit emit) {
  const int shift1 = 2 * (k - 1);
  const XT mask = (XT)(((uint64_t)1 << 2 * k) - 1);
  XT kmer0 = 0, kmer1 = 0;
  MinimizerWindow<W, XT> win;
  win.init(k);
  int l = 0, kmer_span = 0, n = 0;
  auto count_emit = [&](XT x, uint32_t y) { emit((uint64_t)x, y), ++n; };
  for (int i = 0; i < len; ++i) {
    const int c = codes[i] & 0xf;
    XT ix = MinimizerWindow<W, XT>::kMax;
    uint32_t iy = UINT32_MAX;
    if (c < 4) {
      kmer_span = l + 1 < k ? l + 1 : k;
      kmer0 = (kmer0 << 2 | (XT)c) & mask;
      kmer1 = (kmer1 >> 2) | ((XT)3 ^ (XT)c) << shift1;
      if (kmer0 == kmer1) continue;
      const int z = kmer0 < kmer1 ? 0 : 1;
      ++l;
      if (l >= k && kmer_span < 256) {
        const XT key = z ? kmer1 : kmer0;
        const XT hv = sizeof(XT) == 4 ? (XT)hash64_mask_narrow((uint32_t)key, (uint32_t)mask) : (XT)hash64_mask((uint64_t)key, (uint64_t)mask);
        ix = hv << 8 | (XT)kmer_span;
        iy = (uint32_t)i << 1 | (uint32_t)z;
      }
    } else {
      l = 0;
      kmer_span = 0;
    }
    win.step(ix, iy, l, count_emit);
  }
  win.finish(count_emit);
  return n;
}

template <int W, typename Emit>
LGR_HD int sketch_sr(const uint8_t* codes, int len, int k, Emit emit) {
  if (2 * k + 8 <= 32) return sketch_sr_impl<W, uint32_t>(codes, len, k, emit);
  return sketch_sr_impl<W, uint64_t>(codes, len, k, emit);
}

// dispatcher: register-resident window for the reference's w = 5, ring buffer otherwise.
// Stores at most `cap` minimizers through out_x / out_y; returns the full count.
template <typename OutX, typename OutY>
LGR_HD int sketch_any(const uint8_t* codes, int len, int w, int k, OutX out_x, OutY out_y, int cap) {
  if (w == 5) {
    int m = 0;
    return sketch_sr<5>(codes, len, k, [&](uint64_t x, uint32_t y) {
      if (m < cap) out_x[m] = x, out_y[m] = y;
      ++m;
    });
  }
  return sketch(codes, len, w, k, out_x, out_y, cap);
}

// ------------------------------------------------------------------------------------
// seed.c: mm_seed_mz_flt — drop query minimizers that occur more than q_occ_max times in
// the query and more than q_occ_frac of all its minimizers.  Count based, so the unstable
// sort upstream uses to group them does not matter.  In place; returns the new count.
// ------------------------------------------------------------------------------------
template <typename X, typename Y>
LGR_HD int seed_mz_flt(X mz_x, Y mz_y, int n, int q_occ_max, float q_occ_frac) {
  if (n <= q_occ_max || q_occ_frac <= 0.0f || q_occ_max <= 0) return n;
  bool any = false;
  for (int i = 0; i < n; ++i) {
    int cnt = 0;
    const uint64_t xi = mz_x[i];
    for (int j = 0; j < n; ++j) cnt += (mz_x[j] == xi) ? 1 : 0;
    if (cnt > q_occ_max && (float)cnt > (float)n * q_occ_frac) mz_y[i] |= 0x80000000u, any = true;
  }
  if (!any) return n;
  int j = 0;
  for (int i = 0; i < n; ++i) {
    if (mz_y[i] & 0x80000000u) continue;
    mz_x[j] = mz_x[i], mz_y[j] = mz_y[i];
    ++j;
  }
  return j;
}

// ------------------------------------------------------------------------------------
// index.c: mm_idx_cal_max_occ + options.c: mm_mapopt_update's clamp → the mid_occ a
// Genotyper latches from a haplotype (genotyper.cpp:263-266).  idx: sorted table
// (hash<<17 | pos<<1|strand).  thres = (kk-th smallest occurrence count) + 1 with
// kk = (uint32)((1 - f) * n_keys).
// ------------------------------------------------------------------------------------
LGR_HD int32_t hap_mid_occ(const uint64_t* idx, int n, float f, int32_t min_mid_occ, int32_t max_mid_occ) {
  int32_t mid = INT32_MAX;
  if (f > 0.f && n > 0) {
    int n_keys = 0, max_run = 0;
    for (int i = 0; i < n;) {
      int j = i + 1;
      while (j < n && (idx[j] >> 17) == (idx[i] >> 17)) ++j;
      ++n_keys;
      if (j - i > max_run) max_run = j - i;
      i = j;
    }
    const uint32_t kk = (uint32_t)((1. - (double)f) * (double)n_keys);
    for (int v = 1; v <= max_run; ++v) {
      uint32_t le = 0;
      for (int i = 0; i < n;) {
        int j = i + 1;
        while (j < n && (idx[j] >> 17) == (idx[i] >> 17)) ++j;
        if (j - i <= v) ++le;
        i = j;
      }
      if (le > kk) { mid = v + 1; break; }
    }
  }
  if (mid < min_mid_occ) mid = min_mid_occ;
  if (max_mid_occ > min_mid_occ && mid > max_mid_occ) mid = max_mid_occ;
  return mid;
}

// ------------------------------------------------------------------------------------
// exact emulation of ksort.h radix_sort (in-place MSD radix, 8 bits/pass, insertion
// sort for <= 64 elements) on a permutation array: perm[i] holds element ids, key(id)
// their 64-bit sort key.  minimap2's results depend on this (unstable) permutation
// whenever keys tie and n > 64, so it is reproduced move for move.
// ------------------------------------------------------------------------------------
// The pending-range stack holds ranges of more than 64 elements that are pairwise disjoint, so
// n <= 65535 (the 16-bit positions) never needs more than 65535 / 65 = 1008 entries.
struct RadixScratch {     // per-lane, lives in local memory; only touched when n > 64
  uint16_t bb[256], be[256];
  uint16_t st_beg[1024], st_end[1024];
  uint8_t st_s[1024];
};

template <typename Perm, typename KeyFn>
LGR_HD void insertion_sort_perm(Perm perm, int beg, int end, KeyFn key) {
  for (int i = beg + 1; i < end; ++i) {
    const int32_t tmp = perm[i];
    const uint64_t kt = key(tmp);
    if (kt < key(perm[i - 1])) {
      int j;
      for (j = i; j > beg && kt < key(perm[j - 1]); --j) perm[j] = perm[j - 1];
      perm[j] = tmp;
    }
  }
}

template <typename Perm, typename KeyFn>
LGR_HDN void radix_sort_perm(Perm perm, int n, KeyFn key, RadixScratch* rs) {
  if (n <= 64) {
    insertion_sort_perm(perm, 0, n, key);
    return;
  }
  int sp = 0;
  rs->st_beg[0] = 0, rs->st_end[0] = (uint16_t)n, rs->st_s[0] = 56, sp = 1;
  while (sp > 0) {
    --sp;
    const int beg = rs->st_beg[sp], end = rs->st_end[sp];
    int s = rs->st_s[sp];
    {
      // A level at which all keys of the range share the byte puts them in one bucket: the
      // permutation loop moves nothing and (the range being > 64) the next level gets the same
      // range.  Jump straight to the highest byte that differs; none left = nothing to do.
      const uint64_t k0 = key(perm[beg]);
      uint64_t diff = 0;
      for (int i = beg + 1; i < end; ++i) diff |= key(perm[i]) ^ k0;
      if (s < 56) diff &= (1ULL << (s + 8)) - 1;
      if (diff == 0) continue;
      int top = 0;
      for (uint64_t d = diff >> 8; d; d >>= 8) ++top;
      s = 8 * top;
    }
    // only the buckets between the smallest and the largest byte present can be non-empty;
    // everything the full 256-bucket loops would do outside that span is a no-op
    int kmin = 255, kmax = 0;
    for (int i = beg; i < end; ++i) {
      const int b = (int)(key(perm[i]) >> s & 255);
      kmin = b < kmin ? b : kmin, kmax = b > kmax ? b : kmax;
    }
    for (int k = kmin; k <= kmax; ++k) rs->bb[k] = rs->be[k] = (uint16_t)beg;  // be[] = counts first
    for (int i = beg; i < end; ++i) ++rs->be[(int)(key(perm[i]) >> s & 255)];
    // k->e += (k-1)->e - beg ; k->b = (k-1)->e
    for (int k = kmin + 1; k <= kmax; ++k) {
      rs->be[k] = (uint16_t)(rs->be[k] + rs->be[k - 1] - beg);
      rs->bb[k] = rs->be[k - 1];
    }
    for (int k = kmin; k <= kmax;) {
      if (rs->bb[k] != rs->be[k]) {
        int l = (int)(key(perm[rs->bb[k]]) >> s & 255);
        if (l != k) {
          int32_t tmp = perm[rs->bb[k]], swp;
          do {
            swp = tmp;
            tmp = perm[rs->bb[l]];
            perm[rs->bb[l]++] = swp;
            l = (int)(key(tmp) >> s & 255);
          } while (l != k);
          perm[rs->bb[k]++] = tmp;
        } else {
          ++rs->bb[k];
        }
      } else {
        ++k;
      }
    }
    if (s) {
      const int s2 = s > 8 ? s - 8 : 0;
      int b0 = beg;
      for (int k = kmin; k <= kmax; ++k) {
        const int e0 = rs->be[k];
        if (e0 - b0 > 64) {
          rs->st_beg[sp] = (uint16_t)b0, rs->st_end[sp] = (uint16_t)e0, rs->st_s[sp] = (uint8_t)s2;
          ++sp;
        } else if (e0 - b0 > 1) {
          insertion_sort_perm(perm, b0, e0, key);
        }
        b0 = e0;
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// chain scoring (minimap2 lchain.c: comput_sc, mg_log2 with the FMA contraction the
// reference's -O3 -march=x86-64-v3 build applies; see oracle/mm2_restate.cpp)
// ------------------------------------------------------------------------------------
LGR_HD float mg_log2(float x) {
  union {
    float f;
    uint32_t i;
  } z;
  z.f = x;
  float log_2 = (float)(int)(((z.i >> 23) & 255) - 128);
  z.i &= ~(255u << 23);
  z.i += 127u << 23;
#if defined(__CUDA_ARCH__)
  const float t = __fmaf_rn(-0.34484843f, z.f, 2.02466578f);
  log_2 = __fadd_rn(log_2, __fmaf_rn(t, z.f, -0.67487759f));
#else
  const float t = std::fmaf(-0.34484843f, z.f, 2.02466578f);
  log_2 += std::fmaf(t, z.f, -0.67487759f);
#endif
  return log_2;
}

// anchors are kept as two 32-bit words:
//   x32 = rev<<31 | rpos            (upstream x = rev<<63 | rid<<32 | rpos, rid = 0)
//   y32 = tandem<<24 | span<<16 | qpos   (upstream y = flags<<40 | span<<32 | qpos)
LGR_HD int32_t anchor_qpos(uint32_t y32) { return (int32_t)(y32 & 0xffff); }
LGR_HD int32_t anchor_span(uint32_t y32) { return (int32_t)(y32 >> 16 & 0xff); }
LGR_HD int32_t anchor_rpos(uint32_t x32) { return (int32_t)(x32 & 0x7fffffffu); }
LGR_HD uint64_t anchor_x64(uint32_t x32) { return (uint64_t)(x32 >> 31) << 63 | (uint64_t)(x32 & 0x7fffffffu); }
LGR_HD uint64_t anchor_y64(uint32_t y32) {
  return (uint64_t)(y32 >> 24 & 1) << 42 | (uint64_t)(y32 >> 16 & 0xff) << 32 | (uint64_t)(y32 & 0xffff);
}

LGR_HD int32_t comput_sc(uint32_t xi, uint32_t yi, uint32_t xj, uint32_t yj, int32_t max_dist_x,
                         int32_t max_dist_y, int32_t bw, float pen_gap, float pen_skip) {
  const int32_t dq = anchor_qpos(yi) - anchor_qpos(yj);
  if (dq <= 0 || dq > max_dist_x) return INT32_MIN;
  const int32_t dr = anchor_rpos(xi) - anchor_rpos(xj);  // same strand guaranteed by the caller
  if (dr == 0 || dq > max_dist_y) return INT32_MIN;
  const int32_t dd = dr > dq ? dr - dq : dq - dr;
  if (dd > bw) return INT32_MIN;
  const int32_t dg = dr < dq ? dr : dq;
  const int32_t q_span = anchor_span(yj);
  int32_t sc = q_span < dg ? q_span : dg;
  if (dd || dg > q_span) {
#if defined(__CUDA_ARCH__)
    const float lin_pen = __fadd_rn(__fmul_rn(pen_gap, (float)dd), __fmul_rn(pen_skip, (float)dg));
    const float log_pen = dd >= 1 ? mg_log2((float)(dd + 1)) : 0.0f;
    sc -= (int)__fadd_rn(lin_pen, __fmul_rn(.5f, log_pen));
#else
    const float m1 = pen_gap * (float)dd;
    const float m2 = pen_skip * (float)dg;
    const float lin_pen = m1 + m2;
    const float log_pen = dd >= 1 ? mg_log2((float)(dd + 1)) : 0.0f;
    const float hl = .5f * log_pen;
    sc -= (int)(lin_pen + hl);
#endif
  }
  return sc;
}

// ------------------------------------------------------------------------------------
// per-lane workspace: a set of int32 arrays of `cap` elements, interleaved over S lanes
// ------------------------------------------------------------------------------------
enum WsArray {
  A_AX = 0, A_AY, A_SX, A_SY, A_F, A_P, A_T, A_V, A_Z, A_PERM,  // anchors / chaining
  A_SEEDQ, A_SEEDN, A_SEEDS,                                       // seeds
  A_CX, A_CY,                                                      // compacted anchors
  R_SCORE, R_CNT, R_AS, R_HASH, R_QS, R_QE, R_RS, R_RE, R_REV, R_PARENT, R_ID, R_AUX0, R_AUX1,
  A_COUNT
};

// LEAN: the layout of the lean chain kernel, which finishes only sorted co-linear pairs.  It never sorts (the
// sorted arrays ARE the anchor arrays), never needs the seed arrays once the anchors exist (they share the
// slots of f / p, which are written later), never runs the general chain DP or tail (no t, v, z, perm,
// compacted anchors) and holds one reg: 5 anchor-sized arrays instead of 15, so that more CTAs fit an SM.
template <int S, bool LEAN = false>
struct Ws {
  int32_t* base;  // already offset to this lane
  // capacities, packed (keeps the struct at two words: a third member made nvcc lose track of
  // the shared address space of `base` in k_chain_warp and fall back to generic LD/ST):
  // low 16 bits = elements of the anchor-sized arrays (A_*), high bits = elements of the
  // chain/reg-sized arrays (R_*; 0 = same as the anchor arrays).  A pair with more chains
  // than that overflows.
  int caps;
  static constexpr int kSlots = LEAN ? 5 : (int)R_SCORE;
  static LGR_HD constexpr int slot(int k) {
    if (!LEAN) return k;
    switch (k) {
      case A_AX: case A_SX: return 0;
      case A_AY: case A_SY: return 1;
      case A_F: case A_SEEDQ: return 2;
      case A_P: case A_SEEDN: return 3;
      default: return 4;  // A_SEEDS; the arrays of the general DP and tail are not used with this layout
    }
  }
  LGR_HD int cap() const { return caps & 0xffff; }
  LGR_HD int rcap() const { return caps >> 16 ? caps >> 16 : caps; }
  static LGR_HD int pack(int cap_, int rcap_) { return cap_ | rcap_ << 16; }
  LGR_HD Strided<int32_t, S> arr(int k) const {
    const int off = k < R_SCORE ? slot(k) * cap() : kSlots * cap() + (k - R_SCORE) * rcap();
    return Strided<int32_t, S>{base + (size_t)off * S};
  }
  static LGR_HD size_t elems(int cap_, int rcap_) { return (size_t)kSlots * cap_ + (size_t)(A_COUNT - R_SCORE) * rcap_; }
};

// ------------------------------------------------------------------------------------
// records exchanged between the kernels (HBM)
// ------------------------------------------------------------------------------------
struct ExtRec {          // one ksw2 extension (left or right tail of a reg)
  int32_t m;             // query bases in the tail (0 = no extension on this side)
  int32_t n;             // target bases available (full window, before pruning)
  int32_t mqe_t;         // out: target offset of the best last-row cell
  int32_t max;           // out: ez.max
  int32_t n_cig;         // out
  int32_t cig_off;       // out: <0 inline, else offset in the extension cigar arena
  uint32_t inl[kInlineCig];
};

struct RegRec {          // one chain selected for base-level alignment (mm_reg1_t subset)
  int32_t score, cnt;
  uint32_t hash;
  int32_t rev;
  int32_t c_qs, c_qe, c_rs, c_re;  // SR max-stretch core, query coords on the reg's strand
  int32_t rs0, re0;                // extension window on the haplotype
  ExtRec ext[2];                   // [0] = left, [1] = right
};

struct AlnOut {          // mirrors lgr_aln (include/lancet_gpu_realign.h)
  int32_t valid, score, rs, re, qs, qe, rev, dp_score, dp_max, mlen, blen, n_ambi, nm, n_cigar,
      cigar_off, n_regs;
};

struct AssignOut {       // mirrors lgr_assign
  double local_score, local_identity, folded_read_pos;
  int32_t global_score;
  uint32_t ref_nm, own_hap_nm, hap_id;
  int8_t allele;
  uint8_t base_qual, assigned, pad[5];
};

// ------------------------------------------------------------------------------------
// ksw2 extension DP, scalar, pruned to the first T target columns (exact: see DESIGN.md
// "column pruning").  q[j] / t[i] are nt4 codes fetched through functors so that the
// caller can present reversed / reverse-complemented views without copies.
// dir: scratch of m*T bytes.  Emits the cigar through `push(op,len)` in upstream order.
// ------------------------------------------------------------------------------------
LGR_HD int prune_cols(const DevParams& P, int m, int n) {
  const int mm = P.b > P.sc_ambi ? P.b : P.sc_ambi;
  const int X = (P.a + mm) * m - P.q;
  const int D = X < 0 ? 0 : X / P.e;
  const int T = m + D;
  return T < n ? T : n;
}

LGR_HD int sub_score(const DevParams& P, int tc, int qc) {
  if (tc > 3 || qc > 3) return -P.sc_ambi;
  return tc == qc ? P.a : -P.b;
}

struct CigBuf {          // run-length cigar builder (ksw_push_cigar semantics)
  uint32_t* ops;
  int n, cap;
  LGR_HD void push(uint32_t op, int len) {
    if (n > 0 && n <= cap && op == (ops[n - 1] & 0xf)) {
      ops[n - 1] += (uint32_t)len << 4;
    } else {
      if (n < cap) ops[n] = (uint32_t)len << 4 | op;
      ++n;  // n > cap flags an overflow to the caller
    }
  }
};

// One cell of the recurrence (shared by both sweep orders and by the warp kernel's lanes
// in spirit): returns H, writes the direction byte and the E/F values flowing right/down.
LGR_HD int32_t ext_cell(int32_t hd, int32_t ee, int32_t f, int q, int e, bool right, uint8_t* dout, int32_t* e_next,
                        int32_t* f_next) {
  int32_t h;
  uint8_t d;
  if (!right) {
    d = ee > hd ? 1 : 0;
    h = ee > hd ? ee : hd;
    if (f > h) d = 2, h = f;
  } else {
    d = hd > ee ? 0 : 1;
    h = hd > ee ? hd : ee;
    if (!(h > f)) d = 2, h = f;
  }
  const int32_t ho = h - q;
  if (!right) {
    if (ee > ho) d |= 0x08;
    if (f > ho) d |= 0x10;
  } else {
    if (ee >= ho) d |= 0x08;
    if (f >= ho) d |= 0x10;
  }
  *dout = d;
  *e_next = (ee > ho ? ee : ho) - e;
  *f_next = (f > ho ? f : ho) - e;
  return h;
}

// ha/fa: scratch of min(m, T) ints each.  The sweep keeps its line buffers over the
// SHORTER dimension (reads overhanging a haplotype end give m ~ 100, T ~ 3), the values
// are independent of the sweep order.
template <typename QF, typename TF>
LGR_HD void ext_dp_scalar(const DevParams& P, int m, int T, QF qf, TF tf, bool right, uint8_t* dir,
                          int32_t* ha, int32_t* fa, int32_t* out_max, int32_t* out_mqe_t) {
  const int q = P.q, e = P.e;
  int32_t ezmax = 0, mqe = kNegInf, mqe_t = -1;
  if (m <= T) {
    // target-major: ha[j] = H(i-1, j), fa[j] = E(i, j) (flows along the target)
    for (int j = 0; j < m; ++j) {
      ha[j] = -(q + e * (j + 1));
      fa[j] = ha[j] - q - e;
    }
    for (int i = 0; i < T; ++i) {
      int32_t hdiag = i == 0 ? 0 : -(q + e * i);
      int32_t f = -(q + e * (i + 1)) - q - e;
      const int tc = tf(i);
      for (int j = 0; j < m; ++j) {
        const int32_t hd = hdiag + sub_score(P, tc, qf(j));
        int32_t en, fn;
        const int32_t h = ext_cell(hd, fa[j], f, q, e, right, &dir[i * m + j], &en, &fn);
        hdiag = ha[j];
        ha[j] = h;
        fa[j] = en;
        f = fn;
        if (h > ezmax) ezmax = h;
      }
      if (ha[m - 1] > mqe) mqe = ha[m - 1], mqe_t = i;
    }
  } else {
    // query-major: ha[i] = H(i, j-1), fa[i] = F(i, j) (flows along the query)
    for (int i = 0; i < T; ++i) {
      ha[i] = -(q + e * (i + 1));
      fa[i] = ha[i] - q - e;
    }
    for (int j = 0; j < m; ++j) {
      int32_t hdiag = j == 0 ? 0 : -(q + e * j);
      int32_t ee = -(q + e * (j + 1)) - q - e;
      const int qc = qf(j);
      for (int i = 0; i < T; ++i) {
        const int32_t hd = hdiag + sub_score(P, tf(i), qc);
        int32_t en, fn;
        const int32_t h = ext_cell(hd, ee, fa[i], q, e, right, &dir[i * m + j], &en, &fn);
        hdiag = ha[i];
        ha[i] = h;
        ee = en;
        fa[i] = fn;
        if (h > ezmax) ezmax = h;
        if (j == m - 1 && h > mqe) mqe = h, mqe_t = i;
      }
    }
  }
  *out_max = ezmax;
  *out_mqe_t = mqe_t;
}

// ksw2.h: ksw_backtrack from (i0, m-1); dirf(i, j) returns the direction byte of cell
// (target i, query j).  `rev_cigar`: keep the backtrack order (left extension), else
// reverse at the end.
template <typename DirF>
LGR_HD void ext_backtrack(DirF dirf, int m, int i0, bool rev_cigar, CigBuf& cb) {
  int i = i0, j = m - 1, state = 0;
  while (i >= 0 && j >= 0) {
    const uint8_t tmp = dirf(i, j);
    if (state == 0) state = tmp & 7;
    else if (!(tmp >> (state + 2) & 1)) state = 0;
    if (state == 0) state = tmp & 7;
    if (state == 0) cb.push(0, 1), --i, --j;
    else if (state == 1) cb.push(2, 1), --i;
    else cb.push(1, 1), --j;
  }
  if (i >= 0) cb.push(2, i + 1);
  if (j >= 0) cb.push(1, j + 1);
  if (!rev_cigar && cb.n <= cb.cap) {
    for (int a = 0; a < cb.n >> 1; ++a) {
      const uint32_t t = cb.ops[a];
      cb.ops[a] = cb.ops[cb.n - 1 - a];
      cb.ops[cb.n - 1 - a] = t;
    }
  }
}

// ------------------------------------------------------------------------------------
// sequence views
// ------------------------------------------------------------------------------------
struct ReadView {        // read codes, forward strand in memory
  const uint8_t* codes;
  int qlen;
  // nt4 code of base i on strand `rev` (rev = reverse complement, as align.c qseq0[1])
  LGR_HD int at(int rev, int i) const {
    if (!rev) return codes[i] & 0xf;
    const int c = codes[qlen - 1 - i] & 0xf;
    return c < 4 ? 3 - c : 4;
  }
};

struct PairIn {          // everything phase A needs about one (read, haplotype) pair
  ReadView read;
  const uint8_t* hap;    // hap codes
  int hap_len;
  const uint64_t* idx;   // sorted (hash<<17 | pos<<1|strand)
  int idx_n;
  const uint64_t* mz_x;  // read minimizers after mm_seed_mz_flt
  const uint32_t* mz_y;
  int mz_n;
  uint32_t name_hash;
  int mid_occ;
};

struct ChainCounters {
  int64_t chain_evals, n_anchors, dp_cells, dp_cells_full;
};

// lower bound in the sorted minimizer table
LGR_HD int idx_lower_bound(const uint64_t* idx, int n, uint64_t key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (idx[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

constexpr int kIdxShift = 17;  // bits of (pos<<1|strand) below the hash in the table

// ------------------------------------------------------------------------------------
// seed.c: mm_seed_select — called only when some seed occurs more than mid_occ times.
// seedq packs q_pos (pos<<1|strand, 20 bits) | span<<20 | tandem<<28 | flt<<29.
// ------------------------------------------------------------------------------------
template <typename SQ, typename SN>
LGR_HD void seed_select(const DevParams& P, SQ seedq, SN seedn, int n_m, int qlen, int mid_occ) {
  {
    const int max_occ = mid_occ;
    if (P.occ_dist > 0 && P.max_max_occ > max_occ) {
      if (n_m > 1) {
        int last0 = -1;
        for (int i = 0; i <= n_m; ++i) {
          if (i == n_m || seedn[i] <= max_occ) {
            if (i - last0 > 1) {
              const int ps = last0 < 0 ? 0 : (int)(((uint32_t)seedq[last0] & 0xfffff) >> 1);
              const int pe = i == n_m ? qlen : (int)(((uint32_t)seedq[i] & 0xfffff) >> 1);
              const int st = last0 + 1, en = i;
              int max_high_occ = (int)((double)(pe - ps) / P.occ_dist + .499);
              if (max_high_occ > 0) {
                // upstream keeps a max-heap of (n<<32|j); the kept set is "replace the current
                // maximum when a strictly less frequent seed arrives".  max_high_occ <= 4 for
                // reads up to LGR_MAX_READ_LEN with occ_dist >= 256 (validated at create).
                uint64_t hb[8];
                if (max_high_occ > 8) max_high_occ = 8;
                int kb = 0, j = st;
                for (; j < en && kb < max_high_occ; ++j, ++kb) hb[kb] = (uint64_t)(uint32_t)seedn[j] << 32 | (uint32_t)j;
                for (; j < en; ++j) {
                  int top = 0;
                  for (int c = 1; c < kb; ++c)
                    if (hb[c] > hb[top]) top = c;
                  if (seedn[j] < (int32_t)(hb[top] >> 32)) hb[top] = (uint64_t)(uint32_t)seedn[j] << 32 | (uint32_t)j;
                }
                for (int c = 0; c < kb; ++c) seedq[(uint32_t)hb[c]] = (int32_t)((uint32_t)seedq[(uint32_t)hb[c]] | 1u << 29);
              }
              for (int j = st; j < en; ++j) seedq[j] = (int32_t)((uint32_t)seedq[j] ^ 1u << 29);
              for (int j = st; j < en; ++j)
                if (seedn[j] > P.max_max_occ) seedq[j] = (int32_t)((uint32_t)seedq[j] | 1u << 29);
            }
            last0 = i;
          }
        }
      }
    } else {
      for (int i = 0; i < n_m; ++i)
        if (seedn[i] > max_occ) seedq[i] = (int32_t)((uint32_t)seedq[i] | 1u << 29);
    }
  }
}

// status codes of map_chain_phase
enum { kMapNoHit = 0, kMapOk = 1, kMapOverflow = -1 };

// ------------------------------------------------------------------------------------
// Phase A, second half: from the chain DP result (sx/sy sorted anchors, f/p per anchor,
// n_a of them) to the surviving regs with their SR stretch and extension windows.  Scalar;
// run by every lane in the thread-per-pair kernel and by lane 0 in the warp-per-pair one.
// ------------------------------------------------------------------------------------
template <int S>
LGR_HDN int map_chain_tail(const DevParams& P, int qlen, int hap_len, uint32_t name_hash, const Ws<S>& ws,
                           RadixScratch* rsx, int n_a, int* n_regs_out) {
  auto ax = ws.arr(A_AX), ay = ws.arr(A_AY), sx = ws.arr(A_SX), sy = ws.arr(A_SY);
  auto f = ws.arr(A_F), p = ws.arr(A_P), t = ws.arr(A_T), v = ws.arr(A_V), z = ws.arr(A_Z);
  auto perm = ws.arr(A_PERM);
  *n_regs_out = 0;
  // ---- lchain.c: mg_chain_backtrack ------------------------------------------------------
  // z[k] = anchor ids with f >= min_sc sorted by f (radix_sort_128x on x = f); chains are
  // collected from the highest score down.  Output: chain c has score u_sc[c], count
  // u_cnt[c]; its anchors (in backtrack order, i.e. descending) in v[].
  auto u_sc = ws.arr(R_AUX0), u_cnt = ws.arr(R_AUX1);
  int n_u = 0, n_v = 0;
  {
    int n_z = 0;
    for (int i = 0; i < n_a; ++i)
      if (f[i] >= P.min_sc) z[n_z++] = i;
    if (n_z == 0) return kMapNoHit;
    radix_sort_perm(z, n_z, [&](int32_t id) { return (uint64_t)(uint32_t)f[id]; }, rsx);
    for (int i = 0; i < n_a; ++i) t[i] = 0;
    const int32_t max_drop = P.bw;
    for (int k = n_z - 1; k >= 0; --k) {
      const int zi = z[k];
      if (t[zi] != 0) continue;
      const int32_t zx = f[zi];
      // mg_chain_bk_end
      int end_i;
      {
        int i = zi, e_i = -1, max_i = i;
        int32_t max_s = 0;
        do {
          t[i] = 2;
          e_i = i = p[i];
          const int32_t s = i < 0 ? zx : zx - f[i];
          if (s > max_s) max_s = s, max_i = i;
          else if (max_s - s > max_drop) break;
        } while (i >= 0 && t[i] == 0);
        for (i = zi; i >= 0 && i != e_i; i = p[i]) t[i] = 0;
        end_i = max_i;
      }
      const int n_v0 = n_v;
      int i;
      for (i = zi; i != end_i; i = p[i]) v[n_v++] = i, t[i] = 1;
      const int32_t sc = i < 0 ? zx : zx - f[i];
      if (sc >= P.min_sc && n_v > n_v0 && n_v - n_v0 >= P.min_cnt) {
        if (n_u >= ws.rcap()) return kMapOverflow;
        u_sc[n_u] = sc, u_cnt[n_u] = n_v - n_v0;
        ++n_u;
      } else {
        n_v = n_v0;
      }
    }
  }
  if (n_u == 0) return kMapNoHit;
  // ---- lchain.c: compact_a ----------------------------------------------------------------
  // b[] = chains' anchors in ascending order, chain after chain; then chains are re-ordered
  // by the x of their first anchor (radix_sort_128x) and anchors copied in that order.
  auto cx = ws.arr(A_CX), cy = ws.arr(A_CY);
  auto r_score = ws.arr(R_SCORE), r_cnt = ws.arr(R_CNT), r_as = ws.arr(R_AS), r_hash = ws.arr(R_HASH);
  auto r_qs = ws.arr(R_QS), r_qe = ws.arr(R_QE), r_rs = ws.arr(R_RS), r_re = ws.arr(R_RE);
  auto r_rev = ws.arr(R_REV), r_parent = ws.arr(R_PARENT), r_id = ws.arr(R_ID);
  {
    // chain c occupies v[koff[c] .. koff[c]+cnt) reversed; keep offsets in t[] (free now)
    int k = 0;
    for (int c = 0; c < n_u; ++c) t[c] = k, k += u_cnt[c];
    for (int c = 0; c < n_u; ++c) perm[c] = c;
    // key: x of the first (lowest) anchor of the chain = last element of its v[] run
    radix_sort_perm(perm, n_u, [&](int32_t c) { return anchor_x64((uint32_t)sx[v[t[c] + u_cnt[c] - 1]]); }, rsx);
    k = 0;
    for (int i = 0; i < n_u; ++i) {
      const int c = perm[i], n = u_cnt[c], k0 = t[c];
      for (int j = 0; j < n; ++j) {
        const int id = v[k0 + (n - j - 1)];
        cx[k + j] = sx[id], cy[k + j] = sy[id];
      }
      // u2[i] = u[c]: stage in f/p (free now)
      f[i] = u_sc[c], p[i] = n;
      k += n;
    }
  }
  // ---- hit.c: mm_gen_regs --------------------------------------------------------------------
  uint32_t hash = name_hash;
  hash ^= wang_hash((uint32_t)qlen) + wang_hash((uint32_t)P.seed);
  hash = wang_hash(hash);
  {
    // z-sort by (u ^ h) ascending then reversed.  key kept in (A_AX hi, A_AY lo) (free now)
    int k = 0;
    for (int i = 0; i < n_u; ++i) {
      const uint32_t h = (uint32_t)hash64_full((hash64_full(anchor_x64((uint32_t)cx[k])) + hash64_full(anchor_y64((uint32_t)cy[k]))) ^ hash);
      ax[i] = f[i];                         // score (high word of u)
      ay[i] = (int32_t)((uint32_t)p[i] ^ h);  // cnt ^ h (low word)
      t[i] = k;                             // as
      k += p[i];
      perm[i] = i;
    }
    radix_sort_perm(perm, n_u,
                    [&](int32_t i) { return (uint64_t)(uint32_t)ax[i] << 32 | (uint32_t)ay[i]; }, rsx);
    for (int i = 0; i < n_u; ++i) {
      const int src = perm[n_u - 1 - i];
      r_id[i] = i;
      r_parent[i] = -1;
      r_score[i] = ax[src];
      r_hash[i] = ay[src];
      r_cnt[i] = p[src];
      r_as[i] = t[src];
      // mm_reg_set_coor
      const int k0 = t[src], k1 = k0 + p[src] - 1;
      const uint32_t x0 = (uint32_t)cx[k0], y0 = (uint32_t)cy[k0], x1 = (uint32_t)cx[k1], y1 = (uint32_t)cy[k1];
      const int q_span = anchor_span(y0);
      const int rev = (int)(x0 >> 31);
      r_rev[i] = rev;
      r_rs[i] = anchor_rpos(x0) + 1 > q_span ? anchor_rpos(x0) + 1 - q_span : 0;
      r_re[i] = anchor_rpos(x1) + 1;
      if (!rev) {
        r_qs[i] = anchor_qpos(y0) + 1 - q_span;
        r_qe[i] = anchor_qpos(y1) + 1;
      } else {
        r_qs[i] = qlen - (anchor_qpos(y1) + 1);
        r_qe[i] = qlen - (anchor_qpos(y0) + 1 - q_span);
      }
    }
  }
  int n_regs = n_u;
  // ---- map.c: chain_post = mm_set_parent + mm_select_sub(check_strand = 1) ---------------------
  if (n_regs > 1) {
    // w[] (primary list) in A_Z, cov[] as two words in A_AX (start) / A_AY (end)
    auto w = z;
    w[0] = 0, r_parent[0] = 0;
    int kk = 1;
    for (int i = 1; i < n_regs; ++i) {
      const int si = r_qs[i], ei = r_qe[i];
      int n_cov = 0, uncov_len = 0;
      for (int j = 0; j < kk; ++j) {
        int sj = r_qs[w[j]], ej = r_qe[w[j]];
        if (ej <= si || sj >= ei) continue;
        if (sj < si) sj = si;
        if (ej > ei) ej = ei;
        ax[n_cov] = sj, ay[n_cov] = ej;
        ++n_cov;
      }
      int j = kk;
      if (n_cov > 0) {
        // sort cov by (start, end): keys are plain values → any correct sort is exact
        for (int a1 = 1; a1 < n_cov; ++a1) {
          const int cs = ax[a1], ce = ay[a1];
          int b1 = a1;
          while (b1 > 0 && (ax[b1 - 1] > cs || (ax[b1 - 1] == cs && ay[b1 - 1] > ce))) {
            ax[b1] = ax[b1 - 1], ay[b1] = ay[b1 - 1];
            --b1;
          }
          ax[b1] = cs, ay[b1] = ce;
        }
        int x = si;
        for (int c = 0; c < n_cov; ++c) {
          if (ax[c] > x) uncov_len += ax[c] - x;
          x = ay[c] > x ? ay[c] : x;
        }
        if (ei > x) uncov_len += ei - x;
        for (j = 0; j < kk; ++j) {
          const int pj = w[j];
          const int sj = r_qs[pj], ej = r_qe[pj];
          if (ej <= si || sj >= ei) continue;
          const int mn = ej - sj < ei - si ? ej - sj : ei - si;
          const int mx = ej - sj > ei - si ? ej - sj : ei - si;
          const int ol = si < sj ? (ei < sj ? 0 : ei < ej ? ei - sj : ej - sj)
                                 : (ej < si ? 0 : ej < ei ? ej - si : ei - si);
          if ((float)ol / mn - (float)uncov_len / mx > P.mask_level && uncov_len <= P.mask_len) {
            r_parent[i] = r_parent[pj];
            break;
          }
        }
      }
      if (j == kk) w[kk++] = i, r_parent[i] = i;
    }
    // mm_select_sub(pri_ratio, min_diff = 2k, best_n, check_strand = 1, min_strand_sc).
    // Upstream compacts in place (r[k++] = r[i]) while still reading r[p] through the ORIGINAL
    // parent index, so a parent slot that was already overwritten is read as whatever reg now
    // sits there; the arrays are compacted in place here to reproduce exactly that.
    if (P.pri_ratio > 0.0f) {
      int k2 = 0, n_2nd = 0;
      for (int i = 0; i < n_regs; ++i) {
        const int pp = r_parent[i];
        bool keep = false;
        if (pp == i) {
          keep = true;
        } else if (((float)r_score[i] >= (float)r_score[pp] * P.pri_ratio || r_score[i] + P.k * 2 >= r_score[pp]) &&
                   n_2nd < P.best_n) {
          if (!(r_qs[i] == r_qs[pp] && r_qe[i] == r_qe[pp] && r_rs[i] == r_rs[pp] && r_re[i] == r_re[pp]))
            keep = true, ++n_2nd;
        } else if (n_2nd < P.best_n && r_score[i] > P.min_strand_sc && r_rev[pp] != r_rev[i]) {
          keep = true, ++n_2nd;
        }
        if (keep) {
          if (k2 != i) {
            r_score[k2] = r_score[i], r_cnt[k2] = r_cnt[i], r_as[k2] = r_as[i], r_hash[k2] = r_hash[i];
            r_qs[k2] = r_qs[i], r_qe[k2] = r_qe[i], r_rs[k2] = r_rs[i], r_re[k2] = r_re[i];
            r_rev[k2] = r_rev[i], r_parent[k2] = r_parent[i];
          }
          ++k2;
        }
      }
      n_regs = k2;
    }
  } else {
    r_parent[0] = 0;
  }
  // ---- align.c: mm_align1 (SR): mm_max_stretch + extension window per reg -----------------------
  // results: R_QS/R_QE/R_RS/R_RE are overwritten with the core stretch (strand coords),
  // A_F = rs0, A_P = re0.
  for (int r = 0; r < n_regs; ++r) {
    const int as = r_as[r], cnt = r_cnt[r];
    int as1 = as, cnt1 = cnt;
    if (cnt >= 2) {
      int32_t max_score = -1, max_i = -1, max_len = 0;
      int32_t score = anchor_span((uint32_t)cy[as]), len = 1;
      int i;
      for (i = as; i < as + cnt - 1; ++i) {
        const int32_t q_span = anchor_span((uint32_t)cy[i + 1]);
        const int32_t lr = anchor_rpos((uint32_t)cx[i + 1]) - anchor_rpos((uint32_t)cx[i]);
        const int32_t lq = anchor_qpos((uint32_t)cy[i + 1]) - anchor_qpos((uint32_t)cy[i]);
        if (lq == lr) {
          score += lq < q_span ? lq : q_span;
          ++len;
        } else {
          if (score > max_score) max_score = score, max_len = len, max_i = i - len + 1;
          score = q_span;
          len = 1;
        }
      }
      if (score > max_score) max_score = score, max_len = len, max_i = i - len + 1;
      as1 = max_i, cnt1 = max_len;
    }
    const uint32_t y0 = (uint32_t)cy[as1];
    const int32_t rs = anchor_rpos((uint32_t)cx[as1]) + 1 - anchor_span(y0);
    const int32_t qs = anchor_qpos(y0) + 1 - anchor_span(y0);
    const int32_t re = anchor_rpos((uint32_t)cx[as1 + cnt1 - 1]) + 1;
    const int32_t qe = anchor_qpos((uint32_t)cy[as1 + cnt1 - 1]) + 1;
    int32_t l = qs;
    l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
    const int32_t rs0 = rs - l > 0 ? rs - l : 0;
    l = qlen - qe;
    l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
    const int32_t re0 = re + l < hap_len ? re + l : hap_len;
    r_qs[r] = qs, r_qe[r] = qe, r_rs[r] = rs, r_re[r] = re;
    f[r] = rs0, p[r] = re0;
  }
  *n_regs_out = n_regs;
  return kMapOk;
}

// ------------------------------------------------------------------------------------
// Phase A: seeds → anchors → sort → chain DP → backtrack → regs → parent/sub selection
// → per-reg SR stretch + extension windows.  On return (kMapOk) the surviving regs are
// in the R_* arrays [0, *n_regs) and the per-reg stretch in R_AUX*/A_* as documented
// at the end.  Restates minimap2 map.c:mm_map_frag up to (not including) the ksw2 calls.
// ------------------------------------------------------------------------------------
template <int S>
LGR_HDN int map_chain_phase(const DevParams& P, const PairIn& in, const Ws<S>& ws, RadixScratch* rsx,
                            int* n_regs_out, ChainCounters* ctr) {
  const int cap = ws.cap();
  auto ax = ws.arr(A_AX), ay = ws.arr(A_AY), sx = ws.arr(A_SX), sy = ws.arr(A_SY);
  auto f = ws.arr(A_F), p = ws.arr(A_P), t = ws.arr(A_T), v = ws.arr(A_V), z = ws.arr(A_Z);
  auto perm = ws.arr(A_PERM);
  auto seedq = ws.arr(A_SEEDQ), seedn = ws.arr(A_SEEDN), seeds = ws.arr(A_SEEDS);
  const int qlen = in.read.qlen;
  *n_regs_out = 0;
#ifdef LGR_CORE_SELFCHECK
  bool sc_tail_expected = false;
  int32_t sc_tail_score = 0;
#endif

  // ---- seed.c: mm_seed_collect_all -------------------------------------------------
  // seedq: q_pos (pos<<1|strand) | span<<20 | tandem<<28 | flt<<29 ; seedn: occurrences ;
  // seeds: first index in the table
  int n_m = 0, n_high = 0;
  for (int i = 0; i < in.mz_n; ++i) {
    const uint64_t hx = in.mz_x[i] >> 8;
    const int s0 = idx_lower_bound(in.idx, in.idx_n, hx << kIdxShift);
    const int s1 = idx_lower_bound(in.idx, in.idx_n, (hx + 1) << kIdxShift);
    const int occ = s1 - s0;
    if (occ == 0) continue;
    if (n_m >= cap) return kMapOverflow;
    uint32_t tandem = 0;
    if (i > 0 && hx == in.mz_x[i - 1] >> 8) tandem = 1;
    if (i < in.mz_n - 1 && hx == in.mz_x[i + 1] >> 8) tandem = 1;
    seedq[n_m] = (int32_t)(in.mz_y[i] | (uint32_t)(in.mz_x[i] & 0xff) << 20 | tandem << 28);
    seedn[n_m] = occ;
    seeds[n_m] = s0;
    if (occ > in.mid_occ) ++n_high;
    ++n_m;
  }
  // ---- seed.c: mm_seed_select (occ_dist > 0 && max_max_occ > max_occ) or plain cut --
  if (n_high > 0) seed_select(P, seedq, seedn, n_m, qlen, in.mid_occ);
  // ---- map.c: collect_seed_hits -----------------------------------------------------
  int n_a = 0;
  for (int i = 0; i < n_m; ++i) {
    const uint32_t sq = (uint32_t)seedq[i];
    if (sq >> 29 & 1) continue;
    const uint32_t q_pos = sq & 0xfffff, q_span = sq >> 20 & 0xff, tandem = sq >> 28 & 1;
    const int occ = seedn[i], s0 = seeds[i];
    if (n_a + occ > cap) return kMapOverflow;
    for (int k = 0; k < occ; ++k) {
      const uint32_t rk = (uint32_t)(in.idx[s0 + k] & ((1u << kIdxShift) - 1));
      const uint32_t rpos = rk >> 1;
      uint32_t x32, qp;
      if ((rk & 1) == (q_pos & 1)) {
        x32 = rpos;
        qp = q_pos >> 1;
      } else {
        x32 = 1u << 31 | rpos;
        qp = (uint32_t)(qlen - ((int32_t)(q_pos >> 1) + 1 - (int32_t)q_span) - 1);
      }
      ax[n_a] = (int32_t)x32;
      ay[n_a] = (int32_t)(tandem << 24 | q_span << 16 | (qp & 0xffff));
      ++n_a;
    }
  }
  if (ctr) ctr->n_anchors += n_a;
  if (n_a == 0) return kMapNoHit;
  // ---- radix_sort_128x(a) by x --------------------------------------------------------
  {
    bool sorted = true, strict = true;
    for (int i = 1; i < n_a; ++i) {
      if ((uint32_t)ax[i] < (uint32_t)ax[i - 1]) { sorted = false; break; }
      if ((uint32_t)ax[i] == (uint32_t)ax[i - 1]) strict = false;
    }
    if (sorted && (n_a <= 64 || strict)) {
      for (int i = 0; i < n_a; ++i) sx[i] = ax[i], sy[i] = ay[i];
#ifdef LGR_CORE_SELFCHECK
      if (n_a > 64) {  // the skipped in-place radix passes must be the identity on a strictly increasing sequence
        ++lgr_selfcheck_sorted_seen;
        for (int i = 0; i < n_a; ++i) perm[i] = i;
        radix_sort_perm(perm, n_a, [&](int32_t id) { return anchor_x64((uint32_t)ax[id]); }, rsx);
        for (int i = 0; i < n_a; ++i)
          if (perm[i] != i) { ++lgr_selfcheck_failures; break; }
      }
#endif
    } else {
      // NB: for n_a > 64 an already sorted input is still permuted by the in-place radix
      // passes when keys tie, so only a strictly increasing sequence may skip the emulation.
      for (int i = 0; i < n_a; ++i) perm[i] = i;
      radix_sort_perm(perm, n_a, [&](int32_t id) { return anchor_x64((uint32_t)ax[id]); }, rsx);
      for (int i = 0; i < n_a; ++i) sx[i] = ax[perm[i]], sy[i] = ay[perm[i]];
    }
  }
  // ---- lchain.c: mg_lchain_dp ---------------------------------------------------------
  int32_t max_dist_x = P.max_gap_ref > 0 ? P.max_gap_ref : P.max_gap;
  int32_t max_dist_y = qlen > P.max_gap ? qlen : P.max_gap;  // MM_F_SR
  if (max_dist_x < P.bw) max_dist_x = P.bw;
  if (max_dist_y < P.bw) max_dist_y = P.bw;
  {
    int st = 0, max_ii = -1;
    int64_t n_iter = 0;
    for (int i = 0; i < n_a; ++i) t[i] = 0;
    for (int i = 0; i < n_a; ++i) {
      const uint32_t xi = (uint32_t)sx[i], yi = (uint32_t)sy[i];
      int max_j = -1, end_j;
      int32_t max_f = anchor_span(yi), n_skip = 0;
      while (st < i && ((xi >> 31) != ((uint32_t)sx[st] >> 31) ||
                        anchor_rpos(xi) > anchor_rpos((uint32_t)sx[st]) + max_dist_x))
        ++st;
      if (i - st > P.max_iter) st = i - P.max_iter;
      int j;
      for (j = i - 1; j >= st; --j) {
        int32_t sc = comput_sc(xi, yi, (uint32_t)sx[j], (uint32_t)sy[j], max_dist_x, max_dist_y, P.bw,
                               P.pen_gap, P.pen_skip);
        ++n_iter;
        if (sc == INT32_MIN) continue;
        sc += f[j];
        if (sc > max_f) {
          max_f = sc, max_j = j;
          if (n_skip > 0) --n_skip;
        } else if (t[j] == i) {
          if (++n_skip > P.max_skip) break;
        }
        if (p[j] >= 0) t[p[j]] = i;
      }
      end_j = j;
      bool far;
      if (max_ii >= 0) {
        const uint32_t xm = (uint32_t)sx[max_ii];
        far = (xi >> 31) != (xm >> 31) || anchor_rpos(xi) - anchor_rpos(xm) > max_dist_x;
      } else {
        far = true;
      }
      if (max_ii < 0 || far) {
        int32_t mx = INT32_MIN;
        max_ii = -1;
        for (j = i - 1; j >= st; --j)
          if (mx < f[j]) mx = f[j], max_ii = j;
      }
      if (max_ii >= 0 && max_ii < end_j) {
        const int32_t tmp = comput_sc(xi, yi, (uint32_t)sx[max_ii], (uint32_t)sy[max_ii], max_dist_x,
                                      max_dist_y, P.bw, P.pen_gap, P.pen_skip);
        if (tmp != INT32_MIN && max_f < tmp + f[max_ii]) max_f = tmp + f[max_ii], max_j = max_ii;
      }
      f[i] = max_f, p[i] = max_j;
      if (max_ii < 0) {
        max_ii = i;
      } else {
        const uint32_t xm = (uint32_t)sx[max_ii];
        const bool near = (xi >> 31) == (xm >> 31) && anchor_rpos(xi) - anchor_rpos(xm) <= max_dist_x;
        if (near && f[max_ii] < f[i]) max_ii = i;
      }
    }
    if (ctr) ctr->chain_evals += n_iter;
#ifdef LGR_CORE_SELFCHECK
    // host emulation only: whenever the warp kernel's co-linear precondition holds, its closed
    // form (p[i] = i-1, f = prefix sum of min(span, gap), sum of min(i, max_skip+2) iterations)
    // must equal what the scalar loop above just computed
    {
      const uint32_t x0 = (uint32_t)sx[0], y0 = (uint32_t)sy[0];
      const int diag0 = anchor_rpos(x0) - anchor_qpos(y0), span0 = anchor_span(y0);
      bool ok = true;
      for (int i = 0; i < n_a && ok; ++i) {
        const uint32_t x = (uint32_t)sx[i], y = (uint32_t)sy[i];
        ok = (x >> 31) == (x0 >> 31) && anchor_rpos(x) - anchor_qpos(y) == diag0 && anchor_span(y) == span0;
        if (ok && i > 0) ok = anchor_rpos(x) > anchor_rpos((uint32_t)sx[i - 1]);
      }
      const int tot_span = anchor_rpos((uint32_t)sx[n_a - 1]) - anchor_rpos(x0);
      if (ok && P.pen_skip == 0.0f && P.max_skip >= 0 && n_a <= P.max_iter && tot_span <= max_dist_x && tot_span <= max_dist_y &&
          span0 > 0) {
        ++lgr_selfcheck_colinear_seen;
        int32_t acc = span0;
        bool same = f[0] == span0 && p[0] == -1;
        for (int i = 1; i < n_a && same; ++i) {
          const int32_t dq = anchor_rpos((uint32_t)sx[i]) - anchor_rpos((uint32_t)sx[i - 1]);
          acc += dq < span0 ? dq : span0;
          same = f[i] == acc && p[i] == i - 1;
        }
        const long long cap_it = P.max_skip + 2, nm1 = n_a - 1;
        const long long want_iter = nm1 <= cap_it ? nm1 * (nm1 + 1) / 2 : cap_it * (cap_it + 1) / 2 + (nm1 - cap_it) * cap_it;
        if (!same || want_iter != (long long)n_iter) ++lgr_selfcheck_failures;
        // ... and the closed-form tail (warp_chain_tail_colinear): one reg spanning all anchors
        sc_tail_expected = true;
        sc_tail_score = f[n_a - 1];
      }
    }
#endif
  }
#ifdef LGR_CORE_SELFCHECK
  const uint32_t sc_x0 = (uint32_t)ws.arr(A_SX)[0], sc_y0 = (uint32_t)ws.arr(A_SY)[0];
  const uint32_t sc_x1 = n_a > 0 ? (uint32_t)ws.arr(A_SX)[n_a - 1] : 0, sc_y1 = n_a > 0 ? (uint32_t)ws.arr(A_SY)[n_a - 1] : 0;
  const int st_tail = map_chain_tail<S>(P, qlen, in.hap_len, in.name_hash, ws, rsx, n_a, n_regs_out);
  if (sc_tail_expected) {
    ++lgr_selfcheck_tail_seen;
    bool okt;
    if (!(sc_tail_score >= P.min_sc && n_a >= P.min_cnt)) {
      okt = st_tail == kMapNoHit;
    } else {
      uint32_t hash = in.name_hash;
      hash ^= wang_hash((uint32_t)qlen) + wang_hash((uint32_t)P.seed);
      hash = wang_hash(hash);
      const uint32_t h = (uint32_t)hash64_full((hash64_full(anchor_x64(sc_x0)) + hash64_full(anchor_y64(sc_y0))) ^ hash);
      const int32_t span = anchor_span(sc_y0);
      const int32_t rs = anchor_rpos(sc_x0) + 1 - span, qs = anchor_qpos(sc_y0) + 1 - span;
      const int32_t re = anchor_rpos(sc_x1) + 1, qe = anchor_qpos(sc_y1) + 1;
      int32_t l = qs;
      l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
      const int32_t rs0 = rs - l > 0 ? rs - l : 0;
      l = qlen - qe;
      l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
      const int32_t re0 = re + l < in.hap_len ? re + l : in.hap_len;
      okt = st_tail == kMapOk && *n_regs_out == 1 && ws.arr(R_SCORE)[0] == sc_tail_score && ws.arr(R_CNT)[0] == n_a &&
            ws.arr(R_AS)[0] == 0 && (uint32_t)ws.arr(R_HASH)[0] == ((uint32_t)n_a ^ h) && ws.arr(R_REV)[0] == (int32_t)(sc_x0 >> 31) &&
            ws.arr(R_QS)[0] == qs && ws.arr(R_QE)[0] == qe && ws.arr(R_RS)[0] == rs && ws.arr(R_RE)[0] == re &&
            ws.arr(A_F)[0] == rs0 && ws.arr(A_P)[0] == re0;
    }
    if (!okt) ++lgr_selfcheck_failures;
  }
  return st_tail;
#else
  return map_chain_tail<S>(P, qlen, in.hap_len, in.name_hash, ws, rsx, n_a, n_regs_out);
#endif
}

// fill a RegRec (without the extension results) from the workspace after map_chain_phase
template <int S, bool C>
LGR_HD void export_reg(const Ws<S, C>& ws, int r, int qlen, RegRec* out) {
  out->score = ws.arr(R_SCORE)[r];
  out->cnt = ws.arr(R_CNT)[r];
  out->hash = (uint32_t)ws.arr(R_HASH)[r];
  out->rev = ws.arr(R_REV)[r];
  out->c_qs = ws.arr(R_QS)[r], out->c_qe = ws.arr(R_QE)[r];
  out->c_rs = ws.arr(R_RS)[r], out->c_re = ws.arr(R_RE)[r];
  out->rs0 = ws.arr(A_F)[r], out->re0 = ws.arr(A_P)[r];
  // align.c: left extension iff qs > 0 && rs > 0; right iff qe < qlen && re < re0
  ExtRec& L = out->ext[0];
  ExtRec& R = out->ext[1];
  L.m = L.n = 0, L.mqe_t = -1, L.max = 0, L.n_cig = 0, L.cig_off = -1;
  R = L;
  if (out->c_qs > 0 && out->c_rs > 0) L.m = out->c_qs, L.n = out->c_rs - out->rs0;
  if (out->c_qe < qlen && out->c_re < out->re0) R.m = qlen - out->c_qe, R.n = out->re0 - out->c_re;
}

// does this extension run inline in the pair's lane (true) or on a warp (k_ext_big)?
LGR_HD bool ext_is_small(const DevParams& P, const ExtRec& E) {
  if (E.m <= 0) return true;
  return (int64_t)E.m * prune_cols(P, E.m, E.n) <= kSmallCells;
}

// query / target accessors of an extension, as align.c presents them to ksw2
struct ExtQuery {
  ReadView rv;
  int rev, side, c_qs, c_qe;
  // left: qseq0[rev][0..qs) reversed ; right: qseq0[rev][qe..qlen)
  LGR_HD int operator()(int j) const { return side == 0 ? rv.at(rev, c_qs - 1 - j) : rv.at(rev, c_qe + j); }
};
struct ExtTarget {
  const uint8_t* hap;
  int side, c_rs, c_re;
  // left: hap[rs0..rs) reversed ; right: hap[re..re0)
  LGR_HD int operator()(int i) const { return (side == 0 ? hap[c_rs - 1 - i] : hap[c_re + i]) & 0xf; }
};

// Scalar statement of the data-dependent column bound the warp kernel computes with one lane
// per gap length (lgr_kernels_ext.cuh, ext_dp_warp): LB = best score over "main diagonal for p
// bases, one gap of delta in [-15, 16], shifted diagonal to the end"; columns at or beyond
// m + floor((a*m - q - LB) / e) can hold neither the first last-row maximum, nor the global
// maximum, nor a traceback cell.  Same gates and arithmetic as the kernel; the host emulation
// runs it so that the bound is fuzzed against the un-pruned oracle on the CPU.
constexpr int kDynPruneMinRowsCore = 12;
template <typename QF, typename TF>
LGR_HD int dyn_prune_cols(const DevParams& P, int m, int n, int t_static, const QF& qf, const TF& tf) {
  if (!(n >= m && P.e > 0 && m >= kDynPruneMinRowsCore)) return t_static;
  const int32_t sc_match = P.a, sc_mis = -P.b, sc_amb = -P.sc_ambi;
  int32_t lb = kNegInf;
  for (int delta = -15; delta <= 16; ++delta) {
    if (!(delta >= 0 ? m + delta <= n : -delta < m)) continue;
    const int k = delta < 0 ? -delta : 0;  // inserted query bases
    int32_t p0 = 0, ps = 0, best = 0;
    const int steps = m - k;
    for (int p = 0; p < steps; ++p) {
      const int tcp = tf(p), tcs = tf(p + (delta > 0 ? delta : 0)), qcp = qf(p), qcs = qf(p + k);
      p0 += (tcp > 3 || qcp > 3) ? sc_amb : (tcp == qcp ? sc_match : sc_mis);
      ps += (tcs > 3 || qcs > 3) ? sc_amb : (tcs == qcs ? sc_match : sc_mis);
      const int32_t dlt = p0 - ps;
      if (dlt > best) best = dlt;
    }
    const int32_t cand = best + ps - (delta != 0 ? P.q + P.e * (delta < 0 ? -delta : delta) : 0);
    if (cand > lb) lb = cand;
  }
  const int X = P.a * m - P.q - lb;
  const int Dd = X <= 0 ? 0 : X / P.e;
  return m + Dd < t_static ? m + Dd : t_static;
}

// run one extension inline (scalar).  dir/hcol/ecol: scratch sized for m x T.
// `arena`/`arena_used`/`arena_cap`: overflow storage for cigars longer than kInlineCig
// (host emu and device differ only in how `alloc` bumps the counter).
template <typename Alloc>
LGR_HD bool run_ext_scalar(const DevParams& P, const ReadView& rv, const uint8_t* hap, RegRec* reg, int side,
                           uint8_t* dir, int32_t* hcol, int32_t* ecol, uint32_t* cig_tmp, int cig_tmp_cap,
                           uint32_t* arena, Alloc alloc, ChainCounters* ctr) {
  ExtRec& E = reg->ext[side];
  const int m = E.m;
  ExtQuery qf{rv, reg->rev, side, reg->c_qs, reg->c_qe};
  ExtTarget tf{hap, side, reg->c_rs, reg->c_re};
  const int T = dyn_prune_cols(P, m, E.n, prune_cols(P, m, E.n), qf, tf);
  ext_dp_scalar(P, m, T, qf, tf, side == 0, dir, hcol, ecol, &E.max, &E.mqe_t);
  if (ctr) ctr->dp_cells += (int64_t)m * T, ctr->dp_cells_full += (int64_t)m * E.n;
  CigBuf cb{cig_tmp, 0, cig_tmp_cap};
  ext_backtrack([&](int i, int j) { return dir[i * m + j]; }, m, E.mqe_t, side == 0, cb);
  E.n_cig = cb.n;
  if (cb.n > cig_tmp_cap) return false;
#ifdef LGR_CORE_SELFCHECK
  // host emulation only: whenever the warp kernel's exact-match / overhang precondition holds
  // (warp_ext_exact), its closed form must equal what the DP and traceback just produced
  if (P.a > 0 && !(E.n < m && (P.q <= 0 || P.e <= 0))) {
    const int n = E.n, nn = n < m ? n : m;
    bool same = true;
    for (int j = 0; j < nn && same; ++j) same = qf(j) == tf(j) && qf(j) < 4;
    if (same && n < m) same = qf(m - 1) != tf(n - 1);
    if (same) {
      ++lgr_selfcheck_ext_seen;
      bool okc = E.max == nn * P.a && E.mqe_t == nn - 1;
      if (n >= m) {
        okc = okc && cb.n == 1 && cig_tmp[0] == ((uint32_t)m << 4);
      } else {
        const uint32_t mop = (uint32_t)n << 4, iop = (uint32_t)(m - n) << 4 | 1u;
        okc = okc && cb.n == 2 && (side == 0 ? (cig_tmp[0] == iop && cig_tmp[1] == mop) : (cig_tmp[0] == mop && cig_tmp[1] == iop));
      }
      if (!okc) ++lgr_selfcheck_failures;
    }
  }
#endif
  if (cb.n <= kInlineCig) {
    E.cig_off = -1;
    for (int i = 0; i < cb.n; ++i) E.inl[i] = cig_tmp[i];
  } else {
    const int64_t off = alloc(cb.n);
    if (off < 0) return false;
    E.cig_off = (int32_t)off;
    for (int i = 0; i < cb.n; ++i) arena[off + i] = cig_tmp[i];
  }
  return true;
}

// ------------------------------------------------------------------------------------
// Phase C: per pair, after every extension of every reg is available.
//   align.c: mm_append_cigar ×3, coordinates, mm_update_extra (mm_fix_cigar + mlen/blen/
//   dp_max), hit.c: mm_filter_regs, mm_hit_sort, mm_set_parent + mm_select_sub (n_regs only);
//   then regs[0] → AlnOut, BuildCigar's payload, and hts::ComputeEditDistance (NM).
// cig: per-lane scratch of cig_cap ops (assembled cigar of the reg under work);
// best: per-lane scratch holding the best reg's cigar so far.
// ------------------------------------------------------------------------------------
struct FinishScratch {
  uint32_t* cig;   // cap ops
  uint32_t* best;  // cap ops
  int cap;
};

LGR_HD void cig_append(uint32_t* c, int& n, int cap, const uint32_t* src, int ns, bool& ovf) {
  if (ns == 0) return;
  int st = 0;
  if (n > 0 && (c[n - 1] & 0xf) == (src[0] & 0xf)) {
    c[n - 1] += (src[0] >> 4) << 4;
    st = 1;
  }
  for (int i = st; i < ns; ++i) {
    if (n >= cap) { ovf = true; return; }
    c[n++] = src[i];
  }
}

struct RegFinal {
  int32_t rs, re, qs, qe, dp_score, dp_max, mlen, blen, n_ambi, n_cig;
};

// Assembled-but-unscored reg: cigar in c[0..n), coordinates after mm_fix_cigar, and where the
// (strand) query / haplotype walk of mm_update_extra starts.
struct RegAsm {
  int32_t n, rs, re, qs, qe;  // final mm_reg1_t coordinates (qs/qe on the forward read)
  int32_t qb, tb;             // strand-query / haplotype offsets of the first cigar column
  int32_t dp_ext;             // sum of ez.max of the extensions (dp_score without the core)
};

// align.c: mm_append_cigar x3 + coordinates + mm_fix_cigar.  Scalar.  false on scratch overflow.
LGR_HD bool assemble_fix_reg(const ReadView& rv, const uint8_t* hap, const RegRec& reg, const uint32_t* ext_arena,
                             uint32_t* c, int cap, RegAsm* out) {
  const int qlen = rv.qlen;
  const int rev = reg.rev;
  int n = 0;
  bool ovf = false;
  int32_t dp_score = 0;
  int32_t rs1, qs1, re1, qe1;
  const ExtRec& L = reg.ext[0];
  const ExtRec& R = reg.ext[1];
  if (L.m > 0) {
    const uint32_t* src = L.cig_off < 0 ? L.inl : ext_arena + L.cig_off;
    cig_append(c, n, cap, src, L.n_cig, ovf);
    if (L.n_cig > 0) dp_score += L.max;
    rs1 = reg.c_rs - (L.mqe_t + 1);
    qs1 = 0;
  } else {
    rs1 = reg.c_rs, qs1 = reg.c_qs;
  }
  {
    const uint32_t op = (uint32_t)(reg.c_qe - reg.c_qs) << 4;
    cig_append(c, n, cap, &op, 1, ovf);
  }
  re1 = reg.c_re, qe1 = reg.c_qe;
  if (R.m > 0) {
    const uint32_t* src = R.cig_off < 0 ? R.inl : ext_arena + R.cig_off;
    cig_append(c, n, cap, src, R.n_cig, ovf);
    if (R.n_cig > 0) dp_score += R.max;
    re1 = reg.c_re + (R.mqe_t + 1);
    qe1 = qlen;
  }
  if (ovf) return false;
  int32_t r_rs = rs1, r_re = re1, r_qs, r_qe;
  if (rev) r_qs = qlen - qe1, r_qe = qlen - qs1;
  else r_qs = qs1, r_qe = qe1;

  // ---- mm_fix_cigar (qseq = strand query from qs1, tseq = hap from rs1) ----
  int qshift = 0, tshift = 0;
  if (n > 1) {
    int32_t toff = 0, qoff = 0;
    bool to_shrink = false;
    const int nn = n;
    for (int k = 0; k < nn; ++k) {
      const uint32_t op = c[k] & 0xf;
      const int len = (int)(c[k] >> 4);
      if (len == 0) to_shrink = true;
      if (op == 0) {
        toff += len, qoff += len;
      } else if (op == 1 || op == 2) {
        if (k > 0 && k < nn - 1 && (c[k - 1] & 0xf) == 0 && (c[k + 1] & 0xf) == 0) {
          int l;
          const int prev_len = (int)(c[k - 1] >> 4);
          if (op == 1) {
            for (l = 0; l < prev_len; ++l)
              if (rv.at(rev, qs1 + qoff - 1 - l) != rv.at(rev, qs1 + qoff + len - 1 - l)) break;
          } else {
            for (l = 0; l < prev_len; ++l)
              if ((hap[rs1 + toff - 1 - l] & 0xf) != (hap[rs1 + toff + len - 1 - l] & 0xf)) break;
          }
          if (l > 0) c[k - 1] -= (uint32_t)l << 4, c[k + 1] += (uint32_t)l << 4, qoff -= l, toff -= l;
          if (l == prev_len) to_shrink = true;
        }
        if (op == 1) qoff += len;
        else toff += len;
      } else if (op == 3) {
        toff += len;
      }
    }
    for (int k = 0; k + 2 < nn; ++k) {
      if ((c[k] & 0xf) > 0 && (c[k] & 0xf) + (c[k + 1] & 0xf) == 3) {
        int l;
        uint32_t s[3] = {0, 0, 0};
        for (l = k; l < nn; ++l) {
          const uint32_t op = c[l] & 0xf;
          if (op == 1 || op == 2 || c[l] >> 4 == 0) s[op] += c[l] >> 4;
          else break;
        }
        if (s[1] > 0 && s[2] > 0 && l - k > 2) {
          c[k] = s[1] << 4 | 1;
          c[k + 1] = s[2] << 4 | 2;
          for (k += 2; k < l; ++k) c[k] &= 0xf;
          to_shrink = true;
        }
        k = l;
      }
    }
    if (to_shrink) {
      int l = 0;
      for (int k = 0; k < n; ++k)
        if (c[k] >> 4 != 0) c[l++] = c[k];
      n = l;
      l = 0;
      for (int k = 0; k < n; ++k) {
        if (k == n - 1 || (c[k] & 0xf) != (c[k + 1] & 0xf)) c[l++] = c[k];
        else c[k + 1] += c[k] >> 4 << 4;
      }
      n = l;
    }
    if (n > 0 && ((c[0] & 0xf) == 1 || (c[0] & 0xf) == 2)) {
      const int32_t l = (int32_t)(c[0] >> 4);
      if ((c[0] & 0xf) == 1) {
        if (rev) r_qe -= l;
        else r_qs += l;
        qshift = l;
      } else {
        r_rs += l, tshift = l;
      }
      for (int k = 1; k < n; ++k) c[k - 1] = c[k];
      --n;
    }
  }
  out->n = n, out->rs = r_rs, out->re = r_re, out->qs = r_qs, out->qe = r_qe;
  out->qb = qs1 + qshift, out->tb = rs1 + tshift, out->dp_ext = dp_score;
  return true;
}

// align.c: the SR "gap filling" block — ungapped score of the co-linear core (N scores +e2 = +e)
LGR_HD int32_t core_score_scalar(const DevParams& P, const ReadView& rv, const uint8_t* hap, const RegRec& reg) {
  int32_t score = 0;
  const int len = reg.c_qe - reg.c_qs;
  for (int j = 0; j < len; ++j) {
    const int qc = rv.at(reg.rev, reg.c_qs + j), tc = hap[reg.c_rs + j] & 0xf;
    if (qc >= 4 || tc >= 4) score += P.e;
    else score += qc == tc ? P.a : -P.b;
  }
  return score;
}

// align.c: mm_update_extra (is_eqx = 0, log_gap = 0 under MM_F_SR): mlen / blen / n_ambi / dp_max
LGR_HD void update_extra_scalar(const DevParams& P, const ReadView& rv, int rev, const uint8_t* hap, int qb, int tb,
                                const uint32_t* c, int n, RegFinal* out) {
  {
    int32_t toff = 0, qoff = 0, blen = 0, mlen = 0, n_ambi_tot = 0;
    double s = 0.0, mx = 0.0;
    for (int k = 0; k < n; ++k) {
      const uint32_t op = c[k] & 0xf;
      const int len = (int)(c[k] >> 4);
      if (op == 0) {
        int n_ambi = 0, n_diff = 0;
        for (int l = 0; l < len; ++l) {
          const int cq = rv.at(rev, qb + qoff + l), ct = hap[tb + toff + l] & 0xf;
          if (ct > 3 || cq > 3) ++n_ambi;
          else if (ct != cq) ++n_diff;
          s += (double)sub_score(P, ct, cq);
          if (s < 0) s = 0;
          else mx = mx > s ? mx : s;
        }
        blen += len - n_ambi, mlen += len - (n_ambi + n_diff), n_ambi_tot += n_ambi;
        toff += len, qoff += len;
      } else if (op == 1) {
        int n_ambi = 0;
        for (int l = 0; l < len; ++l)
          if (rv.at(rev, qb + qoff + l) > 3) ++n_ambi;
        blen += len - n_ambi, n_ambi_tot += n_ambi;
        s -= (double)(P.q + P.e);
        if (s < 0) s = 0;
        qoff += len;
      } else if (op == 2) {
        int n_ambi = 0;
        for (int l = 0; l < len; ++l)
          if ((hap[tb + toff + l] & 0xf) > 3) ++n_ambi;
        blen += len - n_ambi, n_ambi_tot += n_ambi;
        s -= (double)(P.q + P.e);
        if (s < 0) s = 0;
        toff += len;
      } else if (op == 3) {
        toff += len;
      }
    }
    out->blen = blen, out->mlen = mlen, out->n_ambi = n_ambi_tot;
    out->dp_max = (int32_t)(mx + .499);
  }
}

// align one reg's pieces into its final cigar + stats.  Returns false on scratch overflow.
LGR_HD bool finish_reg(const DevParams& P, const ReadView& rv, const uint8_t* hap, const RegRec& reg,
                       const uint32_t* ext_arena, uint32_t* c, int cap, RegFinal* out) {
  RegAsm ra;
  if (!assemble_fix_reg(rv, hap, reg, ext_arena, c, cap, &ra)) return false;
  update_extra_scalar(P, rv, reg.rev, hap, ra.qb, ra.tb, c, ra.n, out);
  out->rs = ra.rs, out->re = ra.re, out->qs = ra.qs, out->qe = ra.qe;
  out->dp_score = ra.dp_ext + core_score_scalar(P, rv, hap, reg);
  out->n_cig = ra.n;
  return true;
}


// hts::ComputeEditDistance over minimap2's cigar (M/I/D only) with Lancet codes; the S
// bookends of BuildCigar only advance the query (cigar_utils.h:48-94, genotyper.cpp:45-69).
LGR_HD int32_t edit_distance(const uint8_t* read_codes, int qlen, const uint8_t* hap, int rs, int re, int qs,
                             const uint32_t* c, int n) {
  int32_t nm = 0;
  int qpos = qs, tpos = 0;
  const int tn = re - rs;
  for (int k = 0; k < n; ++k) {
    const uint32_t op = c[k] & 0xf;
    const int len = (int)(c[k] >> 4);
    if (op == 0) {
      for (int l = 0; l < len; ++l, ++qpos, ++tpos)
        if (qpos < qlen && tpos < tn && (read_codes[qpos] >> 4) != (hap[rs + tpos] >> 4)) ++nm;
    } else if (op == 1) {
      nm += len, qpos += len;
    } else if (op == 2) {
      nm += len, tpos += len;
    } else if (op == 3) {
      tpos += len;
    }
  }
  return nm;
}

// number of hits mm_map returns for the survivors of mm_filter_regs: mm_hit_sort order,
// mm_set_parent, mm_select_sub(check_strand = 0).  Tracked exactly for up to kTrack survivors.
constexpr int kTrack = 8;
LGR_HD int select_returned(const DevParams& P, int n_surv, const int32_t* s_qs, const int32_t* s_qe, const int32_t* s_rs,
                           const int32_t* s_re, const int32_t* s_score, const uint64_t* s_key) {
  int n_ret = n_surv;
  if (n_surv > 1 && n_surv <= kTrack && P.pri_ratio > 0.0f) {
    int ord[kTrack];
    for (int i = 0; i < n_surv; ++i) ord[i] = i;
    // descending by key, ties: later first
    for (int i = 1; i < n_surv; ++i) {
      const int o = ord[i];
      int j = i;
      while (j > 0 && s_key[ord[j - 1]] <= s_key[o]) ord[j] = ord[j - 1], --j;
      ord[j] = o;
    }
    int parent[kTrack], w[kTrack], kk = 1;
    w[0] = 0, parent[0] = 0;
    for (int i = 1; i < n_surv; ++i) {
      const int si = s_qs[ord[i]], ei = s_qe[ord[i]];
      int cs[kTrack], ce[kTrack], n_cov = 0, uncov_len = 0;
      for (int j = 0; j < kk; ++j) {
        int sj = s_qs[ord[w[j]]], ej = s_qe[ord[w[j]]];
        if (ej <= si || sj >= ei) continue;
        if (sj < si) sj = si;
        if (ej > ei) ej = ei;
        cs[n_cov] = sj, ce[n_cov] = ej, ++n_cov;
      }
      int j = kk;
      if (n_cov > 0) {
        for (int a1 = 1; a1 < n_cov; ++a1) {
          const int xs = cs[a1], xe = ce[a1];
          int b1 = a1;
          while (b1 > 0 && (cs[b1 - 1] > xs || (cs[b1 - 1] == xs && ce[b1 - 1] > xe))) cs[b1] = cs[b1 - 1], ce[b1] = ce[b1 - 1], --b1;
          cs[b1] = xs, ce[b1] = xe;
        }
        int x = si;
        for (int cc = 0; cc < n_cov; ++cc) {
          if (cs[cc] > x) uncov_len += cs[cc] - x;
          x = ce[cc] > x ? ce[cc] : x;
        }
        if (ei > x) uncov_len += ei - x;
        for (j = 0; j < kk; ++j) {
          const int sj = s_qs[ord[w[j]]], ej = s_qe[ord[w[j]]];
          if (ej <= si || sj >= ei) continue;
          const int mn = ej - sj < ei - si ? ej - sj : ei - si;
          const int mx = ej - sj > ei - si ? ej - sj : ei - si;
          const int ol = si < sj ? (ei < sj ? 0 : ei < ej ? ei - sj : ej - sj) : (ej < si ? 0 : ej < ei ? ej - si : ei - si);
          if ((float)ol / mn - (float)uncov_len / mx > P.mask_level && uncov_len <= P.mask_len) {
            parent[i] = parent[w[j]];
            break;
          }
        }
      }
      if (j == kk) w[kk++] = i, parent[i] = i;
    }
    // in-place compaction quirk of mm_select_sub reproduced through cur[]
    int cur[kTrack];
    for (int i = 0; i < n_surv; ++i) cur[i] = ord[i];
    int kept = 0, n_2nd = 0;
    for (int i = 0; i < n_surv; ++i) {
      const int pp = parent[i];
      const int me = cur[i];
      bool keep = false;
      if (pp == i) {
        keep = true;
      } else {
        const int pa = cur[pp];
        if (((float)s_score[me] >= (float)s_score[pa] * P.pri_ratio || s_score[me] + P.k * 2 >= s_score[pa]) &&
            n_2nd < P.best_n) {
          if (!(s_qs[me] == s_qs[pa] && s_qe[me] == s_qe[pa] && s_rs[me] == s_rs[pa] && s_re[me] == s_re[pa]))
            keep = true, ++n_2nd;
        }
      }
      if (keep) cur[kept++] = me;
    }
    n_ret = kept;
  }
  return n_ret;
}

// Finish one pair from its reg records.  regs[0..n_regs) in mm_gen_regs order (after
// chain_post).  Writes the winning alignment to *out and its cigar to out_cig (cap ops;
// returns the op count, or -1 on scratch overflow).
LGR_HD int finish_pair(const DevParams& P, const ReadView& rv, const uint8_t* hap, const RegRec* regs, int n_regs,
                       const uint32_t* ext_arena, FinishScratch& fs, AlnOut* out) {
  const int qlen = rv.qlen;
  // survivors of mm_filter_regs, with the key of mm_hit_sort: (dp_max<<32 | hash).  Ties on
  // the full key keep the LATER reg first (stable ascending sort, then reversed).
  int best = -1, n_surv = 0;
  uint64_t best_key = 0;
  RegFinal bf;
  bf.n_cig = 0;
  // for the final mm_set_parent/mm_select_sub (n_regs only) remember survivors' (qs,qe,rs,re,
  // score,dp_max,rev,cnt) — at most 8 tracked exactly; n_regs output saturates there.
  int32_t s_qs[kTrack], s_qe[kTrack], s_rs[kTrack], s_re[kTrack], s_score[kTrack];
  uint64_t s_key[kTrack];
  for (int r = 0; r < n_regs; ++r) {
    RegFinal rf;
    if (!finish_reg(P, rv, hap, regs[r], ext_arena, fs.cig, fs.cap, &rf)) return -1;
    // mm_filter_regs
    bool flt = false;
    if (regs[r].cnt < P.min_cnt) flt = true;
    if (rf.mlen < P.min_sc) flt = true;
    else if (rf.dp_max < P.min_dp_max) flt = true;
    else if ((float)rf.qs > (float)qlen * P.max_clip_ratio && (float)(qlen - rf.qe) > (float)qlen * P.max_clip_ratio) flt = true;
    if (flt) continue;
    const uint64_t key = (uint64_t)(uint32_t)rf.dp_max << 32 | regs[r].hash;
    if (n_surv < kTrack) {
      s_qs[n_surv] = rf.qs, s_qe[n_surv] = rf.qe, s_rs[n_surv] = rf.rs, s_re[n_surv] = rf.re;
      s_score[n_surv] = regs[r].score, s_key[n_surv] = key;
    }
    ++n_surv;
    if (best < 0 || key >= best_key) {
      best = r, best_key = key, bf = rf;
      uint32_t* tmp = fs.best;
      fs.best = fs.cig;
      fs.cig = tmp;
    }
  }
  out->valid = 0, out->score = 0, out->rs = out->re = out->qs = out->qe = 0, out->rev = 0, out->dp_score = 0;
  out->dp_max = 0, out->mlen = out->blen = out->n_ambi = 0, out->nm = 0, out->n_cigar = 0, out->cigar_off = -1;
  out->n_regs = 0;
  if (best < 0) return 0;
  const int n_ret = select_returned(P, n_surv, s_qs, s_qe, s_rs, s_re, s_score, s_key);
  out->valid = 1;
  out->score = regs[best].score;
  out->rs = bf.rs, out->re = bf.re, out->qs = bf.qs, out->qe = bf.qe;
  out->rev = regs[best].rev;
  out->dp_score = bf.dp_score, out->dp_max = bf.dp_max, out->mlen = bf.mlen, out->blen = bf.blen;
  out->n_ambi = bf.n_ambi;
  out->n_cigar = bf.n_cig;
  out->n_regs = n_ret;
  out->nm = edit_distance(rv.codes, qlen, hap, bf.rs, bf.re, bf.qs, fs.best, bf.n_cig);
  return bf.n_cig;
}

// ------------------------------------------------------------------------------------
// Phase D: ScoreReadAtVariant for one (alignment, variant) — combined_scorer.cpp:60-108 with
// ComputeLocalScore (local_scorer.cpp:166-279), ComputeSoftClipPenalty (:290-305) and
// CigarRefPosToQueryPos (cigar_utils.h:104-139) fused into one walk of the core cigar; the
// S bookends BuildCigar adds are represented by qs / qlen - qe.
// phred_err: 256-entry table 10^(-Q/10).
// ------------------------------------------------------------------------------------
LGR_HD void score_read_variant(const AlnOut& a, const uint32_t* c, const uint8_t* read_codes, const uint8_t* quals,
                               int qlen, const uint8_t* hap, int32_t var_start, int32_t var_len, int allele,
                               int hap_local, uint32_t ref_nm, const double* phred_err, AssignOut* out) {
  const int n = a.n_cigar;
  const int rs = a.rs, tn = a.re - a.rs;
  double pbq = 0.0, raw = 0.0;
  int64_t matches = 0, aligned = 0;
  int min_bq = 255;
  const bool empty = (n == 0);  // BuildCigar returns an empty vector when n_cigar == 0
  if (!empty && var_len != 0) {
    const int32_t var_end = var_start + var_len;
    int32_t tpos = 0;
    int64_t qpos = 0;
    bool stop = false;
    if (a.qs > 0) qpos += a.qs;  // leading S: never consumes reference, never breaks
    for (int k = 0; k < n && !stop; ++k) {
      const uint32_t op = c[k] & 0xf;
      const int len = (int)(c[k] >> 4);
      const bool consumes_ref = op == 0 || op == 2 || op == 3 || op == 7 || op == 8;
      if (rs + tpos >= var_end && consumes_ref) break;
      if (op == 0 || op == 7 || op == 8) {
        for (int i = 0; i < len; ++i, ++tpos, ++qpos) {
          const int32_t abs_pos = rs + tpos;
          if (!(abs_pos >= var_start && abs_pos < var_end)) continue;
          ++aligned;
          if (!(qpos >= qlen || tpos >= tn)) {
            const int tc = hap[rs + tpos] >> 4, qc = read_codes[qpos] >> 4;
            const int r = (tc == 4 || qc == 4) ? 0 : (tc == qc ? 1 : -4);
            raw += (double)r;
            const double weight = 1.0 - phred_err[quals[qpos]];
            pbq += (double)r * weight;
            matches += qc == tc ? 1 : 0;
          }
          if (qpos < qlen && quals[qpos] < min_bq) min_bq = quals[qpos];
        }
      } else if (op == 1) {
        const int32_t abs_pos = rs + tpos;
        const bool in = abs_pos >= var_start && abs_pos < var_end;
        for (int i = 0; i < len; ++i, ++qpos) {
          if (!in) continue;
          ++aligned;
          if (qpos < qlen && quals[qpos] < min_bq) min_bq = quals[qpos];
          pbq += 3.0;
        }
      } else if (op == 2) {
        for (int i = 0; i < len; ++i, ++tpos) {
          const int32_t abs_pos = rs + tpos;
          if (abs_pos >= var_start && abs_pos < var_end) {
            ++aligned;
            pbq += 3.0;
          }
        }
        if (qpos > 0 && qpos - 1 < qlen && quals[qpos - 1] < min_bq) min_bq = quals[qpos - 1];
        if (qpos < qlen && quals[qpos] < min_bq) min_bq = quals[qpos];
      } else if (op == 3) {
        tpos += len;
      }
    }
  }
  const double identity = aligned > 0 ? (double)matches / (double)aligned : 0.0;
  // ComputeSoftClipPenalty: first op S / last op S (size > 1) of the BuildCigar vector
  double sc_pen = 0.0;
  if (!empty) {
    const int32_t c5 = a.qs > 0 ? a.qs : 0;
    const int32_t c3 = a.qe < qlen ? qlen - a.qe : 0;  // vector has >= 2 entries whenever a trailing S exists
    sc_pen = (double)(c5 + c3) * 4;
  }
  const double global_adjusted = (double)a.score - sc_pen;
  out->allele = (int8_t)allele;
  out->global_score = (int32_t)(global_adjusted - raw);
  out->local_score = pbq;
  out->local_identity = identity;
  out->base_qual = (uint8_t)(min_bq == 255 ? 0 : min_bq);
  out->hap_id = (uint32_t)hap_local;
  out->own_hap_nm = (uint32_t)a.nm;
  out->ref_nm = ref_nm;
  out->assigned = 1;
  // folded read position
  int64_t var_start_in_aln = 0;
  if (var_start > a.rs) var_start_in_aln = var_start - a.rs;
  int64_t qpos = 0, tpos = 0;
  bool found = false;
  if (!empty) {
    if (a.qs > 0) qpos += a.qs;
    for (int k = 0; k < n && !found; ++k) {
      const uint32_t op = c[k] & 0xf;
      const int len = (int)(c[k] >> 4);
      if (op == 0 || op == 7 || op == 8) {
        if (var_start_in_aln >= tpos && var_start_in_aln < tpos + len) {
          qpos += var_start_in_aln - tpos;
          found = true;
        } else {
          qpos += len, tpos += len;
        }
      } else if (op == 1) {
        qpos += len;
      } else if (op == 2 || op == 3) {
        if (var_start_in_aln >= tpos && var_start_in_aln < tpos + len) found = true;
        else tpos += len;
      }
    }
    if (!found && a.qe < qlen) qpos += qlen - a.qe;  // trailing S advances the query
  }
  const double rel = qlen > 0 ? (double)qpos / (double)qlen : 0.5;
  const double one_minus = 1.0 - rel;
  out->folded_read_pos = rel < one_minus ? rel : one_minus;
  for (int i = 0; i < 5; ++i) out->pad[i] = 0;
}

}  // namespace lgr
