// lgr_kernels_chain.cuh — seeding + chaining: k_chain_overflow, warp_seed_chain, chain tails, closed-form extensions, k_chain_lean, k_chain_cold
// Part of the single translation unit lgr_gpu.cu (included there, in order); see that file's header.
#ifndef LANCET2_B200_LGR_KERNELS_CHAIN_CUH_
#define LANCET2_B200_LGR_KERNELS_CHAIN_CUH_

namespace {

// ---------------------------------------------------------------------------------------
// k_chain_overflow: phase A for the pairs whose seeds/anchors exceeded the shared-memory cap of
// the chain kernels (tandem repeats: hundreds to thousands of anchors).  One LANE per pair running the
// scalar core (map_chain_phase) over a 16384-anchor HBM workspace interleaved per warp; regs are
// parked exactly like the chain kernels do.  Exits immediately when the overflow list is empty.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_chain_overflow(const __grid_constant__ Dev D) {
  const int lane = threadIdx.x & 31;
  const int gthread = blockIdx.x * blockDim.x + threadIdx.x;
  const int gwarp = gthread >> 5;
  const long long n_work = D.ctr[C_NOVF] < D.ovf_cap ? D.ctr[C_NOVF] : D.ovf_cap;
  if (n_work == 0) return;
  Ws<32> ws;
  ws.caps = D.ws_cap;  // 16384: fits the low half, chain arrays the same size
  ws.base = D.ws + (size_t)gwarp * A_COUNT * D.ws_cap * 32 + lane;
  RadixScratch rsx;
  ChainCounters ctr{0, 0, 0, 0};
  for (;;) {
    long long item = 0;
    if (lane == 0) item = atomicAdd((unsigned long long*)&D.ctr[C_OVFPOS], 32ULL);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= n_work) break;
    if (item + lane < n_work) {
      const int r = D.ovf_read[item + lane];
      // bit 30: the warp kernel had already counted this pair's anchors and chain evaluations when
      // it ran out of chain slots (kRegCap); do not count them twice
      const bool counted = (D.ovf_hap[item + lane] >> 30) & 1;
      const int h = D.ovf_hap[item + lane] & ~(1 << 30);
      const ChainCounters ctr_before = ctr;
      const int g = D.read_grp[r];
      const int64_t pair = D.pair_off[r] + (h - D.grp_hap_begin[g]);
      const int64_t roff = D.read_off[r], hoff = D.hap_off[h];
      const int qlen = (int)(D.read_off[r + 1] - roff);
      const int hlen = (int)(D.hap_off[h + 1] - hoff);
      ReadView rv{D.read_codes + roff, qlen};
      PairIn pin{rv, D.hap_codes + hoff, hlen, D.idx + hoff, D.idx_n[h], D.mz_x + roff, D.mz_y + roff, D.mz_n[r], D.name_hash[r], D.grp_mid[g]};
      int n_regs = 0;
      const int st = qlen > 0 ? map_chain_phase<32>(D.P, pin, ws, &rsx, &n_regs, &ctr) : kMapNoHit;
      if (counted) ctr = ctr_before;
      PairReg pr{0, 0, r, h};
      if (st == kMapOverflow) {
        flag_err(D, g, E_ANCHOR_CAP);
        write_invalid(&D.aln[pair]);
      } else if (st == kMapNoHit) {
        write_invalid(&D.aln[pair]);
      } else {
        const long long first = atomicAdd((unsigned long long*)&D.ctr[C_REGS], (unsigned long long)n_regs);
        if (first + n_regs > D.regs_cap) {
          flag_err(D, g, E_REG_ARENA);
          write_invalid(&D.aln[pair]);
        } else {
          pr = PairReg{(int32_t)first, n_regs, r, h};
          for (int i = 0; i < n_regs; ++i) {
            RegRec* rg = &D.regs[first + i];
            export_reg<32>(ws, i, qlen, rg);
            for (int side = 0; side < 2; ++side) {
              if (rg->ext[side].m <= 0) continue;
              if (!push_task(D, (int32_t)(first + i), side, r, h, rg->ext[side].m, rg->ext[side].n)) flag_err(D, g, E_REG_ARENA);
            }
          }
        }
      }
      D.pair_reg[pair] = pr;
    }
    __syncwarp();
  }
  for (int o = 16; o > 0; o >>= 1) {
    ctr.chain_evals += __shfl_down_sync(0xffffffffu, ctr.chain_evals, o);
    ctr.n_anchors += __shfl_down_sync(0xffffffffu, ctr.n_anchors, o);
  }
  if (lane == 0) {
    atomicAdd((unsigned long long*)&D.ctr[C_EVALS], (unsigned long long)ctr.chain_evals);
    atomicAdd((unsigned long long*)&D.ctr[C_ANCH], (unsigned long long)ctr.n_anchors);
  }
}

// ---------------------------------------------------------------------------------------
// k_map_warp: ONE WARP PER (read, haplotype) PAIR.  A CTA (8 warps) takes a work item =
// (haplotype, up to 64 consecutive reads of its group), stages the haplotype's code bytes and
// minimizer table in shared memory, and its warps walk the reads.  Per pair, all chain state
// (seeds, anchors, f/p/t, chains, regs: A_COUNT arrays of CAP int32) lives in the warp's slice
// of shared memory:
//   seeds     32 minimizers at a time: binary search in the staged table, ballot-compacted
//   anchors   warp prefix sum over occurrence counts
//   chain DP  for anchor i, 32 predecessors j at a time: comput_sc in parallel, then minimap2's
//             sequential max / max_skip / break automaton reproduced exactly with a prefix-max
//             scan, a (max,+) scan for the saturating skip counter and ballots
//   tail      backtrack → regs → stretch: the scalar core (map_chain_tail) on lane 0
//   extension short tails scalar on lane 0, long tails on the whole warp (ext_dp_warp)
//   finish    scalar core on lane 0 (cigar assembly, mm_fix_cigar, mm_update_extra, NM)
// Pairs whose seeds/anchors exceed CAP are appended to the overflow list (k_chain_overflow).
// ---------------------------------------------------------------------------------------
#ifdef LGR_COLD_MINB  // A/B builds only; measured: no gain from more CTAs per SM (the kernel waits for its slowest pairs)
#define LGR_COLD_BOUNDS __launch_bounds__(LGR_WARPS_PER_CTA * 32, LGR_COLD_MINB)
#else
#define LGR_COLD_BOUNDS __launch_bounds__(LGR_WARPS_PER_CTA * 32)
#endif
#ifndef LGR_CHAIN_LOCKSTEP
#define LGR_CHAIN_LOCKSTEP 0
#endif
#ifndef LGR_WARPS_PER_CTA
#define LGR_WARPS_PER_CTA 4
#endif
constexpr int kWarpsPerCta = LGR_WARPS_PER_CTA;
constexpr int kMapOkColinear = 2;  // warp_seed_chain: chain DP done by the co-linear closed form
constexpr int kMapCold = -3;       // lean tier only: a shape whose code lives in the cold kernel (queued, not computed)

// Which chain kernel a pair runs in.  Lean: k_chain_lean, which every pair enters.  It finishes the
// sorted co-linear pairs (93 % on cfg2) and returns kMapCold for every other shape — a seed above
// mid_occ (mm_seed_select), unsorted anchors, a chain the closed form does not cover — so that the
// general chain DP, the general tail and the multi-reg export are not part of its instruction
// footprint, registers or workspace.  Cold: k_chain_cold, the complete code, tables read from HBM.
enum class Tier { Lean, Cold };

// The pair's anchor / evaluation counts are returned to the caller, who commits them only for pairs
// that finish in this tier (a deferred pair is counted where it is computed).
template <int CAP, Tier T>
__device__ __forceinline__ int warp_seed_chain(const Dev& D, const PairIn& in, const uint16_t* bkt, const Ws<1, T == Tier::Lean>& ws,
                                               RadixScratch* rsx, long long* n_eval_out, int* n_a_out, int* need_out) {
  constexpr bool LEAN = T == Tier::Lean;
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const DevParams& P = D.P;
  auto ax = ws.arr(A_AX), ay = ws.arr(A_AY), sx = ws.arr(A_SX), sy = ws.arr(A_SY);
  auto f = ws.arr(A_F), p = ws.arr(A_P), t = ws.arr(A_T), perm = ws.arr(A_PERM);
  auto seedq = ws.arr(A_SEEDQ), seedn = ws.arr(A_SEEDN), seeds = ws.arr(A_SEEDS);
  const int qlen = in.read.qlen;
  // ---- seeds (mm_seed_collect_all) ----
  int n_m = 0, n_high = 0, n_occ = 0;
  for (int base = 0; base < in.mz_n; base += 32) {
    const int i = base + lane;
    int occ = 0, s0 = 0;
    uint32_t sq = 0;
    if (i < in.mz_n) {
      const uint64_t mx = in.mz_x[i];
      const uint64_t hx = mx >> 8;
      {  // bisection restricted to the minimizer's hash bucket (usually 0-2 entries)
        const int b = (int)(hx >> D.bkt_shift);
        int lo = bkt[b];
        int hi = bkt[b + 1];
        const uint64_t key = hx << kIdxShift;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (in.idx[mid] < key) lo = mid + 1;
          else hi = mid;
        }
        s0 = lo;
      }
      int s1 = s0;
      while (s1 < in.idx_n && (in.idx[s1] >> kIdxShift) == hx && s1 - s0 < 8) ++s1;
      if (s1 - s0 == 8) s1 = idx_lower_bound(in.idx, in.idx_n, (hx + 1) << kIdxShift);  // long run: finish by bisection
      occ = s1 - s0;
      if (occ > 0) {
        uint32_t tandem = 0;
        if (i > 0 && hx == in.mz_x[i - 1] >> 8) tandem = 1;
        if (i < in.mz_n - 1 && hx == in.mz_x[i + 1] >> 8) tandem = 1;
        sq = in.mz_y[i] | (uint32_t)(mx & 0xff) << 20 | tandem << 28;
      }
    }
    const unsigned hit = __ballot_sync(full, occ > 0);
    const int pos = n_m + __popc(hit & ((1u << lane) - 1));
    if (occ > 0 && pos < CAP) seedq[pos] = (int32_t)sq, seedn[pos] = occ, seeds[pos] = s0;
    n_high += __popc(__ballot_sync(full, occ > in.mid_occ));
    n_m += __popc(hit);
    n_occ += __reduce_add_sync(full, occ);
  }
  // what the overflow pass must hold for this pair: every seed and every occurrence (seed_select only removes)
  *need_out = n_m > n_occ ? n_m : n_occ;
  if (n_m > CAP) return kMapOverflow;
  __syncwarp();
  if (n_high > 0) {
    if (LEAN) {
      if (lane == 0) atomicAdd((unsigned long long*)&D.ctr[C_COLD_HIGH], 1ULL);
      return kMapCold;
    }
    if (lane == 0) seed_select(P, seedq, seedn, n_m, qlen, in.mid_occ);
    __syncwarp();
  }
  // ---- anchors (collect_seed_hits) ----
  int n_a = 0;
  for (int base = 0; base < n_m; base += 32) {
    const int i = base + lane;
    int occ = 0;
    uint32_t sq = 0;
    if (i < n_m) {
      sq = (uint32_t)seedq[i];
      if (!(sq >> 29 & 1)) occ = seedn[i];
    }
    int inc = occ;
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(full, inc, o);
      if (lane >= o) inc += v;
    }
    const int total = __shfl_sync(full, inc, 31);
    if (n_a + total > CAP) return kMapOverflow;
    if (occ > 0) {
      const uint32_t q_pos = sq & 0xfffff, q_span = sq >> 20 & 0xff, tandem = sq >> 28 & 1;
      const int s0 = seeds[i];
      int off = n_a + inc - occ;
      for (int k = 0; k < occ; ++k, ++off) {
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
        ax[off] = (int32_t)x32;
        ay[off] = (int32_t)(tandem << 24 | q_span << 16 | (qp & 0xffff));
      }
    }
    n_a += total;
  }
  *n_a_out = n_a;
  if (n_a == 0) return kMapNoHit;
  __syncwarp();
  // ---- radix_sort_128x(a): already-sorted fast path, else the exact emulation on lane 0 ----
  {
    // sorted input is left alone by upstream's insertion sort (n <= 64, stable); its in-place
    // radix passes (n > 64) may permute elements whose keys tie, so beyond 64 anchors only a
    // STRICTLY increasing key sequence — which has exactly one sorted order — can skip the emulation
    bool ok = true, strict = true;
    for (int i = lane + 1; i < n_a; i += 32) {
      const uint32_t cur = (uint32_t)ax[i], prev = (uint32_t)ax[i - 1];
      ok &= cur >= prev, strict &= cur > prev;
    }
    const bool sorted = __all_sync(full, ok);
    const bool strictly = __all_sync(full, strict);
    if (sorted && (n_a <= 64 || strictly)) {
      if constexpr (!LEAN)  // the lean layout has no separate sorted arrays: sx/sy are ax/ay
        for (int i = lane; i < n_a; i += 32) sx[i] = ax[i], sy[i] = ay[i];
    } else if (LEAN) {
      if (lane == 0) atomicAdd((unsigned long long*)&D.ctr[C_COLD_SORT], 1ULL);
      return kMapCold;
    } else {
      // upstream's radix_sort_128x is an insertion sort up to 64 elements, i.e. STABLE: the result is
      // the unique stable order, which the warp gets by ranking instead of sorting on one lane
      // (typically two reverse-strand anchors of a short palindrome sit mid-list).  Beyond 64 elements
      // upstream runs its unstable in-place radix passes: if all keys are distinct there is still only
      // one sorted order and ranking gives it; only a list with tied keys needs the move-for-move
      // emulation on lane 0.  Warp-uniform trip counts on purpose: a lane-dependent loop here cost the
      // whole kernel its convergence (measured: +0.8 ms on cfg2 when this ran in the former hot kernel),
      // so these pairs stay with the cold kernel.
      bool tie = false;
      for (int base = 0; base < n_a; base += 32) {
        const int i = base + lane;
        const uint32_t xi = i < n_a ? (uint32_t)ax[i] : 0u;
        int rank = 0;
        for (int j = 0; j < n_a; ++j) {
          const uint32_t xj = (uint32_t)ax[j];
          rank += (xj < xi) || (xj == xi && j < i);
          tie |= xj == xi && j != i && i < n_a;
        }
        __syncwarp();
        if (i < n_a) sx[rank] = (int32_t)xi, sy[rank] = ay[i];
      }
      __syncwarp();
      if (n_a > 64 && __any_sync(full, tie)) {
        if (lane == 0) {
          for (int i = 0; i < n_a; ++i) perm[i] = i;
          radix_sort_perm(perm, n_a, [&](int32_t id) { return anchor_x64((uint32_t)ax[id]); }, rsx);
          for (int i = 0; i < n_a; ++i) sx[i] = ax[perm[i]], sy[i] = ay[perm[i]];
        }
      }
    }
  }
  __syncwarp();
  // ---- mg_lchain_dp ----
  int32_t max_dist_x = P.max_gap_ref > 0 ? P.max_gap_ref : P.max_gap;
  int32_t max_dist_y = qlen > P.max_gap ? qlen : P.max_gap;
  if (max_dist_x < P.bw) max_dist_x = P.bw;
  if (max_dist_y < P.bw) max_dist_y = P.bw;
  int st = 0, max_ii = -1;
  long long n_iter = 0;
  // ---- co-linear fast path ----------------------------------------------------------------
  // All anchors on one strand and one diagonal, strictly increasing, equal spans, no skip
  // penalty: then for every i the best predecessor is i-1 (sc_{i-1} = f[i-1] + min(span, dq) >=
  // f[j] + min(span, dq_ij) for all j < i-1 because sum(min(span, g)) >= min(span, sum g); ties
  // go to the first j scanned, i-1), there is no gap penalty (dd = 0), so f is a prefix sum and
  // p[i] = i-1.  The predecessor scan upstream visits min(i, max_skip + 2) anchors for anchor i
  // (j = i-1 raises the maximum, every further j is stamped by its successor's predecessor link
  // and bumps the skip counter until it exceeds max_skip), which gives its iteration count.
  {
    const uint32_t x0 = (uint32_t)sx[0], y0 = (uint32_t)sy[0];
    const int diag0 = anchor_rpos(x0) - anchor_qpos(y0), span0 = anchor_span(y0);
    bool ok = true;
    for (int i = lane; i < n_a; i += 32) {
      const uint32_t x = (uint32_t)sx[i], y = (uint32_t)sy[i];
      ok &= (x >> 31) == (x0 >> 31) && anchor_rpos(x) - anchor_qpos(y) == diag0 && anchor_span(y) == span0;
      if (i > 0) ok &= anchor_rpos(x) > anchor_rpos((uint32_t)sx[i - 1]);
    }
    const int tot_span = anchor_rpos((uint32_t)sx[n_a - 1]) - anchor_rpos(x0);
    const bool colinear = __all_sync(full, ok) && P.pen_skip == 0.0f && P.max_skip >= 0 && n_a <= P.max_iter &&
                          tot_span <= max_dist_x && tot_span <= max_dist_y && span0 > 0;
    if (colinear) {
      int32_t carry = span0;  // f[0]
      for (int base = 0; base < n_a; base += 32) {
        const int i = base + lane;
        int32_t c = 0;
        if (i > 0 && i < n_a) {
          const int32_t dq = anchor_rpos((uint32_t)sx[i]) - anchor_rpos((uint32_t)sx[i - 1]);
          c = dq < span0 ? dq : span0;
        }
        for (int o = 1; o < 32; o <<= 1) {
          const int32_t v = __shfl_up_sync(full, c, o);
          if (lane >= o) c += v;
        }
        if (i < n_a) f[i] = carry + c, p[i] = i - 1;
        carry += __shfl_sync(full, c, 31);
      }
      const long long cap_it = P.max_skip + 2, nm1 = n_a - 1;  // sum_{i=1}^{n_a-1} min(i, cap_it)
      n_iter = nm1 <= cap_it ? nm1 * (nm1 + 1) / 2 : cap_it * (cap_it + 1) / 2 + (nm1 - cap_it) * cap_it;
      *n_eval_out = n_iter;
      __syncwarp();
      return kMapOkColinear;
    }
  }
  if constexpr (LEAN) {
    return kMapCold;  // the general DP below is not part of the lean kernel
  } else {
    for (int i = lane; i < n_a; i += 32) t[i] = 0;
    __syncwarp();
    for (int i = 0; i < n_a; ++i) {
      const uint32_t xi = (uint32_t)sx[i], yi = (uint32_t)sy[i];
      while (st < i && ((xi >> 31) != ((uint32_t)sx[st] >> 31) || anchor_rpos(xi) > anchor_rpos((uint32_t)sx[st]) + max_dist_x)) ++st;
      if (i - st > P.max_iter) st = i - P.max_iter;
      int32_t max_f = anchor_span(yi);
      int max_j = -1, n_skip = 0, end_j = st - 1;
      for (int jb = i - 1; jb >= st; jb -= 32) {
        const int j = jb - lane;
        int32_t sc = INT32_MIN;
        int pj = -1;
        if (j >= st) {
          sc = comput_sc(xi, yi, (uint32_t)sx[j], (uint32_t)sy[j], max_dist_x, max_dist_y, P.bw, P.pen_gap, P.pen_skip);
          if (sc != INT32_MIN) sc += f[j], pj = p[j];
        }
        const bool valid = sc != INT32_MIN;
        // stamps t[p[j]] = i of this chunk: predecessors processed earlier (higher j, lower lane) are
        // visible to later lanes after the barrier; stamps written by lanes at/after a break only
        // touch entries that are never read again for this i.
        if (valid && pj >= 0) t[pj] = i;
        __syncwarp();
        const bool stamped = valid && t[j] == i;
        // record setters of the sequential "sc > max_f" test: lanes whose score exceeds max_f and
        // every earlier lane of the chunk.  Usually there is at most one, so they are peeled off
        // with ballots instead of a prefix-max scan.
        unsigned nmask_all = 0;
        {
          int32_t cur = max_f;
          unsigned cand = __ballot_sync(full, valid && sc > cur);
          while (cand) {
            const int l = __ffs(cand) - 1;
            nmask_all |= 1u << l;
            cur = __shfl_sync(full, sc, l);
            cand = __ballot_sync(full, valid && sc > cur) & ~((2u << l) - 1);
          }
        }
        const bool newmax = (nmask_all >> lane) & 1;
        const int ev = newmax ? -1 : (stamped ? 1 : 0);
        const unsigned smask = __ballot_sync(full, ev == 1);
        int last = 31;
        unsigned brk = 0;
        // the skip counter only ever decrements on a record setter; when every record setter comes
        // before the first stamped lane and the counter enters at 0 (or there is none), the
        // decrements are no-ops and the counter is a running popcount of the stamped lanes
        const bool simple = nmask_all == 0 || (n_skip == 0 && (smask == 0 || (31 - __clz(nmask_all)) < (__ffs(smask) - 1)));
        if (simple) {
          const int need = P.max_skip + 1 - n_skip;  // stamped lanes until the break
          const int tot = __popc(smask);
          if (need <= tot) {
            last = (int)__fns(smask, 0, need);
            brk = 1u << last;
            n_skip = P.max_skip + 1;
          } else {
            n_skip += tot;
          }
        } else {
          // general case: n -> max(n + a, b) per lane, composed left to right ((max,+) scan)
          int a = ev, b = ev == 1 ? 1 : 0;
          for (int o = 1; o < 32; o <<= 1) {
            const int au = __shfl_up_sync(full, a, o), bu = __shfl_up_sync(full, b, o);
            if (lane >= o) {
              const int nb = bu + a;
              b = nb > b ? nb : b;
              a = au + a;
            }
          }
          int n_after = n_skip + a;
          if (b > n_after) n_after = b;
          brk = __ballot_sync(full, ev == 1 && n_after > P.max_skip);
          last = brk ? __ffs(brk) - 1 : 31;
          n_skip = __shfl_sync(full, n_after, last);
        }
        const unsigned nmask = nmask_all & (last == 31 ? 0xffffffffu : ((2u << last) - 1));
        if (nmask) {
          const int src = 31 - __clz(nmask);
          max_f = __shfl_sync(full, sc, src);
          max_j = jb - src;
        }
        const int n_in = jb - st + 1 < 32 ? jb - st + 1 : 32;
        if (brk) {
          n_iter += last + 1;
          end_j = jb - last;
          break;
        }
        n_iter += n_in;
        __syncwarp();
      }
      bool far = true;
      if (max_ii >= 0) {
        const uint32_t xm = (uint32_t)sx[max_ii];
        far = (xi >> 31) != (xm >> 31) || anchor_rpos(xi) - anchor_rpos(xm) > max_dist_x;
      }
      if (max_ii < 0 || far) {
        int32_t bf = INT32_MIN;
        int bj = -1;
        for (int j = i - 1 - lane; j >= st; j -= 32)
          if (f[j] > bf) bf = f[j], bj = j;
        for (int o = 16; o > 0; o >>= 1) {
          const int32_t of = __shfl_xor_sync(full, bf, o);
          const int oj = __shfl_xor_sync(full, bj, o);
          if (of > bf || (of == bf && oj > bj)) bf = of, bj = oj;
        }
        max_ii = bj;
      }
      if (max_ii >= 0 && max_ii < end_j) {
        const int32_t tmp = comput_sc(xi, yi, (uint32_t)sx[max_ii], (uint32_t)sy[max_ii], max_dist_x, max_dist_y, P.bw, P.pen_gap, P.pen_skip);
        if (tmp != INT32_MIN && max_f < tmp + f[max_ii]) max_f = tmp + f[max_ii], max_j = max_ii;
      }
      __syncwarp();
      if (lane == 0) f[i] = max_f, p[i] = max_j;
      if (max_ii < 0) {
        max_ii = i;
      } else {
        const uint32_t xm = (uint32_t)sx[max_ii];
        const bool near = (xi >> 31) == (xm >> 31) && anchor_rpos(xi) - anchor_rpos(xm) <= max_dist_x;
        if (near && f[max_ii] < max_f) max_ii = i;
      }
      __syncwarp();
    }
    *n_eval_out = n_iter;
    return kMapOk;
  }
}

// ---------------------------------------------------------------------------------------
// warp_chain_tail_fast: map_chain_tail for the overwhelmingly common shape — every anchor with
// f >= min_sc lies on ONE chain that is accepted.  All lanes execute it uniformly on the shared
// arrays.  Returns kMapOk (one reg, R_* / stretch filled exactly as map_chain_tail would),
// kMapNoHit, or -2 when the shape is different (then lane 0 runs the exact scalar map_chain_tail
// from scratch).
// ---------------------------------------------------------------------------------------
template <bool C>
__device__ __noinline__ int warp_chain_tail_fast(const DevParams& P, int qlen, int hap_len, uint32_t name_hash, const Ws<1, C>& ws, int n_a) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  auto sx = ws.arr(A_SX), sy = ws.arr(A_SY), f = ws.arr(A_F), p = ws.arr(A_P), t = ws.arr(A_T), v = ws.arr(A_V);
  auto cx = ws.arr(A_CX), cy = ws.arr(A_CY);
  // z = anchors with f >= min_sc; its top (processed first upstream) is the max (f, index)
  int n_z = 0;
  int32_t bf = INT32_MIN;
  int bi = -1;
  for (int base = 0; base < n_a; base += 32) {
    const int i = base + lane;
    const bool in = i < n_a && f[i] >= P.min_sc;
    n_z += __popc(__ballot_sync(full, in));
    if (in && (f[i] > bf || (f[i] == bf && i > bi))) bf = f[i], bi = i;
    if (i < n_a) t[i] = 0;
  }
  if (n_z == 0) return kMapNoHit;
  for (int o = 16; o > 0; o >>= 1) {
    const int32_t of = __shfl_xor_sync(full, bf, o);
    const int oi = __shfl_xor_sync(full, bi, o);
    if (of > bf || (of == bf && oi > bi)) bf = of, bi = oi;
  }
  if (n_z > 64) {
    // beyond 64 candidates upstream's in-place radix pass orders ties arbitrarily: the chain it
    // starts with is only certain when the maximum is unique (every other candidate is then
    // swallowed by that chain or sends us to the general path below)
    int ties = 0;
    for (int base = 0; base < n_a; base += 32) {
      const int i = base + lane;
      ties += __popc(__ballot_sync(full, i < n_a && f[i] == bf));
    }
    if (ties > 1) return -2;  // exact scalar path
  }
  __syncwarp();
  // mg_chain_bk_end + collection for the top anchor (t[] is all zero: first chain)
  const int zi = bi;
  const int32_t zx = bf;
  int end_i;
  {
    int i = zi, max_i = zi;
    int32_t max_s = 0;
    do {
      i = p[i];
      const int32_t s = i < 0 ? zx : zx - f[i];
      if (s > max_s) max_s = s, max_i = i;
      else if (max_s - s > P.bw) break;
    } while (i >= 0);
    end_i = max_i;
  }
  int cnt = 0;
  int i;
  for (i = zi; i != end_i; i = p[i]) {
    if (lane == 0) v[cnt] = i, t[i] = 1;
    ++cnt;
  }
  const int32_t sc = i < 0 ? zx : zx - f[i];
  __syncwarp();
  if (!(sc >= P.min_sc && cnt >= P.min_cnt)) return -2;  // rejected top chain: general path
  // any other candidate left?  (they would start further chains upstream)
  {
    bool other = false;
    for (int j = lane; j < n_a; j += 32) other |= f[j] >= P.min_sc && t[j] == 0;
    if (__any_sync(full, other)) return -2;
  }
  // compact_a: ascending anchors of the chain
  for (int j = lane; j < cnt; j += 32) {
    const int id = v[cnt - 1 - j];
    cx[j] = sx[id], cy[j] = sy[id];
  }
  __syncwarp();
  // mm_gen_regs for the single chain
  uint32_t hash = name_hash;
  hash ^= wang_hash((uint32_t)qlen) + wang_hash((uint32_t)P.seed);
  hash = wang_hash(hash);
  const uint32_t x0 = (uint32_t)cx[0], y0 = (uint32_t)cy[0];
  const uint32_t h = (uint32_t)hash64_full((hash64_full(anchor_x64(x0)) + hash64_full(anchor_y64(y0))) ^ hash);
  const int rev = (int)(x0 >> 31);
  // mm_max_stretch (uniform sequential scan over the chain)
  int as1 = 0, cnt1 = cnt;
  if (cnt >= 2) {
    int32_t max_score = -1, max_i = -1, max_len = 0;
    int32_t score = anchor_span(y0), len = 1;
    int k;
    uint32_t px = x0, py = y0;
    for (k = 0; k < cnt - 1; ++k) {
      const uint32_t nx = (uint32_t)cx[k + 1], ny = (uint32_t)cy[k + 1];
      const int32_t q_span = anchor_span(ny);
      const int32_t lr = anchor_rpos(nx) - anchor_rpos(px);
      const int32_t lq = anchor_qpos(ny) - anchor_qpos(py);
      if (lq == lr) {
        score += lq < q_span ? lq : q_span;
        ++len;
      } else {
        if (score > max_score) max_score = score, max_len = len, max_i = k - len + 1;
        score = q_span;
        len = 1;
      }
      px = nx, py = ny;
    }
    if (score > max_score) max_score = score, max_len = len, max_i = k - len + 1;
    as1 = max_i, cnt1 = max_len;
  }
  const uint32_t ys = (uint32_t)cy[as1];
  const int32_t rs = anchor_rpos((uint32_t)cx[as1]) + 1 - anchor_span(ys);
  const int32_t qs = anchor_qpos(ys) + 1 - anchor_span(ys);
  const int32_t re = anchor_rpos((uint32_t)cx[as1 + cnt1 - 1]) + 1;
  const int32_t qe = anchor_qpos((uint32_t)cy[as1 + cnt1 - 1]) + 1;
  int32_t l = qs;
  l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
  const int32_t rs0 = rs - l > 0 ? rs - l : 0;
  l = qlen - qe;
  l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
  const int32_t re0 = re + l < hap_len ? re + l : hap_len;
  __syncwarp();
  if (lane == 0) {
    ws.arr(R_SCORE)[0] = sc, ws.arr(R_CNT)[0] = cnt, ws.arr(R_AS)[0] = 0, ws.arr(R_HASH)[0] = (int32_t)((uint32_t)cnt ^ h);
    ws.arr(R_REV)[0] = rev, ws.arr(R_PARENT)[0] = 0, ws.arr(R_ID)[0] = 0;
    ws.arr(R_QS)[0] = qs, ws.arr(R_QE)[0] = qe, ws.arr(R_RS)[0] = rs, ws.arr(R_RE)[0] = re;
    f[0] = rs0, p[0] = re0;
  }
  __syncwarp();
  return kMapOk;
}

// Tail of a co-linear pair in closed form: f is strictly increasing and p[i] = i-1, so the top
// of z is the last anchor, mg_chain_bk_end walks to the start (s = zx - f[i] grows all the way,
// f > 0), the chain is ALL anchors with score f[n_a-1]; if it fails min_sc / min_cnt every other
// candidate is already marked used, so there is no hit.  All anchors share the diagonal, hence
// mm_max_stretch returns the whole chain.  Fills the same R_* slots as map_chain_tail.
template <bool C>
__device__ __forceinline__ int warp_chain_tail_colinear(const DevParams& P, int qlen, int hap_len, uint32_t name_hash,
                                                        const Ws<1, C>& ws, int n_a) {
  const int lane = threadIdx.x & 31;
  auto sx = ws.arr(A_SX), sy = ws.arr(A_SY), f = ws.arr(A_F), p = ws.arr(A_P);
  const int32_t sc = f[n_a - 1];
  if (!(sc >= P.min_sc && n_a >= P.min_cnt)) return kMapNoHit;
  const uint32_t x0 = (uint32_t)sx[0], y0 = (uint32_t)sy[0], x1 = (uint32_t)sx[n_a - 1], y1 = (uint32_t)sy[n_a - 1];
  uint32_t hash = name_hash;
  hash ^= wang_hash((uint32_t)qlen) + wang_hash((uint32_t)P.seed);
  hash = wang_hash(hash);
  const uint32_t h = (uint32_t)hash64_full((hash64_full(anchor_x64(x0)) + hash64_full(anchor_y64(y0))) ^ hash);
  const int32_t span = anchor_span(y0);
  const int32_t rs = anchor_rpos(x0) + 1 - span, qs = anchor_qpos(y0) + 1 - span;
  const int32_t re = anchor_rpos(x1) + 1, qe = anchor_qpos(y1) + 1;
  int32_t l = qs;
  l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
  const int32_t rs0 = rs - l > 0 ? rs - l : 0;
  l = qlen - qe;
  l += l * P.a + P.end_bonus > P.q ? (l * P.a + P.end_bonus - P.q) / P.e : 0;
  const int32_t re0 = re + l < hap_len ? re + l : hap_len;
  __syncwarp();
  if (lane == 0) {
    ws.arr(R_SCORE)[0] = sc, ws.arr(R_CNT)[0] = n_a, ws.arr(R_AS)[0] = 0, ws.arr(R_HASH)[0] = (int32_t)((uint32_t)n_a ^ h);
    ws.arr(R_REV)[0] = (int32_t)(x0 >> 31), ws.arr(R_PARENT)[0] = 0, ws.arr(R_ID)[0] = 0;
    ws.arr(R_QS)[0] = qs, ws.arr(R_QE)[0] = qe, ws.arr(R_RS)[0] = rs, ws.arr(R_RE)[0] = re;
    f[0] = rs0, p[0] = re0;
  }
  __syncwarp();
  return kMapOk;
}

// Closed forms of an extension tail (both proven in DESIGN.md §4, both checked against the DP by
// the parity tests):
//  * exact match, n >= m: the m query bases equal the first m target bases (no ambiguity codes).
//    The only path reaching m*a is the gap-free diagonal ⇒ max = mqe = m*a at target offset m-1,
//    cigar mM.
//  * overhang, n < m: the first n query bases equal the n target bases and the LAST query base
//    differs from the last target base.  Every path ends in column <= n-1, has at most n matches
//    and at least m-n inserted bases; n*a - (q + e(m-n)) is reached only by "n matches, then one
//    insertion of m-n" (an insertion anywhere earlier would have to match t[n-1] with q[m-1]).
//    ⇒ max = n*a, mqe_t = n-1, cigar nM (m-n)I in alignment order (the left extension reports it
//    outward-in as (m-n)I nM).  Needs a, q, e > 0.
__device__ __forceinline__ bool warp_ext_exact(const DevParams& P, const ReadView& rv, const uint8_t* hapc, RegRec* reg, int side,
                                               int64_t* cells_full) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int m = reg->ext[side].m, n = reg->ext[side].n;
  if (P.a <= 0) return false;
  const int nn = n < m ? n : m;  // bases that must match
  if (n < m && (P.q <= 0 || P.e <= 0)) return false;
  ExtQuery qf{rv, reg->rev, side, reg->c_qs, reg->c_qe};
  ExtTarget tf{hapc, side, reg->c_rs, reg->c_re};
  bool same = true;
  for (int j = lane; j < nn; j += 32) {
    const int qc = qf(j), tc = tf(j);
    same &= qc == tc && qc < 4;
  }
  if (n < m && lane == 0) same &= qf(m - 1) != tf(n - 1);
  if (!__all_sync(full, same)) return false;
  if (lane == 0) {
    ExtRec& E = reg->ext[side];
    E.max = nn * P.a, E.mqe_t = nn - 1, E.cig_off = -1;
    if (n >= m) {
      E.n_cig = 1, E.inl[0] = (uint32_t)m << 4;
    } else {
      E.n_cig = 2;
      const uint32_t mop = (uint32_t)n << 4, iop = (uint32_t)(m - n) << 4 | 1u;
      if (side == 0) E.inl[0] = iop, E.inl[1] = mop;
      else E.inl[0] = mop, E.inl[1] = iop;
    }
    *cells_full += (int64_t)m * n;
  }
  __syncwarp();
  return true;
}

constexpr int kCtaItemReads = 32;  // reads per CTA work item (all against one haplotype) in machine-filling batches

// Phase A kernel: seeds → anchors → chain DP → regs, one warp per pair.  Every pair with at least
// one reg is parked: its RegRecs go to the arena and its PairReg slot tells k_finish_warp where.
constexpr int kRegCap = 16;  // chains per pair held in shared memory (more → overflow pass)

constexpr int kTabCap = 512;  // minimizer-table entries of one haplotype staged in shared memory (~1500 bp at w = 5)

__device__ __forceinline__ void cold_push(const Dev& D, int r, int h) {
  const long long o = atomicAdd((unsigned long long*)&D.ctr[C_NCOLD], 1ULL);
  D.cold_read[o] = r, D.cold_hap[o] = h;  // capacity n_pairs: every pair is pushed at most once
}

// One (read, haplotype) pair on one warp: seeds → anchors → chain DP → regs, closed-form extensions,
// the other extensions queued, regs parked for k_finish_warp.  `tab` / `bkt` are the haplotype's
// sorted minimizer table and bucket directory (shared memory in the lean kernel, HBM in the cold one).
template <int CAP, Tier T>
__device__ __forceinline__ void chain_pair(const Dev& D, int r, int h, int g, int h_local, int mid_occ, const uint8_t* hapc, int hlen,
                                           const uint64_t* tab, int idx_n, const uint16_t* bkt, const Ws<1, T == Tier::Lean>& ws, RadixScratch* rsx,
                                           RegRec* s_reg, ChainCounters& ctr) {
  constexpr bool LEAN = T == Tier::Lean;
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int64_t pair = D.pair_off[r] + h_local;
  const int64_t roff = D.read_off[r];
  const int qlen = (int)(D.read_off[r + 1] - roff);
  ReadView rv{D.read_codes + roff, qlen};
  PairIn pin{rv, hapc, hlen, tab, idx_n, D.mz_x + roff, D.mz_y + roff, D.mz_n[r], D.name_hash[r], mid_occ};
  int n_a = 0, n_regs = 0, need = 0;
  long long n_eval = 0;
  int st = qlen > 0 ? warp_seed_chain<CAP, T>(D, pin, bkt, ws, rsx, &n_eval, &n_a, &need) : kMapNoHit;
  if (st == kMapOkColinear) {
    st = warp_chain_tail_colinear(D.P, qlen, hlen, pin.name_hash, ws, n_a);
    n_regs = 1;
  } else if constexpr (!LEAN) {
    if (st == kMapOk) {
      st = warp_chain_tail_fast(D.P, qlen, hlen, pin.name_hash, ws, n_a);
      n_regs = 1;
      if (st == -2) {
        __syncwarp();  // the lanes' reads of the workspace in the fast form are done before lane 0 rewrites it
        if (lane == 0) st = map_chain_tail<1>(D.P, qlen, hlen, pin.name_hash, ws, rsx, n_a, &n_regs);
        st = __shfl_sync(full, st, 0);
        n_regs = __shfl_sync(full, n_regs, 0);
      }
    }
  }
  if (st == kMapCold) {  // computed (and counted) by the cold kernel
    if (lane == 0) {
      atomicAdd((unsigned long long*)&D.ctr[C_LEAN_DEFER], 1ULL);
      cold_push(D, r, h);
    }
    __syncwarp();
    return;
  }
  if (st != kMapOverflow || n_a > 0) ctr.n_anchors += n_a, ctr.chain_evals += n_eval;
  if (st == kMapOverflow || st == kMapNoHit) {
    if (lane == 0) {
      if (st == kMapOverflow) {
        // not refused: listed for the host-driven overflow pass (lgr_gpu.cu overflow_pass), which
        // sizes its HBM workspace from the largest need recorded here
        const long long o = atomicAdd((unsigned long long*)&D.ctr[C_NOVF], 1ULL);
        if (o < D.ovf_cap) D.ovf_read[o] = r, D.ovf_hap[o] = h | (n_a > 0 ? 1 << 30 : 0);  // n_a > 0: overflowed after counting
        else flag_err(D, g, E_ANCHOR_CAP);
        atomicMax((unsigned long long*)&D.ctr[C_OVFNEED], (unsigned long long)need);
      }
      write_invalid(&D.aln[pair]);
      D.pair_reg[pair] = PairReg{0, 0, r, h};
    }
    __syncwarp();
    return;
  }
  if (n_regs == 1) {
    // the common case: the reg stays in shared memory while the closed-form extensions are tried,
    // then goes to the arena in one coalesced write (no HBM round trip between export and extension)
    if (lane == 0) export_reg<1>(ws, 0, qlen, s_reg);
    __syncwarp();
    unsigned task_mask = 0;
    for (int side = 0; side < 2; ++side) {
      if (s_reg->ext[side].m <= 0) continue;
      if (!warp_ext_exact(D.P, rv, hapc, s_reg, side, &ctr.dp_cells_full)) task_mask |= 1u << side;
    }
    long long first = -1;
    if (lane == 0) {
      first = atomicAdd((unsigned long long*)&D.ctr[C_REGS], 1ULL);
      if (first + 1 > D.regs_cap) {
        flag_err(D, g, E_REG_ARENA);
        write_invalid(&D.aln[pair]);
        D.pair_reg[pair] = PairReg{0, 0, r, h};
        first = -1;
      } else {
        D.pair_reg[pair] = PairReg{(int32_t)first, 1, r, h};
        for (int side = 0; side < 2; ++side)
          if ((task_mask >> side & 1u) && !push_task(D, (int32_t)first, side, r, h, s_reg->ext[side].m, s_reg->ext[side].n))
            flag_err(D, g, E_REG_ARENA);
      }
    }
    first = __shfl_sync(full, first, 0);
    if (first >= 0) {
      constexpr int kWords = (int)(sizeof(RegRec) / 4);
      const uint32_t* src = reinterpret_cast<const uint32_t*>(s_reg);
      uint32_t* dst = reinterpret_cast<uint32_t*>(&D.regs[first]);
      for (int w = lane; w < kWords; w += 32) dst[w] = src[w];
    }
    __syncwarp();
    return;
  }
  if constexpr (LEAN) return;  // the lean tier finishes single-reg pairs only
  long long first = -1;
  if (lane == 0) {
    first = atomicAdd((unsigned long long*)&D.ctr[C_REGS], (unsigned long long)n_regs);
    if (first + n_regs > D.regs_cap) {
      flag_err(D, g, E_REG_ARENA);
      write_invalid(&D.aln[pair]);
      D.pair_reg[pair] = PairReg{0, 0, r, h};
      first = -1;
    } else {
      D.pair_reg[pair] = PairReg{(int32_t)first, n_regs, r, h};
      for (int i = 0; i < n_regs; ++i) export_reg<1>(ws, i, qlen, &D.regs[first + i]);
    }
  }
  first = __shfl_sync(full, first, 0);
  __syncwarp();
  if (first >= 0) {
    // extensions: closed forms here (warp-parallel compare), everything else → wavefront queue
    for (int i = 0; i < n_regs; ++i) {
      RegRec* rg = &D.regs[first + i];
      for (int side = 0; side < 2; ++side) {
        if (rg->ext[side].m <= 0) continue;
        if (warp_ext_exact(D.P, rv, hapc, rg, side, &ctr.dp_cells_full)) continue;
        if (lane == 0 && !push_task(D, (int32_t)(first + i), side, r, h, rg->ext[side].m, rg->ext[side].n)) flag_err(D, g, E_REG_ARENA);
      }
    }
  }
  __syncwarp();
}

// shared memory of the chain kernels: per-warp workspace, per-warp RegRec slot, and (lean kernel) the
// staged minimizer table + bucket directory of the CTA's haplotype
__host__ __device__ inline size_t chain_smem_bytes(int cap, bool lean) {
  return (size_t)kWarpsPerCta * ((lean ? Ws<1, true>::elems(cap, 1) : Ws<1>::elems(cap, kRegCap)) * sizeof(int32_t) + sizeof(RegRec)) +
         (lean ? (size_t)kTabCap * sizeof(uint64_t) + (size_t)(kBuckets + 2) * sizeof(uint16_t) : 0) + 16;
}

// Phase A, lean kernel: the first chain launch, which every pair enters.  A CTA takes a work item =
// (haplotype, up to item_reads consecutive reads of its group), stages that haplotype's sorted minimizer
// table and 513-entry bucket directory in shared memory (every seed lookup of every read of the item then
// stays on chip: the dependent minimizer → bucket → table loads were the top stall of the round-1
// kernel), and its warps take the item's reads one at a time from a shared counter.  Only sorted
// co-linear pairs finish here; every other shape is queued for k_chain_cold (Tier::Lean).
template <int CAP>
__global__ void __launch_bounds__(kWarpsPerCta * 32, LGR_CHAIN_MINB) k_chain_lean(const __grid_constant__ Dev D) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* s_tab = reinterpret_cast<uint64_t*>(smem_raw);
  int32_t* s_ws = reinterpret_cast<int32_t*>(smem_raw + (size_t)kTabCap * sizeof(uint64_t));
  using LeanWs = Ws<1, true>;
  RegRec* s_regs = reinterpret_cast<RegRec*>(s_ws + (size_t)kWarpsPerCta * LeanWs::elems(CAP, 1));
  uint16_t* s_bkt = reinterpret_cast<uint16_t*>(s_regs + kWarpsPerCta);
  __shared__ long long s_item;
  __shared__ int s_next;
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  LeanWs ws{s_ws + (size_t)warp * LeanWs::elems(CAP, 1), LeanWs::pack(CAP, 1)};
  ChainCounters ctr{0, 0, 0, 0};
  for (;;) {
    __syncthreads();  // every warp is done with the previous item's table
    if (threadIdx.x == 0) s_item = atomicAdd((unsigned long long*)&D.ctr[C_ITEM], 1ULL), s_next = 0;
    __syncthreads();
    const long long item = s_item;
    if (item >= D.n_items) break;
    const int h = D.item_hap[item], r0 = D.item_r0[item], nr = D.item_n[item];
    const int64_t hoff = D.hap_off[h];
    const int hlen = (int)(D.hap_off[h + 1] - hoff);
    const int idx_n = D.idx_n[h];
    const uint8_t* hapc = D.hap_codes + hoff;
    const int g = D.hap_grp[h];
    const int h_local = h - D.grp_hap_begin[g];
    const int mid_occ = D.grp_mid[g];
    if (idx_n > kTabCap) {
      // a haplotype whose table does not fit the staging block (> ~1500 bp): its pairs go to the cold
      // kernel, which reads the table from HBM
      for (int rr = threadIdx.x; rr < nr; rr += blockDim.x) cold_push(D, r0 + rr, h);
      if (threadIdx.x == 0) atomicAdd((unsigned long long*)&D.ctr[C_COLD_LONG], (unsigned long long)nr);
      continue;
    }
    {
      const uint64_t* idx = D.idx + hoff;
      const uint16_t* bk = D.bkt + (size_t)h * (kBuckets + 1);
      for (int i = threadIdx.x; i < idx_n; i += blockDim.x) s_tab[i] = idx[i];
      for (int b = threadIdx.x; b <= kBuckets; b += blockDim.x) s_bkt[b] = bk[b];
    }
    __syncthreads();
#if LGR_CHAIN_LOCKSTEP
    // the CTA's warps start every pair together: they then run the same stretch of this kernel at about the
    // same time and share its instruction-cache lines, at the price of waiting for the slowest pair of a round
    for (int base = 0; base < nr; base += kWarpsPerCta) {
      __syncthreads();
      const int rr = base + warp;
      if (rr < nr) chain_pair<CAP, Tier::Lean>(D, r0 + rr, h, g, h_local, mid_occ, hapc, hlen, s_tab, idx_n, s_bkt, ws, nullptr, &s_regs[warp], ctr);
    }
#else
    for (;;) {
      int rr = 0;
      if (lane == 0) rr = atomicAdd(&s_next, 1);
      rr = __shfl_sync(full, rr, 0);
      if (rr >= nr) break;
      chain_pair<CAP, Tier::Lean>(D, r0 + rr, h, g, h_local, mid_occ, hapc, hlen, s_tab, idx_n, s_bkt, ws, nullptr, &s_regs[warp], ctr);
    }
#endif
  }
  if (lane == 0) {
    atomicAdd((unsigned long long*)&D.ctr[C_EVALS], (unsigned long long)ctr.chain_evals);
    atomicAdd((unsigned long long*)&D.ctr[C_ANCH], (unsigned long long)ctr.n_anchors);
    atomicAdd((unsigned long long*)&D.ctr[C_CELLSFULL], (unsigned long long)ctr.dp_cells_full);
  }
}

// Phase A, cold kernel: the pairs the lean kernel queued, one warp per pair, the complete code
// (mm_seed_select, the radix-pass emulation, the general chain DP and tail, several regs per pair),
// tables read from HBM (Tier::Cold).
template <int CAP>
__global__ void LGR_COLD_BOUNDS k_chain_cold(const __grid_constant__ Dev D) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t* s_ws = reinterpret_cast<int32_t*>(smem_raw);
  RegRec* s_regs = reinterpret_cast<RegRec*>(s_ws + (size_t)kWarpsPerCta * Ws<1>::elems(CAP, kRegCap));
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gwarp = blockIdx.x * kWarpsPerCta + warp;
  const long long n_cold = D.ctr[C_NCOLD];
  if (n_cold == 0) return;
  Ws<1> ws{s_ws + (size_t)warp * Ws<1>::elems(CAP, kRegCap), Ws<1>::pack(CAP, kRegCap)};
  RadixScratch* rsx = D.rsx_scratch + gwarp;
  ChainCounters ctr{0, 0, 0, 0};
  for (;;) {
    long long i = 0;
    if (lane == 0) i = atomicAdd((unsigned long long*)&D.ctr[C_COLDPOS], 1ULL);
    i = __shfl_sync(full, i, 0);
    if (i >= n_cold) break;
    const int r = D.cold_read[i], h = D.cold_hap[i];
    const int64_t hoff = D.hap_off[h];
    const int g = D.hap_grp[h];
    chain_pair<CAP, Tier::Cold>(D, r, h, g, h - D.grp_hap_begin[g], D.grp_mid[g], D.hap_codes + hoff, (int)(D.hap_off[h + 1] - hoff),
                           D.idx + hoff, D.idx_n[h], D.bkt + (size_t)h * (kBuckets + 1), ws, rsx, &s_regs[warp], ctr);
  }
  if (lane == 0) {
    atomicAdd((unsigned long long*)&D.ctr[C_EVALS], (unsigned long long)ctr.chain_evals);
    atomicAdd((unsigned long long*)&D.ctr[C_ANCH], (unsigned long long)ctr.n_anchors);
    atomicAdd((unsigned long long*)&D.ctr[C_CELLSFULL], (unsigned long long)ctr.dp_cells_full);
  }
}

}  // namespace

#endif  // LANCET2_B200_LGR_KERNELS_CHAIN_CUH_
