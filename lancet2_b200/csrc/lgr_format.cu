// lgr_format.cu — VariantSupport aggregation + FORMAT math on the device (SURVEY.md §8f #2):
// kernels k_fmt_dedup / k_fmt_metrics and the C-ABI entry points lgr_format_* declared in
// include/lancet_gpu_realign.h.  Own translation unit, compiled with -fmad=false so that the
// f64 expressions of lgr_format.cuh are evaluated as written (the host emulation is compiled
// with -ffp-contract=off).  No CPU fallback: a missing device is LGR_E_NO_DEVICE.
#include <cuda_runtime.h>

#include <cstring>

#include <string>
#include <vector>

#include "lgr_format.cuh"
#include "lgr_host.h"

namespace {

using lgr_fmt::Ev;

// global (L1-cached) rather than __constant__: lanes index it with different qualities
__device__ const double g_phred[256] = {
#include "phred_lut.inc"
};

struct FmtDev {
  Ev e;
  const int64_t* sup_begin;
  const int32_t* sup_n_alleles;
  const int32_t* sup_variant_len;
  const int32_t* sup_total_haps;
  uint8_t* keep;
  lgr_format* out;
  int32_t n_supports;
  int64_t n_evidence;
};

// one thread per evidence record: AddEvidence's first-seen rule against the earlier records of
// the same support (variant_support.cpp:28-29).  Supports are a few hundred records, so the scan
// is short and its loads are warp-uniform or coalesced.
__global__ void __launch_bounds__(256) k_fmt_dedup(const __grid_constant__ FmtDev D) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D.n_evidence) return;
  int lo = 0, hi = D.n_supports;  // last support with sup_begin <= i
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (D.sup_begin[mid] <= i) lo = mid;
    else hi = mid;
  }
  D.keep[i] = lgr_fmt::dedup_keep(D.e.allele, D.e.rname_hash, D.sup_begin[lo], i);
}


// ---------------------------------------------------------------------------------------------
// k_evidence_*: AddToTable on the device (SURVEY.md §8f #2, DESIGN.md §10.1).  From the resident
// lgr_assign records of a realignment batch and a few per-read columns, build the SoA evidence of
// every (variant, sample) support exactly as lancet_gpu::EvidenceColumns::AppendJob does on the host
// (genotyper.cpp:423-456): supports in (group, variant, sample-first-seen) order, records in read
// order.  The realignment's X31 name hash stands in for absl::HashOf(qname): the dedup only asks
// whether two records of a support carry the same name.
// ---------------------------------------------------------------------------------------------
constexpr int kEvMaxSamples = 32;

struct EvDev {
  const lgr_assign* assign;       // resident records of the realignment batch
  const int32_t* grp_read_begin;  // [G+1]
  const int32_t* grp_var_begin;   // [G+1]
  const int64_t* grp_asg_begin;   // [G+1] first assign record of the group
  const int32_t* grp_n_haps;      // [G]
  const int32_t* var_grp;         // [NV]
  const int32_t* var_n_alleles;   // [NV]
  const int32_t* var_len;         // [NV]
  const int64_t* r_insert;        // per read
  const int64_t* r_start;
  const uint32_t* r_hash;
  const int32_t* r_sample;
  const uint16_t* r_flag;
  const uint8_t* r_mapq;
  const uint8_t* r_soft;
  int32_t n_vars, n_samples;
  // slots: variant v owns [v * n_samples, (v+1) * n_samples), filled in sample-first-seen order
  int32_t* slot_cnt;
  int32_t* slot_sample;
  int64_t* slot_begin;
  long long* totals;  // [0] supports, [1] evidence records, [2] error flags
  // outputs: the columns of lgr_evidence_in + the support tables
  int64_t* sup_begin;
  int32_t* sup_n_alleles;
  int32_t* sup_variant_len;
  int32_t* sup_total_haps;
  int32_t* sup_key;  // [3 S]: group, variant, sample id
  int64_t* o_insert;
  int64_t* o_start;
  double* o_aln;
  double* o_fold;
  uint32_t* o_hash;
  uint32_t* o_rnm;
  uint32_t* o_onm;
  uint32_t* o_hid;
  uint8_t* o_allele;
  uint8_t* o_flags;
  uint8_t* o_bq;
  uint8_t* o_mq;
};

// one CTA per variant: per-sample record counts and the first read that names each sample
__global__ void __launch_bounds__(128) k_evidence_count(const __grid_constant__ EvDev D) {
  __shared__ int s_cnt[kEvMaxSamples];
  __shared__ int s_first[kEvMaxSamples];
  for (int v = blockIdx.x; v < D.n_vars; v += gridDim.x) {
    const int g = D.var_grp[v];
    const int r0 = D.grp_read_begin[g], R = D.grp_read_begin[g + 1] - r0;
    const int V = D.grp_var_begin[g + 1] - D.grp_var_begin[g], vi = v - D.grp_var_begin[g];
    const lgr_assign* a = D.assign + D.grp_asg_begin[g] + vi;
    __syncthreads();
    if (threadIdx.x < kEvMaxSamples) s_cnt[threadIdx.x] = 0, s_first[threadIdx.x] = 0x7fffffff;
    __syncthreads();
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
      if (!a[(int64_t)r * V].assigned) continue;
      const int sm = D.r_sample[r0 + r];
      atomicAdd(&s_cnt[sm], 1);
      atomicMin(&s_first[sm], r);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      // FindOrCreate's creation order: samples by the first read that contributes to this variant
      int order[kEvMaxSamples], n = 0;
      for (int sm = 0; sm < D.n_samples; ++sm)
        if (s_cnt[sm] > 0) {
          int at = n++;
          while (at > 0 && s_first[order[at - 1]] > s_first[sm]) order[at] = order[at - 1], --at;
          order[at] = sm;
        }
      for (int k = 0; k < D.n_samples; ++k) {
        D.slot_cnt[(int64_t)v * D.n_samples + k] = k < n ? s_cnt[order[k]] : 0;
        D.slot_sample[(int64_t)v * D.n_samples + k] = k < n ? order[k] : -1;
      }
    }
  }
}

// one CTA: exclusive scans over the slots → support numbers and evidence ranges, support tables
__global__ void __launch_bounds__(1024) k_evidence_scan(const __grid_constant__ EvDev D) {
  __shared__ long long s_ev[32];
  __shared__ int s_sup[32];
  __shared__ long long s_carry_ev;
  __shared__ int s_carry_sup;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n_slots = (int64_t)D.n_vars * D.n_samples;
  if (threadIdx.x == 0) s_carry_ev = 0, s_carry_sup = 0;
  __syncthreads();
  for (int64_t base = 0; base < n_slots; base += blockDim.x) {
    const int64_t slot = base + threadIdx.x;
    const int cnt = slot < n_slots ? D.slot_cnt[slot] : 0;
    long long ev = cnt;
    int sup = cnt > 0;
    for (int o = 1; o < 32; o <<= 1) {
      const long long e2 = __shfl_up_sync(0xffffffffu, ev, o);
      const int s2 = __shfl_up_sync(0xffffffffu, sup, o);
      if (lane >= o) ev += e2, sup += s2;
    }
    if (lane == 31) s_ev[warp] = ev, s_sup[warp] = sup;
    __syncthreads();
    if (warp == 0) {
      long long e = s_ev[lane];
      int u = s_sup[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const long long e2 = __shfl_up_sync(0xffffffffu, e, o);
        const int u2 = __shfl_up_sync(0xffffffffu, u, o);
        if (lane >= o) e += e2, u += u2;
      }
      s_ev[lane] = e, s_sup[lane] = u;
    }
    __syncthreads();
    const long long ev_excl = s_carry_ev + (warp > 0 ? s_ev[warp - 1] : 0) + ev - cnt;
    const int sup_excl = s_carry_sup + (warp > 0 ? s_sup[warp - 1] : 0) + sup - (cnt > 0);
    if (slot < n_slots) {
      D.slot_begin[slot] = ev_excl;
      if (cnt > 0) {
        const int v = (int)(slot / D.n_samples), g = D.var_grp[v];
        D.sup_begin[sup_excl] = ev_excl;
        D.sup_n_alleles[sup_excl] = D.var_n_alleles[v];
        D.sup_variant_len[sup_excl] = D.var_len[v];
        D.sup_total_haps[sup_excl] = D.grp_n_haps[g];
        D.sup_key[3 * sup_excl] = g, D.sup_key[3 * sup_excl + 1] = v, D.sup_key[3 * sup_excl + 2] = D.slot_sample[slot];
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_carry_ev += s_ev[31], s_carry_sup += s_sup[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    D.sup_begin[s_carry_sup] = s_carry_ev;
    D.totals[0] = s_carry_sup, D.totals[1] = s_carry_ev;
  }
}

// one warp per slot: the support's records in read order (ballot compaction), every column of ReadEvidence
__global__ void __launch_bounds__(128) k_evidence_scatter(const __grid_constant__ EvDev D) {
  const int lane = threadIdx.x & 31;
  const int64_t n_slots = (int64_t)D.n_vars * D.n_samples;
  for (int64_t slot = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5); slot < n_slots; slot += (int64_t)gridDim.x * 4) {
    if (D.slot_cnt[slot] == 0) continue;
    const int v = (int)(slot / D.n_samples), sm = D.slot_sample[slot], g = D.var_grp[v];
    const int r0 = D.grp_read_begin[g], R = D.grp_read_begin[g + 1] - r0;
    const int V = D.grp_var_begin[g + 1] - D.grp_var_begin[g], vi = v - D.grp_var_begin[g];
    const int K = D.var_n_alleles[v];
    const lgr_assign* ab = D.assign + D.grp_asg_begin[g] + vi;
    int64_t at = D.slot_begin[slot];
    for (int base = 0; base < R; base += 32) {
      const int r = base + lane;
      lgr_assign a;
      bool take = false;
      if (r < R && D.r_sample[r0 + r] == sm) {
        a = ab[(int64_t)r * V];
        take = a.assigned != 0;
      }
      const unsigned m = __ballot_sync(0xffffffffu, take);
      if (take) {
        const int64_t o = at + __popc(m & ((1u << lane) - 1u));
        const int rr = r0 + r;
        D.o_insert[o] = D.r_insert[rr], D.o_start[o] = D.r_start[rr];
        D.o_aln[o] = (double)a.global_score + (a.local_score * a.local_identity);  // CombinedScore(); -fmad=false: as written
        D.o_fold[o] = a.folded_read_pos;
        D.o_hash[o] = D.r_hash[rr], D.o_rnm[o] = a.ref_nm, D.o_onm[o] = a.own_hap_nm, D.o_hid[o] = a.hap_id;
        D.o_allele[o] = (uint8_t)a.allele;
        const unsigned fl = D.r_flag[rr];
        D.o_flags[o] = (uint8_t)(((fl & 0x10u) ? LGR_EV_REV : 0u) | (D.r_soft[rr] ? LGR_EV_SOFTCLIP : 0u) | ((fl & 0x2u) ? LGR_EV_PROPER_PAIR : 0u));
        D.o_bq[o] = a.base_qual, D.o_mq[o] = D.r_mapq[rr];
        if (a.allele < 0 || (int)a.allele >= K) atomicOr((unsigned long long*)&D.totals[2], 1ull);
      }
      at += __popc(m);
    }
  }
}

struct CtaDev {
  int tid;
  __device__ __forceinline__ bool leader() const { return tid == 0; }
#ifdef LGR_FMT_SORT  // DESIGN.md §10.1 #1: not in the default build until it has run on a GPU
  uint64_t* keys_;
  uint8_t* tags_;
  __device__ __forceinline__ uint64_t* sort_keys() const { return keys_; }
  __device__ __forceinline__ uint8_t* sort_tags() const { return tags_; }
  template <class F>
  __device__ __forceinline__ void each(const F& f) {
    f(tid);
    __syncthreads();
  }
#endif
  template <class A, class F>
  __device__ __forceinline__ A reduce(const F& f) {
    constexpr int nd = (int)(sizeof(A::d) / sizeof(double)), ni = (int)(sizeof(A::i) / sizeof(long long));
    __shared__ double s_d[lgr_fmt::kWarps][nd];
    __shared__ long long s_i[lgr_fmt::kWarps][ni];
    A a = f(tid);
#pragma unroll
    for (int off = lgr_fmt::kLanes / 2; off > 0; off >>= 1) {
#pragma unroll
      for (int k = 0; k < nd; ++k) a.d[k] = a.d[k] + __shfl_xor_sync(0xffffffffu, a.d[k], off);
#pragma unroll
      for (int k = 0; k < ni; ++k) a.i[k] = a.i[k] + __shfl_xor_sync(0xffffffffu, a.i[k], off);
    }
    if ((tid & 31) == 0) {
#pragma unroll
      for (int k = 0; k < nd; ++k) s_d[tid >> 5][k] = a.d[k];
#pragma unroll
      for (int k = 0; k < ni; ++k) s_i[tid >> 5][k] = a.i[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < nd; ++k) a.d[k] = (s_d[0][k] + s_d[1][k]) + (s_d[2][k] + s_d[3][k]);
#pragma unroll
    for (int k = 0; k < ni; ++k) a.i[k] = (s_i[0][k] + s_i[1][k]) + (s_i[2][k] + s_i[3][k]);
    __syncthreads();  // the partials may be overwritten by the next reduction of this instantiation
    return a;
  }
};

// one 128-thread CTA per (support, task): blockIdx.y is the task (lgr_fmt::kTask*), supports are
// taken in a grid-stride loop along x.  A batch of a few hundred supports is a few thousand CTAs.
__global__ void __launch_bounds__(lgr_fmt::kThreads) k_fmt_metrics(const __grid_constant__ FmtDev D) {
  const unsigned task = 1u << blockIdx.y;
#ifdef LGR_FMT_SORT
  __shared__ uint64_t s_keys[lgr_fmt::kSortCap];
  __shared__ uint8_t s_tags[lgr_fmt::kSortCap];
  CtaDev w{(int)threadIdx.x, s_keys, s_tags};
#else
  CtaDev w{(int)threadIdx.x};
#endif
  for (int s = (int)blockIdx.x; s < D.n_supports; s += (int)gridDim.x) {
    // a support with more alleles than the record's fixed arrays hold is not computed here (the host marks its
    // record LGR_FMT_WIDE): it runs as an empty one-allele support so that nothing indexes past the arrays
    const int K = D.sup_n_alleles[s];
    const bool wide = K > LGR_FMT_MAX_ALLELES;
    const int64_t b = D.sup_begin[s];
    lgr_fmt::support_metrics(w, D.e, b, wide ? b : D.sup_begin[s + 1], wide ? 1 : K, D.sup_variant_len[s], D.sup_total_haps[s], g_phred,
                             &D.out[s], task);
  }
}

// ---------------------------------------------------------------------------------------------
// Packed windows (lgr_format_pack / lgr_format_metrics_packed).  A block and the device arena of lgr_format_metrics
// share one section order (lgr_format.cu:391-394); fmt_layout gives the 16 offsets from `base` (the header size for a
// block, 0 for the arena) and returns the end.
// ---------------------------------------------------------------------------------------------
constexpr int kSecBegin = 0, kSecK = 5, kSecVl = 6, kSecTh = 7, kSecAllele = 12;
__host__ __device__ constexpr int fmt_sec_size(int k) { return k <= 4 ? 8 : k <= 11 ? 4 : 1; }
__host__ __device__ constexpr bool fmt_sec_per_support(int k) { return k == kSecBegin || (k >= kSecK && k <= kSecTh); }

__host__ __device__ inline uint64_t fmt_layout(int64_t S, int64_t N, uint64_t base, uint64_t* off) {
  uint64_t o = base;
  for (int k = 0; k < LGR_FMT_SECTIONS; ++k) {
    const uint64_t n = k == kSecBegin ? (uint64_t)S + 1 : fmt_sec_per_support(k) ? (uint64_t)S : (uint64_t)N;
    off[k] = o;
    o += (n * fmt_sec_size(k) + 15) & ~(uint64_t)15;
  }
  return o;
}

// offset of section k alone (the kernel's form of fmt_layout: no per-thread offset array in local memory)
__device__ __forceinline__ uint64_t fmt_sec_off(int64_t S, int64_t N, uint64_t base, int k) {
  uint64_t o = base;
#pragma unroll
  for (int j = 0; j < LGR_FMT_SECTIONS; ++j) {
    const uint64_t n = j == kSecBegin ? (uint64_t)S + 1 : fmt_sec_per_support(j) ? (uint64_t)S : (uint64_t)N;
    if (j < k) o += (n * fmt_sec_size(j) + 15) & ~(uint64_t)15;
  }
  return o;
}

struct UnpackDev {
  const uint8_t* slab;      // device copy of the slab
  const lgr_fmt_dir* dir;   // device copy of the directory
  int32_t n_windows, n_supports;
  int64_t n_evidence;
  int64_t n_rec_ctas;       // CTAs [0, n_rec_ctas) copy records, the rest one support per warp
  uint8_t* arena;           // lgr_format_metrics' arena, sections at aoff
  uint64_t aoff[LGR_FMT_SECTIONS];
  int* status;              // set to 1 when a block's records are malformed
};
constexpr int kUnpackThreads = 256, kUnpackWarps = kUnpackThreads / 32;
constexpr int64_t kUnpackChunk = 512;  // records per CTA of the copy half (a cfg2 step: 228 CTAs)

// last window whose base (ev_base or sup_base) is <= x: the window that holds record / support x (windows without any
// share their base with the next one and are skipped)
template <bool kEv>
__device__ __forceinline__ int fmt_window_of(const lgr_fmt_dir* dir, int n_windows, int64_t x) {
  int lo = 0, hi = n_windows;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((kEv ? dir[mid].ev_base : (int64_t)dir[mid].sup_base) <= x) lo = mid;
    else hi = mid;
  }
  return lo;
}

// one warp copies `bytes` bytes: 16-byte vectors when source and destination agree modulo 16, else elements of `es`
// bytes (both are always aligned to their element size)
__device__ __forceinline__ void fmt_copy_span(uint8_t* dst, const uint8_t* src, uint64_t bytes, int es, int lane) {
  const uint64_t mis = ((uintptr_t)dst ^ (uintptr_t)src) & 15;
  if (mis == 0) {
    uint64_t head = (16 - ((uintptr_t)src & 15)) & 15;
    if (head > bytes) head = bytes;
    for (uint64_t i = lane; i < head; i += 32) dst[i] = src[i];
    const uint64_t nvec = (bytes - head) >> 4;
    const uint4* s4 = reinterpret_cast<const uint4*>(src + head);
    uint4* d4 = reinterpret_cast<uint4*>(dst + head);
    for (uint64_t i = lane; i < nvec; i += 32) d4[i] = s4[i];
    for (uint64_t i = head + (nvec << 4) + lane; i < bytes; i += 32) dst[i] = src[i];
  } else if (es == 8) {
    for (uint64_t i = lane; i < bytes / 8; i += 32) reinterpret_cast<uint64_t*>(dst)[i] = reinterpret_cast<const uint64_t*>(src)[i];
  } else if (es == 4) {
    for (uint64_t i = lane; i < bytes / 4; i += 32) reinterpret_cast<uint32_t*>(dst)[i] = reinterpret_cast<const uint32_t*>(src)[i];
  } else {
    for (uint64_t i = lane; i < bytes; i += 32) dst[i] = src[i];
  }
}

// Scatter of the packed blocks into the arena, over two kinds of work item so that one oversized window is spread
// over the GPU like many small ones:
//  * a CTA of the first kind owns kUnpackChunk consecutive records of the batch; its warps take the (window, column)
//    pieces of that range and copy them;
//  * a warp of the second kind owns one support: sup_begin[sup_base + s] = ev_base + local_begin[s] (and the final
//    entry N), the three support columns, and the checks the host skipped.  A support whose range is not inside
//    [0, N] and ordered, whose K < 1, whose records name an allele >= K, or that is wide in a window that declared no
//    wide supports sets *status and is written as a wide (never computed) support with a clamped begin, so that
//    k_fmt_dedup / k_fmt_metrics stay inside the arena whatever the slab holds.
__global__ void __launch_bounds__(kUnpackThreads) k_fmt_unpack(const __grid_constant__ UnpackDev U) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr uint64_t kHdr = sizeof(lgr_fmt_blk_hdr);
  if ((int64_t)blockIdx.x < U.n_rec_ctas) {
    const int64_t lo = (int64_t)blockIdx.x * kUnpackChunk;
    const int64_t hi = lo + kUnpackChunk < U.n_evidence ? lo + kUnpackChunk : U.n_evidence;
    const int w0 = fmt_window_of<true>(U.dir, U.n_windows, lo);
    constexpr int kCols = LGR_FMT_SECTIONS - 4;  // the twelve record columns
    for (int piece = warp;; piece += kUnpackWarps) {
      const int w = w0 + piece / kCols;
      if (w >= U.n_windows) break;
      const lgr_fmt_dir d = U.dir[w];
      if (d.ev_base >= hi) break;
      const int64_t a = lo > d.ev_base ? lo - d.ev_base : 0;
      const int64_t b = hi - d.ev_base < d.n_evidence ? hi - d.ev_base : d.n_evidence;
      if (a >= b) continue;
      const int c = piece % kCols, k = c < 4 ? 1 + c : 4 + c;  // sections 1..4 and 8..15
      const int es = fmt_sec_size(k);
      fmt_copy_span(U.arena + U.aoff[k] + (uint64_t)(d.ev_base + a) * es,
                    U.slab + d.rec_off + fmt_sec_off(d.n_supports, d.n_evidence, kHdr, k) + (uint64_t)a * es,
                    (uint64_t)(b - a) * es, es, lane);
    }
    return;
  }
  const int64_t g = ((int64_t)blockIdx.x - U.n_rec_ctas) * kUnpackWarps + warp;
  if (g >= U.n_supports) return;
  const int w = fmt_window_of<false>(U.dir, U.n_windows, g);
  const lgr_fmt_dir d = U.dir[w];
  const int s = (int)(g - d.sup_base);
  const uint8_t* blk = U.slab + d.rec_off;
  const int64_t* lb = reinterpret_cast<const int64_t*>(blk + kHdr);
  const int64_t N = d.n_evidence, b = lb[s], e = lb[s + 1];
  const int K = reinterpret_cast<const int32_t*>(blk + fmt_sec_off(d.n_supports, N, kHdr, kSecK))[s];
  bool ok = lb[0] == 0 && lb[d.n_supports] == N && 0 <= b && b <= e && e <= N && K >= 1 &&
            (K <= LGR_FMT_MAX_ALLELES || d.n_wide > 0);
  if (ok) {
    const uint8_t* al = blk + fmt_sec_off(d.n_supports, N, kHdr, kSecAllele);
    bool bad = false;
    for (int64_t i = b + lane; i < e; i += 32) bad |= al[i] >= K;
    ok = !__any_sync(0xffffffffu, bad);
  }
  if (lane == 0) {
    reinterpret_cast<int64_t*>(U.arena + U.aoff[kSecBegin])[g] = d.ev_base + (b < 0 ? 0 : b > N ? N : b);
    reinterpret_cast<int32_t*>(U.arena + U.aoff[kSecK])[g] = ok ? K : LGR_FMT_MAX_ALLELES + 1;
    reinterpret_cast<int32_t*>(U.arena + U.aoff[kSecVl])[g] = reinterpret_cast<const int32_t*>(blk + fmt_sec_off(d.n_supports, N, kHdr, kSecVl))[s];
    reinterpret_cast<int32_t*>(U.arena + U.aoff[kSecTh])[g] = reinterpret_cast<const int32_t*>(blk + fmt_sec_off(d.n_supports, N, kHdr, kSecTh))[s];
    if (g == U.n_supports - 1) reinterpret_cast<int64_t*>(U.arena + U.aoff[kSecBegin])[g + 1] = U.n_evidence;
    if (!ok) *U.status = 1;
  }
}

}  // namespace

struct lgr_fmt_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;
  DeviceBuffer b_in, b_keep, b_out;  // one packed input arena, the dedup flags, the results
  DeviceBuffer b_ev, b_key;           // lgr_format_from_assign: per-read / per-variant inputs + slots, support keys
  DeviceBuffer b_slab, b_dir;         // lgr_format_metrics_packed: the slab (+ status word), a directory outside it
  lgr_evidence_in last_ev{};  // device pointers of the columns the last call worked on (lgr_format_debug_evidence)
};

static thread_local std::string g_fmt_create_err;

extern "C" {

int lgr_format_create(int device_ordinal, lgr_fmt_ctx** out) {
  if (!out) return LGR_E_ARG;
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0) {
    g_fmt_create_err = "no CUDA device (this path has no CPU fallback)";
    return LGR_E_NO_DEVICE;
  }
  if (device_ordinal < 0 || device_ordinal >= n_dev) {
    g_fmt_create_err = "device ordinal out of range";
    return LGR_E_ARG;
  }
  lgr_fmt_ctx* c = new lgr_fmt_ctx();
  c->device = device_ordinal;
  cudaError_t e = cudaSetDevice(device_ordinal);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device_ordinal);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
  if (e != cudaSuccess) {
    g_fmt_create_err = std::string("lgr_format_create: ") + cudaGetErrorString(e);
    lgr_format_destroy(c);
    return LGR_E_CUDA;
  }
  *out = c;
  return LGR_OK;
}

void lgr_format_destroy(lgr_fmt_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;  // frees the device buffers
}

const char* lgr_format_last_error(const lgr_fmt_ctx* c) { return c ? c->err.c_str() : g_fmt_create_err.c_str(); }

int lgr_format_metrics(lgr_fmt_ctx* c, const lgr_evidence_in* in, lgr_format* out, float* ms_kernels) {
  if (!c || !in || (!out && in->n_supports > 0)) return LGR_E_ARG;
  c->err.clear();
  if (ms_kernels) *ms_kernels = 0.0f;
  const int S = in->n_supports;
  const int64_t N = in->n_evidence;
  if (S < 0 || N < 0) return c->err = "negative sizes", LGR_E_ARG;
  if (S == 0) return LGR_OK;
  int n_wide = 0;
  if (!in->sup_begin || !in->sup_n_alleles || !in->sup_variant_len || !in->sup_total_haps)
    return c->err = "missing support arrays", LGR_E_ARG;
  if (in->sup_begin[0] != 0 || in->sup_begin[S] != N) return c->err = "sup_begin must span [0, n_evidence]", LGR_E_ARG;
  for (int s = 0; s < S; ++s) {
    if (in->sup_begin[s + 1] < in->sup_begin[s]) return c->err = "sup_begin not monotone", LGR_E_ARG;
    if (in->sup_n_alleles[s] < 1) return c->err = "support with fewer than one allele", LGR_E_ARG;
    n_wide += in->sup_n_alleles[s] > LGR_FMT_MAX_ALLELES;  // not an error of the batch: see LGR_FMT_WIDE
  }
  if (N > 0 && !(in->insert_size && in->aln_start && in->aln_score && in->folded_pos && in->rname_hash && in->ref_nm &&
                 in->own_hap_nm && in->hap_id && in->allele && in->flags && in->base_qual && in->map_qual))
    return c->err = "missing evidence arrays", LGR_E_ARG;
  for (int s = 0; s < S; ++s)
    for (int64_t i = in->sup_begin[s]; i < in->sup_begin[s + 1]; ++i)
      if (in->allele[i] >= in->sup_n_alleles[s]) return c->err = "evidence allele index >= the support's allele count", LGR_E_ARG;

  LGR_CUDA(c, cudaSetDevice(c->device));
  // one packed arena: 8-byte arrays first, then 4-byte, then bytes (every section 16-byte aligned)
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t n = (size_t)N;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += up16(bytes);
    return o;
  };
  const size_t o_begin = take((size_t)(S + 1) * 8), o_isz = take(n * 8), o_start = take(n * 8), o_aln = take(n * 8),
               o_fold = take(n * 8), o_k = take((size_t)S * 4), o_vl = take((size_t)S * 4), o_th = take((size_t)S * 4),
               o_hash = take(n * 4), o_rnm = take(n * 4), o_onm = take(n * 4), o_hid = take(n * 4), o_al = take(n),
               o_fl = take(n), o_bq = take(n), o_mq = take(n);
  int rc;
  if ((rc = c->b_in.ensure(off, false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_keep.ensure(n, false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_out.ensure((size_t)S * sizeof(lgr_format), false, c->err)) != LGR_OK) return rc;
  char* base = (char*)c->b_in.p;
  auto h2d = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
    return bytes ? cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, c->stream) : cudaSuccess;
  };
  LGR_CUDA(c, h2d(o_begin, in->sup_begin, (size_t)(S + 1) * 8));
  LGR_CUDA(c, h2d(o_k, in->sup_n_alleles, (size_t)S * 4));
  LGR_CUDA(c, h2d(o_vl, in->sup_variant_len, (size_t)S * 4));
  LGR_CUDA(c, h2d(o_th, in->sup_total_haps, (size_t)S * 4));
  LGR_CUDA(c, h2d(o_isz, in->insert_size, n * 8));
  LGR_CUDA(c, h2d(o_start, in->aln_start, n * 8));
  LGR_CUDA(c, h2d(o_aln, in->aln_score, n * 8));
  LGR_CUDA(c, h2d(o_fold, in->folded_pos, n * 8));
  LGR_CUDA(c, h2d(o_hash, in->rname_hash, n * 4));
  LGR_CUDA(c, h2d(o_rnm, in->ref_nm, n * 4));
  LGR_CUDA(c, h2d(o_onm, in->own_hap_nm, n * 4));
  LGR_CUDA(c, h2d(o_hid, in->hap_id, n * 4));
  LGR_CUDA(c, h2d(o_al, in->allele, n));
  LGR_CUDA(c, h2d(o_fl, in->flags, n));
  LGR_CUDA(c, h2d(o_bq, in->base_qual, n));
  LGR_CUDA(c, h2d(o_mq, in->map_qual, n));

  FmtDev D;
  D.e.insert_size = (const int64_t*)(base + o_isz), D.e.aln_start = (const int64_t*)(base + o_start);
  D.e.aln_score = (const double*)(base + o_aln), D.e.folded_pos = (const double*)(base + o_fold);
  D.e.rname_hash = (const uint32_t*)(base + o_hash), D.e.ref_nm = (const uint32_t*)(base + o_rnm);
  D.e.own_hap_nm = (const uint32_t*)(base + o_onm), D.e.hap_id = (const uint32_t*)(base + o_hid);
  D.e.allele = (const uint8_t*)(base + o_al), D.e.flags = (const uint8_t*)(base + o_fl);
  D.e.base_qual = (const uint8_t*)(base + o_bq), D.e.map_qual = (const uint8_t*)(base + o_mq);
  D.e.keep = (const uint8_t*)c->b_keep.p;
  D.sup_begin = (const int64_t*)(base + o_begin), D.sup_n_alleles = (const int32_t*)(base + o_k);
  D.sup_variant_len = (const int32_t*)(base + o_vl), D.sup_total_haps = (const int32_t*)(base + o_th);
  D.keep = (uint8_t*)c->b_keep.p, D.out = (lgr_format*)c->b_out.p;
  D.n_supports = S, D.n_evidence = N;

  LGR_CUDA(c, cudaEventRecord(c->ev0, c->stream));
  if (N > 0) {
    const unsigned blocks = (unsigned)((N + 255) / 256);
    k_fmt_dedup<<<blocks, 256, 0, c->stream>>>(D);
    LGR_CUDA(c, cudaGetLastError());
  }
  {
    // one CTA per (support, task); beyond 32 CTAs per SM and task the supports are grid-strided
    const int cap = c->sm_count * 32;
    const dim3 grid((unsigned)(S < cap ? S : cap), (unsigned)lgr_fmt::kNumTasks);
    k_fmt_metrics<<<grid, lgr_fmt::kThreads, 0, c->stream>>>(D);
    LGR_CUDA(c, cudaGetLastError());
  }
  LGR_CUDA(c, cudaEventRecord(c->ev1, c->stream));
  LGR_CUDA(c, cudaMemcpyAsync(out, c->b_out.p, (size_t)S * sizeof(lgr_format), cudaMemcpyDeviceToHost, c->stream));
  LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  if (ms_kernels) LGR_CUDA(c, cudaEventElapsedTime(ms_kernels, c->ev0, c->ev1));
  if (n_wide > 0) {
    for (int s = 0; s < S; ++s)
      if (in->sup_n_alleles[s] > LGR_FMT_MAX_ALLELES) {
        std::memset(&out[s], 0, sizeof(lgr_format));
        out[s].n_alleles = (uint32_t)in->sup_n_alleles[s], out[s].valid = LGR_FMT_WIDE;
      }
    c->err = "some supports have more than LGR_FMT_MAX_ALLELES alleles (records flagged LGR_FMT_WIDE)";
    return LGR_E_PARTIAL;
  }
  return LGR_OK;
}

// AddToTable + FORMAT math without the host round trip: evidence columns are built on the device from the
// realignment's resident lgr_assign records (k_evidence_*), then k_fmt_dedup / k_fmt_metrics run on them.
int lgr_format_from_assign(lgr_fmt_ctx* c, const lgr_assign_batch* in, lgr_format* out, int32_t out_cap, int32_t* sup_key,
                           int32_t* n_supports, float* ms_kernels) {
  if (!c || !in || !n_supports) return LGR_E_ARG;
  c->err.clear();
  *n_supports = 0;
  if (ms_kernels) *ms_kernels = 0.0f;
  const int G = in->n_groups, NR = in->n_reads, NV = in->n_vars, NS = in->n_samples;
  if (G < 0 || NR < 0 || NV < 0 || in->n_assign < 0) return c->err = "negative sizes", LGR_E_ARG;
  if (NS < 1 || NS > kEvMaxSamples) return c->err = "n_samples must be in [1, 32]", LGR_E_LIMIT;
  if (G == 0 || NV == 0 || in->n_assign == 0) return LGR_OK;
  if (!in->dev_assign && !in->host_assign) return c->err = "neither dev_assign nor host_assign", LGR_E_ARG;
  if (!in->grp_read_begin || !in->grp_var_begin || !in->grp_n_haps || !in->var_n_alleles || !in->var_len || !in->read_insert_size ||
      !in->read_aln_start || !in->read_name_hash || !in->read_sample || !in->read_sam_flag || !in->read_map_qual ||
      !in->read_soft_clipped)
    return c->err = "missing input arrays", LGR_E_ARG;
  if (in->grp_read_begin[0] != 0 || in->grp_var_begin[0] != 0 || in->grp_read_begin[G] != NR || in->grp_var_begin[G] != NV)
    return c->err = "group prefix arrays do not span the reads / variants", LGR_E_ARG;
  std::vector<int64_t> asg_begin((size_t)G + 1, 0);
  std::vector<int32_t> var_grp((size_t)NV);
  for (int g = 0; g < G; ++g) {
    const int R = in->grp_read_begin[g + 1] - in->grp_read_begin[g], V = in->grp_var_begin[g + 1] - in->grp_var_begin[g];
    if (R < 0 || V < 0) return c->err = "group prefix arrays must be non-decreasing", LGR_E_ARG;
    asg_begin[(size_t)g + 1] = asg_begin[(size_t)g] + (int64_t)R * V;
    for (int v = in->grp_var_begin[g]; v < in->grp_var_begin[g + 1]; ++v) var_grp[(size_t)v] = g;
  }
  if (asg_begin[(size_t)G] != in->n_assign) return c->err = "n_assign is not the sum of reads x variants over the groups", LGR_E_ARG;
  for (int r = 0; r < NR; ++r)
    if (in->read_sample[r] < 0 || in->read_sample[r] >= NS) return c->err = "read_sample out of range", LGR_E_ARG;
  for (int v = 0; v < NV; ++v)
    if (in->var_n_alleles[v] < 1) return c->err = "variant with fewer than one allele", LGR_E_ARG;
  const int64_t n_slots = (int64_t)NV * NS;
  if (n_slots > out_cap && (!out || !sup_key)) return c->err = "out / sup_key missing", LGR_E_ARG;

  LGR_CUDA(c, cudaSetDevice(c->device));
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += up16(bytes);
    return o;
  };
  // inputs + slots
  const size_t nr = (size_t)NR, nv = (size_t)NV, ng = (size_t)G, na = (size_t)in->n_assign;
  const size_t i_asg = take(in->dev_assign ? 0 : na * sizeof(lgr_assign)), i_grb = take((ng + 1) * 4), i_gvb = take((ng + 1) * 4),
               i_gab = take((ng + 1) * 8), i_gnh = take(ng * 4), i_vg = take(nv * 4), i_vk = take(nv * 4), i_vl = take(nv * 4),
               i_ins = take(nr * 8), i_st = take(nr * 8), i_hash = take(nr * 4), i_smp = take(nr * 4), i_flag = take(nr * 2),
               i_mq = take(nr), i_sc = take(nr), i_scnt = take((size_t)n_slots * 4), i_ssmp = take((size_t)n_slots * 4),
               i_sbeg = take((size_t)n_slots * 8), i_tot = take(3 * 8);
  int rc;
  if ((rc = c->b_ev.ensure(off, false, c->err)) != LGR_OK) return rc;
  char* eb = (char*)c->b_ev.p;
  // columns (capacity: one record per assign record, one support per slot)
  off = 0;
  const size_t S_cap = (size_t)n_slots;
  const size_t o_begin = take((S_cap + 1) * 8), o_isz = take(na * 8), o_start = take(na * 8), o_aln = take(na * 8), o_fold = take(na * 8),
               o_k = take(S_cap * 4), o_vl = take(S_cap * 4), o_th = take(S_cap * 4), o_hash = take(na * 4), o_rnm = take(na * 4),
               o_onm = take(na * 4), o_hid = take(na * 4), o_al = take(na), o_fl = take(na), o_bq = take(na), o_mq = take(na);
  if ((rc = c->b_in.ensure(off, false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_keep.ensure(na, false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_out.ensure(S_cap * sizeof(lgr_format), false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_key.ensure(S_cap * 3 * sizeof(int32_t), false, c->err)) != LGR_OK) return rc;
  char* base = (char*)c->b_in.p;
  auto h2d = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
    return bytes ? cudaMemcpyAsync(eb + o, src, bytes, cudaMemcpyHostToDevice, c->stream) : cudaSuccess;
  };
  if (!in->dev_assign) LGR_CUDA(c, h2d(i_asg, in->host_assign, na * sizeof(lgr_assign)));
  LGR_CUDA(c, h2d(i_grb, in->grp_read_begin, (ng + 1) * 4));
  LGR_CUDA(c, h2d(i_gvb, in->grp_var_begin, (ng + 1) * 4));
  LGR_CUDA(c, h2d(i_gab, asg_begin.data(), (ng + 1) * 8));
  LGR_CUDA(c, h2d(i_gnh, in->grp_n_haps, ng * 4));
  LGR_CUDA(c, h2d(i_vg, var_grp.data(), nv * 4));
  LGR_CUDA(c, h2d(i_vk, in->var_n_alleles, nv * 4));
  LGR_CUDA(c, h2d(i_vl, in->var_len, nv * 4));
  LGR_CUDA(c, h2d(i_ins, in->read_insert_size, nr * 8));
  LGR_CUDA(c, h2d(i_st, in->read_aln_start, nr * 8));
  LGR_CUDA(c, h2d(i_hash, in->read_name_hash, nr * 4));
  LGR_CUDA(c, h2d(i_smp, in->read_sample, nr * 4));
  LGR_CUDA(c, h2d(i_flag, in->read_sam_flag, nr * 2));
  LGR_CUDA(c, h2d(i_mq, in->read_map_qual, nr));
  LGR_CUDA(c, h2d(i_sc, in->read_soft_clipped, nr));
  LGR_CUDA(c, cudaMemsetAsync(eb + i_tot, 0, 3 * 8, c->stream));

  EvDev E;
  E.assign = in->dev_assign ? in->dev_assign : (const lgr_assign*)(eb + i_asg);
  E.grp_read_begin = (const int32_t*)(eb + i_grb), E.grp_var_begin = (const int32_t*)(eb + i_gvb);
  E.grp_asg_begin = (const int64_t*)(eb + i_gab), E.grp_n_haps = (const int32_t*)(eb + i_gnh);
  E.var_grp = (const int32_t*)(eb + i_vg), E.var_n_alleles = (const int32_t*)(eb + i_vk), E.var_len = (const int32_t*)(eb + i_vl);
  E.r_insert = (const int64_t*)(eb + i_ins), E.r_start = (const int64_t*)(eb + i_st), E.r_hash = (const uint32_t*)(eb + i_hash);
  E.r_sample = (const int32_t*)(eb + i_smp), E.r_flag = (const uint16_t*)(eb + i_flag), E.r_mapq = (const uint8_t*)(eb + i_mq);
  E.r_soft = (const uint8_t*)(eb + i_sc);
  E.n_vars = NV, E.n_samples = NS;
  E.slot_cnt = (int32_t*)(eb + i_scnt), E.slot_sample = (int32_t*)(eb + i_ssmp), E.slot_begin = (int64_t*)(eb + i_sbeg);
  E.totals = (long long*)(eb + i_tot);
  E.sup_begin = (int64_t*)(base + o_begin), E.sup_n_alleles = (int32_t*)(base + o_k), E.sup_variant_len = (int32_t*)(base + o_vl);
  E.sup_total_haps = (int32_t*)(base + o_th), E.sup_key = (int32_t*)c->b_key.p;
  E.o_insert = (int64_t*)(base + o_isz), E.o_start = (int64_t*)(base + o_start), E.o_aln = (double*)(base + o_aln);
  E.o_fold = (double*)(base + o_fold), E.o_hash = (uint32_t*)(base + o_hash), E.o_rnm = (uint32_t*)(base + o_rnm);
  E.o_onm = (uint32_t*)(base + o_onm), E.o_hid = (uint32_t*)(base + o_hid), E.o_allele = (uint8_t*)(base + o_al);
  E.o_flags = (uint8_t*)(base + o_fl), E.o_bq = (uint8_t*)(base + o_bq), E.o_mq = (uint8_t*)(base + o_mq);

  LGR_CUDA(c, cudaEventRecord(c->ev0, c->stream));
  k_evidence_count<<<NV < c->sm_count * 16 ? NV : c->sm_count * 16, 128, 0, c->stream>>>(E);
  k_evidence_scan<<<1, 1024, 0, c->stream>>>(E);
  {
    const int64_t want = (n_slots + 3) / 4;
    k_evidence_scatter<<<(unsigned)(want < c->sm_count * 16 ? want : c->sm_count * 16), 128, 0, c->stream>>>(E);
  }
  LGR_CUDA(c, cudaGetLastError());
  long long totals[3] = {0, 0, 0};
  LGR_CUDA(c, cudaMemcpyAsync(totals, eb + i_tot, sizeof(totals), cudaMemcpyDeviceToHost, c->stream));
  LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  const int S = (int)totals[0];
  const int64_t N = totals[1];
  if (totals[2] != 0) return c->err = "an assignment names an allele outside its variant's allele count", LGR_E_ARG;
  *n_supports = S;
  if (S > out_cap) return c->err = "out / sup_key too small for the supports of this batch", LGR_E_ARG;

  FmtDev D;
  D.e.insert_size = E.o_insert, D.e.aln_start = E.o_start, D.e.aln_score = E.o_aln, D.e.folded_pos = E.o_fold;
  D.e.rname_hash = E.o_hash, D.e.ref_nm = E.o_rnm, D.e.own_hap_nm = E.o_onm, D.e.hap_id = E.o_hid;
  D.e.allele = E.o_allele, D.e.flags = E.o_flags, D.e.base_qual = E.o_bq, D.e.map_qual = E.o_mq;
  D.e.keep = (const uint8_t*)c->b_keep.p;
  D.sup_begin = E.sup_begin, D.sup_n_alleles = E.sup_n_alleles, D.sup_variant_len = E.sup_variant_len, D.sup_total_haps = E.sup_total_haps;
  D.keep = (uint8_t*)c->b_keep.p, D.out = (lgr_format*)c->b_out.p;
  D.n_supports = S, D.n_evidence = N;
  c->last_ev = lgr_evidence_in{};
  c->last_ev.n_supports = S, c->last_ev.n_evidence = N;
  c->last_ev.sup_begin = E.sup_begin, c->last_ev.sup_n_alleles = E.sup_n_alleles, c->last_ev.sup_variant_len = E.sup_variant_len;
  c->last_ev.sup_total_haps = E.sup_total_haps, c->last_ev.insert_size = E.o_insert, c->last_ev.aln_start = E.o_start;
  c->last_ev.aln_score = E.o_aln, c->last_ev.folded_pos = E.o_fold, c->last_ev.rname_hash = E.o_hash, c->last_ev.ref_nm = E.o_rnm;
  c->last_ev.own_hap_nm = E.o_onm, c->last_ev.hap_id = E.o_hid, c->last_ev.allele = E.o_allele, c->last_ev.flags = E.o_flags;
  c->last_ev.base_qual = E.o_bq, c->last_ev.map_qual = E.o_mq;
  if (S > 0) {
    if (N > 0) {
      k_fmt_dedup<<<(unsigned)((N + 255) / 256), 256, 0, c->stream>>>(D);
      LGR_CUDA(c, cudaGetLastError());
    }
    const int cap = c->sm_count * 32;
    const dim3 grid((unsigned)(S < cap ? S : cap), (unsigned)lgr_fmt::kNumTasks);
    k_fmt_metrics<<<grid, lgr_fmt::kThreads, 0, c->stream>>>(D);
    LGR_CUDA(c, cudaGetLastError());
  }
  LGR_CUDA(c, cudaEventRecord(c->ev1, c->stream));
  if (S > 0) {
    LGR_CUDA(c, cudaMemcpyAsync(out, c->b_out.p, (size_t)S * sizeof(lgr_format), cudaMemcpyDeviceToHost, c->stream));
    LGR_CUDA(c, cudaMemcpyAsync(sup_key, c->b_key.p, (size_t)S * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  }
  LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  if (ms_kernels) LGR_CUDA(c, cudaEventElapsedTime(ms_kernels, c->ev0, c->ev1));
  int n_wide = 0;
  for (int s = 0; s < S; ++s) {
    const int K = in->var_n_alleles[sup_key[3 * s + 1]];
    if (K > LGR_FMT_MAX_ALLELES) {
      std::memset(&out[s], 0, sizeof(lgr_format));
      out[s].n_alleles = (uint32_t)K, out[s].valid = LGR_FMT_WIDE;
      ++n_wide;
    }
  }
  if (n_wide > 0) {
    c->err = "some supports have more than LGR_FMT_MAX_ALLELES alleles (records flagged LGR_FMT_WIDE)";
    return LGR_E_PARTIAL;
  }
  return LGR_OK;
}

// Test hook: copy the evidence columns the last lgr_format_from_assign built on the device into caller buffers
// (dst's pointers are DESTINATIONS with room for n_evidence / n_supports entries; NULL ones are skipped).
int lgr_format_debug_evidence(lgr_fmt_ctx* c, lgr_evidence_in* dst) {
  if (!c || !dst) return LGR_E_ARG;
  const lgr_evidence_in& L = c->last_ev;
  const size_t n = (size_t)L.n_evidence, S = (size_t)L.n_supports;
  dst->n_supports = L.n_supports, dst->n_evidence = L.n_evidence;
  LGR_CUDA(c, cudaSetDevice(c->device));
  auto cp = [&](const void* d, const void* s, size_t bytes) -> cudaError_t {
    return d && s && bytes ? cudaMemcpy(const_cast<void*>(d), s, bytes, cudaMemcpyDeviceToHost) : cudaSuccess;
  };
  if (S > 0) {
    LGR_CUDA(c, cp(dst->sup_begin, L.sup_begin, (S + 1) * 8));
    LGR_CUDA(c, cp(dst->sup_n_alleles, L.sup_n_alleles, S * 4));
    LGR_CUDA(c, cp(dst->sup_variant_len, L.sup_variant_len, S * 4));
    LGR_CUDA(c, cp(dst->sup_total_haps, L.sup_total_haps, S * 4));
  }
  LGR_CUDA(c, cp(dst->insert_size, L.insert_size, n * 8));
  LGR_CUDA(c, cp(dst->aln_start, L.aln_start, n * 8));
  LGR_CUDA(c, cp(dst->aln_score, L.aln_score, n * 8));
  LGR_CUDA(c, cp(dst->folded_pos, L.folded_pos, n * 8));
  LGR_CUDA(c, cp(dst->rname_hash, L.rname_hash, n * 4));
  LGR_CUDA(c, cp(dst->ref_nm, L.ref_nm, n * 4));
  LGR_CUDA(c, cp(dst->own_hap_nm, L.own_hap_nm, n * 4));
  LGR_CUDA(c, cp(dst->hap_id, L.hap_id, n * 4));
  LGR_CUDA(c, cp(dst->allele, L.allele, n));
  LGR_CUDA(c, cp(dst->flags, L.flags, n));
  LGR_CUDA(c, cp(dst->base_qual, L.base_qual, n));
  LGR_CUDA(c, cp(dst->map_qual, L.map_qual, n));
  return LGR_OK;
}

size_t lgr_format_packed_bytes(const lgr_evidence_in* in) {
  if (!in || in->n_supports < 0 || in->n_evidence < 0) return 0;
  uint64_t off[LGR_FMT_SECTIONS];
  // a window without supports packs as an empty block (lgr_format_metrics returns before looking at its records)
  return in->n_supports == 0 ? fmt_layout(0, 0, sizeof(lgr_fmt_blk_hdr), off)
                             : fmt_layout(in->n_supports, in->n_evidence, sizeof(lgr_fmt_blk_hdr), off);
}

int lgr_format_pack(const lgr_evidence_in* in, void* dst, size_t cap, lgr_fmt_dir* dir) {
  if (!in || !dst || in->n_supports < 0 || in->n_evidence < 0) return LGR_E_ARG;
  const int S = in->n_supports;
  const int64_t N = S == 0 ? 0 : in->n_evidence;
  int n_wide = 0;
  if (S > 0) {  // the checks of lgr_format_metrics (lgr_format.cu:358-379), in the same order
    if (!in->sup_begin || !in->sup_n_alleles || !in->sup_variant_len || !in->sup_total_haps) return LGR_E_ARG;
    if (in->sup_begin[0] != 0 || in->sup_begin[S] != N) return LGR_E_ARG;
    for (int s = 0; s < S; ++s) {
      if (in->sup_begin[s + 1] < in->sup_begin[s] || in->sup_n_alleles[s] < 1) return LGR_E_ARG;
      n_wide += in->sup_n_alleles[s] > LGR_FMT_MAX_ALLELES;
    }
    if (N > 0 && !(in->insert_size && in->aln_start && in->aln_score && in->folded_pos && in->rname_hash && in->ref_nm &&
                   in->own_hap_nm && in->hap_id && in->allele && in->flags && in->base_qual && in->map_qual))
      return LGR_E_ARG;
    for (int s = 0; s < S; ++s)
      for (int64_t i = in->sup_begin[s]; i < in->sup_begin[s + 1]; ++i)
        if (in->allele[i] >= in->sup_n_alleles[s]) return LGR_E_ARG;
  }
  lgr_fmt_blk_hdr h{};
  h.magic = LGR_FMT_MAGIC, h.n_supports = S, h.n_evidence = N;
  h.rec_bytes = fmt_layout(S, N, sizeof(lgr_fmt_blk_hdr), h.off);
  if (cap < h.rec_bytes) return LGR_E_ARG;
  uint8_t* p = static_cast<uint8_t*>(dst);
  std::memcpy(p, &h, sizeof(h));
  const void* src[LGR_FMT_SECTIONS] = {in->sup_begin, in->insert_size, in->aln_start, in->aln_score, in->folded_pos,
                                       in->sup_n_alleles, in->sup_variant_len, in->sup_total_haps, in->rname_hash,
                                       in->ref_nm, in->own_hap_nm, in->hap_id, in->allele, in->flags, in->base_qual,
                                       in->map_qual};
  for (int k = 0; k < LGR_FMT_SECTIONS; ++k) {
    const uint64_t end = k + 1 < LGR_FMT_SECTIONS ? h.off[k + 1] : h.rec_bytes;
    const uint64_t n = S == 0 ? 0 : (k == kSecBegin ? (uint64_t)S + 1 : fmt_sec_per_support(k) ? (uint64_t)S : (uint64_t)N) * fmt_sec_size(k);
    if (n) std::memcpy(p + h.off[k], src[k], n);
    std::memset(p + h.off[k] + n, 0, end - h.off[k] - n);  // padding: the bytes of a block depend on the window only
  }
  if (dir) {
    *dir = lgr_fmt_dir{};
    dir->n_supports = S, dir->n_evidence = N, dir->n_wide = n_wide;
  }
  return LGR_OK;
}

int lgr_format_metrics_packed(lgr_fmt_ctx* c, const lgr_fmt_packed_in* in, lgr_format* out, float* ms_kernels) {
  if (!c || !in) return LGR_E_ARG;
  c->err.clear();
  if (ms_kernels) *ms_kernels = 0.0f;
  const int W = in->n_windows;
  if (W < 0) return c->err = "negative n_windows", LGR_E_ARG;
  if (W == 0) return LGR_OK;
  if (!in->slab || !in->dir) return c->err = "missing slab or directory", LGR_E_ARG;
  // the directory only: each block's header must agree with its entry and the block must lie inside the slab, so that
  // every read of k_fmt_unpack stays inside the device copy of the slab
  const uint8_t* slab = static_cast<const uint8_t*>(in->slab);
  int64_t S = 0, N = 0, n_wide = 0;
  for (int w = 0; w < W; ++w) {
    const lgr_fmt_dir& d = in->dir[w];
    if (d.sup_base != S || d.ev_base != N) return c->err = "sup_base / ev_base are not the prefix sums of the counts", LGR_E_ARG;
    if (d.n_supports < 0 || d.n_evidence < 0 || d.n_wide < 0 || d.n_wide > d.n_supports)
      return c->err = "negative or inconsistent counts in the directory", LGR_E_ARG;
    if (d.rec_off % 16 != 0 || d.rec_off > in->slab_bytes || in->slab_bytes - d.rec_off < sizeof(lgr_fmt_blk_hdr))
      return c->err = "rec_off outside the slab or not 16-byte aligned", LGR_E_ARG;
    lgr_fmt_blk_hdr h;
    std::memcpy(&h, slab + d.rec_off, sizeof(h));
    uint64_t off[LGR_FMT_SECTIONS];
    const uint64_t bytes = fmt_layout(d.n_supports, d.n_evidence, sizeof(lgr_fmt_blk_hdr), off);
    if (h.magic != LGR_FMT_MAGIC) return c->err = "bad block magic", LGR_E_ARG;
    if (h.n_supports != d.n_supports || h.n_evidence != d.n_evidence || h.rec_bytes != bytes)
      return c->err = "block header disagrees with its directory entry", LGR_E_ARG;
    if (in->slab_bytes - d.rec_off < bytes) return c->err = "block runs past the end of the slab", LGR_E_ARG;
    S += d.n_supports, N += d.n_evidence, n_wide += d.n_wide;
    if (S > INT32_MAX) return c->err = "more than 2^31 - 1 supports", LGR_E_ARG;
  }
  if (S == 0) return LGR_OK;
  if (!out) return c->err = "missing out", LGR_E_ARG;

  LGR_CUDA(c, cudaSetDevice(c->device));
  const size_t slab_bytes = (in->slab_bytes + 15) & ~(size_t)15;
  const char* dir_p = reinterpret_cast<const char*>(in->dir);
  const size_t dir_bytes = (size_t)W * sizeof(lgr_fmt_dir);
  const bool dir_inside = dir_p >= (const char*)slab && (size_t)(dir_p - (const char*)slab) <= in->slab_bytes &&
                          in->slab_bytes - (size_t)(dir_p - (const char*)slab) >= dir_bytes && (dir_p - (const char*)slab) % 16 == 0;
  UnpackDev U;
  const uint64_t arena_bytes = fmt_layout(S, N, 0, U.aoff);
  int rc;
  if ((rc = c->b_slab.ensure(slab_bytes + 16, false, c->err)) != LGR_OK) return rc;
  if (!dir_inside && (rc = c->b_dir.ensure(dir_bytes, false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_in.ensure(arena_bytes, false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_keep.ensure((size_t)N, false, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_out.ensure((size_t)S * sizeof(lgr_format), false, c->err)) != LGR_OK) return rc;
  uint8_t* dslab = static_cast<uint8_t*>(c->b_slab.p);
  int* status = reinterpret_cast<int*>(dslab + slab_bytes);
  LGR_CUDA(c, cudaMemcpyAsync(dslab, slab, in->slab_bytes, cudaMemcpyHostToDevice, c->stream));
  if (!dir_inside) LGR_CUDA(c, cudaMemcpyAsync(c->b_dir.p, in->dir, dir_bytes, cudaMemcpyHostToDevice, c->stream));
  LGR_CUDA(c, cudaMemsetAsync(status, 0, sizeof(int), c->stream));

  U.slab = dslab;
  U.dir = dir_inside ? reinterpret_cast<const lgr_fmt_dir*>(dslab + (dir_p - (const char*)slab)) : (const lgr_fmt_dir*)c->b_dir.p;
  U.n_windows = W, U.n_supports = (int32_t)S, U.n_evidence = N;
  U.n_rec_ctas = (N + kUnpackChunk - 1) / kUnpackChunk;
  U.arena = static_cast<uint8_t*>(c->b_in.p);
  U.status = status;
  uint8_t* base = U.arena;
  FmtDev D;
  D.e.insert_size = (const int64_t*)(base + U.aoff[1]), D.e.aln_start = (const int64_t*)(base + U.aoff[2]);
  D.e.aln_score = (const double*)(base + U.aoff[3]), D.e.folded_pos = (const double*)(base + U.aoff[4]);
  D.e.rname_hash = (const uint32_t*)(base + U.aoff[8]), D.e.ref_nm = (const uint32_t*)(base + U.aoff[9]);
  D.e.own_hap_nm = (const uint32_t*)(base + U.aoff[10]), D.e.hap_id = (const uint32_t*)(base + U.aoff[11]);
  D.e.allele = (const uint8_t*)(base + U.aoff[12]), D.e.flags = (const uint8_t*)(base + U.aoff[13]);
  D.e.base_qual = (const uint8_t*)(base + U.aoff[14]), D.e.map_qual = (const uint8_t*)(base + U.aoff[15]);
  D.e.keep = (const uint8_t*)c->b_keep.p;
  D.sup_begin = (const int64_t*)(base + U.aoff[kSecBegin]), D.sup_n_alleles = (const int32_t*)(base + U.aoff[kSecK]);
  D.sup_variant_len = (const int32_t*)(base + U.aoff[kSecVl]), D.sup_total_haps = (const int32_t*)(base + U.aoff[kSecTh]);
  D.keep = (uint8_t*)c->b_keep.p, D.out = (lgr_format*)c->b_out.p;
  D.n_supports = (int32_t)S, D.n_evidence = N;

  LGR_CUDA(c, cudaEventRecord(c->ev0, c->stream));
  {
    const int64_t blocks = U.n_rec_ctas + (S + kUnpackWarps - 1) / kUnpackWarps;
    k_fmt_unpack<<<(unsigned)blocks, kUnpackThreads, 0, c->stream>>>(U);
    LGR_CUDA(c, cudaGetLastError());
  }
  if (N > 0) {  // the grid rule of lgr_format_metrics
    k_fmt_dedup<<<(unsigned)((N + 255) / 256), 256, 0, c->stream>>>(D);
    LGR_CUDA(c, cudaGetLastError());
  }
  {
    const int64_t cap = (int64_t)c->sm_count * 32;
    const dim3 grid((unsigned)(S < cap ? S : cap), (unsigned)lgr_fmt::kNumTasks);
    k_fmt_metrics<<<grid, lgr_fmt::kThreads, 0, c->stream>>>(D);
    LGR_CUDA(c, cudaGetLastError());
  }
  LGR_CUDA(c, cudaEventRecord(c->ev1, c->stream));
  int bad = 0;
  LGR_CUDA(c, cudaMemcpyAsync(out, c->b_out.p, (size_t)S * sizeof(lgr_format), cudaMemcpyDeviceToHost, c->stream));
  LGR_CUDA(c, cudaMemcpyAsync(&bad, status, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  if (ms_kernels) LGR_CUDA(c, cudaEventElapsedTime(ms_kernels, c->ev0, c->ev1));
  if (bad) return c->err = "a packed block holds malformed records (sup_begin, K or an allele >= K)", LGR_E_ARG;
  if (n_wide == 0) return LGR_OK;
  // wide supports: the records lgr_format_metrics gives them, found through the windows that declare some
  int64_t seen = 0;
  for (int w = 0; w < W; ++w) {
    const lgr_fmt_dir& d = in->dir[w];
    if (d.n_wide == 0) continue;
    uint64_t off[LGR_FMT_SECTIONS];
    fmt_layout(d.n_supports, d.n_evidence, sizeof(lgr_fmt_blk_hdr), off);
    for (int s = 0; s < d.n_supports; ++s) {
      int32_t K;
      std::memcpy(&K, slab + d.rec_off + off[kSecK] + 4 * (size_t)s, 4);
      if (K > LGR_FMT_MAX_ALLELES) {
        lgr_format& r = out[d.sup_base + s];
        std::memset(&r, 0, sizeof(lgr_format));
        r.n_alleles = (uint32_t)K, r.valid = LGR_FMT_WIDE;
        ++seen;
      }
    }
  }
  if (seen != n_wide) return c->err = "n_wide of the directory disagrees with the blocks", LGR_E_ARG;
  c->err = "some supports have more than LGR_FMT_MAX_ALLELES alleles (records flagged LGR_FMT_WIDE)";
  return LGR_E_PARTIAL;
}

int lgr_format_reserve(lgr_fmt_ctx* c, int64_t slab_bytes, int32_t n_supports, int64_t n_evidence) {
  if (!c || slab_bytes < 0 || n_supports < 0 || n_evidence < 0) return LGR_E_ARG;
  c->err.clear();
  LGR_CUDA(c, cudaSetDevice(c->device));
  uint64_t off[LGR_FMT_SECTIONS];
  int rc;
  if ((rc = c->b_slab.ensure((((size_t)slab_bytes + 15) & ~(size_t)15) + 16, true, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_in.ensure(fmt_layout(n_supports, n_evidence, 0, off), true, c->err)) != LGR_OK) return rc;
  if ((rc = c->b_keep.ensure((size_t)n_evidence, true, c->err)) != LGR_OK) return rc;
  return c->b_out.ensure((size_t)n_supports * sizeof(lgr_format), true, c->err);
}

int64_t lgr_format_device_bytes(const lgr_fmt_ctx* c) {
  if (!c) return 0;
  return (int64_t)(c->b_in.cap + c->b_keep.cap + c->b_out.cap + c->b_ev.cap + c->b_key.cap + c->b_slab.cap + c->b_dir.cap);
}

}  // extern "C"
