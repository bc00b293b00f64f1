// lgr_repeat.cu — SURVEY.md §8f #3 (first half): repeat detection over the sliding k-mers of
// reference windows, batched.  C-ABI in include/lancet_gpu_realign.h (lgr_repeat_*).
//
// Replaces, per (window sequence, k, max_mismatches) job:
//   cbdg::Graph::HasExactOrApproxRepeat    graph.h:127-131  (HasRepeat(SlidingView(seq, k), 2), once per k of the k-loop)
//   VariantBuilder::ShouldSkipWindow       variant_builder.cpp:116-117 (HasExactRepeat(SlidingView(seq, max_k)))
//   base::HasRepeat / IsWithinHammingDist  base/repeat.cpp:55-217, 348-371
// Answer: do two k-mers at different offsets differ in at most max_mismatches BYTE positions?
//
// The reference compares every k-mer pair (O(n^2) pairs, SIMD compare with early exit).  Here the
// pairs are organised by diagonal: for an offset d, x_d[p] = (seq[p] != seq[p + d]) and the Hamming
// distance of the k-mers at i and i + d is the number of set bits of x_d in [i, i + k) — a sliding
// window sum.  One CTA takes one job and stages the sequence in shared memory; each of its warps
// takes diagonals d = warp, warp + 8, ...: one ballot per 32 positions turns x_d into bit masks with
// a running popcount, then every lane evaluates one window start with two prefix look-ups.  A
// diagonal costs 2 * n / 32 warp steps whatever k is.  The mask does not depend on k at all, so consecutive jobs over the
// same sequence with the same threshold (a window's whole k-loop) share one CTA: the mask of a diagonal is built once and
// every still-open k is answered from it.  A job is closed at its first hit; the CTA stops when all its jobs are closed.
// Byte compares on the raw ASCII, like the reference (case and IUPAC letters count as written).
// A batch of few windows would leave most SMs idle under one CTA per group, so the unit of work is a (group, diagonal
// slice) pair: the host splits each group into S slices (about resident CTAs / groups, at least one diagonal per warp)
// and slice s takes diagonals 1 + s * 8 + warp, stepping by S * 8.  The slices of a group share a found word in global
// memory for the early exit; the last slice to finish writes the answers.  Big batches get S = 1, the one-CTA schedule.
// -DLGR_REPEAT_ONE_SLICE forces S = 1 (A/B builds).
// There is no CPU fallback: lgr_repeat_create returns LGR_E_NO_DEVICE without a GPU.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/lancet_gpu_realign.h"
#include "lgr_host.h"

namespace {

constexpr int kRepThreads = 256;
constexpr int kRepWarps = kRepThreads / 32;
constexpr int kRepMaxLen = LGR_REPEAT_MAX_LEN;        // bases of one job's sequence (staged in shared memory)
constexpr int kRepWords = kRepMaxLen / 32 + 2;        // mask words of one diagonal

constexpr int kRepCtasPerSm = 8;  // CTAs launched per SM: 2,048 threads, all resident with k_repeat_scan<true>'s 32 registers

// one slice of a job group: consecutive jobs over the same sequence with the same max_mismatches share the mismatch masks
struct RepItem {
  int32_t first, n;       // the group's jobs
  int32_t gid;            // the group's found / done words (slices > 1 only)
  int16_t slice, slices;  // diagonals 1 + slice * kRepWarps + warp, stepping by slices * kRepWarps
};

struct RepDev {
  const uint8_t* seqs;
  const lgr_repeat_job* jobs;
  const RepItem* items;
  uint8_t* out;
  int* next_item;    // work counter (groups differ by 20x in cost: a static stride would pair the heavy ones up)
  unsigned* found;   // per sliced group, zeroed before the launch: bit j = job j has its repeat (OR over the slices)
  unsigned* done;    // per sliced group, zeroed before the launch: slices finished
  int n_items;
};

constexpr int kRepGroupJobs = 32;  // k values handled by one group (a window's k-loop has 20)

// One CTA per work item.  The mismatch mask of a diagonal depends on the sequence and the offset only, not on k, so
// the warp builds it once and then answers every still-open k of the group from it: (1 + K) * n / 32 warp steps per
// diagonal instead of 2 K * n / 32 (K = 20 for a window's k-loop: 1.9x fewer steps).  kSliced = false: every item is a
// whole group (S = 1), compiled without the slice arithmetic and the global flags.
template <bool kSliced>
__global__ void __launch_bounds__(kRepThreads) k_repeat_scan(const RepDev D) {
  __shared__ uint8_t s_seq[kRepMaxLen];
  __shared__ uint32_t s_mask[kRepWarps][kRepWords];
  __shared__ uint16_t s_pre[kRepWarps][kRepWords];
  __shared__ int s_k[kRepGroupJobs];
  __shared__ unsigned s_found;  // bit j: job j of the group has its repeat (this CTA's hits; a cache of *g_found when sliced)
  __shared__ bool s_last;
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ int s_item;
  for (;;) {
    __syncthreads();  // the previous item is finished with the shared arrays (and with s_item)
    if (threadIdx.x == 0) s_item = atomicAdd(D.next_item, 1);
    __syncthreads();
    const int item = s_item;
    if (item >= D.n_items) break;
    const RepItem G = D.items[item];
    const bool sliced = kSliced && G.slices > 1;
    unsigned* g_found = D.found + G.gid;  // dereferenced only when sliced
    const lgr_repeat_job j0 = D.jobs[G.first];
    const int len = j0.seq_len, mm = j0.max_mismatches;
    if (threadIdx.x == 0) s_found = 0;
    if (threadIdx.x < G.n) s_k[threadIdx.x] = D.jobs[G.first + threadIdx.x].k;
    if (len > kRepMaxLen) {  // not computed: flagged for the host (such a group has one slice)
      if (threadIdx.x < G.n) D.out[G.first + threadIdx.x] = LGR_REPEAT_TOO_LONG;
      continue;
    }
    const uint8_t* seq = D.seqs + j0.seq_off;
    for (int p = threadIdx.x; p < len; p += kRepThreads) s_seq[p] = seq[p];
    __syncthreads();
    int k_min = s_k[0];
    for (int q = 1; q < G.n; ++q) k_min = s_k[q] < k_min ? s_k[q] : k_min;
    const unsigned all = G.n == 32 ? full : (1u << G.n) - 1u;
    const int d_end = len - k_min + 1;  // diagonals of the smallest k (base::SlidingView: none when the sequence is shorter than k)
    uint32_t* mask = s_mask[warp];
    uint16_t* pre = s_pre[warp];
    const int step = kSliced ? G.slices * kRepWarps : kRepWarps;
    for (int d = 1 + (kSliced ? G.slice * kRepWarps : 0) + warp; d < d_end; d += step) {
      // which jobs are still open: one lane reads the flags (atomics on both sides, no data race) and the whole
      // warp follows its answer, so the lanes can never disagree about leaving the loop
      unsigned found = 0;
      if (lane == 0) {
        found = atomicOr(&s_found, 0u);
        if (sliced) found |= atomicOr(g_found, 0u);  // the other slices' hits
      }
      found = __shfl_sync(full, found, 0);
      if (found == all) break;
      const int span = len - d;  // positions p with a partner p + d
      const int words = (span + 31) >> 5;
      int run = 0;
      for (int c = 0; c < words; ++c) {
        const int p = (c << 5) + lane;
        const unsigned m = __ballot_sync(full, p < span && s_seq[p] != s_seq[p + d]);
        if (lane == 0) mask[c] = m, pre[c] = (uint16_t)run;
        run += __popc(m);
      }
      if (lane == 0) mask[words] = 0, pre[words] = (uint16_t)run;  // P(span) when span is a multiple of 32
      __syncwarp();
      unsigned newly = 0;
      for (int q = 0; q < G.n; ++q) {
        if (found >> q & 1u) continue;
        const int k = s_k[q];
        const int starts = len - k + 1 - d;  // k-mer pairs (i, i + d) of this k on the diagonal
        if (starts <= 0) continue;
        bool hit = false;
        for (int base = 0; base < starts; base += 32) {
          const int i = base + lane;
          if (i < starts) {
            const int e = i + k;
            const int pb = pre[i >> 5] + __popc(mask[i >> 5] & ((1u << (i & 31)) - 1u));
            const int pe = pre[e >> 5] + __popc(mask[e >> 5] & ((1u << (e & 31)) - 1u));
            hit |= pe - pb <= mm;
          }
        }
        if (__any_sync(full, hit)) newly |= 1u << q;
      }
      if (newly && lane == 0) {
        atomicOr(&s_found, newly);
        if (sliced) atomicOr(g_found, newly);
      }
      __syncwarp();
    }
    __syncthreads();
    if (!sliced) {
      if (threadIdx.x < G.n) D.out[G.first + threadIdx.x] = (uint8_t)(s_found >> threadIdx.x & 1u);
      continue;
    }
    // the last slice to finish writes the answers: the OR of the per-diagonal hits over a partition of the diagonals
    if (threadIdx.x == 0) {
      __threadfence();  // this slice's atomicOr on *g_found is ordered before its count
      s_last = atomicAdd(D.done + G.gid, 1) == G.slices - 1;
    }
    __syncthreads();
    if (s_last) {
      __threadfence();
      if (threadIdx.x < G.n) D.out[G.first + threadIdx.x] = (uint8_t)(atomicOr(g_found, 0u) >> threadIdx.x & 1u);
    }
  }
}

}  // namespace

struct lgr_rep_ctx {
  int device = 0, sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  DeviceBuffer d_seq, d_jobs, d_out, d_items, d_ctr;
  struct Group {
    int32_t first, n, k_min;
  };
  std::vector<Group> groups;  // host scratch of lgr_repeat_scan, kept to reuse its storage
  std::vector<RepItem> items;
  std::string err;
};

static thread_local std::string g_rep_create_err;

// device buffers of a batch of n_jobs jobs over seq_bytes bytes: the work items are at most max(n_jobs, resident CTAs)
// (a group gets several slices only while there are fewer groups than resident CTAs), the counter words 1 + 2 per group.
// Half as much again on a regrow inside lgr_repeat_scan, exactly on a reservation.
static int rep_buffers(lgr_rep_ctx* c, size_t seq_bytes, size_t n_jobs, size_t n_items, size_t ctr_words, bool exact) {
  int rc;
  if ((rc = c->d_seq.ensure(seq_bytes, exact, c->err)) != LGR_OK) return rc;
  if ((rc = c->d_jobs.ensure(sizeof(lgr_repeat_job) * n_jobs, exact, c->err)) != LGR_OK) return rc;
  if ((rc = c->d_out.ensure(n_jobs, exact, c->err)) != LGR_OK) return rc;
  if ((rc = c->d_items.ensure(sizeof(RepItem) * n_items, exact, c->err)) != LGR_OK) return rc;
  return c->d_ctr.ensure(sizeof(unsigned) * ctr_words, exact, c->err);
}

extern "C" {

int lgr_repeat_create(int device_ordinal, lgr_rep_ctx** out) {
  if (!out) return LGR_E_ARG;
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0 || device_ordinal < 0 || device_ordinal >= n_dev) {
    g_rep_create_err = "no usable CUDA device (this path has no CPU fallback)";
    (void)cudaGetLastError();
    return LGR_E_NO_DEVICE;
  }
  lgr_rep_ctx* c = new lgr_rep_ctx();
  c->device = device_ordinal;
  cudaDeviceProp prop;
  if (cudaSetDevice(device_ordinal) != cudaSuccess || cudaGetDeviceProperties(&prop, device_ordinal) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_rep_create_err = "cudaSetDevice / cudaStreamCreate failed";
    lgr_repeat_destroy(c);
    return LGR_E_CUDA;
  }
  c->sm_count = prop.multiProcessorCount;
  cudaEventCreate(&c->ev0), cudaEventCreate(&c->ev1);
  *out = c;
  return LGR_OK;
}

void lgr_repeat_destroy(lgr_rep_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;  // frees the device buffers
}

const char* lgr_repeat_last_error(const lgr_rep_ctx* c) { return c ? c->err.c_str() : g_rep_create_err.c_str(); }

int lgr_repeat_scan(lgr_rep_ctx* c, const uint8_t* seqs, int64_t seq_bytes, const lgr_repeat_job* jobs, int32_t n_jobs,
                    uint8_t* has_repeat, float* ms_kernels) {
  if (!c || n_jobs < 0 || seq_bytes < 0 || (n_jobs > 0 && (!jobs || !has_repeat)) || (seq_bytes > 0 && !seqs)) return LGR_E_ARG;
  c->err.clear();
  if (ms_kernels) *ms_kernels = 0.0f;
  if (n_jobs == 0) return LGR_OK;
  bool too_long = false;
  for (int i = 0; i < n_jobs; ++i) {
    const lgr_repeat_job& j = jobs[i];
    if (j.seq_len < 0 || j.seq_off < 0 || j.seq_off + j.seq_len > seq_bytes || j.k <= 0 || j.max_mismatches < 0)
      return c->err = "bad repeat job (offsets outside the sequence buffer, k <= 0 or max_mismatches < 0)", LGR_E_ARG;
    too_long |= j.seq_len > LGR_REPEAT_MAX_LEN;
  }
  // consecutive jobs over the same sequence with the same threshold form a group (sharing its mismatch masks)
  std::vector<lgr_rep_ctx::Group>& groups = c->groups;
  groups.clear();
  for (int i = 0; i < n_jobs;) {
    int n = 1, k_min = jobs[i].k;
    while (i + n < n_jobs && n < kRepGroupJobs && jobs[i + n].seq_off == jobs[i].seq_off && jobs[i + n].seq_len == jobs[i].seq_len &&
           jobs[i + n].max_mismatches == jobs[i].max_mismatches)
      k_min = std::min(k_min, jobs[i + n].k), ++n;
    groups.push_back(lgr_rep_ctx::Group{i, n, k_min});
    i += n;
  }
  // the queue hands out the expensive groups first (cost ~ jobs x length^2): a short tail
  std::stable_sort(groups.begin(), groups.end(), [&](const lgr_rep_ctx::Group& a, const lgr_rep_ctx::Group& b) {
    const int64_t la = jobs[a.first].seq_len, lb = jobs[b.first].seq_len;
    return (int64_t)(a.n + 1) * la * la > (int64_t)(b.n + 1) * lb * lb;
  });
  // slices per group: enough work items to fill the resident CTAs, at least one diagonal per warp of a slice
  const int n_groups = (int)groups.size(), resident = c->sm_count * kRepCtasPerSm;
#ifdef LGR_REPEAT_ONE_SLICE
  const int per_group = 1;
#else
  const int per_group = std::min(std::max(resident / n_groups, 1), (int)INT16_MAX);
#endif
  std::vector<RepItem>& items = c->items;
  items.clear();
  int n_sliced = 0;
  for (const lgr_rep_ctx::Group& g : groups) {
    const int len = jobs[g.first].seq_len, diagonals = len - g.k_min;  // d = 1 .. len - k_min
    const int slices = len > kRepMaxLen ? 1 : std::max(1, std::min(per_group, diagonals / kRepWarps));
    const int gid = slices > 1 ? n_sliced++ : 0;
    for (int s = 0; s < slices; ++s) items.push_back(RepItem{g.first, g.n, gid, (int16_t)s, (int16_t)slices});
  }
  const int n_items = (int)items.size();
  const size_t ctr_words = 1 + 2 * (size_t)n_sliced;  // queue counter, then found[n_sliced], done[n_sliced]
  LGR_CUDA(c, cudaSetDevice(c->device));
  int rc;
  if ((rc = rep_buffers(c, (size_t)seq_bytes, (size_t)n_jobs, (size_t)n_items, ctr_words, false)) != LGR_OK) return rc;
  LGR_CUDA(c, cudaMemsetAsync(c->d_ctr.p, 0, sizeof(unsigned) * ctr_words, c->stream));
  if (seq_bytes > 0) LGR_CUDA(c, cudaMemcpyAsync(c->d_seq.p, seqs, (size_t)seq_bytes, cudaMemcpyHostToDevice, c->stream));
  LGR_CUDA(c, cudaMemcpyAsync(c->d_jobs.p, jobs, sizeof(lgr_repeat_job) * (size_t)n_jobs, cudaMemcpyHostToDevice, c->stream));
  LGR_CUDA(c, cudaMemcpyAsync(c->d_items.p, items.data(), sizeof(RepItem) * items.size(), cudaMemcpyHostToDevice, c->stream));
  unsigned* ctr = (unsigned*)c->d_ctr.p;
  RepDev D{(const uint8_t*)c->d_seq.p, (const lgr_repeat_job*)c->d_jobs.p, (const RepItem*)c->d_items.p, (uint8_t*)c->d_out.p,
           (int*)ctr, ctr + 1, ctr + 1 + n_sliced, n_items};
  LGR_CUDA(c, cudaEventRecord(c->ev0, c->stream));
  const int grid = n_items < resident ? n_items : resident;
  if (n_sliced > 0)
    k_repeat_scan<true><<<grid, kRepThreads, 0, c->stream>>>(D);
  else
    k_repeat_scan<false><<<grid, kRepThreads, 0, c->stream>>>(D);
  LGR_CUDA(c, cudaGetLastError());
  LGR_CUDA(c, cudaEventRecord(c->ev1, c->stream));
  LGR_CUDA(c, cudaMemcpyAsync(has_repeat, c->d_out.p, (size_t)n_jobs, cudaMemcpyDeviceToHost, c->stream));
  LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  if (ms_kernels) LGR_CUDA(c, cudaEventElapsedTime(ms_kernels, c->ev0, c->ev1));
  if (too_long) {
    c->err = "some sequences are longer than LGR_REPEAT_MAX_LEN (their answers are LGR_REPEAT_TOO_LONG)";
    return LGR_E_PARTIAL;
  }
  return LGR_OK;
}

int lgr_repeat_reserve(lgr_rep_ctx* c, int64_t seq_bytes, int32_t n_jobs) {
  if (!c || seq_bytes < 0 || n_jobs < 0) return LGR_E_ARG;
  c->err.clear();
  LGR_CUDA(c, cudaSetDevice(c->device));
  const size_t resident = (size_t)c->sm_count * kRepCtasPerSm;
  const int rc = rep_buffers(c, (size_t)seq_bytes, (size_t)n_jobs, std::max((size_t)n_jobs, resident), 1 + 2 * (size_t)n_jobs, true);
  c->groups.reserve((size_t)n_jobs);
  c->items.reserve(std::max((size_t)n_jobs, resident));
  return rc;
}

}  // extern "C"
