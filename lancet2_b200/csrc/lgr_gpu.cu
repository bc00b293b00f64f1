// lgr_gpu.cu — the C-ABI (include/lancet_gpu_realign.h) and host side of the B200 read→haplotype
// realignment path; the sm_100a kernels live in the headers included below (one translation unit).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
//
// Pipeline per batch (12 launches, two streams, no host sync inside; DESIGN.md has layout and rooflines):
//   lgr_kernels_index.cuh
//     k_encode            ASCII → code bytes (nt4 | Lancet code) for haplotypes and reads
//     k_hap_sketch_warp   one warp per haplotype, one lane per position: minimizer sketch → unsorted table
//     k_hap_sort          one CTA per haplotype: bitonic sort of the table (the "index"), hash-bucket
//                         directory, mid_occ the haplotype would latch
//     k_group_mid         effective mid_occ per group
//     k_read_sketch       one lane per read: sketch (second stream); k_read_filter: mm_seed_mz_flt
//   lgr_kernels_chain.cuh
//     k_chain_lean        ONE WARP PER (read, haplotype) PAIR: seeds → anchors → co-linear chain in
//                         closed form → reg; closed-form extensions; regs parked in HBM (RegRec), the
//                         other extensions queued (TaskRec); every other shape queued for k_chain_cold
//     k_chain_cold        the same, one warp per queued pair, with sort, chain DP, backtrack, several
//                         regs and SR stretch
//     k_chain_overflow    the same for pairs whose anchors exceed the shared-memory cap (lane per pair)
//   lgr_kernels_ext.cuh
//     k_ext_warp          one warp per queued extension: anti-diagonal wavefront DP with shuffle
//                         neighbour exchange, exact data-dependent column bound, warp traceback
//   lgr_kernels_finish.cuh
//     k_finish_warp       one warp per parked pair: cigar assembly, mm_fix_cigar, mm_update_extra,
//                         filter/sort, NM → lgr_aln
//     k_assign            one lane per (read, variant): local scoring + best-allele selection
//   lgr_dev.cuh           device descriptor, counters, records, launch-shape knobs
//   lgr_core.cuh          __host__ __device__ per-lane core shared with tests/hostemu
// Graph mode (lgr_set_graph_mode) captures the same launch list (enqueue_pass) as a CUDA graph and replays it.
// There is no host fallback: every entry point fails with an error code when CUDA fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/lancet_gpu_realign.h"
#include "lgr_core.cuh"
#include "lgr_host.h"

#include "lgr_pack.h"

#include "lgr_dev.cuh"
#include "lgr_kernels_unpack.cuh"
#include "lgr_kernels_index.cuh"
#include "lgr_kernels_ext.cuh"
#include "lgr_kernels_finish.cuh"
#include "lgr_kernels_chain.cuh"

namespace {

// =========================================================================================
// host side
// =========================================================================================
// graph mode (lgr_set_graph_mode): one executable per topology of the captured pass, least recently used evicted
constexpr int kGraphCache = 8;
struct GraphSlot {
  cudaGraphExec_t exec = nullptr;
  uint32_t key = 0;
  uint64_t used = 0;
};

// timing events of a pass (stage times of lgr_stats) and of the copies around it (ms_h2d / ms_d2h)
enum Ev {
  EV_PASS_BEGIN, EV_INDEXED, EV_FILTERED, EV_CHAINED, EV_EXTENDED, EV_PASS_END,
  EV_H2D_BEGIN, EV_H2D_END, EV_D2H_BEGIN, EV_D2H_END,
  EV_COUNT
};

}  // namespace

struct lgr_ctx {
  int device = 0;
  cudaStream_t stream = nullptr, stream2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  lgr_params prm;
  DevParams P;
  std::string err;
  int sm_count = 0;
  // ONE grow-only device arena per context; every per-batch array of D is a view into it, laid out afresh by
  // plan_batch.  A batch larger than any before costs one cudaFree + one cudaMalloc (cudaFree synchronises the
  // whole device; sixty separately growing buffers made that sixty stalls per regrow and dominated the batcher's
  // submit time in the first round-2 measurement).
  DeviceBuffer arena;
  DeviceBuffer ws_big;  // the overflow pass's chain workspace, sized to measure
  Dev D;
  bool resident = false, packed = false;
  int occ_cap = 0, warp_blocks_full = 0, ext_blocks_full = 0, fin_blocks_full = 0, overflow_passes = 0;
  int max_read_len = 0, max_hap_len = 0;
  int64_t hap_bytes = 0, read_bytes = 0;
  int ext_blocks = 0, fin_blocks = 0, warp_blocks = 0, cold_blocks = 0, cold_blocks_full = 0, warp_cap = 64;
  size_t warp_smem = 0, cold_smem = 0;
  cudaEvent_t ev[EV_COUNT] = {};
  long long* h_ctr = nullptr;  // pinned copy of the device counters
  int launches = 0;
  // graph mode of the blocking calls: the pass is captured and replayed as a CUDA graph (run_launch_graph)
  bool graph_mode = false, capturing = false;
  GraphSlot graphs[kGraphCache];
  uint64_t graph_tick = 0;
  int64_t graph_instantiated = 0, graph_updated = 0, graph_replayed = 0;
  // asynchronous submissions (lgr_submit/lgr_wait): child contexts, one per slot in flight
  lgr_ctx* slot[LGR_MAX_INFLIGHT] = {};
  bool slot_busy[LGR_MAX_INFLIGHT] = {};
  lgr_batch_out* slot_out[LGR_MAX_INFLIGHT] = {};
  int64_t slot_h2d[LGR_MAX_INFLIGHT] = {}, slot_d2h[LGR_MAX_INFLIGHT] = {};
  lgr_notify_fn notify_fn = nullptr;
  void* notify_user = nullptr;
  struct Note { lgr_ctx* ctx; int ticket; } slot_note[LGR_MAX_INFLIGHT] = {};
  // host staging of helper arrays
  std::vector<int32_t> h_read_grp, h_hap_grp, h_item_hap, h_item_r0, h_item_n, h_grp_mid;
  std::vector<int64_t> h_pair_off, h_asg_off;
};

static thread_local std::string g_create_err;

// the chain kernels of one anchor cap: their launch attributes, and how many blocks of each an SM holds
template <int CAP>
static bool chain_occupancy(const lgr_ctx* c, int* per_sm, int* per_sm_cold) {
  const cudaError_t e1 = cudaFuncSetAttribute(k_chain_lean<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->warp_smem);
  cudaFuncSetAttribute(k_chain_lean<CAP>, cudaFuncAttributePreferredSharedMemoryCarveout, LGR_CHAIN_CARVEOUT);
  const cudaError_t e2 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, k_chain_lean<CAP>, kWarpsPerCta * 32, c->warp_smem);
  const cudaError_t e3 = cudaFuncSetAttribute(k_chain_cold<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->cold_smem);
  const cudaError_t e4 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm_cold, k_chain_cold<CAP>, kWarpsPerCta * 32, c->cold_smem);
  return e1 == cudaSuccess && e2 == cudaSuccess && e3 == cudaSuccess && e4 == cudaSuccess;
}

template <int CAP>
static void launch_chain(const lgr_ctx* c, const Dev& D, cudaStream_t s) {
  k_chain_lean<CAP><<<c->warp_blocks, kWarpsPerCta * 32, c->warp_smem, s>>>(D);
  k_chain_cold<CAP><<<c->cold_blocks, kWarpsPerCta * 32, c->cold_smem, s>>>(D);
}

// one host→device copy into the arena view dst (a const input field of D): `count` elements, as layout_arena
// sized the view; adds the bytes to h2d
template <class T>
static cudaError_t copy_in(lgr_ctx* c, const T* dst, const void* src, size_t count, int64_t& h2d) {
  const size_t bytes = count * sizeof(T);
  h2d += bytes;
  return bytes ? cudaMemcpyAsync(const_cast<T*>(dst), src, bytes, cudaMemcpyHostToDevice, c->stream) : cudaSuccess;
}

extern "C" {

int lgr_abi_version(void) { return LGR_ABI_VERSION; }

void lgr_default_params(lgr_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->k = 11, p->w = 5;
  p->a = 1, p->b = 4, p->q = 12, p->e = 3, p->sc_ambi = 1;
  p->bw = 10000, p->zdrop = 100000, p->end_bonus = 10000;
  p->max_gap = 200, p->max_gap_ref = 5000;
  p->max_chain_skip = 25, p->max_chain_iter = 5000, p->min_cnt = 3, p->min_chain_score = 40;
  p->min_dp_max = 80;
  p->mid_occ = 0, p->min_mid_occ = 10, p->max_mid_occ = 1000000, p->max_max_occ = 4095;
  p->occ_dist = 500, p->best_n = 1, p->seed = 11;
  p->mid_occ_frac = 2e-4f, p->q_occ_frac = 0.01f, p->chain_gap_scale = 0.8f, p->chain_skip_scale = 0.0f;
  p->mask_level = 0.5f, p->pri_ratio = 0.8f, p->max_clip_ratio = 1.0f;
  p->mask_len = INT_MAX;
  p->cigar_arena_ops = 1 << 20;
}

const char* lgr_strerror(int code) {
  if (code == LGR_E_BUSY) return "all submission slots in flight";
  switch (code) {
    case LGR_OK: return "ok";
    case LGR_E_ARG: return "bad argument or inconsistent batch";
    case LGR_E_CUDA: return "CUDA runtime failure";
    case LGR_E_NO_DEVICE: return "no usable CUDA device (this path has no CPU fallback)";
    case LGR_E_LIMIT: return "a sequence or intermediate exceeds a device-path cap";
    case LGR_E_CIGAR_OVERFLOW: return "cigar overflow arena exhausted";
    case LGR_E_NOMEM: return "out of device memory";
    case LGR_E_PARTIAL: return "some groups hit a device-path cap (see grp_status); the others are complete";
    default: return "unknown error";
  }
}

const char* lgr_last_error(const lgr_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

uint32_t lgr_x31_hash(const char* s) {
  uint32_t h = (uint32_t)(int32_t)(signed char)*s;
  if (h)
    for (++s; *s; ++s) h = (h << 5) - h + (uint32_t)(int32_t)(signed char)*s;
  return h;
}

int lgr_pair_offsets(const lgr_batch_in* in, int64_t* pair_off, int64_t* asg_off) {
  if (!in || !pair_off || !asg_off) return LGR_E_ARG;
  int64_t po = 0, ao = 0;
  for (int g = 0; g < in->n_groups; ++g) {
    const int P = in->grp_hap_begin[g + 1] - in->grp_hap_begin[g];
    const int V = in->grp_var_begin[g + 1] - in->grp_var_begin[g];
    for (int r = in->grp_read_begin[g]; r < in->grp_read_begin[g + 1]; ++r) {
      pair_off[r] = po, asg_off[r] = ao;
      po += P, ao += V;
    }
  }
  pair_off[in->n_reads] = po, asg_off[in->n_reads] = ao;
  return LGR_OK;
}

static int validate_params(const lgr_params* p, std::string& err) {
  auto bad = [&](const char* m) { err = m; return LGR_E_ARG; };
  if (p->k < 1 || 2 * p->k + kIdxShift > 64) return bad("k must satisfy 2k+17 <= 64 (k <= 23)");
  if (p->w < 1 || p->w > kMaxWindow) return bad("w must be in [1,32]");
  if (p->a < 0 || p->b < 0 || p->q < 0 || p->e < 1 || p->sc_ambi < 0) return bad("scores must be non-negative, e >= 1");
  if (p->b > 2 * (p->q + p->e)) return bad("mismatch penalty exceeds 2(q+e): ksw2 returns early, unsupported");
  // regime of the reference: the extension always reaches the query end and never z-drops
  if (p->end_bonus < (p->a + std::max(p->b, p->sc_ambi)) * LGR_MAX_READ_LEN + p->q + p->e * LGR_MAX_READ_LEN)
    return bad("end_bonus too small: device path requires reach_end for every extension (reference uses 10000)");
  if (p->zdrop < 16 * LGR_MAX_READ_LEN) return bad("zdrop too small: device path requires that z-drop never fires (reference uses 100000)");
  if (p->occ_dist != 0 && p->occ_dist < 256) return bad("occ_dist must be 0 or >= 256");
  if (p->min_cnt < 1 || p->best_n < 0) return bad("min_cnt >= 1, best_n >= 0");
  return LGR_OK;
}

int lgr_create(int device_ordinal, const lgr_params* params, lgr_ctx** out) {
  if (!out) return LGR_E_ARG;
  *out = nullptr;
  lgr_params p;
  if (params) p = *params;
  else lgr_default_params(&p);
  int rc = validate_params(&p, g_create_err);
  if (rc != LGR_OK) return rc;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0 || device_ordinal < 0 || device_ordinal >= n_dev) {
    g_create_err = "no usable CUDA device";
    (void)cudaGetLastError();
    return LGR_E_NO_DEVICE;
  }
  lgr_ctx* c = new lgr_ctx();
  c->device = device_ordinal;
  c->prm = p;
  if (cudaSetDevice(device_ordinal) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_create_err = "cudaSetDevice/cudaStreamCreate failed";
    lgr_destroy(c);
    return LGR_E_CUDA;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device_ordinal);
  c->sm_count = prop.multiProcessorCount;
  for (auto& e : c->ev) cudaEventCreate(&e);
  if (cudaMallocHost((void**)&c->h_ctr, sizeof(long long) * (C_COUNT + 8)) != cudaSuccess) {
    g_create_err = "cudaMallocHost failed";
    lgr_destroy(c);
    return LGR_E_CUDA;
  }
  cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
  DevParams& d = c->P;
  std::memset(&d, 0, sizeof(d));
  d.k = p.k, d.w = p.w, d.a = p.a, d.b = p.b, d.q = p.q, d.e = p.e, d.sc_ambi = p.sc_ambi, d.bw = p.bw;
  d.end_bonus = p.end_bonus, d.max_gap = p.max_gap, d.max_gap_ref = p.max_gap_ref, d.max_skip = p.max_chain_skip;
  d.max_iter = p.max_chain_iter, d.min_cnt = p.min_cnt, d.min_sc = p.min_chain_score, d.min_dp_max = p.min_dp_max;
  d.max_max_occ = p.max_max_occ, d.occ_dist = p.occ_dist, d.best_n = p.best_n, d.seed = p.seed, d.mask_len = p.mask_len;
  d.pen_gap = (float)(p.chain_gap_scale * 0.01 * p.k);
  d.pen_skip = (float)(p.chain_skip_scale * 0.01 * p.k);
  d.mask_level = p.mask_level, d.pri_ratio = p.pri_ratio, d.max_clip_ratio = p.max_clip_ratio, d.q_occ_frac = p.q_occ_frac;
  d.min_strand_sc = (int32_t)(p.max_gap * 0.8);
  *out = c;
  return LGR_OK;
}

void lgr_destroy(lgr_ctx* c) {
  if (!c) return;
  for (lgr_ctx*& ch : c->slot) {
    lgr_destroy(ch);
    ch = nullptr;
  }
  cudaSetDevice(c->device);
  for (GraphSlot& g : c->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  if (c->h_ctr) cudaFreeHost(c->h_ctr);
  for (cudaEvent_t e : c->ev)
    if (e) cudaEventDestroy(e);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->stream2) cudaStreamDestroy(c->stream2);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;  // frees the device buffers
}

#ifdef LGR_EXT_HIST
int lgr_debug_ext_hist(unsigned long long* out256, int reset) {
  if (cudaMemcpyFromSymbol(out256, g_ext_hist, sizeof(unsigned long long) * 256) != cudaSuccess) return LGR_E_CUDA;
  if (reset) {
    static const unsigned long long zero[256] = {};
    cudaMemcpyToSymbol(g_ext_hist, zero, sizeof(zero));
  }
  return LGR_OK;
}
#endif

void* lgr_alloc_pinned(size_t bytes) {
  void* p = nullptr;
  // portable: usable from every device of the process (one batcher per GPU shares this allocator)
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    (void)cudaGetLastError();
    return nullptr;
  }
  return p;
}

void lgr_free_pinned(void* p) {
  if (p) cudaFreeHost(p);
}

void* lgr_stream(lgr_ctx* c) { return c ? (void*)c->stream : nullptr; }

static constexpr int kBigLanesMax = 4 * 19 * 32;  // lanes of the overflow pass (one pair each)
static constexpr int kBigCapMax = 65535;          // anchors per pair the chain workspace can index (16-bit positions)

// everything the buffer plan needs to know about a batch (from lgr_batch_in or from the packed directory)
struct BatchSizes {
  bool ascii = true;                       // plain form (ASCII strings) or packed slab
  size_t slab_bytes = 0, dir_entries = 0;  // packed form: bytes of the slab / directory entries outside the slab
  int G = 0, NH = 0, NR = 0, NV = 0;
  int64_t hap_bytes = 0, read_bytes = 0, nvh = 0, n_pairs = 0, n_assign = 0, n_items = 0;
  int item_reads = 1, max_read_len = 0, max_hap_len = 0;
};

// reads per warp work item: several reads of one haplotype amortise the item's fixed cost when the
// batch fills the machine many times over; a small batch (one Genotype() call) is latency bound
// instead and wants every pair on its own warp
static int choose_item_reads(const lgr_ctx* c, int64_t pairs_total) {
  // a work item is taken by a CTA (4 warps) that stages the haplotype's table once for all its reads
  const int64_t warps_resident = (int64_t)c->sm_count * 36;
  return pairs_total >= 8 * warps_resident ? kCtaItemReads : (pairs_total >= 3 * warps_resident ? 8 : kWarpsPerCta);
}

// static caps of the device path for one payload shape; NULL when inside them
static const char* limit_message(const lgr_params& prm, int max_hap_len, int max_read_len) {
  if (max_hap_len > LGR_MAX_HAP_LEN) return "haplotype longer than LGR_MAX_HAP_LEN";
  if (max_read_len > LGR_MAX_READ_LEN) return "read longer than LGR_MAX_READ_LEN";
  {  // the warp wavefront exchanges H/F as packed int16: bound |H| for the longest read
    const int Lm = max_read_len, mm = std::max(prm.b, prm.sc_ambi);
    const int64_t Tm = Lm + ((int64_t)(prm.a + mm) * Lm) / prm.e + 2;
    if (prm.q + (int64_t)prm.e * (Tm + Lm) + (int64_t)(mm + prm.a) * Lm > 32000)
      return "scores could leave the int16 range of the extension kernel for this read length / scoring";
  }
  // ksw2 band (w = 1.5*bw + 1) must never bind
  if ((int64_t)max_hap_len + max_read_len >= (int64_t)(prm.bw * 1.5))
    return "haplotype+read length reaches the ksw2 band; unsupported by the device path";
  return nullptr;
}

static int check_limits(lgr_ctx* c, const BatchSizes& z) {
  if (const char* m = limit_message(c->prm, z.max_hap_len, z.max_read_len)) { c->err = m; return LGR_E_LIMIT; }
  if (z.n_pairs > (int64_t)1 << 30) { c->err = "more than 2^30 (read, haplotype) pairs in one batch"; return LGR_E_LIMIT; }
  return LGR_OK;
}

static int validate_batch(lgr_ctx* c, const lgr_batch_in* in, BatchSizes* z) {
  auto bad = [&](const std::string& m, int code = LGR_E_ARG) { c->err = m; return code; };
  if (!in || in->n_groups < 0 || in->n_haps < 0 || in->n_reads < 0 || in->n_vars < 0) return bad("null or negative counts");
  if (in->n_groups > 0 && (!in->grp_hap_begin || !in->grp_read_begin || !in->grp_var_begin)) return bad("null group arrays");
  z->G = in->n_groups, z->NH = in->n_haps, z->NR = in->n_reads, z->NV = in->n_vars;
  if (in->n_groups == 0) return LGR_OK;
  if (in->grp_hap_begin[0] != 0 || in->grp_read_begin[0] != 0 || in->grp_var_begin[0] != 0) return bad("group prefix arrays must start at 0");
  if (in->grp_hap_begin[in->n_groups] != in->n_haps || in->grp_read_begin[in->n_groups] != in->n_reads ||
      in->grp_var_begin[in->n_groups] != in->n_vars)
    return bad("group prefix arrays do not end at the totals");
  if ((in->n_haps > 0 && (!in->hap_off || in->hap_off[0] != 0)) || (in->n_reads > 0 && (!in->read_off || in->read_off[0] != 0)) ||
      (in->n_vars > 0 && (!in->var_hap_off || in->var_hap_off[0] != 0)))
    return bad("hap_off / read_off / var_hap_off must start at 0");
  for (int g = 0; g < in->n_groups; ++g) {
    if (in->grp_hap_begin[g + 1] < in->grp_hap_begin[g] || in->grp_read_begin[g + 1] < in->grp_read_begin[g] ||
        in->grp_var_begin[g + 1] < in->grp_var_begin[g])
      return bad("group prefix arrays must be non-decreasing");
    const int P = in->grp_hap_begin[g + 1] - in->grp_hap_begin[g];
    const int R = in->grp_read_begin[g + 1] - in->grp_read_begin[g];
    if (R > 0 && P == 0) return bad("a group with reads needs at least the REF haplotype");
    // k_assign reads var_*[var_hap_off[v] + h] for h < P: every variant owns exactly P entries
    for (int v = in->grp_var_begin[g]; v < in->grp_var_begin[g + 1]; ++v)
      if (in->var_hap_off[v + 1] - in->var_hap_off[v] != P) return bad("every variant needs one bounds entry per haplotype of its group");
    z->n_pairs += (int64_t)R * P;
    z->n_assign += (int64_t)R * (in->grp_var_begin[g + 1] - in->grp_var_begin[g]);
  }
  for (int h = 0; h < in->n_haps; ++h) {
    const int64_t l = in->hap_off[h + 1] - in->hap_off[h];
    if (l < 0) return bad("hap_off must be non-decreasing");
    if (l > LGR_MAX_HAP_LEN) return bad("haplotype longer than LGR_MAX_HAP_LEN", LGR_E_LIMIT);
    z->max_hap_len = std::max<int>(z->max_hap_len, (int)l);
  }
  for (int r = 0; r < in->n_reads; ++r) {
    const int64_t l = in->read_off[r + 1] - in->read_off[r];
    if (l < 0) return bad("read_off must be non-decreasing");
    if (l > LGR_MAX_READ_LEN) return bad("read longer than LGR_MAX_READ_LEN", LGR_E_LIMIT);
    z->max_read_len = std::max<int>(z->max_read_len, (int)l);
  }
  z->hap_bytes = in->n_haps ? in->hap_off[in->n_haps] : 0;
  z->read_bytes = in->n_reads ? in->read_off[in->n_reads] : 0;
  z->nvh = in->n_vars ? in->var_hap_off[in->n_vars] : 0;
  for (int64_t x = 0; x < z->nvh; ++x)
    if (in->var_allele[x] < -1) return bad("var_allele must be -1 (absent) or an allele index");
  z->item_reads = choose_item_reads(c, z->n_pairs);
  for (int g = 0; g < in->n_groups; ++g) {
    const int64_t P = in->grp_hap_begin[g + 1] - in->grp_hap_begin[g], R = in->grp_read_begin[g + 1] - in->grp_read_begin[g];
    z->n_items += P * ((R + z->item_reads - 1) / z->item_reads);
  }
  return check_limits(c, *z);
}

// The Dev descriptor of a batch of these sizes: its scalars, and every per-batch array as a view into the arena at
// `base`, in one fixed order, each rounded up to 256 bytes and so 256-byte aligned (k_encode relies on that).
// base == 0 only measures.  Returns the arena bytes the batch needs.  The grids (plan_batch) must be set.
static size_t layout_arena(Dev& D, const lgr_ctx* c, const BatchSizes& z, uintptr_t base) {
  std::memset(&D, 0, sizeof(D));  // D.ws / D.ws_cap: k_chain_overflow's workspace, set by overflow_pass
  D.P = c->P;
  D.n_groups = z.G, D.n_haps = z.NH, D.n_reads = z.NR, D.n_vars = z.NV, D.n_pairs = z.n_pairs, D.n_assign = z.n_assign;
  D.n_items = (int)z.n_items, D.item_reads = z.item_reads, D.mid_occ_param = c->prm.mid_occ;
  D.bkt_shift = 2 * c->prm.k > kBucketBits ? 2 * c->prm.k - kBucketBits : 0;
  const int Lm = std::max(z.max_read_len, 1);
  const int Tmax = Lm + ((c->prm.a + std::max(c->prm.b, c->prm.sc_ambi)) * Lm) / c->prm.e + 2;
  D.fin_cap = 2 * z.max_read_len + 16;
  D.regs_cap = z.n_pairs + z.n_pairs / 4 + 1024;
  D.tasks_cap = D.regs_cap * 2;
  D.ext_arena_cap = 4 * z.n_pairs + (1 << 20);
  D.ovf_cap = z.n_pairs;
  D.dir_per_warp = (int64_t)((Lm + 31) / 32) * (Tmax + 32) * 32;
  D.bnd_per_warp = 2 * (int64_t)(Tmax + 32);
  D.wcig_cap = 2 * Lm + 8;
  D.cigar_arena_cap = std::max<int64_t>(c->prm.cigar_arena_ops, 1024);
  // per-warp scratch follows the grid that indexes it: extension / finish kernels vs the cold chain kernel
  const size_t ext_warps = (size_t)std::max(c->ext_blocks, c->fin_blocks) * 4;
  const size_t chain_warps = (size_t)c->cold_blocks * kWarpsPerCta;  // the cold kernel's radix scratch
  const size_t G = z.G, NH = z.NH, NR = z.NR, NV = z.NV, nvh = z.nvh, pairs = z.n_pairs;
  const size_t hap_bytes = z.hap_bytes, read_bytes = z.read_bytes;
  size_t off = 0;
  auto take = [&](auto*& field, size_t count) {
    field = reinterpret_cast<std::remove_reference_t<decltype(field)>>(base + off);
    off += (std::max<size_t>(256, count * sizeof(*field)) + 255) & ~(size_t)255;
  };
  take(D.grp_hap_begin, G + 1), take(D.grp_read_begin, G + 1), take(D.grp_var_begin, G + 1);
  take(D.hap_off, NH + 1), take(D.read_off, NR + 1), take(D.var_hap_off, NV + 1);
  take(D.read_quals, read_bytes), take(D.name_hash, NR);
  take(D.var_start, nvh), take(D.var_len, nvh), take(D.var_allele, nvh);
  take(D.read_grp, NR), take(D.hap_grp, NH);
  take(D.pair_off, NR + 1), take(D.asg_off, NR + 1);
  take(D.item_hap, z.n_items), take(D.item_r0, z.n_items), take(D.item_n, z.n_items);
  take(D.grp_mid_req, G), take(D.grp_mid, G), take(D.grp_err, G + 1);
  take(D.hap_codes, hap_bytes), take(D.read_codes, read_bytes);
  take(D.idx, hap_bytes), take(D.idx_n, NH), take(D.hap_mid, NH);
  take(D.bkt, NH * (kBuckets + 1));
  take(D.mz_x, read_bytes), take(D.mz_y, read_bytes), take(D.mz_n, NR);
  take(D.mz_cnt, 2 * NR);
  take(D.rsx_scratch, chain_warps);
  take(D.fin_scratch, ext_warps * 2 * D.fin_cap);
  take(D.regs, D.regs_cap), take(D.pair_reg, pairs);
  take(D.tasks, D.tasks_cap * kExtClasses);
  take(D.ext_arena, D.ext_arena_cap);
  take(D.ovf_read, pairs + 32), take(D.ovf_hap, pairs + 32);
  take(D.cold_read, pairs + 32), take(D.cold_hap, pairs + 32);
  take(D.dir_scratch, ext_warps * D.dir_per_warp);
  take(D.bnd_scratch, ext_warps * D.bnd_per_warp);
  take(D.wcig_scratch, ext_warps * D.wcig_cap);
  take(D.aln, pairs);
  take(D.cigar_inline, pairs * LGR_CIGAR_INLINE);
  take(D.cigar_arena, D.cigar_arena_cap);
  take(D.assign, z.n_assign), take(D.ctr, C_COUNT);
  // inputs as they arrive: ASCII strings (plain form) or the slab (+ directory, + directory scans) of the packed form
  take(D.hap_bases, z.ascii ? hap_bytes : 0), take(D.read_bases, z.ascii ? read_bytes : 0);
  take(D.slab, z.slab_bytes), take(D.dir, z.dir_entries);
  take(D.grp_hapbase, G + 1), take(D.grp_readbase, G + 1), take(D.grp_vh, G + 1);
  take(D.grp_pair, G + 1), take(D.grp_asg, G + 1), take(D.grp_item, G + 1);
  take(D.hap_plane, z.ascii ? 0 : NH), take(D.read_plane, z.ascii ? 0 : NR);
  take(D.read_qoff, z.ascii ? 0 : NR), take(D.grp_lut, z.ascii ? 0 : 4 * G);
  return off;
}

// grids, arena and Dev descriptor for a batch of these sizes (grow-only; no copies here)
static int plan_batch(lgr_ctx* c, const BatchSizes& z) {
  LGR_CUDA(c, cudaSetDevice(c->device));
  const int64_t n_pairs = z.n_pairs;
  c->max_read_len = z.max_read_len, c->max_hap_len = z.max_hap_len;
  c->hap_bytes = z.hap_bytes, c->read_bytes = z.read_bytes;
  // warp-per-pair kernel: CAP anchors per pair in shared memory
  c->warp_cap = c->max_read_len <= 160 ? 64 : 128;
  c->warp_smem = chain_smem_bytes(c->warp_cap, true);
  c->cold_smem = chain_smem_bytes(c->warp_cap, false);
  if (c->occ_cap != c->warp_cap) {  // occupancy of the persistent kernels: once per context and shape
    int per_sm = 0, per_sm_cold = 0;
    const bool ok = c->warp_cap == 64 ? chain_occupancy<64>(c, &per_sm, &per_sm_cold) : chain_occupancy<128>(c, &per_sm, &per_sm_cold);
    if (!ok || per_sm < 1 || per_sm_cold < 1) {
      c->err = "the chain kernels do not fit on this device (shared memory / registers)";
      return LGR_E_CUDA;
    }
    c->warp_blocks_full = c->sm_count * per_sm;
    c->cold_blocks_full = c->sm_count * per_sm_cold;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ext_warp, 128, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
    c->ext_blocks_full = c->sm_count * per_sm;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_finish_warp, 128, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
    c->fin_blocks_full = c->sm_count * per_sm;
    c->occ_cap = c->warp_cap;
  }
  // a small batch (one Genotype() call) needs neither the full grids nor their per-warp scratch
  c->warp_blocks = (int)std::max<int64_t>(1, std::min<int64_t>(c->warp_blocks_full, z.n_items));
  c->cold_blocks = (int)std::max<int64_t>(1, std::min<int64_t>(c->cold_blocks_full, (n_pairs + kWarpsPerCta - 1) / kWarpsPerCta));
  c->ext_blocks = (int)std::max<int64_t>(1, std::min<int64_t>(c->ext_blocks_full, (n_pairs + 15) / 16));  // ~0.3 queued extensions per pair
  c->fin_blocks = (int)std::max<int64_t>(1, std::min<int64_t>(c->fin_blocks_full, (n_pairs + 4 * kFinChunk - 1) / (4 * kFinChunk)));
  Dev measured;
  const int rc = c->arena.ensure(layout_arena(measured, c, z, 0), false, c->err);
  if (rc != LGR_OK) return rc;
  layout_arena(c->D, c, z, reinterpret_cast<uintptr_t>(c->arena.p));
  return LGR_OK;
}

// plain form: 13 caller arrays + the host-derived helper arrays, one copy each
static int upload_impl(lgr_ctx* c, const lgr_batch_in* in, int64_t* h2d_bytes) {
  BatchSizes z;
  int rc = validate_batch(c, in, &z);
  if (rc != LGR_OK) return rc;
  if ((rc = plan_batch(c, z)) != LGR_OK) return rc;
  int64_t h2d = 0;
  const int G = z.G, NH = z.NH, NR = z.NR, NV = z.NV;
  c->h_read_grp.resize(NR + 1), c->h_hap_grp.resize(NH + 1), c->h_pair_off.resize(NR + 1), c->h_asg_off.resize(NR + 1);
  c->h_grp_mid.resize(G + 1);
  c->h_item_hap.clear(), c->h_item_r0.clear(), c->h_item_n.clear();
  int64_t po = 0, ao = 0;
  for (int g = 0; g < G; ++g) {
    const int h0 = in->grp_hap_begin[g], h1 = in->grp_hap_begin[g + 1];
    const int r0 = in->grp_read_begin[g], r1 = in->grp_read_begin[g + 1];
    const int V = in->grp_var_begin[g + 1] - in->grp_var_begin[g];
    for (int h = h0; h < h1; ++h) c->h_hap_grp[h] = g;
    for (int r = r0; r < r1; ++r) {
      c->h_read_grp[r] = g, c->h_pair_off[r] = po, c->h_asg_off[r] = ao;
      po += h1 - h0, ao += V;
    }
    for (int h = h0; h < h1; ++h)  // z.n_items work items in all (validate_batch counts them the same way)
      for (int r = r0; r < r1; r += z.item_reads) {
        c->h_item_hap.push_back(h), c->h_item_r0.push_back(r), c->h_item_n.push_back(std::min(z.item_reads, r1 - r));
      }
    int32_t mid = c->prm.mid_occ;
    if (in->grp_mid_occ && in->grp_mid_occ[g] > 0) mid = in->grp_mid_occ[g];
    c->h_grp_mid[g] = mid;
  }
  c->h_pair_off[NR] = po, c->h_asg_off[NR] = ao;
  const Dev& D = c->D;
  LGR_CUDA(c, copy_in(c, D.grp_hap_begin, in->grp_hap_begin, G + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.grp_read_begin, in->grp_read_begin, G + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.grp_var_begin, in->grp_var_begin, G + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.hap_off, in->hap_off, NH + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.read_off, in->read_off, NR + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.var_hap_off, in->var_hap_off, NV + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.hap_bases, in->hap_bases, z.hap_bytes, h2d));
  LGR_CUDA(c, copy_in(c, D.read_bases, in->read_bases, z.read_bytes, h2d));
  LGR_CUDA(c, copy_in(c, D.read_quals, in->read_quals, z.read_bytes, h2d));
  LGR_CUDA(c, copy_in(c, D.name_hash, in->read_name_hash, NR, h2d));
  LGR_CUDA(c, copy_in(c, D.var_start, in->var_start, z.nvh, h2d));
  LGR_CUDA(c, copy_in(c, D.var_len, in->var_len, z.nvh, h2d));
  LGR_CUDA(c, copy_in(c, D.var_allele, in->var_allele, z.nvh, h2d));
  LGR_CUDA(c, copy_in(c, D.read_grp, c->h_read_grp.data(), NR, h2d));
  LGR_CUDA(c, copy_in(c, D.hap_grp, c->h_hap_grp.data(), NH, h2d));
  LGR_CUDA(c, copy_in(c, D.pair_off, c->h_pair_off.data(), NR + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.asg_off, c->h_asg_off.data(), NR + 1, h2d));
  LGR_CUDA(c, copy_in(c, D.item_hap, c->h_item_hap.data(), z.n_items, h2d));
  LGR_CUDA(c, copy_in(c, D.item_r0, c->h_item_r0.data(), z.n_items, h2d));
  LGR_CUDA(c, copy_in(c, D.item_n, c->h_item_n.data(), z.n_items, h2d));
  LGR_CUDA(c, copy_in(c, D.grp_mid_req, c->h_grp_mid.data(), G, h2d));
  c->packed = false;
  c->resident = true;
  if (h2d_bytes) *h2d_bytes = h2d;
  return LGR_OK;
}

// packed form: the slab in one copy (plus the directory when it lives outside the slab); every
// other array is derived on the device by k_unpack_scan / k_unpack_group (enqueued by run_launch)
static int upload_packed_impl(lgr_ctx* c, const lgr_packed_in* in, int64_t* h2d_bytes) {
  auto bad = [&](const std::string& m, int code = LGR_E_ARG) { c->err = m; return code; };
  if (!in || in->n_groups < 0 || (in->n_groups > 0 && (!in->slab || !in->dir))) return bad("null packed batch");
  BatchSizes z;
  z.G = in->n_groups;
  for (int g = 0; g < z.G; ++g) {
    const lgr_group_dir& d = in->dir[g];
    if (d.n_haps < 0 || d.n_reads < 0 || d.n_vars < 0 || d.hap_bases < 0 || d.read_bases < 0 || (d.n_reads > 0 && d.n_haps == 0))
      return bad("bad group directory entry");
    if ((d.rec_off & 15) || d.rec_off + sizeof(lgr_group_rec_hdr) > in->slab_bytes) return bad("group record outside the slab");
    const lgr_group_rec_hdr* hdr = reinterpret_cast<const lgr_group_rec_hdr*>(static_cast<const uint8_t*>(in->slab) + d.rec_off);
    if (hdr->magic != LGR_PACK_MAGIC || d.rec_off + hdr->rec_bytes > in->slab_bytes) return bad("group record corrupt or truncated");
    if (hdr->qual_bits != 2 && hdr->qual_bits != 4 && hdr->qual_bits != 8) return bad("group record: bad qual_bits");
    z.NH += d.n_haps, z.NR += d.n_reads, z.NV += d.n_vars;
    z.hap_bytes += d.hap_bases, z.read_bytes += d.read_bases;
    z.nvh += (int64_t)d.n_vars * d.n_haps, z.n_pairs += (int64_t)d.n_reads * d.n_haps, z.n_assign += (int64_t)d.n_reads * d.n_vars;
    z.max_hap_len = std::max(z.max_hap_len, d.max_hap_len), z.max_read_len = std::max(z.max_read_len, d.max_read_len);
    if (z.NH < 0 || z.NR < 0 || z.NV < 0) return bad("batch too large", LGR_E_LIMIT);
  }
  z.item_reads = choose_item_reads(c, z.n_pairs);
  for (int g = 0; g < z.G; ++g)
    z.n_items += (int64_t)in->dir[g].n_haps * ((in->dir[g].n_reads + z.item_reads - 1) / z.item_reads);
  int rc = check_limits(c, z);
  if (rc != LGR_OK) return rc;
  const uint8_t* slab = static_cast<const uint8_t*>(in->slab);
  const uint8_t* dirp = reinterpret_cast<const uint8_t*>(in->dir);
  const bool dir_inside = z.G > 0 && dirp >= slab && dirp + sizeof(lgr_group_dir) * (size_t)z.G <= slab + in->slab_bytes;
  z.ascii = false, z.slab_bytes = in->slab_bytes, z.dir_entries = dir_inside ? 0 : z.G;
  if ((rc = plan_batch(c, z)) != LGR_OK) return rc;
  int64_t h2d = 0;
  Dev& D = c->D;
  LGR_CUDA(c, copy_in(c, D.slab, in->slab, z.slab_bytes, h2d));
  if (dir_inside) D.dir = reinterpret_cast<const lgr_group_dir*>(D.slab + (dirp - slab));
  else LGR_CUDA(c, copy_in(c, D.dir, in->dir, z.dir_entries, h2d));
  c->packed = true;
  c->resident = true;
  if (h2d_bytes) *h2d_bytes = h2d;
  return LGR_OK;
}

// phase B (extensions, finish), used by the main pass and the overflow pass
static void launch_tail(lgr_ctx* c, const Dev& D, cudaStream_t s, int* launches) {
  k_ext_warp<<<c->ext_blocks, 128, 0, s>>>(D);
  k_finish_warp<<<c->fin_blocks, 128, 0, s>>>(D);
  *launches += 2;
}

// assignment, after phase B of the main pass and of the overflow pass
static void launch_assign(const Dev& D, cudaStream_t s, int* launches) {
  if (D.n_assign <= 0) return;
  k_assign<<<(unsigned)((D.n_assign + 127) / 128), 128, 0, s>>>(D);
  *launches += 1;
}

// which k_hap_sketch instance the parameters select: 0 / 1 = warp kernel on 32- / 64-bit keys, 2 = generic
static int hap_sketch_variant(const DevParams& P) {
  if (P.w == 5 && (P.k & 1)) return 2 * P.k + 8 <= 32 ? 0 : 1;
  return 2;
}

// timing event i: an event-record node when the pass is being captured, so that the stage times of lgr_stats
// stay meaningful in graph mode (a plain record inside a capture only orders the streams)
static void mark(lgr_ctx* c, Ev i, cudaStream_t s) {
  if (c->capturing) cudaEventRecordWithFlags(c->ev[i], s, cudaEventRecordExternal);
  else cudaEventRecord(c->ev[i], s);
}

// enqueue one pass of the whole path on the context's streams; no host synchronisation.  Graph mode captures
// exactly this code.
static int enqueue_pass(lgr_ctx* c) {
  Dev& D = c->D;
  cudaStream_t s = c->stream;
  int launches = 0;
  LGR_CUDA(c, cudaMemsetAsync(D.ctr, 0, sizeof(long long) * C_COUNT, s));
  LGR_CUDA(c, cudaMemsetAsync(D.grp_err, 0, sizeof(int32_t) * (D.n_groups + 1), s));
  mark(c, EV_PASS_BEGIN, s);
  const int64_t hb = c->hap_bytes, rb = c->read_bytes;
  if (c->packed && D.n_groups > 0) {
    k_unpack_scan<<<1, 1024, 0, s>>>(D);
    k_unpack_group<<<std::min(D.n_groups, c->sm_count * 8), kUnpackThreads, 0, s>>>(D);
    const long long n_seq = (long long)D.n_haps + D.n_reads;
    if (n_seq > 0) {
      k_unpack_decode<<<(unsigned)std::min<long long>((n_seq + 7) / 8, (long long)c->sm_count * 16), kUnpackThreads, 0, s>>>(D);
      ++launches;
    }
    launches += 2;
  }
  if (D.n_pairs > 0) {
    const int enc_blocks = c->sm_count * 8;
    // read side (encode + sketch) on the second stream, haplotype side (encode, sketch, sort,
    // mid_occ) on the main one; they join before the minimizer filter
    cudaStream_t s2 = c->stream2;
    cudaEventRecord(c->ev_fork, s);
    cudaStreamWaitEvent(s2, c->ev_fork, 0);
    if (!c->packed) k_encode<<<enc_blocks, 256, 0, s2>>>(D.read_bases, D.read_codes, rb), ++launches;
    k_read_sketch<<<(D.n_reads + 127) / 128, 128, 0, s2>>>(D);
    cudaEventRecord(c->ev_join, s2);
    if (!c->packed) k_encode<<<enc_blocks, 256, 0, s>>>(D.hap_bases, D.hap_codes, hb), ++launches;
    const int sketch = hap_sketch_variant(D.P);
    if (sketch == 0) k_hap_sketch_warp<uint32_t><<<(D.n_haps + 3) / 4, 128, 0, s>>>(D);
    else if (sketch == 1) k_hap_sketch_warp<uint64_t><<<(D.n_haps + 3) / 4, 128, 0, s>>>(D);
    else k_hap_sketch<<<(D.n_haps + 63) / 64, 64, 0, s>>>(D);
    k_hap_sort<<<D.n_haps, 128, 2048 * sizeof(uint64_t), s>>>(D, c->prm.mid_occ_frac, c->prm.min_mid_occ, c->prm.max_mid_occ);
    k_group_mid<<<(D.n_groups + 127) / 128, 128, 0, s>>>(D, c->prm.min_mid_occ);
    cudaStreamWaitEvent(s, c->ev_join, 0);
    launches += 4;
    mark(c, EV_INDEXED, s);
    k_read_filter<<<(D.n_reads + 127) / 128, 128, 0, s>>>(D);
    launches += 1;
    mark(c, EV_FILTERED, s);
    c->warp_cap == 64 ? launch_chain<64>(c, D, s) : launch_chain<128>(c, D, s);
    launches += 2;
    mark(c, EV_CHAINED, s);
    launch_tail(c, D, s, &launches);
    mark(c, EV_EXTENDED, s);
    launch_assign(D, s, &launches);
  } else {
    if (D.n_groups > 0) k_group_mid<<<(D.n_groups + 127) / 128, 128, 0, s>>>(D, c->prm.min_mid_occ), ++launches;
    mark(c, EV_INDEXED, s), mark(c, EV_FILTERED, s), mark(c, EV_CHAINED, s), mark(c, EV_EXTENDED, s);
  }
  mark(c, EV_PASS_END, s);
  LGR_CUDA(c, cudaMemcpyAsync(c->h_ctr, D.ctr, sizeof(long long) * C_COUNT, cudaMemcpyDeviceToHost, s));
  c->launches = launches;
  return LGR_OK;
}

// every batch-dependent branch of enqueue_pass: batches with equal keys capture graphs of the same topology
static uint32_t graph_key(const lgr_ctx* c) {
  const Dev& D = c->D;
  return (uint32_t)c->packed | (uint32_t)(D.n_groups > 0) << 1 | (uint32_t)((long long)D.n_haps + D.n_reads > 0) << 2 |
         (uint32_t)(D.n_pairs > 0) << 3 | (uint32_t)(D.n_assign > 0) << 4 | (uint32_t)(c->warp_cap == 128) << 5 |
         (uint32_t)hap_sketch_variant(D.P) << 6;
}

// Graph mode: capture enqueue_pass on the context's streams, bring the cached executable of its topology up to
// this batch with cudaGraphExecUpdate (grid sizes and the Dev descriptor are captured by value, so batches of any
// size share one executable) or instantiate one when there is none or the update is refused, and launch it.  One
// cudaGraphLaunch replaces the pass's dozen dependent launches and the gaps between them.
static int run_launch_graph(lgr_ctx* c) {
  cudaStream_t s = c->stream;
  LGR_CUDA(c, cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  c->capturing = true;
  int rc = enqueue_pass(c);
  c->capturing = false;
  cudaGraph_t graph = nullptr;
  const cudaError_t ec = cudaStreamEndCapture(s, &graph);  // always ends the capture, also after a failed enqueue
  if (rc != LGR_OK || ec != cudaSuccess) {
    if (graph) cudaGraphDestroy(graph);
    const cudaError_t el = cudaGetLastError();  // a launch that invalidated the capture
    if (rc == LGR_OK) {
      c->err = std::string("stream capture of the pass: ") + cudaGetErrorString(el != cudaSuccess ? el : ec);
      rc = LGR_E_CUDA;
    }
    return rc;
  }
  const uint32_t key = graph_key(c);
  GraphSlot* slot = nullptr;
  for (GraphSlot& g : c->graphs)
    if (g.exec && g.key == key) slot = &g;
  if (slot) {
    cudaGraphExecUpdateResultInfo info;
    if (cudaGraphExecUpdate(slot->exec, graph, &info) == cudaSuccess) {
      ++c->graph_updated;
    } else {  // topology or a parameter the update cannot take: instantiate afresh
      (void)cudaGetLastError();
      cudaGraphExecDestroy(slot->exec);
      slot->exec = nullptr;
    }
  } else {
    slot = &c->graphs[0];
    for (GraphSlot& g : c->graphs)
      if (!g.exec || (slot->exec && g.used < slot->used)) slot = &g;
    if (slot->exec) cudaGraphExecDestroy(slot->exec);
    slot->exec = nullptr;
  }
  if (!slot->exec) {
    const cudaError_t ei = cudaGraphInstantiate(&slot->exec, graph, 0);
    if (ei != cudaSuccess) {
      (void)cudaGetLastError();
      slot->exec = nullptr;
      cudaGraphDestroy(graph);
      c->err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ei);
      return LGR_E_CUDA;
    }
    slot->key = key;
    ++c->graph_instantiated;
  }
  slot->used = ++c->graph_tick;
  cudaGraphDestroy(graph);
  LGR_CUDA(c, cudaGraphLaunch(slot->exec, s));
  ++c->graph_replayed;
  return LGR_OK;
}

// one pass of the whole path, as separate launches or (graph = true) as one CUDA graph
static int run_launch(lgr_ctx* c, bool graph) {
  if (!c->resident) { c->err = "no batch uploaded"; return LGR_E_ARG; }
  LGR_CUDA(c, cudaSetDevice(c->device));
  return graph ? run_launch_graph(c) : enqueue_pass(c);
}

// Overflow pass, host driven, after the main pass has drained: the pairs whose seeds / anchors /
// chains did not fit the shared-memory workspace of the chain kernels (reads inside tandem repeats) were
// listed, not refused.  Now their number and the largest anchor count among them are known, so the
// HBM workspace is allocated to measure (nothing is reserved up front), k_chain_overflow maps them,
// and extension / finish / assignment run again over what they added.  Rare: the price is one extra
// host round trip for a batch that holds such a pair.
static int overflow_pass(lgr_ctx* c) {
  Dev& D = c->D;
  cudaStream_t s = c->stream;
  const long long n_ovf = std::min<long long>(c->h_ctr[C_NOVF], D.ovf_cap);
  if (n_ovf <= 0) return LGR_OK;
  long long need = std::max<long long>(c->h_ctr[C_OVFNEED], 256);
  need = std::min<long long>((need + 255) / 256 * 256, kBigCapMax);
  const int lanes = (int)std::min<long long>((n_ovf + 127) / 128 * 128, kBigLanesMax);
  int rc = c->ws_big.ensure(sizeof(int32_t) * (size_t)lanes * A_COUNT * (size_t)need, false, c->err);
  if (rc != LGR_OK) return rc;
  Dev D2 = D;
  D2.ws = (int32_t*)c->ws_big.p, D2.ws_cap = (int)need;
  // restart the queues of phase B: extensions continue after the tasks already done, finish and
  // assignment redo every pair (idempotent; the overflow cigar arena is refilled from 0)
  long long* hc = c->h_ctr + C_COUNT + 2;  // pinned staging of the counter patch
  for (int cls = 0; cls < kExtClasses; ++cls) hc[cls] = std::min<long long>(c->h_ctr[C_NTASK + cls], D.tasks_cap);
  LGR_CUDA(c, cudaMemcpyAsync(D.ctr + C_TASKPOS, hc, sizeof(long long) * kExtClasses, cudaMemcpyHostToDevice, s));
  LGR_CUDA(c, cudaMemsetAsync(D.ctr + C_FINPOS, 0, sizeof(long long), s));
  LGR_CUDA(c, cudaMemsetAsync(D.ctr + C_CIGARENA, 0, sizeof(long long), s));
  LGR_CUDA(c, cudaMemsetAsync(D.ctr + C_ALIGNED, 0, sizeof(long long), s));
  LGR_CUDA(c, cudaMemsetAsync(D.ctr + C_OVFPOS, 0, sizeof(long long), s));
  int launches = 0;
  k_chain_overflow<<<lanes / 128, 128, 0, s>>>(D2);
  ++launches;
  launch_tail(c, D, s, &launches);
  launch_assign(D, s, &launches);
  LGR_CUDA(c, cudaMemcpyAsync(c->h_ctr, D.ctr, sizeof(long long) * C_COUNT, cudaMemcpyDeviceToHost, s));
  LGR_CUDA(c, cudaStreamSynchronize(s));
  c->launches += launches;
  c->overflow_passes += 1;
  return LGR_OK;
}

// after the stream has drained: overflow pass when needed, statistics, device-side limit flags
static int run_finish(lgr_ctx* c, lgr_stats* st) {
  LGR_CUDA(c, cudaGetLastError());
  Dev& D = c->D;
  if (c->h_ctr[C_NOVF] > 0) {
    const int rc = overflow_pass(c);
    if (rc != LGR_OK) return rc;
    LGR_CUDA(c, cudaGetLastError());
  }
  const long long* hctr = c->h_ctr;
  const int launches = c->launches;
  if (st) {
    cudaEventElapsedTime(&st->ms_kernels, c->ev[EV_PASS_BEGIN], c->ev[EV_PASS_END]);
    cudaEventElapsedTime(&st->ms_k_index, c->ev[EV_PASS_BEGIN], c->ev[EV_INDEXED]);
    cudaEventElapsedTime(&st->ms_k_sketch, c->ev[EV_INDEXED], c->ev[EV_FILTERED]);
    cudaEventElapsedTime(&st->ms_k_map, c->ev[EV_FILTERED], c->ev[EV_CHAINED]);
    cudaEventElapsedTime(&st->ms_k_ext, c->ev[EV_CHAINED], c->ev[EV_EXTENDED]);
    cudaEventElapsedTime(&st->ms_k_assign, c->ev[EV_EXTENDED], c->ev[EV_PASS_END]);
    st->n_pairs = D.n_pairs, st->n_aligned = hctr[C_ALIGNED];
    st->dp_cells = hctr[C_CELLS], st->dp_cells_full = hctr[C_CELLSFULL];
    st->chain_evals = hctr[C_EVALS], st->n_anchors = hctr[C_ANCH];
    st->kernel_launches = launches;
    st->reserved = (int32_t)std::min<long long>(hctr[C_NOVF], INT32_MAX);  // pairs that took the overflow pass
  }
  if (hctr[C_ERR]) {
    char buf[200];
    snprintf(buf, sizeof(buf), "device path limit hit (flags 0x%llx: 1 reg arena, 2 ext arena, 4 cigar arena, 8 anchor cap, 16 cigar scratch, 32 minimizer cap)",
             hctr[C_ERR]);
    c->err = buf;
    return (hctr[C_ERR] == E_CIG_ARENA) ? LGR_E_CIGAR_OVERFLOW : LGR_E_LIMIT;
  }
  return LGR_OK;
}

static int run_impl(lgr_ctx* c, lgr_stats* st) {
  int rc = run_launch(c, c->graph_mode);
  if (rc != LGR_OK) return rc;
  LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  return run_finish(c, st);
}

// enqueue the device→host copies whose sizes are known up front (records, inline cigars,
// assignments, per-group status); the overflow cigar arena follows in download_finish once its
// fill is known
static int download_launch(lgr_ctx* c, lgr_batch_out* out, int64_t* d2h_bytes) {
  if (!c->resident || !out) { c->err = "nothing to download"; return LGR_E_ARG; }
  LGR_CUDA(c, cudaSetDevice(c->device));
  Dev& D = c->D;
  int64_t d2h = 0;
  if (out->aln) {
    if (out->n_pairs < D.n_pairs) { c->err = "out->n_pairs too small"; return LGR_E_ARG; }
    LGR_CUDA(c, cudaMemcpyAsync(out->aln, D.aln, sizeof(AlnOut) * D.n_pairs, cudaMemcpyDeviceToHost, c->stream));
    d2h += sizeof(AlnOut) * D.n_pairs;
    if (out->cigar_inline) {
      LGR_CUDA(c, cudaMemcpyAsync(out->cigar_inline, D.cigar_inline, sizeof(uint32_t) * D.n_pairs * LGR_CIGAR_INLINE, cudaMemcpyDeviceToHost, c->stream));
      d2h += sizeof(uint32_t) * D.n_pairs * LGR_CIGAR_INLINE;
    }
    LGR_CUDA(c, cudaMemcpyAsync(c->h_ctr + C_COUNT, D.ctr + C_CIGARENA, sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
  }
  if (out->assign && D.n_assign > 0) {
    if (out->n_assign < D.n_assign) { c->err = "out->n_assign too small"; return LGR_E_ARG; }
    LGR_CUDA(c, cudaMemcpyAsync(out->assign, D.assign, sizeof(AssignOut) * D.n_assign, cudaMemcpyDeviceToHost, c->stream));
    d2h += sizeof(AssignOut) * D.n_assign;
  }
  if (out->grp_status && D.n_groups > 0) {
    LGR_CUDA(c, cudaMemcpyAsync(out->grp_status, D.grp_err, sizeof(int32_t) * D.n_groups, cudaMemcpyDeviceToHost, c->stream));
    d2h += sizeof(int32_t) * D.n_groups;
  }
  if (out->grp_mid_occ && D.n_groups > 0) {
    LGR_CUDA(c, cudaMemcpyAsync(out->grp_mid_occ, D.grp_mid, sizeof(int32_t) * D.n_groups, cudaMemcpyDeviceToHost, c->stream));
    d2h += sizeof(int32_t) * D.n_groups;
  }
  if (d2h_bytes) *d2h_bytes = d2h;
  return LGR_OK;
}

// stream already drained by the caller.  ErrBits → LGR_E_* per group.
static int download_finish(lgr_ctx* c, lgr_batch_out* out, int64_t* d2h_bytes) {
  Dev& D = c->D;
  if (out->grp_status)
    for (int g = 0; g < D.n_groups; ++g) {
      const int bits = out->grp_status[g];
      out->grp_status[g] = bits == 0 ? LGR_OK : (bits == E_CIG_ARENA ? LGR_E_CIGAR_OVERFLOW : LGR_E_LIMIT);
    }
  if (out->aln) {
    const long long used = c->h_ctr[C_COUNT];
    out->cigar_arena_used = used;
    if (used > 0) {
      if (!out->cigar_arena || out->cigar_arena_cap < used) { c->err = "host cigar arena too small"; return LGR_E_CIGAR_OVERFLOW; }
      LGR_CUDA(c, cudaMemcpyAsync(out->cigar_arena, D.cigar_arena, sizeof(uint32_t) * used, cudaMemcpyDeviceToHost, c->stream));
      LGR_CUDA(c, cudaStreamSynchronize(c->stream));
      if (d2h_bytes) *d2h_bytes += sizeof(uint32_t) * used;
    }
  }
  return LGR_OK;
}

static int download_impl(lgr_ctx* c, lgr_batch_out* out, int64_t* d2h_bytes) {
  int rc = download_launch(c, out, d2h_bytes);
  if (rc != LGR_OK) return rc;
  LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  return download_finish(c, out, d2h_bytes);
}

// a device-path limit hit some pairs: with a per-group status array the call is a partial success
static int limit_code(int run_rc, const lgr_batch_out* out) {
  if ((run_rc == LGR_E_LIMIT || run_rc == LGR_E_CIGAR_OVERFLOW) && out && out->grp_status) return LGR_E_PARTIAL;
  return run_rc;
}

int lgr_upload(lgr_ctx* c, const lgr_batch_in* in) {
  if (!c) return LGR_E_ARG;
  int rc = upload_impl(c, in, nullptr);
  if (rc == LGR_OK) LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  return rc;
}

int lgr_upload_packed(lgr_ctx* c, const lgr_packed_in* in) {
  if (!c) return LGR_E_ARG;
  int rc = upload_packed_impl(c, in, nullptr);
  if (rc == LGR_OK) LGR_CUDA(c, cudaStreamSynchronize(c->stream));
  return rc;
}

int lgr_run_resident(lgr_ctx* c, lgr_stats* stats) {
  if (!c) return LGR_E_ARG;
  if (stats) std::memset(stats, 0, sizeof(*stats));
  return run_impl(c, stats);
}

int lgr_download(lgr_ctx* c, lgr_batch_out* out) {
  if (!c) return LGR_E_ARG;
  return download_impl(c, out, nullptr);
}

// ms_h2d / ms_d2h of lgr_stats: the events genotype_sync and submit_async record around the copies
static void copy_times(const lgr_ctx* c, lgr_stats* st) {
  cudaEventElapsedTime(&st->ms_h2d, c->ev[EV_H2D_BEGIN], c->ev[EV_H2D_END]);
  cudaEventElapsedTime(&st->ms_d2h, c->ev[EV_D2H_BEGIN], c->ev[EV_D2H_END]);
}

// synchronous: upload (either form), all kernels, download
typedef int (*upload_fn)(lgr_ctx*, const void*, int64_t*);
static int up_plain(lgr_ctx* c, const void* in, int64_t* b) { return upload_impl(c, static_cast<const lgr_batch_in*>(in), b); }
static int up_packed(lgr_ctx* c, const void* in, int64_t* b) { return upload_packed_impl(c, static_cast<const lgr_packed_in*>(in), b); }

static int genotype_sync(lgr_ctx* c, const void* in, lgr_batch_out* out, lgr_stats* stats, upload_fn up) {
  if (!c || !in || !out) return LGR_E_ARG;
  lgr_stats st;
  std::memset(&st, 0, sizeof(st));
  int64_t h2d = 0, d2h = 0;
  cudaEventRecord(c->ev[EV_H2D_BEGIN], c->stream);
  int rc = up(c, in, &h2d);
  if (rc != LGR_OK) return rc;
  cudaEventRecord(c->ev[EV_H2D_END], c->stream);
  rc = run_impl(c, &st);
  if (rc != LGR_OK && rc != LGR_E_LIMIT && rc != LGR_E_CIGAR_OVERFLOW) return rc;
  const int run_rc = limit_code(rc, out);
  cudaEventRecord(c->ev[EV_D2H_BEGIN], c->stream);
  rc = download_impl(c, out, &d2h);
  cudaEventRecord(c->ev[EV_D2H_END], c->stream);
  cudaStreamSynchronize(c->stream);
  copy_times(c, &st);
  st.h2d_bytes = h2d, st.d2h_bytes = d2h;
  if (stats) *stats = st;
  return run_rc != LGR_OK ? run_rc : rc;
}

int lgr_genotype_batch(lgr_ctx* c, const lgr_batch_in* in, lgr_batch_out* out, lgr_stats* stats) {
  return genotype_sync(c, in, out, stats, up_plain);
}

int lgr_genotype_packed(lgr_ctx* c, const lgr_packed_in* in, lgr_batch_out* out, lgr_stats* stats) {
  return genotype_sync(c, in, out, stats, up_packed);
}

static int submit_async(lgr_ctx* c, const void* in, lgr_batch_out* out, lgr_ticket* ticket, upload_fn up) {
  if (!c || !in || !out || !ticket) return LGR_E_ARG;
  int t = -1;
  for (int i = 0; i < LGR_MAX_INFLIGHT && t < 0; ++i)
    if (!c->slot_busy[i]) t = i;
  if (t < 0) { c->err = "all submission slots are in flight; lgr_wait one first"; return LGR_E_BUSY; }
  if (!c->slot[t]) {
    int rc = lgr_create(c->device, &c->prm, &c->slot[t]);
    if (rc != LGR_OK) { c->err = g_create_err; return rc; }
  }
  lgr_ctx* ch = c->slot[t];
  int64_t h2d = 0, d2h = 0;
  cudaEventRecord(ch->ev[EV_H2D_BEGIN], ch->stream);
  int rc = up(ch, in, &h2d);
  if (rc == LGR_OK) {
    cudaEventRecord(ch->ev[EV_H2D_END], ch->stream);
    rc = run_launch(ch, false);  // the pipelined path hides its launches behind the batch in flight
  }
  if (rc == LGR_OK) {
    cudaEventRecord(ch->ev[EV_D2H_BEGIN], ch->stream);
    rc = download_launch(ch, out, &d2h);
    cudaEventRecord(ch->ev[EV_D2H_END], ch->stream);
  }
  if (rc != LGR_OK) {
    cudaStreamSynchronize(ch->stream);  // leave the slot idle
    c->err = ch->err;
    return rc;
  }
  c->slot_busy[t] = true, c->slot_out[t] = out, c->slot_h2d[t] = h2d, c->slot_d2h[t] = d2h;
  *ticket = t;
  if (c->notify_fn) {
    c->slot_note[t] = lgr_ctx::Note{c, t};
    cudaLaunchHostFunc(ch->stream, [](void* p) {
      const lgr_ctx::Note* n = static_cast<const lgr_ctx::Note*>(p);
      if (n->ctx->notify_fn) n->ctx->notify_fn(n->ctx->notify_user, n->ticket);
    }, &c->slot_note[t]);
  }
  return LGR_OK;
}

int lgr_reserve(lgr_ctx* c, int64_t arena_bytes, int n_slots) {
  if (!c || arena_bytes < 0 || n_slots < 0 || n_slots > LGR_MAX_INFLIGHT) return LGR_E_ARG;
  LGR_CUDA(c, cudaSetDevice(c->device));
  for (int t = 0; t < n_slots; ++t) {
    if (c->slot_busy[t]) continue;  // in flight: its arena is in use, leave it alone
    if (!c->slot[t]) {
      int rc = lgr_create(c->device, &c->prm, &c->slot[t]);
      if (rc != LGR_OK) { c->err = g_create_err; return rc; }
    }
    const int rc = c->slot[t]->arena.ensure((size_t)arena_bytes, false, c->err);
    if (rc != LGR_OK) return rc;
  }
  return LGR_OK;
}

int lgr_resident_assign(lgr_ctx* c, const lgr_assign** dev_assign, int64_t* n_assign) {
  if (!c || !dev_assign || !n_assign) return LGR_E_ARG;
  static_assert(sizeof(AssignOut) == sizeof(lgr_assign), "device and ABI records must coincide");
  *dev_assign = reinterpret_cast<const lgr_assign*>(c->D.assign);
  *n_assign = c->D.n_assign;
  return c->D.assign ? LGR_OK : LGR_E_ARG;
}

int64_t lgr_arena_bytes(const lgr_ctx* c) {
  if (!c) return 0;
  int64_t b = (int64_t)c->arena.cap;
  for (int t = 0; t < LGR_MAX_INFLIGHT; ++t)
    if (c->slot[t]) b += (int64_t)c->slot[t]->arena.cap;
  return b;
}

// Diagnostics: the device counters of the last finished batch of this context (enum Ctr in lgr_dev.cuh: work
// queues, cold-path reasons, extension tasks per size class).  Not part of the stable ABI.
int lgr_debug_counters(lgr_ctx* c, long long* out, int n) {
  if (!c || !out) return LGR_E_ARG;
  for (int i = 0; i < n; ++i) out[i] = i < C_COUNT ? c->h_ctr[i] : 0;
  return C_COUNT;
}

int lgr_set_notify(lgr_ctx* c, lgr_notify_fn fn, void* user) {
  if (!c) return LGR_E_ARG;
  c->notify_fn = fn, c->notify_user = user;
  return LGR_OK;
}

int lgr_set_graph_mode(lgr_ctx* c, int on) {
  if (!c) return LGR_E_ARG;
  c->graph_mode = on != 0;  // the cached executables stay: switching back on reuses them
  return LGR_OK;
}

int lgr_graph_counters(lgr_ctx* c, int64_t* instantiated, int64_t* updated, int64_t* replayed) {
  if (!c) return LGR_E_ARG;
  if (instantiated) *instantiated = c->graph_instantiated;
  if (updated) *updated = c->graph_updated;
  if (replayed) *replayed = c->graph_replayed;
  return LGR_OK;
}

int lgr_check_limits(const lgr_params* params, int32_t max_hap_len, int32_t max_read_len) {
  lgr_params p;
  if (params) p = *params;
  else lgr_default_params(&p);
  return limit_message(p, max_hap_len, max_read_len) ? LGR_E_LIMIT : LGR_OK;
}

int lgr_submit(lgr_ctx* c, const lgr_batch_in* in, lgr_batch_out* out, lgr_ticket* ticket) {
  return submit_async(c, in, out, ticket, up_plain);
}

int lgr_submit_packed(lgr_ctx* c, const lgr_packed_in* in, lgr_batch_out* out, lgr_ticket* ticket) {
  return submit_async(c, in, out, ticket, up_packed);
}

int lgr_wait(lgr_ctx* c, lgr_ticket t, lgr_stats* stats) {
  if (!c || t < 0 || t >= LGR_MAX_INFLIGHT || !c->slot_busy[t]) {
    if (c) c->err = "lgr_wait: unknown ticket";
    return LGR_E_ARG;
  }
  lgr_ctx* ch = c->slot[t];
  c->slot_busy[t] = false;
  if (cudaStreamSynchronize(ch->stream) != cudaSuccess) {
    c->err = std::string("lgr_wait: ") + cudaGetErrorString(cudaGetLastError());
    return LGR_E_CUDA;
  }
  lgr_stats st;
  std::memset(&st, 0, sizeof(st));
  const int passes0 = ch->overflow_passes;
  int run_rc = run_finish(ch, &st);
  int rc = LGR_OK;
  int64_t d2h = c->slot_d2h[t];
  if (run_rc == LGR_OK || run_rc == LGR_E_LIMIT || run_rc == LGR_E_CIGAR_OVERFLOW) {
    // the overflow pass rewrote results after the copies of lgr_submit were taken: copy again
    if (ch->overflow_passes != passes0) rc = download_launch(ch, c->slot_out[t], &d2h);
    if (rc == LGR_OK && ch->overflow_passes != passes0 && cudaStreamSynchronize(ch->stream) != cudaSuccess) rc = LGR_E_CUDA;
    if (rc == LGR_OK) rc = download_finish(ch, c->slot_out[t], &d2h);
  }
  run_rc = limit_code(run_rc, c->slot_out[t]);
  copy_times(ch, &st);
  st.h2d_bytes = c->slot_h2d[t], st.d2h_bytes = d2h;
  if (stats) *stats = st;
  if (run_rc != LGR_OK || rc != LGR_OK) c->err = ch->err;
  return run_rc != LGR_OK ? run_rc : rc;
}

size_t lgr_packed_group_bytes(const lgr_group_desc* g) {
  const lgr_pack::Plan p = lgr_pack::plan_group(g);
  return p.rc == LGR_OK ? p.bytes : 0;
}

int lgr_pack_group(const lgr_group_desc* g, void* dst, size_t cap, lgr_group_dir* dir) {
  if (!g || !dst || (reinterpret_cast<uintptr_t>(dst) & 7)) return LGR_E_ARG;
  const lgr_pack::Plan p = lgr_pack::plan_group(g);
  if (p.rc != LGR_OK) return p.rc;
  if (p.bytes > cap) return LGR_E_ARG;
  return lgr_pack::pack_group(g, p, dst, dir);
}

int lgr_hap_mid_occ(lgr_ctx* c, const uint8_t* hap, int32_t hap_len, int32_t* mid_occ) {
  if (!c || !hap || hap_len < 0 || !mid_occ) return LGR_E_ARG;
  if (hap_len > LGR_MAX_HAP_LEN) { c->err = "haplotype longer than LGR_MAX_HAP_LEN"; return LGR_E_LIMIT; }
  // a one-haplotype, zero-read batch through the index kernels
  const int32_t gb[2] = {0, 1}, zero2[2] = {0, 0};
  const int64_t ho[2] = {0, hap_len}, ro[1] = {0}, vo[1] = {0};
  lgr_batch_in in;
  std::memset(&in, 0, sizeof(in));
  in.n_groups = 1, in.n_haps = 1, in.n_reads = 0, in.n_vars = 0;
  in.grp_hap_begin = gb, in.grp_read_begin = zero2, in.grp_var_begin = zero2;
  in.hap_off = ho, in.hap_bases = hap, in.read_off = ro, in.var_hap_off = vo;
  int rc = upload_impl(c, &in, nullptr);
  if (rc != LGR_OK) return rc;
  Dev& D = c->D;
  cudaStream_t s = c->stream;
  LGR_CUDA(c, cudaMemsetAsync(D.ctr, 0, sizeof(long long) * C_COUNT, s));
  k_encode<<<8, 256, 0, s>>>(D.hap_bases, D.hap_codes, hap_len);
  k_hap_sketch<<<1, 64, 0, s>>>(D);
  k_hap_sort<<<1, 128, 2048 * sizeof(uint64_t), s>>>(D, c->prm.mid_occ_frac, c->prm.min_mid_occ, c->prm.max_mid_occ);
  LGR_CUDA(c, cudaMemcpyAsync(mid_occ, D.hap_mid, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  LGR_CUDA(c, cudaStreamSynchronize(s));
  LGR_CUDA(c, cudaGetLastError());
  c->resident = false;
  return LGR_OK;
}

}  // extern "C"
