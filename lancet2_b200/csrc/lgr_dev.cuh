// lgr_dev.cuh — device descriptor, counters, parked-pair records, launch-shape knobs, result writers
// Part of the single translation unit lgr_gpu.cu (included there, in order); see that file's header.
#ifndef LANCET2_B200_LGR_DEV_CUH_
#define LANCET2_B200_LGR_DEV_CUH_

namespace {

using namespace lgr;

__constant__ double c_phred_err[256] = {
#include "phred_lut.inc"
};

// counters (int64 slots in device memory)
enum Ctr {
  C_ITEM = 0, C_NTASK, C_NTASK1, C_NTASK2, C_NTASK3, C_NTASK4, C_REGS, C_EXTARENA, C_CIGARENA, C_NOVF, C_ERR, C_EVALS, C_ANCH, C_CELLS, C_CELLSFULL,
  C_ALIGNED, C_TASKPOS, C_TASKPOS1, C_TASKPOS2, C_TASKPOS3, C_TASKPOS4, C_FINPOS, C_OVFPOS, C_OVFNEED, C_NCOLD, C_COLDPOS,
  C_COLD_HIGH, C_COLD_SORT, C_COLD_LONG,  // why pairs went to the cold kernel (diagnostics)
  C_LEAN_DEFER,                           // pairs the lean chain kernel queued for the cold kernel (every shape but sorted co-linear)
  C_COUNT
};
enum ErrBits { E_REG_ARENA = 1, E_EXT_ARENA = 2, E_CIG_ARENA = 4, E_ANCHOR_CAP = 8, E_CIG_SCRATCH = 16, E_MZ_CAP = 32 };

constexpr int kBucketBits = 9;
constexpr int kBuckets = 1 << kBucketBits;

struct TaskRec {  // one extension that needs the wavefront DP
  int32_t reg, side, read, hap;
};

// Extension tasks are queued by size class so that short tails share a warp (k_ext_warp):
//   class 0: m <= 8 query rows, 4 tails per warp (8 lanes each)
//   class 1: m <= 16, 2 tails per warp
//   class 2: everything else, one tail per warp (row blocks of 32)
//   class 3: n <= 8 target columns and fewer columns than rows (a read overhanging a haplotype end:
//            ~100 rows x ~5 columns), TRANSPOSED — lanes own columns — 4 tails per warp
//   class 4: the same with n <= 16, 2 tails per warp
// A sub-warp tail must also keep its staged codes and direction bytes in its share of the warp's
// shared-memory slice.
constexpr int kExtClasses = 5;
constexpr int kDirSmemPerWarp = 6144;  // staged codes + direction bytes of the tails a warp works on, in shared memory
constexpr int kSegHead = 96;           // bytes at the start of a sub-warp segment's slice: staged query + target codes

struct PairReg {  // per pair: its parked RegRecs in the arena (n == 0: nothing to finish)
  int32_t first, n, read, hap;
};

struct Dev {      // everything the kernels need, passed by value
  DevParams P;
  int n_groups, n_haps, n_reads, n_vars;
  int64_t n_pairs, n_assign;
  // inputs
  const int32_t *grp_hap_begin, *grp_read_begin, *grp_var_begin;
  const int64_t *hap_off, *read_off, *var_hap_off;
  const uint8_t *hap_bases, *read_bases, *read_quals;
  const uint32_t* name_hash;
  const int32_t *var_start, *var_len;
  const int8_t* var_allele;
  const int32_t* read_grp;      // [NR]
  const int32_t* hap_grp;       // [NH]
  const int64_t *pair_off, *asg_off;  // [NR+1]
  const int32_t *item_hap, *item_r0, *item_n;  // phase-A work items: (hap, first read, #reads<=32)
  int n_items;
  // derived
  uint8_t *hap_codes, *read_codes;
  uint64_t* idx;                // [hap_off-indexed] sorted minimizer tables
  int32_t *idx_n, *hap_mid;     // [NH]
  uint16_t* bkt;                // [NH][kBuckets+1] start of every hash bucket (top hash bits) in the sorted table
  int bkt_shift;                // hash >> bkt_shift = bucket
  const int32_t* grp_mid_req;   // [G] requested: >0 fixed (the worker's latched value), <=0 derive from the REF haplotype
  int32_t* grp_mid;             // [G] effective mid_occ (k_group_mid)
  int32_t* grp_err;             // [G] ErrBits that hit a pair of the group (0 = complete)
  // packed wire format (lgr_submit_packed): the slab as copied + its directory, and the per-group
  // prefix sums k_unpack_scan derives from the directory ([G+1] each)
  const uint8_t* slab;
  const lgr_group_dir* dir;
  int64_t *grp_hapbase, *grp_readbase, *grp_vh, *grp_pair, *grp_asg;
  int32_t* grp_item;
  uint64_t *hap_plane, *read_plane;  // [NH] / [NR] slab offset of every sequence's first plane word (| kSeqHasExc)
  uint64_t* read_qoff;               // [NR] slab offset of the read's quality data | quality plane count << 56
  uint32_t* grp_lut;                 // [G][4] the groups' quality dictionaries
  int item_reads;               // reads per phase-A work item
  int mid_occ_param;            // lgr_params::mid_occ
  uint64_t* mz_x;               // [read_off-indexed]
  uint32_t* mz_y;
  int32_t* mz_n;                // [NR]
  uint64_t* mz_cnt;             // [NR][2] bucket counters of the read's minimizer hashes
  // phase A workspace
  int32_t* ws;                  // k_chain_overflow: [warps][A_COUNT][cap][32 lanes] workspace
  int ws_cap;
  uint32_t* fin_scratch;        // [warps][2][fin_cap] cigar staging of k_finish_warp
  int fin_cap;
  // parked pairs / tails
  RegRec* regs;  int64_t regs_cap;
  PairReg* pair_reg;             // [n_pairs]
  TaskRec* tasks; int64_t tasks_cap;   // [kExtClasses][tasks_cap]
  uint32_t* ext_arena; int64_t ext_arena_cap;
  int32_t* ovf_read; int32_t* ovf_hap; int64_t ovf_cap;
  int32_t* cold_read; int32_t* cold_hap;   // [n_pairs] pairs the lean chain kernel left to k_chain_cold
  // k_ext_big scratch
  uint8_t* dir_scratch; int64_t dir_per_warp;
  int32_t* bnd_scratch; int64_t bnd_per_warp;   // Hb/Fb boundary rows
  uint32_t* wcig_scratch; int wcig_cap;
  RadixScratch* rsx_scratch;     // [warps]
  // outputs
  AlnOut* aln; uint32_t* cigar_inline; uint32_t* cigar_arena; int64_t cigar_arena_cap;
  AssignOut* assign;
  long long* ctr;
};

#ifndef LGR_CHAIN_CARVEOUT
#define LGR_CHAIN_CARVEOUT -1  // cudaSharedmemCarveoutDefault: the chain kernel gains from every KB left to L1 (measured)
#endif
#ifndef LGR_CHAIN_MINB
#define LGR_CHAIN_MINB 9
#endif
#ifndef LGR_EXT_MINB
#define LGR_EXT_MINB 6
#endif
#ifndef LGR_FIN_MINB
#define LGR_FIN_MINB 6
#endif
// a device-path limit hit one pair: remember it for the batch and for the pair's group (the other
// groups of the batch stay valid, lgr_batch_out::grp_status)
__device__ __forceinline__ void flag_err(const Dev& D, int g, int bit) {
  atomicOr((unsigned long long*)&D.ctr[C_ERR], (unsigned long long)bit);
  if (g >= 0 && g < D.n_groups) atomicOr(&D.grp_err[g], bit);
}

__device__ __forceinline__ int ext_class(const DevParams& P, int m, int n) {
  if (n < m && n <= 16) {  // transposed: head = m query + n target codes, direction bytes [m + n - 1][n]
    const int seg = n <= 8 ? 8 : 16;
    if (m + n + n * (m + n - 1) <= kDirSmemPerWarp / (32 / seg)) return n <= 8 ? 3 : 4;
  }
  if (m > 16) return 2;
  const int T = prune_cols(P, m, n);
  const int seg = m <= 8 ? 8 : 16;
  const int need = kSegHead + m * (T + m - 1);          // staged codes + direction bytes [step][row]
  if (T + 1 > kSegHead - seg || need > kDirSmemPerWarp / (32 / seg)) return 2;
  return m <= 8 ? 0 : 1;
}

// queue one extension (lane 0 of the pair's warp); false when the queue is full
__device__ __forceinline__ bool push_task(const Dev& D, int reg, int side, int r, int h, int m, int n) {
  const int cls = ext_class(D.P, m, n);
  const long long ti = atomicAdd((unsigned long long*)&D.ctr[C_NTASK + cls], 1ULL);
  if (ti >= D.tasks_cap) return false;
  D.tasks[(size_t)cls * D.tasks_cap + ti] = TaskRec{reg, side, r, h};
  return true;
}

__device__ __forceinline__ void write_invalid(AlnOut* o) {
  o->valid = 0, o->score = 0, o->rs = 0, o->re = 0, o->qs = 0, o->qe = 0, o->rev = 0, o->dp_score = 0, o->dp_max = 0;
  o->mlen = 0, o->blen = 0, o->n_ambi = 0, o->nm = 0, o->n_cigar = 0, o->cigar_off = -1, o->n_regs = 0;
}

__device__ __forceinline__ void store_final(const Dev& D, int g, int64_t pair, const AlnOut& a, const uint32_t* cig, int nc) {
  AlnOut o = a;
  if (nc <= LGR_CIGAR_INLINE) {
    o.cigar_off = -1;
    uint32_t* dst = D.cigar_inline + pair * LGR_CIGAR_INLINE;
    if (nc == 1) dst[0] = cig[0];  // the common case: one M run
    else
      for (int i = 0; i < nc; ++i) dst[i] = cig[i];
  } else {
    const long long off = atomicAdd((unsigned long long*)&D.ctr[C_CIGARENA], (unsigned long long)nc);
    if (off + nc > D.cigar_arena_cap) {
      flag_err(D, g, E_CIG_ARENA);
      o.cigar_off = -2, o.n_cigar = 0;
    } else {
      o.cigar_off = (int32_t)off;
      for (int i = 0; i < nc; ++i) D.cigar_arena[off + i] = cig[i];
    }
  }
  // 64-byte record, 64-byte aligned: four 16-byte stores straight from registers (taking the record's
  // address would park it in local memory)
  uint4* dst = reinterpret_cast<uint4*>(&D.aln[pair]);
  dst[0] = make_uint4((uint32_t)o.valid, (uint32_t)o.score, (uint32_t)o.rs, (uint32_t)o.re);
  dst[1] = make_uint4((uint32_t)o.qs, (uint32_t)o.qe, (uint32_t)o.rev, (uint32_t)o.dp_score);
  dst[2] = make_uint4((uint32_t)o.dp_max, (uint32_t)o.mlen, (uint32_t)o.blen, (uint32_t)o.n_ambi);
  dst[3] = make_uint4((uint32_t)o.nm, (uint32_t)o.n_cigar, (uint32_t)o.cigar_off, (uint32_t)o.n_regs);
}

}  // namespace

#endif  // LANCET2_B200_LGR_DEV_CUH_
