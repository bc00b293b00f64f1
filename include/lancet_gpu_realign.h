/*
 * lancet_gpu_realign.h — C ABI of the B200 read→haplotype realignment path.
 *
 * This is the drop-in boundary for the hot path of nygenome/Lancet2's
 * `caller::Genotyper`.  The reference has no FFI layer; the seam is the C++
 * member `Genotyper::Genotype(haps, reads, variant_set)`
 * (reference: src/lancet/caller/genotyper.h:213-220, genotyper.cpp:224-235).
 * One *group* below is the payload of exactly one `Genotype()` call (one graph
 * component of one window): P haplotypes, R reads, V variants.  A *batch* is
 * many groups, so that windows from many worker threads fill one GPU.
 *
 * What each entry point replaces in the reference:
 *   lgr_create            Genotyper::Genotyper()            genotyper.cpp:89-191
 *                         (mm_set_opt + the 10 option overrides, mm_tbuf_init)
 *   lgr_genotype_batch    Genotyper::ResetData              genotyper.cpp:243-267
 *                         + AlignToAllHaplotypes (mm_map)   genotyper.cpp:376-411
 *                         + AssignReadToAlleles             genotyper.cpp:269-321
 *                         + ScoreReadAtVariant              combined_scorer.cpp:60-108
 *                         + ComputeLocalScore               local_scorer.cpp:166-279
 *   lgr_hap_mid_occ       mm_mapopt_update (mid_occ latch)  genotyper.cpp:263-266
 *   lgr_destroy           ~Genotyper (mm_idx_destroy, mm_tbuf_destroy)
 *                                                           genotyper.h:226-250
 * `Genotyper::AddToTable` (genotyper.cpp:423-456) stays on the host: it needs
 * absl's per-process salted hash and string_view sample names; the adapter in
 * lancet2_b200/host/ performs it from the lgr_assign records, in read order.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on
 * success and a negative LGR_E_* code on failure (no CPU fallback exists — a
 * missing GPU is an error).  All buffers are caller-owned HOST memory unless a
 * function name ends in `_dev`.  A context is bound to one GPU and may be used
 * by one thread at a time; use one context per GPU/worker.
 */
#ifndef LANCET_GPU_REALIGN_H_
#define LANCET_GPU_REALIGN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGR_ABI_VERSION 2

/* error codes */
#define LGR_OK 0
#define LGR_E_ARG (-1)            /* bad argument / inconsistent batch      */
#define LGR_E_CUDA (-2)           /* CUDA runtime failure (see lgr_last_error) */
#define LGR_E_NO_DEVICE (-3)      /* no usable GPU                          */
#define LGR_E_LIMIT (-4)          /* a sequence exceeds a compile-time cap  */
#define LGR_E_CIGAR_OVERFLOW (-5) /* cigar overflow arena exhausted         */
#define LGR_E_NOMEM (-6)
#define LGR_E_BUSY (-7)           /* all LGR_MAX_INFLIGHT submission slots in use */
#define LGR_E_PARTIAL (-8)        /* some groups failed, the others are complete: see lgr_batch_out::grp_status */

/* compile-time caps of the device path (checked, never silently truncated) */
#define LGR_MAX_READ_LEN 1024
#define LGR_MAX_HAP_LEN 65535
#define LGR_MAX_INFLIGHT 4         /* lgr_submit tickets outstanding per ctx */
#define LGR_CIGAR_INLINE 8 /* u32 cigar ops stored inline per pair */

/*
 * Alignment / mapping parameters.  Defaults (lgr_default_params) are the
 * reference's effective minimap2 option set: mm_set_opt(0) defaults plus the
 * overrides in genotyper.cpp:109-190.
 */
typedef struct lgr_params {
  int32_t k, w;                /* minimizer k-mer / window: 11, 5 (genotyper.cpp:189-190) */
  int32_t a, b, q, e;          /* 1, 4, 12, 3 (scoring_constants.h:17-20)   */
  int32_t sc_ambi;             /* 1 (minimap2 default)                      */
  int32_t bw;                  /* 10000 (genotyper.cpp:140)                 */
  int32_t zdrop;               /* 100000 (genotyper.cpp:131)                */
  int32_t end_bonus;           /* 10000 (genotyper.cpp:181)                 */
  int32_t max_gap;             /* 200 (genotyper.cpp:158)                   */
  int32_t max_gap_ref;         /* 5000 (genotyper.cpp:159)                  */
  int32_t max_chain_skip;      /* 25                                        */
  int32_t max_chain_iter;      /* 5000                                      */
  int32_t min_cnt;             /* 3                                         */
  int32_t min_chain_score;     /* 40                                        */
  int32_t min_dp_max;          /* 80 = 40 * a(default 2), never recomputed  */
  int32_t mid_occ;             /* <=0: latch from first haplotype (mm_mapopt_update); else fixed */
  int32_t min_mid_occ;         /* 10                                        */
  int32_t max_mid_occ;         /* 1000000                                   */
  int32_t max_max_occ;         /* 4095                                      */
  int32_t occ_dist;            /* 500                                       */
  int32_t best_n;              /* 1 (genotyper.cpp:110)                     */
  int32_t seed;                /* 11                                        */
  float mid_occ_frac;          /* 2e-4                                      */
  float q_occ_frac;            /* 0.01                                      */
  float chain_gap_scale;       /* 0.8                                       */
  float chain_skip_scale;      /* 0.0                                       */
  float mask_level;            /* 0.5                                       */
  float pri_ratio;             /* 0.8                                       */
  float max_clip_ratio;        /* 1.0                                       */
  int32_t mask_len;            /* INT_MAX                                   */
  int32_t cigar_arena_ops;     /* capacity (u32 ops) of the overflow cigar arena per batch */
  int32_t reserved[7];
} lgr_params;

/*
 * One batch of G groups.  Index spaces:
 *   haplotypes 0..NH-1, group g owns [grp_hap_begin[g], grp_hap_begin[g+1]); its
 *     first haplotype is the REF haplotype (genotyper.h REF_HAP_IDX = 0).
 *   reads 0..NR-1, group g owns [grp_read_begin[g], grp_read_begin[g+1]), in
 *     the reference's ReadCollector order (it is the evidence-append order).
 *   variants 0..NV-1, group g owns [grp_var_begin[g], grp_var_begin[g+1]).
 *   per-(variant,haplotype) bounds: variant v of group g with P_g haplotypes
 *     owns var_start[var_hap_off[v] + h], h in [0,P_g)  (ExtractHapBounds,
 *     genotyper.cpp:329-352): var_allele = -1 when haplotype h does not carry
 *     the variant, 0 for the REF haplotype row, a+1 for ALT a.
 * Sequences are the ASCII strings the reference passes (hap: std::string,
 * genotyper.cpp:249; read: cbdg::Read::SeqPtr()); qualities are raw Phred
 * bytes; read_name_hash is minimap2's __ac_X31_hash_string(qname), see
 * lgr_x31_hash (mm_map mixes the read name into the hit-sort tie-break).
 */
typedef struct lgr_batch_in {
  int32_t n_groups;
  int32_t n_haps, n_reads, n_vars;
  const int32_t* grp_hap_begin;  /* [G+1] */
  const int32_t* grp_read_begin; /* [G+1] */
  const int32_t* grp_var_begin;  /* [G+1] */
  const int64_t* hap_off;        /* [NH+1] byte offsets into hap_bases  */
  const uint8_t* hap_bases;      /* ASCII                               */
  const int64_t* read_off;       /* [NR+1] byte offsets into read_bases/read_quals */
  const uint8_t* read_bases;     /* ASCII                               */
  const uint8_t* read_quals;     /* raw Phred                           */
  const uint32_t* read_name_hash;/* [NR]                                */
  const int64_t* var_hap_off;    /* [NV+1] offsets into var_* (P_g entries per variant) */
  const int32_t* var_start;      /* mVarStart per (variant,hap)         */
  const int32_t* var_len;        /* mVarLen   per (variant,hap)         */
  const int8_t* var_allele;      /* allele index or -1                  */
  const int32_t* grp_mid_occ;    /* [G] or NULL: per-group mid_occ (>0) overriding params.mid_occ */
} lgr_batch_in;

/* Result of mm_map(read, hap)[0] as consumed by AlignToAllHaplotypes
 * (genotyper.cpp:396-404), one per (read, haplotype-of-its-group) pair.
 * Pair index of read r (global) and local haplotype h: pair_off[r] + h, where
 * pair_off[r] = sum over earlier reads of their group's P (lgr_pair_offsets). */
typedef struct lgr_aln {
  int32_t valid;     /* 0: mm_map returned no hit → haplotype skipped (genotyper.cpp:390-393) */
  int32_t score;     /* mm_reg1_t::score   → Mm2AlnResult::mScore    */
  int32_t rs, re;    /* mm_reg1_t::rs/re   → mRefStart/mRefEnd       */
  int32_t qs, qe;    /* mm_reg1_t::qs/qe   → leading/trailing S in BuildCigar (genotyper.cpp:45-69) */
  int32_t rev;       /* mm_reg1_t::rev (never inspected by the reference) */
  int32_t dp_score;  /* mm_extra_t::dp_score */
  int32_t dp_max;    /* mm_extra_t::dp_max   */
  int32_t mlen, blen;/* mm_reg1_t::mlen/blen */
  int32_t n_ambi;    /* mm_extra_t::n_ambi   */
  int32_t nm;        /* hts::ComputeEditDistance(cigar, read, hap[rs,re)) (cigar_utils.h:48-94) */
  int32_t n_cigar;   /* core ops (without the S bookends)            */
  int32_t cigar_off; /* <0: ops are inline at cigar_inline[pair*LGR_CIGAR_INLINE]; else offset in cigar_arena */
  int32_t n_regs;    /* number of hits mm_map would return            */
} lgr_aln;

/* ReadAlleleAssignment (genotyper.h:152-171), one per (read, variant-of-its-
 * group): index asg_off[r] + v, asg_off[r] = sum over earlier reads of V_g. */
typedef struct lgr_assign {
  double local_score;     /* mLocalScore    */
  double local_identity;  /* mLocalIdentity */
  double folded_read_pos; /* mFoldedReadPos */
  int32_t global_score;   /* mGlobalScore   */
  uint32_t ref_nm;        /* mRefNm         */
  uint32_t own_hap_nm;    /* mOwnHapNm      */
  uint32_t hap_id;        /* mAssignedHaplotypeId */
  int8_t allele;          /* mAllele        */
  uint8_t base_qual;      /* mBaseQualAtVar */
  uint8_t assigned;       /* 0: read has no assignment for this variant */
  uint8_t pad[5];
} lgr_assign;

typedef struct lgr_batch_out {
  int64_t n_pairs;         /* capacity of aln / cigar_inline (in pairs)  */
  int64_t n_assign;        /* capacity of assign                         */
  lgr_aln* aln;            /* [n_pairs]                                  */
  uint32_t* cigar_inline;  /* [n_pairs * LGR_CIGAR_INLINE] BAM-encoded len<<4|op */
  uint32_t* cigar_arena;   /* [cigar_arena_cap] overflow ops             */
  int64_t cigar_arena_cap;
  int64_t cigar_arena_used;/* out */
  lgr_assign* assign;      /* [n_assign]                                 */
  int32_t* grp_status;     /* [n_groups] or NULL.  Per group: LGR_OK or the LGR_E_* code that hit one of ITS pairs (the
                              group's records are then undefined; every other group is complete and the call returns
                              LGR_E_PARTIAL).  NULL: any failing group fails the call with that code.  mm_map itself never
                              refuses an input (genotyper.cpp:387-393), so a host that wants the reference's behaviour
                              passes this array and re-submits or reports only the offending Genotype() payloads. */
  int32_t* grp_mid_occ;    /* [n_groups] or NULL: out, the mid_occ each group ran with (a worker latches the value of its
                              first group, mm_mapopt_update at genotyper.cpp:263-266)                                   */
} lgr_batch_out;

/* per-batch device timing + work counters (filled by lgr_genotype_batch) */
typedef struct lgr_stats {
  float ms_h2d, ms_kernels, ms_d2h; /* CUDA-event times on the ctx stream */
  float ms_k_index;                 /* encode + haplotype sketch/sort/mid_occ, with the read sketch beside it on the second stream */
  float ms_k_sketch;                /* k_read_filter (mm_seed_mz_flt), after the two streams join */
  float ms_k_map;                   /* the chain kernels (k_chain_lean + k_chain_cold) */
  float ms_k_ext;                   /* k_chain_overflow + k_ext_warp + k_finish_warp */
  float ms_k_assign;                /* k_assign */
  int64_t n_pairs, n_aligned;
  int64_t dp_cells;        /* extension-DP cells actually computed       */
  int64_t dp_cells_full;   /* cells of the un-pruned rectangles the reference computes */
  int64_t chain_evals;     /* anchor-pair evaluations in the chain DP    */
  int64_t n_anchors;
  int64_t h2d_bytes, d2h_bytes;
  int32_t kernel_launches;
  int32_t reserved;
} lgr_stats;

typedef struct lgr_ctx lgr_ctx;

int lgr_abi_version(void);
void lgr_default_params(lgr_params* p);
const char* lgr_strerror(int code);
/* last CUDA / argument error message of this ctx (or of creation when ctx==NULL) */
const char* lgr_last_error(const lgr_ctx* ctx);

/* minimap2's __ac_X31_hash_string over a NUL-terminated read name (khash.h). */
uint32_t lgr_x31_hash(const char* qname);

/* helper: fills pair_off[NR+1] / asg_off[NR+1] for a batch (host side). */
int lgr_pair_offsets(const lgr_batch_in* in, int64_t* pair_off, int64_t* asg_off);

int lgr_create(int device_ordinal, const lgr_params* params, lgr_ctx** out);
void lgr_destroy(lgr_ctx* ctx);

/* mid_occ that mm_mapopt_update would latch from this haplotype
 * (mm_idx_cal_max_occ with mid_occ_frac, clamped to [min_mid_occ, max_mid_occ]). */
int lgr_hap_mid_occ(lgr_ctx* ctx, const uint8_t* hap, int32_t hap_len, int32_t* mid_occ);

/* Synchronous: H2D of the batch, all kernels, D2H of the results. */
int lgr_genotype_batch(lgr_ctx* ctx, const lgr_batch_in* in, lgr_batch_out* out, lgr_stats* stats);

/* Asynchronous form of lgr_genotype_batch (SURVEY.md §8b/§8e: "one lgr_ctx + >=2 streams +
 * double-buffered staging per GPU; results return via ticket").  lgr_submit enqueues H2D,
 * kernels and D2H of one batch on a private slot (own streams and device buffers) and returns
 * at once; up to LGR_MAX_INFLIGHT batches may be outstanding, so the copies of one batch
 * overlap the kernels of another.  `in`/`out` buffers must stay valid (and should be pinned
 * for real overlap) until lgr_wait(ticket) returns; lgr_wait reports the batch's status and
 * statistics exactly as lgr_genotype_batch would.  Tickets may be waited in any order.
 * Replaces the synchronous per-window call at core/variant_builder.cpp:258-259 for a host that
 * pipelines windows (SURVEY.md §8f #1). */
typedef int32_t lgr_ticket;
int lgr_submit(lgr_ctx* ctx, const lgr_batch_in* in, lgr_batch_out* out, lgr_ticket* ticket);
int lgr_wait(lgr_ctx* ctx, lgr_ticket ticket, lgr_stats* stats);
/* Completion without polling: after lgr_set_notify, every later lgr_submit / lgr_submit_packed on this ctx ends with a
 * host callback (cudaLaunchHostFunc) that runs fn(user, ticket) on a CUDA-owned thread once the batch's last copy is
 * done; lgr_wait(ticket) then returns without blocking.  fn must not call into this library or CUDA.  NULL disables. */
typedef void (*lgr_notify_fn)(void* user, lgr_ticket ticket);
int lgr_set_notify(lgr_ctx* ctx, lgr_notify_fn fn, void* user);
/* Device memory is one grow-only arena per in-flight slot, and growing it (cudaFree + cudaMalloc) synchronises the whole
 * device.  lgr_reserve creates the first n_slots (<= LGR_MAX_INFLIGHT) submission slots now and gives each an arena of
 * at least arena_bytes, so that a pipelined caller pays neither inside its steady state; a batch that needs more still
 * grows its slot.  lgr_arena_bytes = device bytes this ctx currently holds in arenas (its own and its slots'). */
int lgr_reserve(lgr_ctx* ctx, int64_t arena_bytes, int n_slots);
int64_t lgr_arena_bytes(const lgr_ctx* ctx);
/* LGR_OK when a Genotype() payload whose longest haplotype / read have these lengths is inside the device path's static
 * caps for `params` (NULL = defaults), else LGR_E_LIMIT — the check lgr_submit applies to a whole batch, exposed so that
 * a host batching many payloads can refuse the one offender instead (no CUDA call, any thread). */
int lgr_check_limits(const lgr_params* params, int32_t max_hap_len, int32_t max_read_len);

/* Device-resident variant for kernel-only timing: upload once, run many times,
 * download when wanted.  `lgr_upload` keeps a device copy of `in` inside ctx. */
int lgr_upload(lgr_ctx* ctx, const lgr_batch_in* in);
int lgr_run_resident(lgr_ctx* ctx, lgr_stats* stats);
int lgr_download(lgr_ctx* ctx, lgr_batch_out* out);

/* Graph mode (off by default) for the blocking calls lgr_genotype_batch, lgr_genotype_packed and lgr_run_resident:
 * the device pass (its memsets, kernels and counter copy) is captured as a CUDA graph and launched as one, instead of
 * a dozen dependent launches (on a B200 this saves 0.015-0.02 ms of a 0.54 ms Genotype()-sized call).  Results and
 * lgr_stats are the same in both modes.  The input / result copies and the rare overflow pass stay outside the graph.
 * A context caches one executable per topology of the pass (plain or packed input, reads longer than 160 bases or
 * not, variants present or not, ...) and updates it for every batch of that topology, whatever its size.
 * lgr_submit / lgr_submit_packed never use it.  Counters since lgr_create: executables instantiated (first batch of a
 * topology, or an update the driver refused), executables updated in place, and graph launches; in graph mode
 * instantiated + updated = replayed = passes run in graph mode.  Any of the three pointers may be NULL. */
int lgr_set_graph_mode(lgr_ctx* ctx, int on);
int lgr_graph_counters(lgr_ctx* ctx, int64_t* instantiated, int64_t* updated, int64_t* replayed);

/* ------------------------------------------------------------------------------------------
 * Packed wire format (north_star: "2-bit-packed SoA buffers ... through a thin C-ABI layer").
 *
 * lgr_batch_in above is the plain form (ASCII strings, 13 arrays, one host->device copy each).  A host
 * that feeds the GPU from many worker threads packs every Genotype() payload ONCE, on the thread that
 * owns it, straight into one pinned slab, and the whole batch crosses PCIe in ONE copy:
 *
 *   slab  := group record, group record, ...  [directory]           (records 16-byte aligned)
 *   group record := lgr_group_rec_hdr | hap_len i32[P] | read_len u16[R] | name_hash u32[R]
 *                   | var_start i32[V*P] | var_len i32[V*P] | var_allele i8[V*P]
 *                   | hap planes | read planes | qualities | exceptions
 *   planes: bases as two bit planes per 32-base chunk {u32 lo, u32 hi} (A,C,G,T = 0..3, the nt4 code of
 *           minimap2's seq_nt4_table; every sequence starts a new chunk);
 *   exceptions: positions whose code byte is not plain A/C/G/T (N and other IUPAC letters, U: the
 *           minimap2 and Lancet2 code tables differ there, scoring_constants.h:48-74) as
 *           {u32 pos | 1<<31 for read space} + {u8 code} — lossless for any input byte;
 *   qualities: when the group uses at most 4 (16) distinct Phred values, 2 (4) bit planes per 32-base
 *           chunk indexing a 16-entry dictionary in the record header (binned instruments), else raw bytes.
 * Offsets, group/pair/assignment prefix sums and the work-item list are derived on the device
 * (k_unpack_scan / k_unpack_group); nothing but the slab is copied.
 *
 * lgr_packed_group_bytes / lgr_pack_group are pure host functions (no CUDA call, any thread).
 */
typedef struct lgr_group_desc {    /* one Genotype() payload as the caller holds it */
  int32_t n_haps, n_reads, n_vars;
  int32_t mid_occ;                  /* > 0: the worker's latched mid_occ; <= 0: derive from this group's REF haplotype */
  const uint8_t* const* hap_seq;    /* [n_haps] ASCII, hap 0 = REF haplotype   */
  const int32_t* hap_len;           /* [n_haps]                                */
  const uint8_t* const* read_seq;   /* [n_reads] ASCII                         */
  const uint8_t* const* read_qual;  /* [n_reads] raw Phred, read_len entries   */
  const int32_t* read_len;          /* [n_reads]                               */
  const uint32_t* read_name_hash;   /* [n_reads] lgr_x31_hash(qname)           */
  const int32_t* var_start;         /* [n_vars * n_haps] dense ExtractHapBounds table, variant-major */
  const int32_t* var_len;
  const int8_t* var_allele;
} lgr_group_desc;

typedef struct lgr_group_dir {     /* directory entry of one packed group (40 bytes) */
  uint64_t rec_off;                 /* byte offset of the group record in the slab (multiple of 16) */
  int32_t n_haps, n_reads, n_vars;
  int32_t hap_bases, read_bases;    /* total bases of the group                */
  int32_t mid_occ;
  int32_t max_hap_len, max_read_len;
} lgr_group_dir;

typedef struct lgr_group_rec_hdr { /* first 64 bytes of a group record */
  uint32_t magic;                   /* LGR_PACK_MAGIC */
  uint32_t qual_bits;               /* 2, 4 or 8 */
  uint32_t n_exc;
  uint32_t rec_bytes;               /* size of the record (multiple of 16) */
  uint8_t qual_lut[16];
  uint32_t off_hap_len, off_read_len, off_name_hash, off_var, off_hap_planes, off_read_planes, off_qual, off_exc;
} lgr_group_rec_hdr;
#define LGR_PACK_MAGIC 0x3252474cu /* "LGR2" */

typedef struct lgr_packed_in {
  int32_t n_groups;
  int32_t reserved;
  const void* slab;                 /* host memory (pinned for an asynchronous copy) */
  size_t slab_bytes;                /* bytes to copy                                 */
  const lgr_group_dir* dir;         /* [n_groups]; inside [slab, slab + slab_bytes) => ONE copy, else a second small one */
} lgr_packed_in;

/* bytes lgr_pack_group will write for this payload (upper bound, multiple of 16); 0 on a bad descriptor */
size_t lgr_packed_group_bytes(const lgr_group_desc* g);
/* pack one payload into dst[0..cap); fills *dir except rec_off (the caller places the record).  LGR_E_LIMIT when a
 * sequence exceeds LGR_MAX_READ_LEN / LGR_MAX_HAP_LEN, LGR_E_ARG on a bad descriptor or too small a buffer. */
int lgr_pack_group(const lgr_group_desc* g, void* dst, size_t cap, lgr_group_dir* dir);
/* the packed forms of lgr_genotype_batch / lgr_submit (same outputs, same tickets, same lgr_wait) */
int lgr_genotype_packed(lgr_ctx* ctx, const lgr_packed_in* in, lgr_batch_out* out, lgr_stats* stats);
int lgr_submit_packed(lgr_ctx* ctx, const lgr_packed_in* in, lgr_batch_out* out, lgr_ticket* ticket);
/* kernel-only timing on a packed batch: copy + unpack once, then lgr_run_resident / lgr_download */
int lgr_upload_packed(lgr_ctx* ctx, const lgr_packed_in* in);

/* Page-locked host memory for batch buffers (cudaMallocHost / cudaFreeHost): with pinned `in`/`out`
 * buffers the copies of lgr_submit are truly asynchronous.  NULL when it cannot be had (the
 * caller may fall back to ordinary memory; only the overlap is lost). */
void* lgr_alloc_pinned(size_t bytes);
void lgr_free_pinned(void* p);

/* raw CUDA stream (cudaStream_t) the ctx launches on, for external event timing */
void* lgr_stream(lgr_ctx* ctx);

/* ------------------------------------------------------------------------------------------
 * SURVEY.md §8f #2 — the direct consumer of the path: VariantSupport aggregation + FORMAT math.
 *
 * One *support* is one `caller::VariantSupport` object (one variant x one sample): a stream of
 * `VariantSupport::ReadEvidence` records in AddToTable's append order
 * (reference: src/lancet/caller/variant_support.h:64-84, genotyper.cpp:423-456).
 * lgr_format_metrics replaces, per support:
 *   VariantSupport::AddEvidence (first-seen read-name dedup)   variant_support.cpp:23-67
 *   FwdCount/RevCount/TotalAlleleCov, RawPosteriorBaseQual     variant_support.cpp:140-171, posterior_base_qual.cpp:13-40
 *   RmsMappingQual, StrandBiasLogOR, MeanAlnScore              variant_support.cpp:173-209
 *   SoftClipAsymmetry, FragLengthDelta                         variant_support.cpp:211-232
 *   MappingQualCohenD / ReadPosCohenD / BaseQualCohenD         variant_support.cpp:234-263, base/mann_whitney.h:13-65
 *   AlleleMismatchDelta, ComputeFSSE, ComputeAHDD, ComputeHSE  variant_support.cpp:265-291, variant_support.h:362-412
 *   ComputePLs / ComputeGQ                                     variant_support.cpp:294-310, genotype_likelihood.cpp:109-163
 *   ComputeContinuousMixtureLods                               variant_support.cpp:312-335, genotype_likelihood.cpp:165-205
 * Counts and the three Mann-Whitney effect sizes are exact by construction (integer rank
 * statistics); PL/GQ are rounded lgamma differences and equal the reference's in every test; the
 * other f64 metrics are tree sums with CUDA's libm (log10/log2/log/lgamma/pow), i.e. equal to the
 * reference within 1e-9 relative (the reference's own tests use 1e-6, and its entropy sums run
 * in abseil's salted hash-map order, so it does not reproduce its own last bits either).
 * Own context (device buffers + stream), independent of lgr_ctx; a context is bound to one GPU
 * and may be used by one thread at a time (one per worker, like lgr_ctx); the call returns when
 * `out` is filled.  No CPU fallback: lgr_format_create returns LGR_E_NO_DEVICE without a GPU.
 */
#define LGR_FMT_MAX_ALLELES 8
#define LGR_FMT_MAX_GENOTYPES 36 /* K(K+1)/2 at K = 8 */
/* lgr_evidence_in::flags bits */
#define LGR_EV_REV 1u         /* ReadEvidence::mStrand == REV   */
#define LGR_EV_SOFTCLIP 2u    /* ReadEvidence::mIsSoftClipped   */
#define LGR_EV_PROPER_PAIR 4u /* ReadEvidence::mIsProperPair    */
/* lgr_format::valid bits (std::optional has a value) */
#define LGR_FMT_HAS_FLD 1u
#define LGR_FMT_HAS_MQCD 2u
#define LGR_FMT_HAS_RPCD 4u
#define LGR_FMT_HAS_BQCD 8u
#define LGR_FMT_HAS_ASMD 16u
#define LGR_FMT_HAS_FSSE 32u
#define LGR_FMT_HAS_AHDD 64u
#define LGR_FMT_HAS_HSE 128u
/* The support's variant has more than LGR_FMT_MAX_ALLELES alleles (the reference's ComputePLs /
 * ComputeContinuousMixtureLods take any K; a record here has fixed arrays).  Such a support is NOT computed: its record
 * is zero except n_alleles and this bit, lgr_format_metrics returns LGR_E_PARTIAL, and every other support of the call is
 * complete.  The integrating host keeps such sites (STR loci with many ALTs) on its own VariantSupport code. */
#define LGR_FMT_WIDE 256u

typedef struct lgr_evidence_in {
  int32_t n_supports;
  int32_t reserved;
  int64_t n_evidence;
  const int64_t* sup_begin;        /* [S+1] support s owns evidence [sup_begin[s], sup_begin[s+1]) */
  const int32_t* sup_n_alleles;    /* [S] K: alleles of the variant (ComputePLs/ComputeContinuousMixtureLods argument) */
  const int32_t* sup_variant_len;  /* [S] AlleleMismatchDelta(variant_length) */
  const int32_t* sup_total_haps;   /* [S] ComputeHSE(total_haplotypes)        */
  const int64_t* insert_size;      /* [N] mInsertSize     */
  const int64_t* aln_start;        /* [N] mAlignmentStart */
  const double* aln_score;         /* [N] mAlnScore       */
  const double* folded_pos;        /* [N] mFoldedReadPos  */
  const uint32_t* rname_hash;      /* [N] mRnameHash      */
  const uint32_t* ref_nm;          /* [N] mRefNm          */
  const uint32_t* own_hap_nm;      /* [N] mOwnHapNm       */
  const uint32_t* hap_id;          /* [N] mAssignedHaplotypeId */
  const uint8_t* allele;           /* [N] mAllele (< K)   */
  const uint8_t* flags;            /* [N] LGR_EV_*        */
  const uint8_t* base_qual;        /* [N] mBaseQual       */
  const uint8_t* map_qual;         /* [N] mMapQual        */
} lgr_evidence_in;

typedef struct lgr_format {
  double raw_pbq[LGR_FMT_MAX_ALLELES];  /* RawPosteriorBaseQual(a) */
  double rms_mq[LGR_FMT_MAX_ALLELES];   /* RmsMappingQual(a)       */
  double mean_aln[LGR_FMT_MAX_ALLELES]; /* MeanAlnScore(a)         */
  double cmlod[LGR_FMT_MAX_ALLELES];    /* ComputeContinuousMixtureLods(K)[a] */
  double sb, sca;                       /* StrandBiasLogOR, SoftClipAsymmetry */
  double fld, mqcd, rpcd, bqcd, asmd, fsse, ahdd, hse; /* optionals: see `valid` */
  uint32_t fwd[LGR_FMT_MAX_ALLELES], rev[LGR_FMT_MAX_ALLELES]; /* FwdCount/RevCount */
  uint32_t soft_clip[LGR_FMT_MAX_ALLELES];                     /* PerAlleleData::mSoftClipCount */
  uint32_t pl[LGR_FMT_MAX_GENOTYPES];   /* ComputePLs(K), VCF order j*(j+1)/2+i */
  uint32_t gq;                          /* ComputeGQ(pl) */
  uint32_t n_alleles;                   /* K */
  uint32_t valid;                       /* LGR_FMT_HAS_* */
  uint32_t n_kept;                      /* evidence records that survived the read-name dedup */
} lgr_format;

typedef struct lgr_fmt_ctx lgr_fmt_ctx;
int lgr_format_create(int device_ordinal, lgr_fmt_ctx** out);
void lgr_format_destroy(lgr_fmt_ctx* ctx);
const char* lgr_format_last_error(const lgr_fmt_ctx* ctx);
/* H2D of the evidence, k_fmt_dedup + k_fmt_metrics, D2H of out[S]; ms_kernels (may be NULL) =
 * CUDA-event time of the two kernels. */
int lgr_format_metrics(lgr_fmt_ctx* ctx, const lgr_evidence_in* in, lgr_format* out, float* ms_kernels);

/* AddToTable on the device (SURVEY.md §8f #2, second step): the evidence of every (variant, sample) support is built
 * from the realignment's lgr_assign records — read straight from the device when dev_assign comes from
 * lgr_resident_assign() of a context on the same GPU, so the records never visit the host — plus the per-read fields
 * AddToTable takes from cbdg::Read (genotyper.cpp:423-456), in the order lancet_gpu::EvidenceColumns::AppendJob defines:
 * supports by (group, variant, first read of each sample), records in read order.  Then the FORMAT math runs as in
 * lgr_format_metrics.  read_name_hash replaces absl::HashOf(qname): the dedup only compares names of one support.
 * Returns the number of supports in *n_supports, their records in out[0..S) and sup_key[3 s + 0..2] = group, variant
 * (index in the batch) and sample id of support s; S <= n_vars * n_samples (out_cap must cover the actual S). */
typedef struct lgr_assign_batch {
  const lgr_assign* dev_assign;      /* DEVICE pointer (lgr_resident_assign), or NULL to upload host_assign     */
  const lgr_assign* host_assign;     /* [n_assign] host records, used when dev_assign is NULL                   */
  int64_t n_assign;                  /* sum over groups of reads x variants, group-major, read-major inside     */
  int32_t n_groups, n_reads, n_vars, n_samples; /* n_samples <= 32 */
  const int32_t* grp_read_begin;     /* [G+1] as in lgr_batch_in                                                */
  const int32_t* grp_var_begin;      /* [G+1]                                                                   */
  const int32_t* grp_n_haps;         /* [G]  ComputeHSE(total_haplotypes)                                       */
  const int32_t* var_n_alleles;      /* [NV] 1 + ALT alleles                                                    */
  const int32_t* var_len;            /* [NV] max |ALT length| (AlleleMismatchDelta)                             */
  const int64_t* read_insert_size;   /* [NR] */
  const int64_t* read_aln_start;     /* [NR] */
  const uint32_t* read_name_hash;    /* [NR] */
  const int32_t* read_sample;        /* [NR] dense sample id in [0, n_samples)                                  */
  const uint16_t* read_sam_flag;     /* [NR] 0x10 reverse strand, 0x2 proper pair                               */
  const uint8_t* read_map_qual;      /* [NR] */
  const uint8_t* read_soft_clipped;  /* [NR] */
} lgr_assign_batch;
int lgr_format_from_assign(lgr_fmt_ctx* ctx, const lgr_assign_batch* in, lgr_format* out, int32_t out_cap, int32_t* sup_key,
                           int32_t* n_supports, float* ms_kernels);
/* the device-resident lgr_assign records of the batch ctx last ran (lgr_genotype_*, lgr_run_resident); valid until the
 * next batch on ctx.  For lgr_assign_batch::dev_assign. */
int lgr_resident_assign(lgr_ctx* ctx, const lgr_assign** dev_assign, int64_t* n_assign);
/* test hook: the evidence columns lgr_format_from_assign built last, copied into dst's (caller-allocated) arrays */
int lgr_format_debug_evidence(lgr_fmt_ctx* ctx, lgr_evidence_in* dst);

/* Packed evidence (one block per window).  Lancet2 computes FORMAT fields per window on the worker thread right after
 * Genotype() (CollectSupportedCalls -> VariantCall); lgr_format_metrics copies every column of a call separately.  Here
 * each worker packs its window ONCE into a slab (pure host code, any thread), and a whole batch of windows crosses PCIe
 * in ONE copy:
 *
 *   slab  := block, block, ...  [directory]                        (blocks 16-byte aligned)
 *   block := lgr_fmt_blk_hdr | sup_begin i64[S+1] (window-local, [0, N]) | insert_size, aln_start, aln_score,
 *            folded_pos (8-byte)[N] | sup_n_alleles, sup_variant_len, sup_total_haps i32[S] | rname_hash, ref_nm,
 *            own_hap_nm, hap_id u32[N] | allele, flags, base_qual, map_qual u8[N]
 *   every section 16-byte aligned, zero padded; the order is that of the device arena of lgr_format_metrics.
 * The device scatters the blocks into that arena (sup_begin rebased to the batch) and runs the same two kernels, so a
 * window's records equal lgr_format_metrics on that window alone, byte for byte, whatever batch it travels in. */
#define LGR_FMT_MAGIC 0x31544d46u /* "FMT1" */
#define LGR_FMT_SECTIONS 16
typedef struct lgr_fmt_blk_hdr {   /* first 160 bytes of a block */
  uint32_t magic;                   /* LGR_FMT_MAGIC */
  int32_t n_supports;               /* S */
  int64_t n_evidence;               /* N */
  uint64_t rec_bytes;               /* size of the block (multiple of 16) */
  uint64_t reserved;
  uint64_t off[LGR_FMT_SECTIONS];   /* byte offset of each section from the block start, in the order above */
} lgr_fmt_blk_hdr;

typedef struct lgr_fmt_dir {       /* directory entry of one window (48 bytes) */
  uint64_t rec_off;                 /* byte offset of the block in the slab (multiple of 16) */
  int64_t n_evidence;               /* N of the block */
  int64_t ev_base;                  /* first record of the window in the batch: sum of n_evidence of the windows before */
  int32_t n_supports;               /* S of the block */
  int32_t sup_base;                 /* first support of the window in the batch: sum of n_supports of the windows before */
  int32_t n_wide;                   /* supports with more than LGR_FMT_MAX_ALLELES alleles */
  int32_t reserved[3];
} lgr_fmt_dir;

typedef struct lgr_fmt_packed_in {
  int32_t n_windows;
  int32_t reserved;
  const void* slab;                 /* host memory (pinned for an asynchronous copy) */
  size_t slab_bytes;                /* bytes to copy */
  const lgr_fmt_dir* dir;           /* [n_windows]; inside [slab, slab + slab_bytes) => ONE copy, else a second small one */
} lgr_fmt_packed_in;

/* bytes lgr_format_pack writes for this window (upper bound, multiple of 16); 0 on a malformed input (NULL, negative
 * sizes) */
size_t lgr_format_packed_bytes(const lgr_evidence_in* in);
/* Pack one window into dst[0..cap).  Validates what lgr_format_metrics validates (lgr_format.cu:358-379: negative sizes,
 * missing arrays, sup_begin spanning [0, N] and monotone, K >= 1, allele < K) and returns LGR_E_ARG for a malformed
 * window or a too small cap.  Fills *dir (may be NULL) except rec_off / sup_base / ev_base: the caller places the block.
 * Pure host code (no CUDA call), safe on any thread.  A window without supports packs as an empty block. */
int lgr_format_pack(const lgr_evidence_in* in, void* dst, size_t cap, lgr_fmt_dir* dir);
/* lgr_format_metrics over many packed windows: ONE H2D of the slab (plus the directory when it lies outside),
 * k_fmt_unpack scatters the blocks into the arena lgr_format_metrics builds, then the same k_fmt_dedup / k_fmt_metrics,
 * ONE D2H of out[S] for S = the windows' supports in directory order.  The host checks the directory only (magic,
 * counts and rec_bytes of each block's header, blocks inside the slab, sup_base / ev_base the prefix sums of the
 * counts): anything else is LGR_E_ARG before any CUDA call.  Records the device finds malformed (sup_begin outside
 * [0, N] or not monotone, K < 1, allele >= K, a wide support in a window whose n_wide is 0) are computed as empty
 * supports and the call returns LGR_E_ARG.  Wide supports as in lgr_format_metrics (LGR_FMT_WIDE, LGR_E_PARTIAL).
 * ms_kernels (may be NULL) = CUDA-event time of the three kernels. */
int lgr_format_metrics_packed(lgr_fmt_ctx* ctx, const lgr_fmt_packed_in* in, lgr_format* out, float* ms_kernels);
/* allocate every device buffer of a packed call of up to slab_bytes bytes (directory inside), n_supports supports and
 * n_evidence records now: lgr_format_metrics_packed then never regrows them within these sizes (a regrow frees and
 * allocates device memory, which synchronises the whole device) */
int lgr_format_reserve(lgr_fmt_ctx* ctx, int64_t slab_bytes, int32_t n_supports, int64_t n_evidence);
/* device bytes the context holds (all its buffers) */
int64_t lgr_format_device_bytes(const lgr_fmt_ctx* ctx);

/* ------------------------------------------------------------------------------------------
 * SURVEY.md §8f #3 (first half) — repeat detection over the sliding k-mers of reference windows.
 *
 * One *job* = one (sequence, k, max_mismatches) question: do two k-mers of the sequence, taken at different
 * offsets, differ in at most max_mismatches byte positions?  lgr_repeat_scan replaces, per job:
 *   cbdg::Graph::HasExactOrApproxRepeat   src/lancet/cbdg/graph.h:127-131   (max_mismatches = 2, once per k of the k-loop)
 *   VariantBuilder::ShouldSkipWindow      src/lancet/core/variant_builder.cpp:116-117 (HasExactRepeat at max_k)
 *   base::HasRepeat / HasExactRepeat      src/lancet/base/repeat.cpp:348-375 over base::SlidingView (sliding.h:17-34)
 * Bytes are compared raw, as the reference does; fewer than two k-mers give 0.  A sequence longer than
 * LGR_REPEAT_MAX_LEN is not computed: its answer is LGR_REPEAT_TOO_LONG and the call returns LGR_E_PARTIAL
 * (Lancet2's windows are <= 2.5 kb).  Own context, bound to one GPU, one thread at a time; the call returns when
 * has_repeat[0..n_jobs) is filled.  No CPU fallback: lgr_repeat_create returns LGR_E_NO_DEVICE without a GPU.
 * The k-mer insertion of Graph::AddNodes (the second half of §8f #3) is not part of this library.
 */
#define LGR_REPEAT_MAX_LEN 8192
#define LGR_REPEAT_TOO_LONG 255
typedef struct lgr_repeat_job {
  int64_t seq_off;          /* byte offset of the sequence in `seqs`            */
  int32_t seq_len;          /* bases                                            */
  int32_t k;                /* k-mer length (> 0)                               */
  int32_t max_mismatches;   /* 0 = exact repeat; Graph uses 2                   */
  int32_t reserved;
} lgr_repeat_job;
typedef struct lgr_rep_ctx lgr_rep_ctx;
int lgr_repeat_create(int device_ordinal, lgr_rep_ctx** out);
void lgr_repeat_destroy(lgr_rep_ctx* ctx);
const char* lgr_repeat_last_error(const lgr_rep_ctx* ctx);
/* H2D of the sequences and jobs, k_repeat_scan, D2H of one byte per job (0 / 1 / LGR_REPEAT_TOO_LONG).  Consecutive
 * jobs with the same seq_off, seq_len and max_mismatches (a window's k-loop) are answered together from shared mismatch
 * masks — keep them adjacent in `jobs`.  A batch of fewer such groups than the GPU has resident CTAs spreads each group's
 * diagonals over several CTAs (same answers);
 * ms_kernels (may be NULL) = CUDA-event time of the kernel. */
int lgr_repeat_scan(lgr_rep_ctx* ctx, const uint8_t* seqs, int64_t seq_bytes, const lgr_repeat_job* jobs, int32_t n_jobs,
                    uint8_t* has_repeat, float* ms_kernels);
/* allocate the device buffers of a batch of up to n_jobs jobs over up to seq_bytes bytes now: lgr_repeat_scan then never
 * regrows them within these sizes (a regrow frees and allocates device memory, which synchronises the whole device and
 * so stalls other work on it, e.g. a realignment batcher on the same GPU). */
int lgr_repeat_reserve(lgr_rep_ctx* ctx, int64_t seq_bytes, int32_t n_jobs);

#ifdef __cplusplus
}
#endif
#endif /* LANCET_GPU_REALIGN_H_ */
