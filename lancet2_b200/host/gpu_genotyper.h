// gpu_genotyper.h — host-side mirror of lancet::caller::Genotyper over the lgr_* C-ABI.
//
// Same call shape as the reference class (src/lancet/caller/genotyper.h:213-220):
//   Genotyper();   Result Genotype(Haplotypes, Reads, VariantSet const&);
// with plain std types instead of abseil / cbdg types so that it builds without the
// reference's dependencies; INTEGRATION.md shows the three-line glue that maps
// cbdg::Read / RawVariant onto ReadIn / VariantIn inside Lancet2.
//
// What runs where:
//   GPU  (lgr_genotype_batch): ResetData + AlignToAllHaplotypes + AssignReadToAlleles
//        (genotyper.cpp:243-321, 376-411) for every read of every queued Genotype() call
//   host (this file): AddToTable → VariantSupport::AddEvidence (genotyper.cpp:423-456,
//        variant_support.cpp:23-67), in the reference's read order, because it needs the
//        per-process salted absl::HashOf(qname) and string_view sample names
// Errors: any non-zero lgr code becomes std::runtime_error — the reference's
// terminate-on-exception behaviour (core/async_worker.cpp:73-97) is preserved, there is no
// CPU fallback.
#ifndef LANCET2_B200_HOST_GPU_GENOTYPER_H_
#define LANCET2_B200_HOST_GPU_GENOTYPER_H_

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <functional>
#include <future>
#include <memory>
#include <mutex>
#include <string>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/lancet_gpu_realign.h"

namespace lancet_gpu {

using AlleleIndex = std::uint8_t;  // variant_support.h:32
enum class Strand : bool { FWD, REV };  // per_allele_data.h:12

// what Genotype() reads from a cbdg::Read (cbdg/read.h:100-117)
struct ReadIn {
  std::string_view qname;        // QnameView()
  std::string_view seq;          // SeqView()
  const std::uint8_t* qual;      // QualView().data(), seq.size() entries
  std::string_view sample_name;  // SampleName()
  std::int64_t start0;           // StartPos0()
  std::int64_t insert_size;      // InsertSize()
  std::uint16_t sam_flag;        // Flag(): 0x10 reverse strand, 0x2 proper pair
  std::uint8_t map_qual;         // MapQual()
  bool is_soft_clipped;          // IsSoftClipped()
};

// what ExtractHapBounds reads from a RawVariant (genotyper.cpp:329-352; raw_variant.h:64-80,
// alt_allele.h:29-52)
struct AltAlleleIn {
  std::size_t seq_len;                                             // mSequence.size()
  std::vector<std::pair<std::size_t, std::size_t>> hap_start0;     // mLocalHapStart0Idxs (hap → start)
  std::int64_t length = 0;                                         // mLength (alt_allele.h:50), for ASMD only
};
struct VariantIn {
  const void* key;                 // RawVariant const* (the Result key)
  std::size_t local_ref_start0;    // mLocalRefStart0Idx
  std::size_t ref_allele_len;      // mRefAllele.size()
  std::vector<AltAlleleIn> alts;   // mAlts, in order
};

struct ReadEvidence {  // variant_support.h:64-84
  std::int64_t mInsertSize, mAlignmentStart;
  double mAlnScore, mFoldedReadPos;
  std::uint32_t mRnameHash, mRefNm, mOwnHapNm, mAssignedHaplotypeId;
  AlleleIndex mAllele;
  Strand mStrand;
  std::uint8_t mBaseQual, mMapQual;
  bool mIsSoftClipped, mIsProperPair;
};

struct PerAlleleData {  // per_allele_data.h:25-73
  std::unordered_map<std::uint32_t, Strand> mNameHashes;
  std::vector<std::uint8_t> mFwdBaseQuals, mRevBaseQuals, mMapQuals;
  std::vector<double> mAlnScores, mProperPairIsizes, mFoldedReadPositions, mRefNmValues, mOwnHapNmValues;
  std::vector<std::int64_t> mAlignmentStarts;
  std::vector<std::uint32_t> mHaplotypeIds;
  std::size_t mSoftClipCount = 0;
};

class VariantSupport {  // the AddEvidence half of variant_support.h
 public:
  void AddEvidence(ReadEvidence const& evidence);  // variant_support.cpp:23-67
  [[nodiscard]] const std::vector<PerAlleleData>& AlleleData() const noexcept { return mAlleleData; }

 private:
  std::vector<PerAlleleData> mAlleleData;
};

class SupportArray {  // support_array.h:25-43
 public:
  struct NamedSupport {
    std::string_view mSampleName;
    std::unique_ptr<VariantSupport> mData;
  };
  VariantSupport& FindOrCreate(std::string_view sample_name);  // support_array.cpp:19-28
  [[nodiscard]] auto begin() const { return mItems.begin(); }
  [[nodiscard]] auto end() const { return mItems.end(); }

 private:
  std::vector<NamedSupport> mItems;
};

using Result = std::unordered_map<const void*, SupportArray>;  // genotyper.h:217

// hash of the read name used for the dedup key; inside Lancet2 pass
//   [](std::string_view q) { return static_cast<std::uint32_t>(absl::HashOf(q)); }
using NameHashFn = std::function<std::uint32_t(std::string_view)>;

// One payload of Genotyper::Genotype (borrowed for the duration of the call that consumes it)
struct GenotypeJob {
  const std::string* haps;
  std::size_t n_haps;
  const ReadIn* reads;
  std::size_t n_reads;
  const VariantIn* variants;
  std::size_t n_variants;
  // mm_mapopt_update's latch (genotyper.cpp:263-266) of the logical worker this payload belongs to:
  // 0 = not latched yet (set from this payload's REF haplotype), NULL = the calling thread's own latch
  std::int32_t* mid_occ_latch = nullptr;
};

// ---------------------------------------------------------------------------------------------
// SURVEY.md §8f #2: the evidence as SoA columns for the device FORMAT math (lgr_format_metrics)
// ---------------------------------------------------------------------------------------------
// Identity of one support = one VariantSupport of the reference's Result (variant → sample).
struct SupportKey {
  const void* variant;      // RawVariant const*
  std::string_view sample;  // aliases ReadIn::sample_name, like SupportArray's names (support_array.h:25-29)
};

// AddToTable (genotyper.cpp:423-456) with the evidence written as lgr_evidence_in columns instead
// of per-allele vectors: supports in (job, variant, sample-first-seen) order, records of a support
// in read order — the append order AddEvidence sees — so the device dedup (first seen per allele
// and name hash) keeps exactly the records VariantSupport would keep.
class EvidenceColumns {
 public:
  void Clear();
  void AppendJob(const GenotypeJob& job, const lgr_assign* assign, const NameHashFn& name_hash);
  [[nodiscard]] const lgr_evidence_in& In();
  [[nodiscard]] const std::vector<SupportKey>& Keys() const noexcept { return mKeys; }
  [[nodiscard]] std::size_t NumSupports() const noexcept { return mKeys.size(); }

 private:
  std::vector<SupportKey> mKeys;
  std::vector<std::int64_t> mSupBegin{0}, mInsertSize, mAlnStart;
  std::vector<std::int32_t> mNumAlleles, mVariantLen, mTotalHaps;
  std::vector<double> mAlnScore, mFoldedPos;
  std::vector<std::uint32_t> mRnameHash, mRefNm, mOwnHapNm, mHapId;
  std::vector<std::uint8_t> mAllele, mFlags, mBaseQual, mMapQual;
  lgr_evidence_in mIn{};
};

// Owner of one lgr_fmt_ctx: every FORMAT accessor of every support in one device call
// (variant_support.cpp:140-335 → k_fmt_dedup / k_fmt_metrics).  Throws std::runtime_error on any
// non-zero return code, like the rest of the adapter; no CPU fallback.
class GpuFormatMetrics {
 public:
  explicit GpuFormatMetrics(int device_ordinal = 0);
  ~GpuFormatMetrics();
  GpuFormatMetrics(const GpuFormatMetrics&) = delete;
  GpuFormatMetrics& operator=(const GpuFormatMetrics&) = delete;
  std::vector<lgr_format> Compute(EvidenceColumns& columns, float* ms_kernels = nullptr);

 private:
  lgr_fmt_ctx* mCtx = nullptr;
};

// One Genotype() payload already in the C-ABI's SoA layout, offsets relative to the job.  Built by
// the thread that owns the payload (the per-read work — copies, X31 name hash, ExtractHapBounds'
// dense table — parallelises over the workers); PackedBatch then only concatenates blocks.
struct PackedJob {
  std::vector<std::uint8_t> hap_bases, read_bases, read_quals;
  std::vector<std::int64_t> hap_off, read_off, var_hap_off;  // each starts at 0
  std::vector<std::uint32_t> x31;
  std::vector<std::int32_t> var_start, var_len;
  std::vector<std::int8_t> var_allele;
  std::size_t n_haps = 0, n_reads = 0, n_variants = 0;
  void Build(const GenotypeJob& job);  // ResetData's inputs + ExtractHapBounds (genotyper.cpp:243-267, 329-352)
};

// SoA staging of many GenotypeJobs in the C-ABI's layout (pinned host memory when available) and
// the host half of the path: AddToTable from the returned lgr_assign records.
class PackedBatch {
 public:
  PackedBatch() = default;
  ~PackedBatch();
  PackedBatch(const PackedBatch&) = delete;
  PackedBatch& operator=(const PackedBatch&) = delete;
  // ResetData's inputs + ExtractHapBounds' dense table for every job (genotyper.cpp:243-267, 329-352)
  void Pack(const GenotypeJob* jobs, std::size_t n_jobs, std::int32_t latched_mid_occ);
  // the same from payloads their owners have packed already (block copies + offset rebasing only)
  void PackPrepared(const PackedJob* const* jobs, std::size_t n_jobs, std::int32_t latched_mid_occ);
  [[nodiscard]] const lgr_batch_in& In() const noexcept { return mIn; }
  [[nodiscard]] lgr_batch_out& Out() noexcept { return mOut; }
  [[nodiscard]] std::int64_t Pairs() const noexcept { return mPairs; }
  // the lgr_assign records of job j ([read][variant], n_reads * n_variants of them)
  [[nodiscard]] const lgr_assign* JobAssign(std::size_t j) const noexcept { return mAssign.p + mJobAsg[j]; }
  // AddToTable (genotyper.cpp:423-456) for one job, reads in the caller's order
  static Result BuildResult(const GenotypeJob& job, const lgr_assign* assign, const NameHashFn& name_hash);

 private:
  template <typename T>
  struct Buf {  // grow-only; lgr_alloc_pinned with a malloc fallback
    T* p = nullptr;
    std::size_t n = 0, cap = 0;
    bool pinned = false;
  };
  template <typename T> static void Reserve(Buf<T>& b, std::size_t n);
  template <typename T> static void Push(Buf<T>& b, T v);
  template <typename T> static void Append(Buf<T>& b, const T* src, std::size_t n);
  template <typename T> static void Free(Buf<T>& b);
  Buf<std::int32_t> mGhb, mGrb, mGvb, mGmid, mVarStart, mVarLen;
  Buf<std::int64_t> mHapOff, mReadOff, mVarHapOff;
  Buf<std::uint8_t> mHapBases, mReadBases, mReadQuals;
  Buf<std::uint32_t> mX31;
  Buf<std::int8_t> mVarAllele;
  Buf<lgr_assign> mAssign;
  std::vector<std::int64_t> mJobAsg;
  lgr_batch_in mIn{};
  lgr_batch_out mOut{};
  std::int64_t mPairs = 0;
};

class GpuGenotyper {
 public:
  explicit GpuGenotyper(int device_ordinal = 0, const lgr_params* params = nullptr);
  ~GpuGenotyper();
  GpuGenotyper(const GpuGenotyper&) = delete;
  GpuGenotyper& operator=(const GpuGenotyper&) = delete;

  // drop-in for Genotyper::Genotype (genotyper.cpp:224-235): one group, synchronous
  [[nodiscard]] Result Genotype(const std::string* haps, std::size_t n_haps, const ReadIn* reads, std::size_t n_reads,
                                const VariantIn* variants, std::size_t n_variants, const NameHashFn& name_hash);

  // many Genotype() payloads in ONE device batch (what fills a B200); results in job order
  [[nodiscard]] std::vector<Result> GenotypeMany(const std::vector<GenotypeJob>& jobs, const NameHashFn& name_hash);

  [[nodiscard]] const lgr_stats& LastStats() const noexcept { return mStats; }

  // lgr_set_graph_mode on this genotyper's context: every later call runs its device pass as one CUDA graph
  // (same results, one launch per call instead of a dozen)
  void SetGraphMode(bool on);

 private:
  lgr_ctx* mCtx = nullptr;
  lgr_params mParams;
  std::int32_t mLatchedMidOcc = 0;  // mm_mapopt_update latches mid_occ from the first index it sees
  lgr_stats mStats{};
  std::unique_ptr<PackedBatch> mBatch;
};

// Cross-thread batcher (SURVEY.md §8f #1): the reference runs one Genotyper per worker thread
// (core/variant_builder.h:94, core/pipeline_executor.cpp:174-197) and each Genotype() call
// carries only ~10^3-10^4 pairs.  One GenotypeBatcher per GPU lets all workers share the device.
//
// Data path (north_star: "batches (read, haplotype) pairs across many windows into ... 2-bit-packed
// SoA buffers"): the ENQUEUING worker packs its payload once, straight into the pinned slab that is
// currently being filled (lgr_pack.h: bit planes, quality dictionary, ExtractHapBounds' table, X31
// name hashes) — a reservation under the lock, the packing itself outside it.  The batcher thread
// only seals a slab (appends the directory) and hands it to lgr_submit_packed: ONE host→device copy
// per device batch, every derived array built on the device.  Up to `depth` slabs are in flight;
// completion arrives through lgr_set_notify (no polling).  The collecting worker reads its
// lgr_assign records in place from the slab's pinned result block and runs AddToTable; the slab
// returns to the pool when its last payload has been collected.
//
// Failure isolation (mm_map never refuses, genotyper.cpp:387-393; an exception terminates Lancet2,
// core/async_worker.cpp:73-97): a payload beyond the device path's static caps throws in ITS
// Enqueue and never joins a batch; a device-side cap that hits one payload's pairs is reported per
// group (lgr_batch_out::grp_status), that payload alone is re-run in a batch of its own, and only if
// that fails too does its Collect throw.  Every other payload of the batch is unaffected.
//
// mid_occ latch (mm_mapopt_update, genotyper.cpp:263-266): the reference latches per Genotyper, i.e.
// per worker thread, from the first REF haplotype that worker sees.  Here the latch is per CALLING
// THREAD (or per explicit GenotypeJob::mid_occ_latch), computed once from that thread's first
// payload — independent of how payloads from different threads meet in a device batch and of the
// GPU they are routed to, hence deterministic for a deterministic window-to-worker schedule.
class GenotypeBatcher {
 public:
  struct Options {
    int device = 0;
    int depth = 4;                       // device batches in flight (<= LGR_MAX_INFLIGHT); 4 measured best on one B200
    std::int64_t max_pairs = 1 << 18;    // (read, haplotype) pairs per device batch (the kernels are saturated well below;
                                         // the reserved arena covers a batch of this size)
    std::size_t max_jobs = 8192;         // Genotype() payloads per device batch
    int linger_us = 100;                 // idle GPU: wait this long for more workers to arrive before launching
    int max_wait_us = 400;               // busy GPU: a slab waits at most this long for min_pairs_busy
    std::int64_t min_pairs_busy = 98304; // busy GPU: pairs that make a batch worth its launch overhead (measured: 16 workers x 32
                                         // payloads in flight give 98-111 M pairs/s with 96 K, 41-96 M with 48 K)
    std::size_t slab_bytes = 32u << 20;  // pinned staging per slab (a payload larger than this travels alone)
    std::size_t result_records = 1u << 18;  // lgr_assign records per pinned result block: a slab is sealed before it would
                                            // hold more (only a single payload beyond this grows a block)
    std::int64_t arena_reserve_bytes = 1ll << 30;    // device arena reserved per in-flight slot at construction (lgr_reserve;
                                                     // a cfg2-sized batch of 233 K pairs needs 0.75 GiB, mostly per-warp scratch):
                                                     // a regrow inside the steady state synchronises the whole device
    int direct_blocking_callers = 8;  // Genotype() (the blocking call shape) runs on a device context owned by the calling
                                      // thread while at most this many callers are inside it: no thread hand-offs.  Further
                                      // callers go through the batcher and are coalesced.  Measured calls/s with 1 / 4 / 8 /
                                      // 16 blocking threads: 2.2 K / 7.6 K / 10.7 K / 11.8 K, against 1.3 K / 3.6 K / 6.7 K /
                                      // 10.5 K with everything through the batcher (0) and 3.9 K at 16 threads with
                                      // everything direct (the callers then contend inside the driver)
    bool direct_graph = false;        // the direct contexts above run their device pass as one CUDA graph
                                      // (lgr_set_graph_mode): same results, one launch per call instead of a dozen
    const lgr_params* params = nullptr;
  };
  struct Counters {
    std::uint64_t batches = 0, jobs = 0, pairs = 0, max_jobs_in_batch = 0, retried_alone = 0, h2d_bytes = 0, d2h_bytes = 0;
    std::uint64_t ns_pack = 0;     // worker time: sizing + packing into the slab (summed over workers)
    std::uint64_t ns_submit = 0;   // batcher thread: seal + lgr_submit_packed
    std::uint64_t ns_seal_wait = 0;  // ... of which waiting for workers that were still writing their record
    std::uint64_t ns_wait = 0;     // batcher thread: lgr_wait (statistics, rare overflow pass)
    std::uint64_t ns_deliver = 0;  // worker time: AddToTable (summed over workers)
    std::uint64_t graph_launches = 0;  // direct calls whose device pass ran as a CUDA graph (Options::direct_graph)
  };
  GenotypeBatcher(const Options& opt, NameHashFn name_hash);
  ~GenotypeBatcher();  // drains what is queued, then joins
  GenotypeBatcher(const GenotypeBatcher&) = delete;
  GenotypeBatcher& operator=(const GenotypeBatcher&) = delete;

  // thread-safe drop-in for Genotyper::Genotype (genotyper.cpp:224-235); blocks the calling worker
  [[nodiscard]] Result Genotype(const std::string* haps, std::size_t n_haps, const ReadIn* reads, std::size_t n_reads,
                                const VariantIn* variants, std::size_t n_variants);
  [[nodiscard]] Result Genotype(const GenotypeJob& job);  // the same, with the job's own mid_occ latch if it names one

  // The two halves of Genotype() for a caller that has split ProcessWindow (SURVEY.md §8f #1):
  // Enqueue packs and returns at once, the worker goes on to assemble its next window, and Collect
  // (on any thread) waits for the device and runs AddToTable.  The job's buffers are borrowed until
  // Collect returns.  With many windows enqueued per worker the batches fill the GPU.
  struct Slab;
  struct ResultBlock;
  struct Ticket {
    GenotypeJob job{};
    ResultBlock* res = nullptr;
    std::uint32_t slot = 0;
    std::shared_ptr<std::vector<lgr_assign>> alone;  // results of a payload that travelled alone (larger than a slab)
  };
  [[nodiscard]] Ticket Enqueue(const GenotypeJob& job);
  [[nodiscard]] Result Collect(Ticket& ticket);
  // the lgr_assign records of a ticket ([read][variant]) without AddToTable; valid until Release
  [[nodiscard]] const lgr_assign* WaitAssign(Ticket& ticket, std::vector<lgr_assign>* retry_storage);
  void Release(Ticket& ticket);
  [[nodiscard]] Counters Stats();
  [[nodiscard]] const lgr_params& Params() const noexcept { return mParams; }

 private:
  void Run();
  void SealAndSubmit(Slab* s);
  void Complete(Slab* s);
  Slab* TakeFreeSlabLocked(std::unique_lock<std::mutex>& lk, std::size_t need_bytes);
  std::int32_t LatchFor(const GenotypeJob& job);
  std::vector<lgr_assign> RunAlone(const GenotypeJob& job, std::int32_t mid_occ);
  struct DirectSlot;                     // per calling thread: device context + pinned staging of the blocking path
  DirectSlot* DirectFor();
  Result GenotypeDirect(const GenotypeJob& job);
  std::mutex mDirectMu;
  std::atomic<int> mBlockingCallers{0};
  std::vector<std::unique_ptr<DirectSlot>> mDirect;
  static void OnDeviceDone(void* self, lgr_ticket ticket);
  Options mOpt;
  NameHashFn mNameHash;
  lgr_ctx* mCtx = nullptr;       // batcher thread only
  lgr_ctx* mAuxCtx = nullptr;    // latch computation and single-payload re-runs, under mAuxMu
  std::mutex mAuxMu;
  lgr_params mParams;
  std::uint64_t mUid = 0;        // key of the per-thread latch
  std::mutex mMu;
  std::condition_variable mCv;       // batcher thread: work arrived / a batch finished on the device
  std::condition_variable mFreeCv;   // workers waiting for a free slab
  std::condition_variable mDoneCv;   // workers waiting for their slab's results
  std::vector<std::unique_ptr<Slab>> mSlabs;
  std::vector<Slab*> mFree;
  std::vector<std::unique_ptr<ResultBlock>> mResults;
  std::vector<ResultBlock*> mFreeResults;
  Slab* mOpen = nullptr;             // the slab being filled
  std::deque<Slab*> mSealable;       // full slabs waiting for a device slot, in order
  std::deque<Slab*> mInFlight;       // submitted, oldest first
  int mLingerCredit = 8;              // batches still allowed the idle-GPU linger (see Run)
  std::uint32_t mDeviceDone = 0;     // tickets whose device work has finished (bit per ticket)
  bool mStop = false;
  Counters mCounters;
  std::thread mThread;
};

// Several GPUs of one box (SURVEY.md §8e): one GenotypeBatcher per device behind one entry point.
// Whole Genotype() payloads are routed — never split, the per-variant arg-max needs all haplotype
// pairs of a read together — to the device with the least outstanding work (cost = reads x
// total haplotype length, the same estimate lancet2_b200/dispatch.py uses).  No collective: the
// results come back to the caller that enqueued them, and output order is the caller's order.
class GenotypeDispatcher {
 public:
  GenotypeDispatcher(const std::vector<int>& devices, NameHashFn name_hash, GenotypeBatcher::Options base = {});
  struct Ticket {
    std::size_t device_slot = 0;
    std::int64_t cost = 0;
    GenotypeBatcher::Ticket inner;
  };
  [[nodiscard]] Ticket Enqueue(const GenotypeJob& job);
  [[nodiscard]] Result Collect(Ticket& ticket);
  // thread-safe drop-in for Genotyper::Genotype (genotyper.cpp:224-235)
  [[nodiscard]] Result Genotype(const std::string* haps, std::size_t n_haps, const ReadIn* reads, std::size_t n_reads,
                                const VariantIn* variants, std::size_t n_variants);
  [[nodiscard]] std::size_t Devices() const noexcept { return mBatchers.size(); }
  [[nodiscard]] GenotypeBatcher::Counters Stats(std::size_t device_slot) { return mBatchers[device_slot]->Stats(); }
  static std::int64_t Cost(const GenotypeJob& job);

 private:
  std::vector<std::unique_ptr<GenotypeBatcher>> mBatchers;
  std::unique_ptr<std::atomic<std::int64_t>[]> mOutstanding;
  std::uint64_t mUid = 0;  // key of the per-thread mid_occ latch
};

}  // namespace lancet_gpu

#endif  // LANCET2_B200_HOST_GPU_GENOTYPER_H_
