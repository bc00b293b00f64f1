// gpu_format.h — thread-safe per-window FORMAT calculator over lgr_format_metrics_packed (SURVEY.md §8f #2).
//
// Lancet2 computes the FORMAT fields of a window on its worker thread right after Genotype()
// (CollectSupportedCalls -> VariantCall, one VariantSupport per variant and sample).  A FormatCalculator keeps that
// call shape: Compute() blocks the calling worker until its window's records are back.  Behind it:
//  * the worker sizes its window (lgr_format_packed_bytes), reserves a byte range and a directory slot in the open
//    pinned slab under the mutex, and packs the window there itself (lgr_format_pack) outside the mutex;
//  * one calculator thread seals the open slab as soon as the device is free: it waits for workers still writing,
//    writes the directory behind the blocks and makes ONE lgr_format_metrics_packed (one copy in, the records out into
//    a pinned result block).  The other slab fills meanwhile.  No CUDA call is made under the mutex, and every buffer
//    (two slabs, two result blocks, the device context's buffers) is allocated at construction.
// A window larger than a slab travels alone through a context of its own (Counters::alone counts them; their buffers
// are allocated for them).
//
// Errors: a malformed window (what lgr_format_metrics refuses) throws std::invalid_argument in its caller only and
// leaves an empty block in the batch; a failed device call throws std::runtime_error in every caller of that batch.
// Supports with more than LGR_FMT_MAX_ALLELES alleles come back flagged LGR_FMT_WIDE, as from GpuFormatMetrics.
// No CPU fallback: the constructor throws without a GPU.
#ifndef LANCET2_B200_HOST_GPU_FORMAT_H_
#define LANCET2_B200_HOST_GPU_FORMAT_H_

#include <atomic>
#include <condition_variable>
#include <cstddef>
#include <cstdint>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/lancet_gpu_realign.h"
#include "gpu_genotyper.h"

namespace lancet_gpu {

class FormatCalculator {
 public:
  struct Options {
    int device = 0;
    // per slab (two of each, allocated at construction); a slab is sealed before it would exceed any of the three
    std::size_t slab_bytes = 8u << 20;
    std::size_t max_supports = 1u << 15;
    std::size_t max_evidence = 1u << 20;
  };
  struct Counters {
    std::uint64_t batches = 0, windows = 0, supports = 0, evidence = 0, max_windows_in_batch = 0;
    std::uint64_t alone = 0;         // windows larger than a slab, computed on their own
    std::uint64_t ns_pack = 0;       // callers: sizing + reservation + packing (summed over callers)
    std::uint64_t ns_seal_wait = 0;  // calculator thread: waiting for callers still packing into a sealed slab
    std::uint64_t ns_device = 0;     // calculator thread: inside lgr_format_metrics_packed
  };

  explicit FormatCalculator(const Options& opt);
  explicit FormatCalculator(int device_ordinal = 0) : FormatCalculator(Options{device_ordinal}) {}
  ~FormatCalculator();  // answers every pending window, joins the calculator thread, waits for the callers to leave
  FormatCalculator(const FormatCalculator&) = delete;
  FormatCalculator& operator=(const FormatCalculator&) = delete;

  // One record per support of the window, in the window's support order.  Thread-safe and blocking; the window's
  // columns are read before the call returns and not kept.
  [[nodiscard]] std::vector<lgr_format> Compute(EvidenceColumns& window);
  [[nodiscard]] std::vector<lgr_format> Compute(const lgr_evidence_in& window);
  [[nodiscard]] Counters Stats();
  [[nodiscard]] std::size_t Callers();  // threads inside Compute now

 private:
  struct Slab {
    std::uint8_t* mem = nullptr;  // pinned: blocks, then (at seal time) the directory
    lgr_format* res = nullptr;    // pinned: the records of the batch
    std::vector<lgr_fmt_dir> dir; // one entry per window, written by its caller; bases and rec_off at seal time
    std::size_t used = 0, n_windows = 0, n_supports = 0, n_evidence = 0;
    std::atomic<int> packing{0};  // callers still writing their block
    int readers = 0;              // callers that have not yet taken their records
    bool done = false, failed = false;
    std::string error;
  };
  void Run();
  void RunBatch(Slab* s);
  std::vector<lgr_format> ComputeAlone(const lgr_evidence_in& window, std::size_t bytes);

  Options mOpt;
  std::size_t mMaxWindows = 0;    // directory entries per slab (every block holds at least its header)
  lgr_fmt_ctx* mCtx = nullptr;    // calculator thread only (after construction)
  std::mutex mAloneMu;            // windows larger than a slab
  lgr_fmt_ctx* mAloneCtx = nullptr;
  Slab mSlabs[2];
  Slab* mOpen = &mSlabs[0];       // the slab being filled
  std::mutex mMu;
  std::condition_variable mWorkCv;  // calculator thread: windows arrived / readers left / stop
  std::condition_variable mDoneCv;  // callers: their batch finished or a new slab opened; destructor: last caller left
  std::size_t mCallers = 0, mSpaceWaiters = 0;
  bool mStop = false;
  Counters mCounters;
  std::thread mThread;
};

}  // namespace lancet_gpu

#endif  // LANCET2_B200_HOST_GPU_FORMAT_H_
