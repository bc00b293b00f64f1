// gpu_repeat.h — thread-safe repeat check of the graph's k-loop over the lgr_repeat_* C-ABI (SURVEY.md §8f #3).
//
// The reference asks base::HasRepeat from every worker thread, one window at a time
// (cbdg/graph.h:127-131 once per k, core/variant_builder.cpp:116-117 exactly at max_k).  A RepeatChecker
// keeps that call shape: Check() blocks the calling worker until its window's answers are back.  Behind it
// one checker thread takes every request pending at that moment, lays their questions out in one job table
// and makes ONE lgr_repeat_scan; while the device runs, the next batch gathers (group commit).  A lone
// window is spread over the whole GPU by the kernel's slice schedule, so a batch of one is not slow.
//
// Errors: a malformed question (k <= 0, max_mismatches < 0) throws std::invalid_argument in its caller
// only; a failed device call throws std::runtime_error in every caller of that batch.  No CPU fallback:
// the constructor throws without a GPU.
#ifndef LANCET2_B200_HOST_GPU_REPEAT_H_
#define LANCET2_B200_HOST_GPU_REPEAT_H_

#include <condition_variable>
#include <cstddef>
#include <cstdint>
#include <deque>
#include <mutex>
#include <string>
#include <string_view>
#include <thread>
#include <vector>

#include "../../include/lancet_gpu_realign.h"

namespace lancet_gpu {

// one HasRepeat(SlidingView(seq, k), max_mismatches) question about a window
struct RepeatQuestion {
  std::int32_t k;
  std::int32_t max_mismatches;  // 2 for the graph's k-loop, 0 for ShouldSkipWindow
};

class RepeatChecker {
 public:
  struct Options {
    int device = 0;
    // reserved per batch (device buffers and pinned staging, allocated at construction); a batch is sealed before it
    // would exceed either.  A single window larger than max_seq_bytes is longer than LGR_REPEAT_MAX_LEN: it is answered
    // LGR_REPEAT_TOO_LONG without the device.
    std::size_t max_seq_bytes = 4u << 20;
    std::size_t max_questions = 1u << 16;
  };
  struct Counters {
    std::uint64_t batches = 0, windows = 0, questions = 0, max_windows_in_batch = 0;
    std::uint64_t ns_wait = 0;  // checker thread: inside lgr_repeat_scan (copies, kernel, synchronise)
  };

  explicit RepeatChecker(const Options& opt);
  explicit RepeatChecker(int device_ordinal = 0) : RepeatChecker(Options{device_ordinal}) {}
  ~RepeatChecker();  // answers every pending request, then joins the checker thread and waits for the callers to leave
  RepeatChecker(const RepeatChecker&) = delete;
  RepeatChecker& operator=(const RepeatChecker&) = delete;

  // One byte per question, in the caller's order: 0, 1 or LGR_REPEAT_TOO_LONG.  Thread-safe and blocking; `seq` and
  // `questions` are borrowed until the call returns.
  [[nodiscard]] std::vector<std::uint8_t> Check(std::string_view seq, const RepeatQuestion* questions, std::size_t n);
  [[nodiscard]] Counters Stats();
  [[nodiscard]] std::size_t Callers();  // threads inside Check now, waiting for their answers

 private:
  struct Request {
    std::string_view seq;
    const RepeatQuestion* questions;
    std::size_t n;
    std::vector<std::uint8_t>* answers;
    std::string error;  // the device call's message when the batch failed
    bool failed = false, done = false;
  };
  void Run();
  void RunBatch(const std::vector<Request*>& batch);

  Options mOpt;
  lgr_rep_ctx* mCtx = nullptr;  // checker thread only (after construction)
  std::uint8_t* mSeqs = nullptr;  // pinned staging of one batch
  lgr_repeat_job* mJobs = nullptr;
  std::uint8_t* mAnswers = nullptr;
  std::mutex mMu;
  std::condition_variable mWorkCv;  // checker thread: requests arrived / stop
  std::condition_variable mDoneCv;  // callers: their batch finished; destructor: the last caller left
  std::deque<Request*> mPending;
  std::size_t mCallers = 0;  // threads inside Check
  bool mStop = false;
  Counters mCounters;
  std::thread mThread;
};

}  // namespace lancet_gpu

#endif  // LANCET2_B200_HOST_GPU_REPEAT_H_
