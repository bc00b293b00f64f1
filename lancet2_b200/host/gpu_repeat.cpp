// gpu_repeat.cpp — lancet_gpu::RepeatChecker (see gpu_repeat.h).
#include "gpu_repeat.h"

#include <algorithm>
#include <chrono>
#include <cstring>
#include <numeric>
#include <stdexcept>
#include <string>

namespace lancet_gpu {

RepeatChecker::RepeatChecker(const Options& opt) : mOpt(opt) {
  mOpt.max_seq_bytes = std::max<std::size_t>(mOpt.max_seq_bytes, LGR_REPEAT_MAX_LEN);
  mOpt.max_questions = std::max<std::size_t>(mOpt.max_questions, 1);
  if (mOpt.max_questions > (std::size_t)INT32_MAX) throw std::invalid_argument("RepeatChecker: max_questions too large");
  int rc = lgr_repeat_create(mOpt.device, &mCtx);
  if (rc != LGR_OK) throw std::runtime_error(std::string("lgr_repeat_create: ") + lgr_repeat_last_error(nullptr));
  // everything a batch needs is allocated now: a device regrow later would synchronise the whole GPU
  rc = lgr_repeat_reserve(mCtx, (std::int64_t)mOpt.max_seq_bytes, (std::int32_t)mOpt.max_questions);
  mSeqs = static_cast<std::uint8_t*>(lgr_alloc_pinned(mOpt.max_seq_bytes));
  mJobs = static_cast<lgr_repeat_job*>(lgr_alloc_pinned(sizeof(lgr_repeat_job) * mOpt.max_questions));
  mAnswers = static_cast<std::uint8_t*>(lgr_alloc_pinned(mOpt.max_questions));
  if (rc != LGR_OK || !mSeqs || !mJobs || !mAnswers) {
    const std::string msg = rc != LGR_OK ? lgr_repeat_last_error(mCtx) : "pinned staging allocation failed";
    lgr_free_pinned(mSeqs), lgr_free_pinned(mJobs), lgr_free_pinned(mAnswers);
    lgr_repeat_destroy(mCtx);
    throw std::runtime_error("RepeatChecker: " + msg);
  }
  mThread = std::thread([this] { Run(); });
}

RepeatChecker::~RepeatChecker() {
  {
    std::lock_guard<std::mutex> lk(mMu);
    mStop = true;
  }
  mWorkCv.notify_all();
  mThread.join();  // Run drains mPending before it returns
  {
    // a caller woken by the last batch may still be on its way out of Check (it touches mMu and mDoneCv)
    std::unique_lock<std::mutex> lk(mMu);
    mDoneCv.wait(lk, [&] { return mCallers == 0; });
  }
  lgr_free_pinned(mSeqs), lgr_free_pinned(mJobs), lgr_free_pinned(mAnswers);
  lgr_repeat_destroy(mCtx);
}

std::vector<std::uint8_t> RepeatChecker::Check(std::string_view seq, const RepeatQuestion* questions, std::size_t n) {
  for (std::size_t i = 0; i < n; ++i)
    if (questions[i].k <= 0 || questions[i].max_mismatches < 0)
      throw std::invalid_argument("RepeatChecker::Check: k must be > 0 and max_mismatches >= 0");
  if (n > mOpt.max_questions) throw std::invalid_argument("RepeatChecker::Check: more questions than a batch holds");
  std::vector<std::uint8_t> answers(n);
  if (n == 0) return answers;
  if (seq.size() > mOpt.max_seq_bytes) {  // longer than LGR_REPEAT_MAX_LEN: the device would not compute it either
    std::fill(answers.begin(), answers.end(), (std::uint8_t)LGR_REPEAT_TOO_LONG);
    return answers;
  }
  Request req{seq, questions, n, &answers, {}};
  std::unique_lock<std::mutex> lk(mMu);
  if (mStop) throw std::runtime_error("RepeatChecker::Check: the checker is being destroyed");
  ++mCallers;
  mPending.push_back(&req);
  mWorkCv.notify_one();
  mDoneCv.wait(lk, [&] { return req.done; });
  --mCallers;
  if (mStop && mCallers == 0) mDoneCv.notify_all();  // under the lock: the destructor cannot run ahead of this notify
  if (req.failed) throw std::runtime_error("RepeatChecker: " + req.error);
  return answers;
}

RepeatChecker::Counters RepeatChecker::Stats() {
  std::lock_guard<std::mutex> lk(mMu);
  return mCounters;
}

std::size_t RepeatChecker::Callers() {
  std::lock_guard<std::mutex> lk(mMu);
  return mCallers;
}

void RepeatChecker::Run() {
  std::vector<Request*> batch;
  for (;;) {
    batch.clear();
    {
      std::unique_lock<std::mutex> lk(mMu);
      mWorkCv.wait(lk, [&] { return mStop || !mPending.empty(); });
      if (mPending.empty()) return;  // stopping, and nothing is left to answer
      // seal at the reserved size; every single request fits (Check routes larger ones elsewhere)
      std::size_t bytes = 0, questions = 0;
      while (!mPending.empty()) {
        Request* r = mPending.front();
        if (!batch.empty() && (bytes + r->seq.size() > mOpt.max_seq_bytes || questions + r->n > mOpt.max_questions)) break;
        bytes += r->seq.size(), questions += r->n;
        batch.push_back(r);
        mPending.pop_front();
      }
    }
    RunBatch(batch);  // no lock held: callers keep appending the next batch meanwhile
  }
}

void RepeatChecker::RunBatch(const std::vector<Request*>& batch) {
  // one window's questions adjacent and grouped by threshold: each threshold's k values form one job group of the
  // kernel and share its mismatch masks.  order[] maps a job back to its question.
  std::size_t bytes = 0, n_jobs = 0;
  std::vector<std::size_t> order;
  for (Request* r : batch) {
    std::memcpy(mSeqs + bytes, r->seq.data(), r->seq.size());
    const std::size_t j0 = n_jobs;
    order.resize(j0 + r->n);
    std::iota(order.begin() + (std::ptrdiff_t)j0, order.end(), std::size_t{0});
    std::stable_sort(order.begin() + (std::ptrdiff_t)j0, order.end(), [&](std::size_t a, std::size_t b) {
      return r->questions[a].max_mismatches < r->questions[b].max_mismatches;
    });
    for (std::size_t j = j0; j < j0 + r->n; ++j) {
      const RepeatQuestion& q = r->questions[order[j]];
      mJobs[j] = lgr_repeat_job{(std::int64_t)bytes, (std::int32_t)r->seq.size(), q.k, q.max_mismatches, 0};
    }
    bytes += r->seq.size(), n_jobs += r->n;
  }
  const auto t0 = std::chrono::steady_clock::now();
  const int rc = lgr_repeat_scan(mCtx, mSeqs, (std::int64_t)bytes, mJobs, (std::int32_t)n_jobs, mAnswers, nullptr);
  const auto t1 = std::chrono::steady_clock::now();
  const bool failed = rc != LGR_OK && rc != LGR_E_PARTIAL;  // PARTIAL: some windows are too long, their bytes say so
  const std::string error = failed ? std::string("lgr_repeat_scan: ") + lgr_strerror(rc) + ": " + lgr_repeat_last_error(mCtx) : "";
  if (!failed) {
    std::size_t j = 0;
    for (Request* r : batch)
      for (std::size_t i = 0; i < r->n; ++i, ++j) (*r->answers)[order[j]] = mAnswers[j];
  }
  {
    std::lock_guard<std::mutex> lk(mMu);
    for (Request* r : batch) {
      r->done = true;
      if (failed) r->failed = true, r->error = error;
    }
    mCounters.batches += 1, mCounters.windows += batch.size(), mCounters.questions += n_jobs;
    mCounters.max_windows_in_batch = std::max<std::uint64_t>(mCounters.max_windows_in_batch, batch.size());
    mCounters.ns_wait += (std::uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
  }
  mDoneCv.notify_all();
}

}  // namespace lancet_gpu
