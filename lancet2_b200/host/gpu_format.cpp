// gpu_format.cpp — lancet_gpu::FormatCalculator (see gpu_format.h).
#include "gpu_format.h"

#include <algorithm>
#include <chrono>
#include <cstring>
#include <stdexcept>
#include <string>

namespace lancet_gpu {

namespace {

std::uint64_t NowNs() {
  return (std::uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

std::size_t Up16(std::size_t x) { return (x + 15) & ~(std::size_t)15; }

}  // namespace

FormatCalculator::FormatCalculator(const Options& opt) : mOpt(opt) {
  if (mOpt.max_supports < 1 || mOpt.max_supports > (std::size_t)INT32_MAX || mOpt.max_evidence < 1)
    throw std::invalid_argument("FormatCalculator: max_supports must be in [1, 2^31) and max_evidence >= 1");
  // the smallest block (no supports) is its header plus one sup_begin entry, and each window takes a directory entry
  const std::size_t min_window = sizeof(lgr_fmt_blk_hdr) + 16 + sizeof(lgr_fmt_dir);
  mOpt.slab_bytes = Up16(std::max(mOpt.slab_bytes, 64 * min_window));
  mMaxWindows = mOpt.slab_bytes / min_window;
  int rc = lgr_format_create(mOpt.device, &mCtx);
  if (rc != LGR_OK) throw std::runtime_error(std::string("lgr_format_create: ") + lgr_format_last_error(nullptr));
  // everything a batch needs is allocated now: a device regrow later would synchronise the whole GPU
  rc = lgr_format_reserve(mCtx, (std::int64_t)mOpt.slab_bytes, (std::int32_t)mOpt.max_supports, (std::int64_t)mOpt.max_evidence);
  bool pinned = true;
  for (Slab& s : mSlabs) {
    s.mem = static_cast<std::uint8_t*>(lgr_alloc_pinned(mOpt.slab_bytes));
    s.res = static_cast<lgr_format*>(lgr_alloc_pinned(sizeof(lgr_format) * mOpt.max_supports));
    pinned = pinned && s.mem && s.res;
    s.dir.resize(mMaxWindows);
  }
  if (rc != LGR_OK || !pinned) {
    const std::string msg = rc != LGR_OK ? lgr_format_last_error(mCtx) : "pinned staging allocation failed";
    for (Slab& s : mSlabs) lgr_free_pinned(s.mem), lgr_free_pinned(s.res);
    lgr_format_destroy(mCtx);
    throw std::runtime_error("FormatCalculator: " + msg);
  }
  mThread = std::thread([this] { Run(); });
}

FormatCalculator::~FormatCalculator() {
  {
    std::lock_guard<std::mutex> lk(mMu);
    mStop = true;
  }
  mWorkCv.notify_all();
  mThread.join();  // Run seals every window reserved before it returns
  {
    // a caller woken by the last batch may still be on its way out of Compute (it touches mMu and mDoneCv)
    std::unique_lock<std::mutex> lk(mMu);
    mDoneCv.wait(lk, [&] { return mCallers == 0; });
  }
  for (Slab& s : mSlabs) lgr_free_pinned(s.mem), lgr_free_pinned(s.res);
  lgr_format_destroy(mCtx);
  lgr_format_destroy(mAloneCtx);
}

std::vector<lgr_format> FormatCalculator::Compute(EvidenceColumns& window) { return Compute(window.In()); }

std::vector<lgr_format> FormatCalculator::Compute(const lgr_evidence_in& in) {
  const std::uint64_t t0 = NowNs();
  const std::size_t bytes = lgr_format_packed_bytes(&in);
  if (bytes == 0) throw std::invalid_argument("FormatCalculator::Compute: negative sizes");
  if (in.n_supports == 0) return {};
  const std::size_t S = (std::size_t)in.n_supports, N = (std::size_t)in.n_evidence;
  // every caller is counted, so that the destructor cannot free what a caller still uses
  struct CallerScope {
    FormatCalculator* self;
    ~CallerScope() {
      std::lock_guard<std::mutex> lk(self->mMu);
      if (--self->mCallers == 0 && self->mStop) self->mDoneCv.notify_all();
    }
  };
  {
    std::lock_guard<std::mutex> lk(mMu);
    if (mStop) throw std::runtime_error("FormatCalculator::Compute: the calculator is being destroyed");
    ++mCallers;
  }
  CallerScope scope{this};
  if (bytes + sizeof(lgr_fmt_dir) > mOpt.slab_bytes || S > mOpt.max_supports || N > mOpt.max_evidence)
    return ComputeAlone(in, bytes);

  std::unique_lock<std::mutex> lk(mMu);
  Slab* s = nullptr;
  for (;;) {
    s = mOpen;
    const bool fits = s->n_windows < mMaxWindows &&
                      Up16(s->used + bytes) + (s->n_windows + 1) * sizeof(lgr_fmt_dir) <= mOpt.slab_bytes &&
                      s->n_supports + S <= mOpt.max_supports && s->n_evidence + N <= mOpt.max_evidence;
    if (fits) break;
    // full: the calculator thread seals it as soon as the device is free, then a fresh slab opens
    ++mSpaceWaiters;
    mWorkCv.notify_one();
    mDoneCv.wait(lk, [&] { return mOpen != s || s->n_windows == 0; });  // or s itself reopened empty meanwhile
    --mSpaceWaiters;
  }
  const std::size_t slot = s->n_windows++, off = s->used;
  s->used += bytes, s->n_supports += S, s->n_evidence += N;
  ++s->readers;
  s->packing.fetch_add(1, std::memory_order_relaxed);
  lk.unlock();
  mWorkCv.notify_one();

  int rc = lgr_format_pack(&in, s->mem + off, bytes, &s->dir[slot]);
  if (rc != LGR_OK) {  // refused here; the batch gets an empty block in its place
    const lgr_evidence_in empty{};
    lgr_format_pack(&empty, s->mem + off, bytes, &s->dir[slot]);
  }
  s->dir[slot].rec_off = off;
  s->packing.fetch_sub(1, std::memory_order_release);
  const std::uint64_t t1 = NowNs();

  lk.lock();
  mCounters.ns_pack += t1 - t0;
  std::vector<lgr_format> out;
  if (rc == LGR_OK) {
    mDoneCv.wait(lk, [&] { return s->done; });
    if (!s->failed) {
      const lgr_format* r = s->res + s->dir[slot].sup_base;
      out.assign(r, r + S);
    }
  }
  const bool failed = rc == LGR_OK && s->failed;
  const std::string error = failed ? s->error : "";
  if (--s->readers == 0) mWorkCv.notify_one();  // the slab may be reopened
  lk.unlock();
  if (rc != LGR_OK) throw std::invalid_argument("FormatCalculator::Compute: malformed window (what lgr_format_metrics refuses)");
  if (failed) throw std::runtime_error("FormatCalculator: " + error);
  return out;
}

std::vector<lgr_format> FormatCalculator::ComputeAlone(const lgr_evidence_in& in, std::size_t bytes) {
  const std::uint64_t t0 = NowNs();
  std::vector<std::uint8_t> block(bytes);
  lgr_fmt_dir dir;
  if (lgr_format_pack(&in, block.data(), bytes, &dir) != LGR_OK)
    throw std::invalid_argument("FormatCalculator::Compute: malformed window (what lgr_format_metrics refuses)");
  dir.rec_off = 0, dir.sup_base = 0, dir.ev_base = 0;
  const std::uint64_t t1 = NowNs();
  lgr_fmt_packed_in pk{1, 0, block.data(), bytes, &dir};
  std::vector<lgr_format> out((std::size_t)in.n_supports);
  {
    std::lock_guard<std::mutex> lk(mAloneMu);
    if (!mAloneCtx && lgr_format_create(mOpt.device, &mAloneCtx) != LGR_OK)
      throw std::runtime_error(std::string("FormatCalculator: lgr_format_create: ") + lgr_format_last_error(nullptr));
    const int rc = lgr_format_metrics_packed(mAloneCtx, &pk, out.data(), nullptr);
    if (rc != LGR_OK && rc != LGR_E_PARTIAL)
      throw std::runtime_error(std::string("FormatCalculator: lgr_format_metrics_packed: ") + lgr_strerror(rc) + ": " +
                               lgr_format_last_error(mAloneCtx));
  }
  std::lock_guard<std::mutex> lk(mMu);
  mCounters.alone += 1, mCounters.ns_pack += t1 - t0;
  return out;
}

FormatCalculator::Counters FormatCalculator::Stats() {
  std::lock_guard<std::mutex> lk(mMu);
  return mCounters;
}

std::size_t FormatCalculator::Callers() {
  std::lock_guard<std::mutex> lk(mMu);
  return mCallers;
}

void FormatCalculator::Run() {
  for (;;) {
    Slab* s = nullptr;
    {
      std::unique_lock<std::mutex> lk(mMu);
      auto other = [&] { return mOpen == &mSlabs[0] ? &mSlabs[1] : &mSlabs[0]; };
      // the other slab reopens once every caller of its batch has taken its records
      mWorkCv.wait(lk, [&] {
        return (mOpen->n_windows > 0 && other()->readers == 0) || (mStop && mOpen->n_windows == 0 && mSpaceWaiters == 0);
      });
      if (mOpen->n_windows == 0) return;  // stopping, and nothing is left to answer
      s = mOpen;
      Slab* next = other();
      next->used = next->n_windows = next->n_supports = next->n_evidence = 0;
      next->done = next->failed = false;
      next->error.clear();
      mOpen = next;
    }
    mDoneCv.notify_all();  // callers waiting for room
    RunBatch(s);           // no lock held: callers keep packing into the other slab meanwhile
  }
}

void FormatCalculator::RunBatch(Slab* s) {
  const std::uint64_t t0 = NowNs();
  while (s->packing.load(std::memory_order_acquire) != 0) std::this_thread::yield();  // callers finishing their block
  const std::uint64_t t1 = NowNs();
  // the directory behind the blocks: the whole batch is one copy
  const std::size_t W = s->n_windows, dir_off = Up16(s->used);
  std::int64_t sup = 0, ev = 0;
  for (std::size_t w = 0; w < W; ++w) {
    lgr_fmt_dir& d = s->dir[w];
    d.sup_base = (std::int32_t)sup, d.ev_base = ev;
    sup += d.n_supports, ev += d.n_evidence;
  }
  std::memcpy(s->mem + dir_off, s->dir.data(), W * sizeof(lgr_fmt_dir));
  const lgr_fmt_packed_in in{(std::int32_t)W, 0, s->mem, dir_off + W * sizeof(lgr_fmt_dir),
                             reinterpret_cast<const lgr_fmt_dir*>(s->mem + dir_off)};
  const int rc = lgr_format_metrics_packed(mCtx, &in, s->res, nullptr);
  const std::uint64_t t2 = NowNs();
  const bool failed = rc != LGR_OK && rc != LGR_E_PARTIAL;  // PARTIAL: wide supports, their records say so
  {
    std::lock_guard<std::mutex> lk(mMu);
    s->done = true;
    if (failed) s->failed = true, s->error = std::string("lgr_format_metrics_packed: ") + lgr_strerror(rc) + ": " + lgr_format_last_error(mCtx);
    mCounters.batches += 1, mCounters.windows += W, mCounters.supports += (std::uint64_t)sup, mCounters.evidence += (std::uint64_t)ev;
    mCounters.max_windows_in_batch = std::max<std::uint64_t>(mCounters.max_windows_in_batch, W);
    mCounters.ns_seal_wait += t1 - t0, mCounters.ns_device += t2 - t1;
  }
  mDoneCv.notify_all();
}

}  // namespace lancet_gpu
