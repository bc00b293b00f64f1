// adapter_capi.cpp — C hooks around lancet_gpu::GpuGenotyper so that the pytest suite can
// drive the C++ adapter (ctypes) without a C++ test runner.  Test support only; the product
// boundary is include/lancet_gpu_realign.h + host/gpu_genotyper.h.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <deque>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "gpu_format.h"
#include "gpu_genotyper.h"
#include "gpu_repeat.h"

namespace {

void AppI(std::string& s, long long v) { char b[32]; std::snprintf(b, sizeof(b), "%lld,", v); s += b; }
void AppD(std::string& s, double v) { char b[48]; std::snprintf(b, sizeof(b), "%a,", v); s += b; }

// plain snprintf/std::string on purpose (no iostreams)
void DumpAllele(std::string& s, const lancet_gpu::PerAlleleData& d) {
  s += "fwdbq:";
  for (auto v : d.mFwdBaseQuals) AppI(s, v);
  s += "|revbq:";
  for (auto v : d.mRevBaseQuals) AppI(s, v);
  s += "|mapq:";
  for (auto v : d.mMapQuals) AppI(s, v);
  s += "|aln:";
  for (auto v : d.mAlnScores) AppD(s, v);
  s += "|isz:";
  for (auto v : d.mProperPairIsizes) AppD(s, v);
  s += "|fold:";
  for (auto v : d.mFoldedReadPositions) AppD(s, v);
  s += "|refnm:";
  for (auto v : d.mRefNmValues) AppD(s, v);
  s += "|ownnm:";
  for (auto v : d.mOwnHapNmValues) AppD(s, v);
  s += "|starts:";
  for (auto v : d.mAlignmentStarts) AppI(s, v);
  s += "|hapids:";
  for (auto v : d.mHaplotypeIds) AppI(s, v);
  s += "|sc:" + std::to_string(d.mSoftClipCount) + "|hashes:";
  std::vector<std::pair<std::uint32_t, int>> hs;
  for (auto& kv : d.mNameHashes) hs.emplace_back(kv.first, (int)(kv.second == lancet_gpu::Strand::REV));
  std::sort(hs.begin(), hs.end());
  for (auto& kv : hs) s += std::to_string(kv.first) + ":" + std::to_string(kv.second) + ",";
}

int WriteOut(const std::string& s, char* out, long long cap) {
  if ((long long)s.size() + 1 > cap) return -1;
  std::memcpy(out, s.c_str(), s.size() + 1);
  return (int)s.size();
}

}  // namespace

extern "C" {

// Feed one evidence stream through lancet_gpu::VariantSupport::AddEvidence and dump the
// per-allele vectors (same text format as oracle/ref_shim/ref_capi.cpp:ref_add_evidence_dump).
int lgr_adapter_add_evidence_dump(int n, const long long* isize, const long long* start, const double* aln,
                                  const double* fold, const unsigned* hash, const unsigned* ref_nm, const unsigned* own_nm,
                                  const unsigned* hap_id, const unsigned char* allele, const unsigned char* rev,
                                  const unsigned char* bq, const unsigned char* mapq, const unsigned char* softclip,
                                  const unsigned char* proper, char* out, long long cap) {
  lancet_gpu::VariantSupport vs;
  for (int i = 0; i < n; ++i) {
    lancet_gpu::ReadEvidence ev;
    ev.mInsertSize = isize[i], ev.mAlignmentStart = start[i], ev.mAlnScore = aln[i], ev.mFoldedReadPos = fold[i];
    ev.mRnameHash = hash[i], ev.mRefNm = ref_nm[i], ev.mOwnHapNm = own_nm[i], ev.mAssignedHaplotypeId = hap_id[i];
    ev.mAllele = allele[i], ev.mStrand = rev[i] ? lancet_gpu::Strand::REV : lancet_gpu::Strand::FWD;
    ev.mBaseQual = bq[i], ev.mMapQual = mapq[i], ev.mIsSoftClipped = softclip[i] != 0, ev.mIsProperPair = proper[i] != 0;
    vs.AddEvidence(ev);
  }
  std::string os;
  for (std::size_t a = 0; a < vs.AlleleData().size(); ++a) {
    os += "A" + std::to_string(a) + "|";
    DumpAllele(os, vs.AlleleData()[a]);
    os += "\n";
  }
  return WriteOut(os, out, cap);
}

}  // extern "C"

namespace {

// Rebuilds the C++-side view (strings, ReadIn, VariantIn, one GenotypeJob per group) of a batch
// given in the C-ABI's SoA form plus the per-read metadata AddToTable needs.
struct JobSet {
  std::vector<std::string_view> qn, sn;
  std::vector<std::string> haps;
  std::vector<lancet_gpu::ReadIn> reads;
  std::vector<lancet_gpu::VariantIn> vars;
  std::vector<lancet_gpu::GenotypeJob> jobs;
};

void BuildJobs(const lgr_batch_in* in, const char* names, const char* samples, const int* sample_id, const long long* start0,
               const long long* isize, const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
               JobSet& js) {
  for (const char* p = names; (int)js.qn.size() < in->n_reads; p += std::strlen(p) + 1) js.qn.emplace_back(p);
  int n_samples = 0;
  for (int r = 0; r < in->n_reads; ++r) n_samples = std::max(n_samples, sample_id[r] + 1);
  for (const char* p = samples; (int)js.sn.size() < n_samples; p += std::strlen(p) + 1) js.sn.emplace_back(p);
  js.haps.resize(in->n_haps);
  for (int h = 0; h < in->n_haps; ++h)
    js.haps[h].assign(reinterpret_cast<const char*>(in->hap_bases) + in->hap_off[h], (size_t)(in->hap_off[h + 1] - in->hap_off[h]));
  js.reads.resize(in->n_reads);
  for (int r = 0; r < in->n_reads; ++r) {
    const size_t len = (size_t)(in->read_off[r + 1] - in->read_off[r]);
    js.reads[r] = lancet_gpu::ReadIn{js.qn[r], std::string_view(reinterpret_cast<const char*>(in->read_bases) + in->read_off[r], len),
                                     in->read_quals + in->read_off[r], js.sn[sample_id[r]], start0[r], isize[r], sam_flag[r],
                                     mapq[r], softclip[r] != 0};
  }
  js.vars.resize(in->n_vars);
  for (int g = 0; g < in->n_groups; ++g) {
    const int h0 = in->grp_hap_begin[g], P = in->grp_hap_begin[g + 1] - h0;
    for (int v = in->grp_var_begin[g]; v < in->grp_var_begin[g + 1]; ++v) {
      lancet_gpu::VariantIn& vi = js.vars[v];
      vi.key = &js.vars[v];
      const long long o = in->var_hap_off[v];
      vi.local_ref_start0 = (size_t)in->var_start[o], vi.ref_allele_len = (size_t)in->var_len[o];
      int max_al = 0;
      for (int h = 1; h < P; ++h) max_al = std::max(max_al, (int)in->var_allele[o + h]);
      vi.alts.resize(max_al);
      for (int h = 1; h < P; ++h) {
        const int al = in->var_allele[o + h];
        if (al <= 0) continue;
        vi.alts[al - 1].seq_len = (size_t)in->var_len[o + h];
        vi.alts[al - 1].length = (long long)in->var_len[o + h] - (long long)vi.ref_allele_len;
        vi.alts[al - 1].hap_start0.emplace_back((size_t)h, (size_t)in->var_start[o + h]);
      }
    }
    js.jobs.push_back(lancet_gpu::GenotypeJob{js.haps.data() + h0, (size_t)P, js.reads.data() + in->grp_read_begin[g],
                                              (size_t)(in->grp_read_begin[g + 1] - in->grp_read_begin[g]),
                                              js.vars.data() + in->grp_var_begin[g],
                                              (size_t)(in->grp_var_begin[g + 1] - in->grp_var_begin[g])});
  }
}

std::string DumpResults(const lgr_batch_in* in, const JobSet& js, const std::vector<lancet_gpu::Result>& res) {
  std::string os;
  for (int g = 0; g < in->n_groups; ++g) {
    for (int v = in->grp_var_begin[g]; v < in->grp_var_begin[g + 1]; ++v) {
      auto it = res[g].find(&js.vars[v]);
      if (it == res[g].end()) continue;
      for (const auto& ns : it->second) {
        const auto& ad = ns.mData->AlleleData();
        for (std::size_t a = 0; a < ad.size(); ++a) {
          os += "G" + std::to_string(g) + " V" + std::to_string(v - in->grp_var_begin[g]) + " S" + std::string(ns.mSampleName) +
                " A" + std::to_string(a) + "|";
          DumpAllele(os, ad[a]);
          os += "\n";
        }
      }
    }
  }
  return os;
}

std::uint32_t X31OfView(std::string_view q) { return lgr_x31_hash(std::string(q).c_str()); }

}  // namespace

extern "C" {

// Run GpuGenotyper::GenotypeMany on the batch; dump every (group, variant, sample, allele)
// evidence block.  names: NUL-separated read names; samples: NUL-separated sample names,
// sample_id per read.  The name hash is X31 of the name (deterministic stand-in for
// absl::HashOf in tests).
int lgr_adapter_genotype_dump(int device, const lgr_batch_in* in, const char* names, const char* samples,
                              const int* sample_id, const long long* start0, const long long* isize,
                              const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
                              char* out, long long cap) {
  try {
    JobSet js;
    BuildJobs(in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, js);
    lancet_gpu::GpuGenotyper gt(device);
    std::vector<lancet_gpu::Result> res = gt.GenotypeMany(js.jobs, X31OfView);
    return WriteOut(DumpResults(in, js, res), out, cap);
  } catch (const std::exception& e) {
    std::snprintf(out, (size_t)cap, "EXCEPTION: %s", e.what());
    return -2;
  }
}

// Host logic without a GPU (CPU test suite): pack the batch's groups through PackedJob/PackedBatch
// and compare the resulting C-ABI SoA arrays with the arrays the batch came from (a round trip
// through the C++ view), then run AddToTable (PackedBatch::BuildResult) on caller-provided
// lgr_assign records (the oracle's, in the tests) and dump the evidence.  Returns the number of
// mismatching array elements of the packing round trip in *pack_mismatches.
int lgr_adapter_host_logic_dump(const lgr_batch_in* in, const char* names, const char* samples, const int* sample_id,
                                const long long* start0, const long long* isize, const unsigned short* sam_flag,
                                const unsigned char* mapq, const unsigned char* softclip, const lgr_assign* assign,
                                long long* pack_mismatches, char* out, long long cap) {
  try {
    JobSet js;
    BuildJobs(in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, js);
    lancet_gpu::PackedBatch pb;
    pb.Pack(js.jobs.data(), js.jobs.size(), 0);
    const lgr_batch_in& p = pb.In();
    long long bad = 0;
    bad += p.n_groups != in->n_groups || p.n_haps != in->n_haps || p.n_reads != in->n_reads || p.n_vars != in->n_vars;
    if (!bad) {
      for (int g = 0; g <= in->n_groups; ++g)
        bad += p.grp_hap_begin[g] != in->grp_hap_begin[g] || p.grp_read_begin[g] != in->grp_read_begin[g] ||
               p.grp_var_begin[g] != in->grp_var_begin[g];
      for (int h = 0; h <= in->n_haps; ++h) bad += p.hap_off[h] != in->hap_off[h];
      for (int r = 0; r <= in->n_reads; ++r) bad += p.read_off[r] != in->read_off[r];
      for (int v = 0; v <= in->n_vars; ++v) bad += p.var_hap_off[v] != in->var_hap_off[v];
      bad += std::memcmp(p.hap_bases, in->hap_bases, (size_t)in->hap_off[in->n_haps]) != 0;
      bad += std::memcmp(p.read_bases, in->read_bases, (size_t)in->read_off[in->n_reads]) != 0;
      bad += std::memcmp(p.read_quals, in->read_quals, (size_t)in->read_off[in->n_reads]) != 0;
      for (int r = 0; r < in->n_reads; ++r) bad += p.read_name_hash[r] != in->read_name_hash[r];
      for (long long x = 0; x < in->var_hap_off[in->n_vars]; ++x)
        bad += p.var_start[x] != in->var_start[x] || p.var_len[x] != in->var_len[x] || p.var_allele[x] != in->var_allele[x];
      bad += p.grp_mid_occ != nullptr;  // latched value 0 → per-group derivation left to the device
    }
    if (pack_mismatches) *pack_mismatches = bad;
    std::vector<lancet_gpu::Result> res(js.jobs.size());
    long long off = 0;
    for (std::size_t g = 0; g < js.jobs.size(); ++g) {
      res[g] = lancet_gpu::PackedBatch::BuildResult(js.jobs[g], assign + off, X31OfView);
      off += (long long)(js.jobs[g].n_reads * js.jobs[g].n_variants);
    }
    return WriteOut(DumpResults(in, js, res), out, cap);
  } catch (const std::exception& e) {
    std::snprintf(out, (size_t)cap, "EXCEPTION: %s", e.what());
    return -2;
  }
}

// Same batch, but every group is a separate blocking GenotypeBatcher::Genotype() call issued
// from `n_threads` worker threads (round-robin over the groups, `rounds` times), the way
// Lancet2's workers would call it.  counters[9] = batches, jobs, pairs, max jobs in one batch,
// wall nanoseconds of the worker phase, batcher-thread nanoseconds in pack / submit / wait / deliver.  cap <= 0 skips the dump (timing runs).  window > 1:
// every worker keeps that many groups enqueued (Enqueue/Collect) instead of blocking per group.
// n_devices > 1: a GenotypeDispatcher over devices device .. device+n_devices-1; counters[9 + d] =
// payloads that went to device d (counters must hold 17 entries).
static int BatcherRun(int device, const lgr_batch_in* in, const char* names, const char* samples,
                             const int* sample_id, const long long* start0, const long long* isize,
                             const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
                             int n_threads, int rounds, int window, int n_devices, unsigned long long* counters, int n_counters,
                             char* out, long long cap, bool dump, bool direct_graph = false) {
  try {
    JobSet js;
    BuildJobs(in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, js);
    std::vector<lancet_gpu::Result> res(js.jobs.size());
    std::vector<std::string> errors((size_t)n_threads);
    {
      std::vector<int> devices;
      for (int d = 0; d < (n_devices > 1 ? n_devices : 1); ++d) devices.push_back(device + d);
      lancet_gpu::GenotypeBatcher::Options opt;
      opt.direct_graph = direct_graph;
      lancet_gpu::GenotypeDispatcher batcher(devices, X31OfView, opt);
      std::vector<std::thread> workers;
      const auto t0 = std::chrono::steady_clock::now();
      for (int t = 0; t < n_threads; ++t) {
        workers.emplace_back([&, t] {
          try {
            // split ProcessWindow: up to `window` groups enqueued per worker before the oldest is collected.  The
            // window rolls across rounds (a worker of the caller has thousands of windows queued, it never drains
            // its pipeline between two of them); everything is collected before the clock stops.
            std::deque<std::pair<std::size_t, lancet_gpu::GenotypeDispatcher::Ticket>> open_t;
            for (int round = 0; round < rounds; ++round) {
              if (window <= 1) {  // the reference's call shape: one blocking call per group
                for (std::size_t g = (size_t)t; g < js.jobs.size(); g += (size_t)n_threads) {
                  const lancet_gpu::GenotypeJob& j = js.jobs[g];
                  res[g] = batcher.Genotype(j.haps, j.n_haps, j.reads, j.n_reads, j.variants, j.n_variants);
                }
              } else {
                for (std::size_t g = (size_t)t; g < js.jobs.size(); g += (size_t)n_threads) {
                  if ((int)open_t.size() == window) {
                    res[open_t.front().first] = batcher.Collect(open_t.front().second);
                    open_t.pop_front();
                  }
                  open_t.emplace_back(g, batcher.Enqueue(js.jobs[g]));
                }
              }
            }
            for (auto& ot : open_t) res[ot.first] = batcher.Collect(ot.second);
          } catch (const std::exception& e) {
            errors[(size_t)t] = e.what();
          }
        });
      }
      for (auto& w : workers) w.join();
      const auto t1 = std::chrono::steady_clock::now();
      lancet_gpu::GenotypeBatcher::Counters c;  // summed over the devices; counters[9 + d] = jobs of device d
      for (std::size_t d = 0; d < batcher.Devices(); ++d) {
        const auto cd = batcher.Stats(d);
        c.batches += cd.batches, c.jobs += cd.jobs, c.pairs += cd.pairs;
        c.max_jobs_in_batch = std::max(c.max_jobs_in_batch, cd.max_jobs_in_batch);
        c.ns_pack += cd.ns_pack, c.ns_submit += cd.ns_submit, c.ns_wait += cd.ns_wait, c.ns_deliver += cd.ns_deliver;
        c.h2d_bytes += cd.h2d_bytes, c.d2h_bytes += cd.d2h_bytes, c.retried_alone += cd.retried_alone, c.ns_seal_wait += cd.ns_seal_wait;
        c.graph_launches += cd.graph_launches;
        if (counters && d < 8) counters[9 + d] = cd.jobs;
      }
      if (counters && n_counters >= 20) counters[17] = c.h2d_bytes, counters[18] = c.d2h_bytes, counters[19] = c.retried_alone;
      if (counters && n_counters >= 21) counters[20] = c.ns_seal_wait;
      if (counters && n_counters >= 22) counters[21] = c.graph_launches;
      if (counters) {
        counters[0] = c.batches, counters[1] = c.jobs, counters[2] = c.pairs, counters[3] = c.max_jobs_in_batch;
        counters[4] = (unsigned long long)std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
        counters[5] = c.ns_pack, counters[6] = c.ns_submit, counters[7] = c.ns_wait, counters[8] = c.ns_deliver;
      }
    }
    for (const auto& e : errors)
      if (!e.empty()) throw std::runtime_error(e);
    if (!dump || cap <= 0) return 0;
    return WriteOut(DumpResults(in, js, res), out, cap);
  } catch (const std::exception& e) {
    if (out && cap > 0) std::snprintf(out, (size_t)cap, "EXCEPTION: %s", e.what());
    return -2;
  }
}

int lgr_adapter_batcher_dump(int device, const lgr_batch_in* in, const char* names, const char* samples,
                             const int* sample_id, const long long* start0, const long long* isize,
                             const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
                             int n_threads, int rounds, int window, int n_devices, unsigned long long* counters, char* out,
                             long long cap) {
  return BatcherRun(device, in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, n_threads, rounds, window,
                    n_devices, counters, 17, out, cap, true);
}

// the same without the dump, for bench.py's e2e arm: counters[21] adds [17] bytes copied host→device, [18] device→host,
// [19] payloads re-run alone, [20] batcher-thread ns spent waiting for workers still packing when a slab was sealed
int lgr_adapter_batcher_bench(int device, const lgr_batch_in* in, const char* names, const char* samples,
                              const int* sample_id, const long long* start0, const long long* isize,
                              const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
                              int n_threads, int rounds, int window, int n_devices, unsigned long long* counters, char* err,
                              long long err_cap) {
  const int rc = BatcherRun(device, in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, n_threads, rounds,
                            window, n_devices, counters, 21, err, err_cap, false);
  return rc;
}

// The blocking call shape on one device with GenotypeBatcher::Options::direct_graph off (0) or on: every group is a
// Genotype() call from one of n_threads threads, `rounds` times.  counters[22] as lgr_adapter_batcher_bench plus
// [21] calls whose device pass ran as a CUDA graph.  cap <= 0 skips the dump (timing runs).
int lgr_adapter_direct_graph_run(int device, const lgr_batch_in* in, const char* names, const char* samples,
                                 const int* sample_id, const long long* start0, const long long* isize,
                                 const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
                                 int n_threads, int rounds, int direct_graph, unsigned long long* counters, char* out,
                                 long long cap) {
  return BatcherRun(device, in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, n_threads, rounds, 1, 1,
                    counters, 22, out, cap, true, direct_graph != 0);
}

// Failure isolation of the batcher: ONE worker enqueues every group before it collects the first (so they
// share device batches), catching per payload.  job_status[g] = 0 ok, 1 Enqueue threw, 2 Collect threw; the dump
// holds the evidence of the groups that succeeded.  mid_occ > 0 overrides lgr_params::mid_occ (to provoke a
// device-side cap).  counters[0] = payloads re-run alone.
int lgr_adapter_isolation_dump(int device, const lgr_batch_in* in, const char* names, const char* samples,
                               const int* sample_id, const long long* start0, const long long* isize,
                               const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
                               int mid_occ, int* job_status, unsigned long long* counters, char* out, long long cap) {
  try {
    JobSet js;
    BuildJobs(in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, js);
    std::vector<lancet_gpu::Result> res(js.jobs.size());
    lgr_params prm;
    lgr_default_params(&prm);
    if (mid_occ > 0) prm.mid_occ = mid_occ;
    lancet_gpu::GenotypeBatcher::Options opt;
    opt.device = device, opt.params = &prm, opt.linger_us = 50000;  // all payloads of the probe share one device batch
    {
      lancet_gpu::GenotypeBatcher batcher(opt, X31OfView);
      std::vector<lancet_gpu::GenotypeBatcher::Ticket> tickets(js.jobs.size());
      for (std::size_t g = 0; g < js.jobs.size(); ++g) {
        job_status[g] = 0;
        try {
          tickets[g] = batcher.Enqueue(js.jobs[g]);
        } catch (const std::exception&) {
          job_status[g] = 1;
        }
      }
      for (std::size_t g = 0; g < js.jobs.size(); ++g) {
        if (job_status[g]) continue;
        try {
          res[g] = batcher.Collect(tickets[g]);
        } catch (const std::exception&) {
          job_status[g] = 2;
        }
      }
      if (counters) counters[0] = batcher.Stats().retried_alone, counters[1] = batcher.Stats().batches;
    }
    return WriteOut(DumpResults(in, js, res), out, cap);
  } catch (const std::exception& e) {
    if (out && cap > 0) std::snprintf(out, (size_t)cap, "EXCEPTION: %s", e.what());
    return -2;
  }
}

// SURVEY.md §8f #2 — EvidenceColumns::AppendJob over every group of the batch on caller-provided
// lgr_assign records (no device involved).  Returns the columns as a lgr_evidence_in that stays
// valid until the next call on this thread; key_out[3 s + 0..2] = group, variant (index within
// the group) and sample id of support s (at most key_cap supports are described).
const lgr_evidence_in* lgr_adapter_evidence_columns(const lgr_batch_in* in, const char* names, const char* samples,
                                                    const int* sample_id, const long long* start0, const long long* isize,
                                                    const unsigned short* sam_flag, const unsigned char* mapq,
                                                    const unsigned char* softclip, const lgr_assign* assign, int* key_out,
                                                    int key_cap) {
  static thread_local lancet_gpu::EvidenceColumns cols;
  static thread_local JobSet js;
  try {
    js = JobSet();
    BuildJobs(in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, js);
    cols.Clear();
    long long off = 0;
    std::vector<int> job_of_support;
    for (std::size_t g = 0; g < js.jobs.size(); ++g) {
      cols.AppendJob(js.jobs[g], assign + off, X31OfView);
      off += (long long)(js.jobs[g].n_reads * js.jobs[g].n_variants);
      job_of_support.resize(cols.NumSupports(), (int)g);
    }
    for (std::size_t s = 0; s < cols.NumSupports() && (int)s < key_cap; ++s) {
      const auto& k = cols.Keys()[s];
      const int v = (int)(static_cast<const lancet_gpu::VariantIn*>(k.variant) - js.vars.data());
      int sid = -1;
      for (std::size_t i = 0; i < js.sn.size(); ++i)
        if (js.sn[i] == k.sample) sid = (int)i;
      key_out[3 * s] = job_of_support[s], key_out[3 * s + 1] = v - in->grp_var_begin[job_of_support[s]], key_out[3 * s + 2] = sid;
    }
    return &cols.In();
  } catch (const std::exception&) {
    return nullptr;
  }
}

// The same columns through lancet_gpu::GpuFormatMetrics::Compute on `device`: out must hold one
// lgr_format per support (n_out of them); returns the number of supports, < 0 on error (message in err).
int lgr_adapter_format_metrics(int device, const lgr_batch_in* in, const char* names, const char* samples, const int* sample_id,
                               const long long* start0, const long long* isize, const unsigned short* sam_flag,
                               const unsigned char* mapq, const unsigned char* softclip, const lgr_assign* assign,
                               lgr_format* out, int n_out, char* err, int err_cap) {
  try {
    JobSet js;
    BuildJobs(in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, js);
    lancet_gpu::EvidenceColumns cols;
    long long off = 0;
    for (std::size_t g = 0; g < js.jobs.size(); ++g) {
      cols.AppendJob(js.jobs[g], assign + off, X31OfView);
      off += (long long)(js.jobs[g].n_reads * js.jobs[g].n_variants);
    }
    if ((int)cols.NumSupports() > n_out) throw std::runtime_error("output too small");
    lancet_gpu::GpuFormatMetrics fm(device);
    const std::vector<lgr_format> res = fm.Compute(cols);
    std::memcpy(out, res.data(), res.size() * sizeof(lgr_format));
    return (int)res.size();
  } catch (const std::exception& e) {
    std::snprintf(err, (size_t)err_cap, "%s", e.what());
    return -2;
  }
}

}  // extern "C"

namespace {

// The windows of a RepeatChecker run: window w = seqs[seq_off[w], seq_off[w] + seq_len[w]) with questions
// q_begin[w] .. q_begin[w + 1] of (q_k, q_mm); its answers go to answers[q_begin[w] ..].
struct RepeatWindows {
  const unsigned char* seqs;
  const long long* seq_off;
  const int* seq_len;
  int n_windows;
  const int* q_begin;
  const int* q_k;
  const int* q_mm;
  std::string_view Seq(int w) const { return {reinterpret_cast<const char*>(seqs) + seq_off[w], (std::size_t)seq_len[w]}; }
  std::vector<lancet_gpu::RepeatQuestion> Questions(int w) const {
    std::vector<lancet_gpu::RepeatQuestion> q;
    for (int i = q_begin[w]; i < q_begin[w + 1]; ++i) q.push_back(lancet_gpu::RepeatQuestion{q_k[i], q_mm[i]});
    return q;
  }
};

// n_threads threads; thread t asks windows t, t + n_threads, ... (only window t when one_each), one blocking call each,
// in order.  ask(w, t) returns the answers of window w; status[w] = 0 ok, 1 std::invalid_argument, 2 any other
// exception.  after_start(returned) runs on the calling thread once every thread is running; returned counts the calls
// that have come back.  Returns the wall nanoseconds from the start to the last join.
template <typename Ask, typename AfterStart>
unsigned long long RunWindows(const RepeatWindows& win, int n_threads, bool one_each, unsigned char* answers, int* status,
                              Ask ask, AfterStart after_start) {
  std::atomic<int> started{0}, returned{0};
  std::vector<std::thread> threads;
  const auto t0 = std::chrono::steady_clock::now();
  for (int t = 0; t < n_threads; ++t) {
    threads.emplace_back([&, t] {
      started.fetch_add(1);
      for (int w = t; w < win.n_windows; w += n_threads) {
        try {
          const std::vector<std::uint8_t> a = ask(w, t);
          std::memcpy(answers + win.q_begin[w], a.data(), a.size());
          status[w] = 0;
        } catch (const std::invalid_argument&) {
          status[w] = 1;
        } catch (const std::exception&) {
          status[w] = 2;
        }
        returned.fetch_add(1);
        if (one_each) break;
      }
    });
  }
  while (started.load() < n_threads) std::this_thread::yield();
  after_start(returned);
  for (auto& th : threads) th.join();
  return (unsigned long long)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace

extern "C" {

// lancet_gpu::RepeatChecker for the tests and tools/bench_repeat_checker.py.  NULL (message in err) when construction
// throws, e.g. without a GPU.
void* lgr_adapter_repeat_checker_create(int device, long long max_seq_bytes, long long max_questions, char* err, int err_cap) {
  try {
    lancet_gpu::RepeatChecker::Options opt;
    opt.device = device;
    if (max_seq_bytes > 0) opt.max_seq_bytes = (std::size_t)max_seq_bytes;
    if (max_questions > 0) opt.max_questions = (std::size_t)max_questions;
    return new lancet_gpu::RepeatChecker(opt);
  } catch (const std::exception& e) {
    if (err && err_cap > 0) std::snprintf(err, (size_t)err_cap, "%s", e.what());
    return nullptr;
  }
}

void lgr_adapter_repeat_checker_destroy(void* checker) { delete static_cast<lancet_gpu::RepeatChecker*>(checker); }

// n_threads C++ threads call RepeatChecker::Check on their share of the windows (see RunWindows).  counters[7] =
// batches, windows, questions, max windows in a batch, checker-thread ns inside lgr_repeat_scan, wall ns of the run,
// callers waiting when the checker was destroyed.  destroy != 0: thread t asks window t only (status of the windows
// beyond n_threads: -1), and once every thread is inside Check or back from it, the checker is destroyed while its
// callers wait (the caller must not destroy it again; counters[0..4] are then 0).
int lgr_adapter_repeat_checker_run(void* checker, const unsigned char* seqs, const long long* seq_off, const int* seq_len,
                                   int n_windows, const int* q_begin, const int* q_k, const int* q_mm, int n_threads,
                                   int destroy, unsigned char* answers, int* status, unsigned long long* counters) {
  if (!checker || n_threads <= 0 || n_windows < 0) return -1;
  auto* chk = static_cast<lancet_gpu::RepeatChecker*>(checker);
  const RepeatWindows win{seqs, seq_off, seq_len, n_windows, q_begin, q_k, q_mm};
  for (int i = 0; i < 7; ++i) counters[i] = 0;
  for (int w = 0; w < n_windows; ++w) status[w] = -1;
  const int askers = destroy ? std::min(n_threads, n_windows) : n_threads;
  const unsigned long long wall = RunWindows(
      win, askers, destroy != 0, answers, status,
      [&](int w, int) {
        const std::vector<lancet_gpu::RepeatQuestion> q = win.Questions(w);
        return chk->Check(win.Seq(w), q.data(), q.size());
      },
      [&](const std::atomic<int>& returned) {
        if (!destroy) return;
        // a thread that has not reached Check yet must not find the checker gone: wait until every one is inside
        // (counted by Callers) or back (returned, read first so that no thread is missed by both reads)
        for (;;) {
          const int back = returned.load();
          const std::size_t inside = chk->Callers();
          if (back + (int)inside >= askers) {
            counters[6] = inside;
            break;
          }
          std::this_thread::yield();
        }
        delete chk;
      });
  if (!destroy) {
    const lancet_gpu::RepeatChecker::Counters c = chk->Stats();
    counters[0] = c.batches, counters[1] = c.windows, counters[2] = c.questions, counters[3] = c.max_windows_in_batch;
    counters[4] = c.ns_wait;
  }
  counters[5] = wall;
  return 0;
}

// The binding without the checker, for comparison: every thread owns an lgr_rep_ctx (created before the clock starts)
// and makes one lgr_repeat_scan per window.  Returns the wall ns of the run, < 0 when a context cannot be created.
long long lgr_adapter_repeat_private_run(int device, const unsigned char* seqs, const long long* seq_off, const int* seq_len,
                                         int n_windows, const int* q_begin, const int* q_k, const int* q_mm, int n_threads,
                                         unsigned char* answers, int* status) {
  if (n_threads <= 0 || n_windows < 0) return -1;
  std::vector<lgr_rep_ctx*> ctx((size_t)n_threads, nullptr);
  bool ok = true;
  for (auto& c : ctx) ok = ok && lgr_repeat_create(device, &c) == LGR_OK;
  long long wall = -1;
  if (ok) {
    const RepeatWindows win{seqs, seq_off, seq_len, n_windows, q_begin, q_k, q_mm};
    wall = (long long)RunWindows(
        win, n_threads, false, answers, status,
        [&](int w, int t) {
          const int n = win.q_begin[w + 1] - win.q_begin[w];
          std::vector<lgr_repeat_job> jobs((size_t)n);
          for (int i = 0; i < n; ++i) jobs[(size_t)i] = lgr_repeat_job{0, win.seq_len[w], win.q_k[win.q_begin[w] + i], win.q_mm[win.q_begin[w] + i], 0};
          std::vector<std::uint8_t> a((size_t)n);
          const int rc = lgr_repeat_scan(ctx[(size_t)t], seqs + win.seq_off[w], win.seq_len[w], jobs.data(), n, a.data(), nullptr);
          if (rc != LGR_OK && rc != LGR_E_PARTIAL) throw std::runtime_error(lgr_repeat_last_error(ctx[(size_t)t]));
          return a;
        },
        [](const std::atomic<int>&) {});
  }
  for (auto* c : ctx) lgr_repeat_destroy(c);
  return wall;
}

}  // extern "C"

namespace {

// The windows of a FormatCalculator run: window w = supports win_sup_begin[w] .. win_sup_begin[w + 1] of the flat
// columns `all`, as a window-local lgr_evidence_in (sup_begin rebased to 0, columns offset to its first record).
// Built before any clock starts; records go to out[win_sup_begin[w] ..].
struct FormatWindows {
  std::vector<std::vector<std::int64_t>> begin;
  std::vector<lgr_evidence_in> in;
  const int* win_sup_begin;
  FormatWindows(const lgr_evidence_in* all, const int* wsb, int n_windows) : begin((std::size_t)n_windows), in((std::size_t)n_windows), win_sup_begin(wsb) {
    for (int w = 0; w < n_windows; ++w) {
      const int s0 = wsb[w], s1 = wsb[w + 1];
      const std::int64_t e0 = all->sup_begin[s0];
      auto& b = begin[(std::size_t)w];
      for (int s = s0; s <= s1; ++s) b.push_back(all->sup_begin[s] - e0);
      lgr_evidence_in& x = in[(std::size_t)w];
      x = *all;
      x.n_supports = s1 - s0, x.n_evidence = b.back();
      x.sup_begin = b.data(), x.sup_n_alleles = all->sup_n_alleles + s0, x.sup_variant_len = all->sup_variant_len + s0;
      x.sup_total_haps = all->sup_total_haps + s0;
      x.insert_size = all->insert_size + e0, x.aln_start = all->aln_start + e0, x.aln_score = all->aln_score + e0;
      x.folded_pos = all->folded_pos + e0, x.rname_hash = all->rname_hash + e0, x.ref_nm = all->ref_nm + e0;
      x.own_hap_nm = all->own_hap_nm + e0, x.hap_id = all->hap_id + e0, x.allele = all->allele + e0, x.flags = all->flags + e0;
      x.base_qual = all->base_qual + e0, x.map_qual = all->map_qual + e0;
    }
  }
};

// n_threads threads; thread t computes windows t, t + n_threads, ... in order, one blocking call each.  ask(w, t)
// returns the records of window w; status[w] = 0 ok, 1 std::invalid_argument, 2 any other exception.  Returns the wall
// nanoseconds from the start to the last join.
template <typename Ask>
unsigned long long RunFormatWindows(const FormatWindows& win, int n_threads, lgr_format* out, int* status, Ask ask) {
  const int n_windows = (int)win.in.size();
  std::vector<std::thread> threads;
  const auto t0 = std::chrono::steady_clock::now();
  for (int t = 0; t < n_threads; ++t) {
    threads.emplace_back([&, t] {
      for (int w = t; w < n_windows; w += n_threads) {
        try {
          const std::vector<lgr_format> r = ask(w, t);
          std::memcpy(out + win.win_sup_begin[w], r.data(), r.size() * sizeof(lgr_format));
          status[w] = 0;
        } catch (const std::invalid_argument&) {
          status[w] = 1;
        } catch (const std::exception&) {
          status[w] = 2;
        }
      }
    });
  }
  for (auto& th : threads) th.join();
  return (unsigned long long)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace

extern "C" {

// lancet_gpu::FormatCalculator for the tests and tools/bench_format_calculator.py.  Sizes <= 0 keep the defaults.
// NULL (message in err) when construction throws, e.g. without a GPU.
void* lgr_adapter_format_calculator_create(int device, long long slab_bytes, long long max_supports, long long max_evidence,
                                           char* err, int err_cap) {
  try {
    lancet_gpu::FormatCalculator::Options opt;
    opt.device = device;
    if (slab_bytes > 0) opt.slab_bytes = (std::size_t)slab_bytes;
    if (max_supports > 0) opt.max_supports = (std::size_t)max_supports;
    if (max_evidence > 0) opt.max_evidence = (std::size_t)max_evidence;
    return new lancet_gpu::FormatCalculator(opt);
  } catch (const std::exception& e) {
    if (err && err_cap > 0) std::snprintf(err, (size_t)err_cap, "%s", e.what());
    return nullptr;
  }
}

void lgr_adapter_format_calculator_destroy(void* calc) { delete static_cast<lancet_gpu::FormatCalculator*>(calc); }

// n_threads C++ threads call FormatCalculator::Compute on their share of the windows (see RunFormatWindows).
// counters[10] = batches, windows, supports, evidence, max windows in a batch, alone, ns_pack, ns_seal_wait, ns_device,
// wall ns of the run.
int lgr_adapter_format_calculator_run(void* calc, const lgr_evidence_in* all, const int* win_sup_begin, int n_windows,
                                      int n_threads, lgr_format* out, int* status, unsigned long long* counters) {
  if (!calc || !all || n_threads <= 0 || n_windows < 0) return -1;
  auto* fc = static_cast<lancet_gpu::FormatCalculator*>(calc);
  const FormatWindows win(all, win_sup_begin, n_windows);
  const unsigned long long wall = RunFormatWindows(win, n_threads, out, status, [&](int w, int) { return fc->Compute(win.in[(std::size_t)w]); });
  const lancet_gpu::FormatCalculator::Counters c = fc->Stats();
  const std::uint64_t v[10] = {c.batches, c.windows, c.supports, c.evidence, c.max_windows_in_batch, c.alone, c.ns_pack,
                               c.ns_seal_wait, c.ns_device, wall};
  for (int i = 0; i < 10; ++i) counters[i] = v[i];
  return 0;
}

// The binding without the calculator, for comparison: every thread owns an lgr_fmt_ctx (what GpuFormatMetrics wraps,
// created before the clock starts) and makes one lgr_format_metrics per window.  Returns the wall ns of the run, < 0
// when a context cannot be created.
long long lgr_adapter_format_private_run(int device, const lgr_evidence_in* all, const int* win_sup_begin, int n_windows,
                                         int n_threads, lgr_format* out, int* status) {
  if (!all || n_threads <= 0 || n_windows < 0) return -1;
  std::vector<lgr_fmt_ctx*> ctx((size_t)n_threads, nullptr);
  bool ok = true;
  for (auto& c : ctx) ok = ok && lgr_format_create(device, &c) == LGR_OK;
  long long wall = -1;
  if (ok) {
    const FormatWindows win(all, win_sup_begin, n_windows);
    wall = (long long)RunFormatWindows(win, n_threads, out, status, [&](int w, int t) {
      const lgr_evidence_in& x = win.in[(std::size_t)w];
      std::vector<lgr_format> r((std::size_t)std::max(x.n_supports, 0));
      const int rc = lgr_format_metrics(ctx[(size_t)t], &x, r.data(), nullptr);
      if (rc == LGR_E_ARG) throw std::invalid_argument(lgr_format_last_error(ctx[(size_t)t]));
      if (rc != LGR_OK && rc != LGR_E_PARTIAL) throw std::runtime_error(lgr_format_last_error(ctx[(size_t)t]));
      return r;
    });
  }
  for (auto* c : ctx) lgr_format_destroy(c);
  return wall;
}

// End to end: EvidenceColumns::AppendJob of every group of a realignment batch (the inputs of
// lgr_adapter_format_metrics), one window per group.  n_threads threads compute the windows through one
// FormatCalculator (out_calc), and GpuFormatMetrics::Compute computes the same columns (out_plain), both in the batch's
// support order.  Returns the number of supports, < 0 on error (message in err).
int lgr_adapter_format_calculator_columns(int device, const lgr_batch_in* in, const char* names, const char* samples,
                                          const int* sample_id, const long long* start0, const long long* isize,
                                          const unsigned short* sam_flag, const unsigned char* mapq, const unsigned char* softclip,
                                          const lgr_assign* assign, int n_threads, lgr_format* out_calc, lgr_format* out_plain,
                                          int n_out, char* err, int err_cap) {
  try {
    JobSet js;
    BuildJobs(in, names, samples, sample_id, start0, isize, sam_flag, mapq, softclip, js);
    std::vector<lancet_gpu::EvidenceColumns> cols(js.jobs.size());
    std::vector<int> first(js.jobs.size() + 1, 0);
    long long off = 0;
    for (std::size_t g = 0; g < js.jobs.size(); ++g) {
      cols[g].AppendJob(js.jobs[g], assign + off, X31OfView);
      off += (long long)(js.jobs[g].n_reads * js.jobs[g].n_variants);
      first[g + 1] = first[g] + (int)cols[g].NumSupports();
    }
    if (first.back() > n_out) throw std::runtime_error("output too small");
    lancet_gpu::GpuFormatMetrics fm(device);
    for (std::size_t g = 0; g < cols.size(); ++g) {
      const std::vector<lgr_format> r = fm.Compute(cols[g]);
      std::memcpy(out_plain + first[g], r.data(), r.size() * sizeof(lgr_format));
    }
    lancet_gpu::FormatCalculator fc(device);
    std::vector<std::thread> threads;
    std::vector<std::string> errors((std::size_t)std::max(n_threads, 1));
    for (int t = 0; t < n_threads; ++t)
      threads.emplace_back([&, t] {
        try {
          for (std::size_t g = (std::size_t)t; g < cols.size(); g += (std::size_t)n_threads) {
            const std::vector<lgr_format> r = fc.Compute(cols[g]);
            std::memcpy(out_calc + first[g], r.data(), r.size() * sizeof(lgr_format));
          }
        } catch (const std::exception& e) {
          errors[(std::size_t)t] = e.what();
        }
      });
    for (auto& th : threads) th.join();
    for (const std::string& e : errors)
      if (!e.empty()) throw std::runtime_error(e);
    return first.back();
  } catch (const std::exception& e) {
    std::snprintf(err, (size_t)err_cap, "%s", e.what());
    return -2;
  }
}

}  // extern "C"
