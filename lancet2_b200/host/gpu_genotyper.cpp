// gpu_genotyper.cpp — see gpu_genotyper.h.  Host logic only: batch building, the C-ABI call,
// and AddToTable/AddEvidence in the reference's read order.
#include "gpu_genotyper.h"

#include "../csrc/lgr_pack.h"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

namespace lancet_gpu {

// variant_support.cpp:23-67 (EnsureAlleleSlot + first-seen-wins dedup on the name hash)
void VariantSupport::AddEvidence(ReadEvidence const& ev) {
  if (mAlleleData.size() <= ev.mAllele) mAlleleData.resize(static_cast<std::size_t>(ev.mAllele) + 1);
  PerAlleleData& data = mAlleleData[ev.mAllele];
  if (!data.mNameHashes.try_emplace(ev.mRnameHash, ev.mStrand).second) return;
  if (ev.mStrand == Strand::FWD) data.mFwdBaseQuals.push_back(ev.mBaseQual);
  else data.mRevBaseQuals.push_back(ev.mBaseQual);
  data.mMapQuals.push_back(ev.mMapQual);
  data.mAlnScores.push_back(ev.mAlnScore);
  if (ev.mIsSoftClipped) ++data.mSoftClipCount;
  if (ev.mIsProperPair && ev.mInsertSize != 0) data.mProperPairIsizes.push_back(static_cast<double>(ev.mInsertSize));
  data.mFoldedReadPositions.push_back(ev.mFoldedReadPos);
  data.mRefNmValues.push_back(static_cast<double>(ev.mRefNm));
  data.mAlignmentStarts.push_back(ev.mAlignmentStart);
  data.mOwnHapNmValues.push_back(static_cast<double>(ev.mOwnHapNm));
  data.mHaplotypeIds.push_back(ev.mAssignedHaplotypeId);
}

// support_array.cpp:19-28
VariantSupport& SupportArray::FindOrCreate(std::string_view sample_name) {
  for (auto& item : mItems)
    if (item.mSampleName == sample_name) return *item.mData;
  mItems.push_back(NamedSupport{sample_name, std::make_unique<VariantSupport>()});
  return *mItems.back().mData;
}

static void Check(lgr_ctx* ctx, int rc) {
  if (rc != LGR_OK) {
    std::string msg = lgr_strerror(rc);
    const char* detail = lgr_last_error(ctx);
    if (detail && *detail) msg += std::string(": ") + detail;
    throw std::runtime_error("lancet_gpu::GpuGenotyper: " + msg);
  }
}

// ---------------------------------------------------------------------------------------------
// PackedBatch
// ---------------------------------------------------------------------------------------------
template <typename T>
void PackedBatch::Free(Buf<T>& b) {
  if (b.p) {
    if (b.pinned) lgr_free_pinned(b.p);
    else std::free(b.p);
  }
  b.p = nullptr, b.n = b.cap = 0;
}

template <typename T>
void PackedBatch::Reserve(Buf<T>& b, std::size_t n) {
  if (n <= b.cap) return;
  std::size_t cap = b.cap ? b.cap : 256;
  while (cap < n) cap = cap * 2 + 64;  // pinned allocations are slow: grow rarely
  bool pinned = true;
  T* p = static_cast<T*>(lgr_alloc_pinned(cap * sizeof(T)));
  if (!p) {
    pinned = false;
    p = static_cast<T*>(std::malloc(cap * sizeof(T)));
    if (!p) throw std::bad_alloc();
  }
  if (b.n) std::memcpy(p, b.p, b.n * sizeof(T));
  const std::size_t keep = b.n;
  Free(b);
  b.p = p, b.n = keep, b.cap = cap, b.pinned = pinned;
}

template <typename T>
void PackedBatch::Push(Buf<T>& b, T v) {
  if (b.n == b.cap) Reserve(b, b.n + 1);
  b.p[b.n++] = v;
}

template <typename T>
void PackedBatch::Append(Buf<T>& b, const T* src, std::size_t n) {
  Reserve(b, b.n + n + 1);
  if (n) std::memcpy(b.p + b.n, src, n * sizeof(T));
  b.n += n;
}

PackedBatch::~PackedBatch() {
  Free(mGhb), Free(mGrb), Free(mGvb), Free(mGmid), Free(mVarStart), Free(mVarLen);
  Free(mHapOff), Free(mReadOff), Free(mVarHapOff);
  Free(mHapBases), Free(mReadBases), Free(mReadQuals);
  Free(mX31), Free(mVarAllele), Free(mAssign);
}

void PackedJob::Build(const GenotypeJob& j) {
  n_haps = j.n_haps, n_reads = j.n_reads, n_variants = j.n_variants;
  hap_bases.clear(), read_bases.clear(), read_quals.clear(), x31.clear();
  var_start.clear(), var_len.clear(), var_allele.clear();
  hap_off.assign(1, 0), read_off.assign(1, 0), var_hap_off.assign(1, 0);
  std::size_t hap_total = 0, read_total = 0;
  for (std::size_t h = 0; h < j.n_haps; ++h) hap_total += j.haps[h].size();
  for (std::size_t r = 0; r < j.n_reads; ++r) read_total += j.reads[r].seq.size();
  hap_bases.reserve(hap_total), read_bases.reserve(read_total), read_quals.reserve(read_total);
  x31.reserve(j.n_reads), read_off.reserve(j.n_reads + 1), hap_off.reserve(j.n_haps + 1);
  for (std::size_t h = 0; h < j.n_haps; ++h) {
    hap_bases.insert(hap_bases.end(), j.haps[h].begin(), j.haps[h].end());
    hap_off.push_back(static_cast<std::int64_t>(hap_bases.size()));
  }
  std::string qn;
  for (std::size_t r = 0; r < j.n_reads; ++r) {
    const ReadIn& rd = j.reads[r];
    read_bases.insert(read_bases.end(), rd.seq.begin(), rd.seq.end());
    read_quals.insert(read_quals.end(), rd.qual, rd.qual + rd.seq.size());
    read_off.push_back(static_cast<std::int64_t>(read_bases.size()));
    qn.assign(rd.qname);  // mm_map receives the NUL-terminated QnamePtr()
    x31.push_back(lgr_x31_hash(qn.c_str()));
  }
  for (std::size_t v = 0; v < j.n_variants; ++v) {
    const VariantIn& var = j.variants[v];
    for (std::size_t h = 0; h < j.n_haps; ++h) {  // ExtractHapBounds (genotyper.cpp:329-352)
      std::int32_t st = -1, ln = 0;
      std::int8_t al = -1;
      if (h == 0) {
        st = static_cast<std::int32_t>(var.local_ref_start0), ln = static_cast<std::int32_t>(var.ref_allele_len), al = 0;
      } else {
        for (std::size_t a = 0; a < var.alts.size() && al < 0; ++a)
          for (const auto& kv : var.alts[a].hap_start0)
            if (kv.first == h) {
              st = static_cast<std::int32_t>(kv.second), ln = static_cast<std::int32_t>(var.alts[a].seq_len);
              al = static_cast<std::int8_t>(a + 1);
              break;
            }
      }
      var_start.push_back(st), var_len.push_back(ln), var_allele.push_back(al);
    }
    var_hap_off.push_back(static_cast<std::int64_t>(var_start.size()));
  }
}

void PackedBatch::Pack(const GenotypeJob* jobs, std::size_t n_jobs, std::int32_t latched_mid_occ) {
  std::vector<PackedJob> packed(n_jobs);
  std::vector<const PackedJob*> ptrs(n_jobs);
  for (std::size_t g = 0; g < n_jobs; ++g) packed[g].Build(jobs[g]), ptrs[g] = &packed[g];
  PackPrepared(ptrs.data(), n_jobs, latched_mid_occ);
}

void PackedBatch::PackPrepared(const PackedJob* const* jobs, std::size_t n_jobs, std::int32_t latched_mid_occ) {
  for (auto* b : {&mGhb, &mGrb, &mGvb, &mGmid, &mVarStart, &mVarLen}) b->n = 0;
  for (auto* b : {&mHapOff, &mReadOff, &mVarHapOff}) b->n = 0;
  for (auto* b : {&mHapBases, &mReadBases, &mReadQuals}) b->n = 0;
  mX31.n = 0, mVarAllele.n = 0;
  mJobAsg.clear();
  // sizes first: one reservation per array, then straight block copies
  std::size_t nh = 0, nr = 0, nv = 0, hb = 0, rb = 0, vh = 0;
  for (std::size_t g = 0; g < n_jobs; ++g) {
    const PackedJob& j = *jobs[g];
    nh += j.n_haps, nr += j.n_reads, nv += j.n_variants;
    hb += j.hap_bases.size(), rb += j.read_bases.size(), vh += j.var_start.size();
  }
  Reserve(mGhb, n_jobs + 2), Reserve(mGrb, n_jobs + 2), Reserve(mGvb, n_jobs + 2), Reserve(mGmid, n_jobs + 1);
  Reserve(mHapOff, nh + 2), Reserve(mReadOff, nr + 2), Reserve(mVarHapOff, nv + 2);
  Reserve(mHapBases, hb + 1), Reserve(mReadBases, rb + 1), Reserve(mReadQuals, rb + 1);
  Reserve(mX31, nr + 1), Reserve(mVarStart, vh + 1), Reserve(mVarLen, vh + 1), Reserve(mVarAllele, vh + 1);
  Push<std::int32_t>(mGhb, 0), Push<std::int32_t>(mGrb, 0), Push<std::int32_t>(mGvb, 0);
  Push<std::int64_t>(mHapOff, 0), Push<std::int64_t>(mReadOff, 0), Push<std::int64_t>(mVarHapOff, 0);
  std::int64_t n_assign = 0;
  mPairs = 0;
  auto rebase = [](Buf<std::int64_t>& dst, const std::vector<std::int64_t>& rel, std::int64_t base) {
    for (std::size_t i = 1; i < rel.size(); ++i) dst.p[dst.n++] = rel[i] + base;
  };
  for (std::size_t g = 0; g < n_jobs; ++g) {
    const PackedJob& j = *jobs[g];
    rebase(mHapOff, j.hap_off, static_cast<std::int64_t>(mHapBases.n));
    rebase(mReadOff, j.read_off, static_cast<std::int64_t>(mReadBases.n));
    rebase(mVarHapOff, j.var_hap_off, static_cast<std::int64_t>(mVarStart.n));
    Append(mHapBases, j.hap_bases.data(), j.hap_bases.size());
    Append(mReadBases, j.read_bases.data(), j.read_bases.size());
    Append(mReadQuals, j.read_quals.data(), j.read_quals.size());
    Append(mX31, j.x31.data(), j.x31.size());
    Append(mVarStart, j.var_start.data(), j.var_start.size());
    Append(mVarLen, j.var_len.data(), j.var_len.size());
    Append(mVarAllele, j.var_allele.data(), j.var_allele.size());
    Push(mGhb, mGhb.p[g] + static_cast<std::int32_t>(j.n_haps));
    Push(mGrb, mGrb.p[g] + static_cast<std::int32_t>(j.n_reads));
    Push(mGvb, mGvb.p[g] + static_cast<std::int32_t>(j.n_variants));
    Push(mGmid, latched_mid_occ);
    mJobAsg.push_back(n_assign);
    n_assign += static_cast<std::int64_t>(j.n_reads) * static_cast<std::int64_t>(j.n_variants);
    mPairs += static_cast<std::int64_t>(j.n_reads) * static_cast<std::int64_t>(j.n_haps);
  }
  Reserve(mAssign, static_cast<std::size_t>(n_assign) + 1);
  mAssign.n = static_cast<std::size_t>(n_assign);
  const int G = static_cast<int>(n_jobs);
  std::memset(&mIn, 0, sizeof(mIn));
  mIn.n_groups = G, mIn.n_haps = mGhb.p[G], mIn.n_reads = mGrb.p[G], mIn.n_vars = mGvb.p[G];
  mIn.grp_hap_begin = mGhb.p, mIn.grp_read_begin = mGrb.p, mIn.grp_var_begin = mGvb.p;
  mIn.hap_off = mHapOff.p, mIn.hap_bases = mHapBases.p;
  mIn.read_off = mReadOff.p, mIn.read_bases = mReadBases.p, mIn.read_quals = mReadQuals.p;
  mIn.read_name_hash = mX31.p;
  mIn.var_hap_off = mVarHapOff.p, mIn.var_start = mVarStart.p, mIn.var_len = mVarLen.p, mIn.var_allele = mVarAllele.p;
  mIn.grp_mid_occ = latched_mid_occ > 0 ? mGmid.p : nullptr;
  std::memset(&mOut, 0, sizeof(mOut));
  mOut.n_assign = n_assign;
  mOut.assign = mAssign.p;  // out.aln stays NULL: the adapter only needs the assignments
}

Result PackedBatch::BuildResult(const GenotypeJob& j, const lgr_assign* assign, const NameHashFn& name_hash) {
  Result table;
  for (std::size_t r = 0; r < j.n_reads; ++r) {
    const ReadIn& rd = j.reads[r];
    std::uint32_t rname_hash = 0;
    bool hashed = false;
    for (std::size_t v = 0; v < j.n_variants; ++v) {
      const lgr_assign& a = assign[r * j.n_variants + v];
      if (!a.assigned) continue;
      if (!hashed) rname_hash = name_hash(rd.qname), hashed = true;
      VariantSupport& support = table[j.variants[v].key].FindOrCreate(rd.sample_name);
      ReadEvidence ev;
      ev.mInsertSize = rd.insert_size;
      ev.mAlignmentStart = rd.start0;
      ev.mAlnScore = static_cast<double>(a.global_score) + (a.local_score * a.local_identity);  // CombinedScore()
      ev.mFoldedReadPos = a.folded_read_pos;
      ev.mRnameHash = rname_hash;
      ev.mRefNm = a.ref_nm, ev.mOwnHapNm = a.own_hap_nm, ev.mAssignedHaplotypeId = a.hap_id;
      ev.mAllele = static_cast<AlleleIndex>(a.allele);
      ev.mStrand = (rd.sam_flag & 0x10) ? Strand::REV : Strand::FWD;
      ev.mBaseQual = a.base_qual, ev.mMapQual = rd.map_qual;
      ev.mIsSoftClipped = rd.is_soft_clipped;
      ev.mIsProperPair = (rd.sam_flag & 0x2) != 0;
      support.AddEvidence(ev);
    }
  }
  return table;
}

// ---------------------------------------------------------------------------------------------
// EvidenceColumns / GpuFormatMetrics (SURVEY.md §8f #2)
// ---------------------------------------------------------------------------------------------
void EvidenceColumns::Clear() {
  mKeys.clear();
  mSupBegin.assign(1, 0);
  for (auto* v : {&mInsertSize, &mAlnStart}) v->clear();
  for (auto* v : {&mNumAlleles, &mVariantLen, &mTotalHaps}) v->clear();
  for (auto* v : {&mAlnScore, &mFoldedPos}) v->clear();
  for (auto* v : {&mRnameHash, &mRefNm, &mOwnHapNm, &mHapId}) v->clear();
  for (auto* v : {&mAllele, &mFlags, &mBaseQual, &mMapQual}) v->clear();
}

void EvidenceColumns::AppendJob(const GenotypeJob& j, const lgr_assign* assign, const NameHashFn& name_hash) {
  // name hashes once per read that has any assignment (AddToTable hashes once per read, genotyper.cpp:426)
  std::vector<std::uint32_t> hash(j.n_reads, 0);
  for (std::size_t r = 0; r < j.n_reads; ++r)
    for (std::size_t v = 0; v < j.n_variants; ++v)
      if (assign[r * j.n_variants + v].assigned) {
        hash[r] = name_hash(j.reads[r].qname);
        break;
      }
  std::vector<std::string_view> samples;  // FindOrCreate's creation order for this variant
  for (std::size_t v = 0; v < j.n_variants; ++v) {
    const VariantIn& var = j.variants[v];
    samples.clear();
    for (std::size_t r = 0; r < j.n_reads; ++r) {
      if (!assign[r * j.n_variants + v].assigned) continue;
      const std::string_view s = j.reads[r].sample_name;
      bool seen = false;
      for (const auto& x : samples) seen = seen || x == s;
      if (!seen) samples.push_back(s);
    }
    std::int64_t max_len = 0;  // variant_call.cpp:179-182: max |mLength| over the ALTs
    for (const auto& alt : var.alts) max_len = std::max<std::int64_t>(max_len, alt.length < 0 ? -alt.length : alt.length);
    for (const auto& sample : samples) {
      for (std::size_t r = 0; r < j.n_reads; ++r) {
        const lgr_assign& a = assign[r * j.n_variants + v];
        const ReadIn& rd = j.reads[r];
        if (!a.assigned || rd.sample_name != sample) continue;
        mInsertSize.push_back(rd.insert_size);
        mAlnStart.push_back(rd.start0);
        mAlnScore.push_back(static_cast<double>(a.global_score) + (a.local_score * a.local_identity));  // CombinedScore()
        mFoldedPos.push_back(a.folded_read_pos);
        mRnameHash.push_back(hash[r]);
        mRefNm.push_back(a.ref_nm), mOwnHapNm.push_back(a.own_hap_nm), mHapId.push_back(a.hap_id);
        mAllele.push_back(static_cast<std::uint8_t>(a.allele));
        mFlags.push_back(static_cast<std::uint8_t>(((rd.sam_flag & 0x10) ? LGR_EV_REV : 0u) | (rd.is_soft_clipped ? LGR_EV_SOFTCLIP : 0u) |
                                                   ((rd.sam_flag & 0x2) ? LGR_EV_PROPER_PAIR : 0u)));
        mBaseQual.push_back(a.base_qual), mMapQual.push_back(rd.map_qual);
      }
      mKeys.push_back(SupportKey{var.key, sample});
      mSupBegin.push_back(static_cast<std::int64_t>(mAllele.size()));
      mNumAlleles.push_back(static_cast<std::int32_t>(1 + var.alts.size()));
      mVariantLen.push_back(static_cast<std::int32_t>(max_len));
      mTotalHaps.push_back(static_cast<std::int32_t>(j.n_haps));
    }
  }
}

const lgr_evidence_in& EvidenceColumns::In() {
  mIn = lgr_evidence_in{};
  mIn.n_supports = static_cast<std::int32_t>(mKeys.size());
  mIn.n_evidence = static_cast<std::int64_t>(mAllele.size());
  mIn.sup_begin = mSupBegin.data(), mIn.sup_n_alleles = mNumAlleles.data();
  mIn.sup_variant_len = mVariantLen.data(), mIn.sup_total_haps = mTotalHaps.data();
  mIn.insert_size = mInsertSize.data(), mIn.aln_start = mAlnStart.data();
  mIn.aln_score = mAlnScore.data(), mIn.folded_pos = mFoldedPos.data();
  mIn.rname_hash = mRnameHash.data(), mIn.ref_nm = mRefNm.data(), mIn.own_hap_nm = mOwnHapNm.data(), mIn.hap_id = mHapId.data();
  mIn.allele = mAllele.data(), mIn.flags = mFlags.data(), mIn.base_qual = mBaseQual.data(), mIn.map_qual = mMapQual.data();
  return mIn;
}

GpuFormatMetrics::GpuFormatMetrics(int device_ordinal) {
  const int rc = lgr_format_create(device_ordinal, &mCtx);
  if (rc != LGR_OK)
    throw std::runtime_error(std::string("lancet_gpu::GpuFormatMetrics: ") + lgr_strerror(rc) + ": " + lgr_format_last_error(nullptr));
}

GpuFormatMetrics::~GpuFormatMetrics() { lgr_format_destroy(mCtx); }

std::vector<lgr_format> GpuFormatMetrics::Compute(EvidenceColumns& columns, float* ms_kernels) {
  std::vector<lgr_format> out(columns.NumSupports());
  const int rc = lgr_format_metrics(mCtx, &columns.In(), out.data(), ms_kernels);
  // LGR_E_PARTIAL: supports of sites with more than LGR_FMT_MAX_ALLELES alleles come back flagged LGR_FMT_WIDE
  // (variant_support.cpp:294-335 takes any K); they do not fail the batch
  if (rc != LGR_OK && rc != LGR_E_PARTIAL)
    throw std::runtime_error(std::string("lancet_gpu::GpuFormatMetrics: ") + lgr_strerror(rc) + ": " + lgr_format_last_error(mCtx));
  return out;
}

// ---------------------------------------------------------------------------------------------
// GpuGenotyper
// ---------------------------------------------------------------------------------------------
GpuGenotyper::GpuGenotyper(int device_ordinal, const lgr_params* params) {
  if (params) mParams = *params;
  else lgr_default_params(&mParams);
  Check(nullptr, lgr_create(device_ordinal, &mParams, &mCtx));
  mBatch = std::make_unique<PackedBatch>();
}

GpuGenotyper::~GpuGenotyper() {
  mBatch.reset();
  lgr_destroy(mCtx);
}

void GpuGenotyper::SetGraphMode(bool on) { Check(mCtx, lgr_set_graph_mode(mCtx, on ? 1 : 0)); }

Result GpuGenotyper::Genotype(const std::string* haps, std::size_t n_haps, const ReadIn* reads, std::size_t n_reads,
                              const VariantIn* variants, std::size_t n_variants, const NameHashFn& name_hash) {
  std::vector<GenotypeJob> jobs{GenotypeJob{haps, n_haps, reads, n_reads, variants, n_variants}};
  return std::move(GenotypeMany(jobs, name_hash)[0]);
}

// mm_mapopt_update latches mid_occ from the first index a Genotyper ever builds
// (genotyper.cpp:263-266); later haplotypes never refresh it.
static void LatchMidOcc(lgr_ctx* ctx, const lgr_params& prm, const GenotypeJob* jobs, std::size_t n, std::int32_t* latched) {
  if (prm.mid_occ > 0 || *latched > 0) return;
  for (std::size_t i = 0; i < n; ++i) {
    if (jobs[i].n_haps == 0) continue;
    Check(ctx, lgr_hap_mid_occ(ctx, reinterpret_cast<const std::uint8_t*>(jobs[i].haps[0].data()),
                               static_cast<std::int32_t>(jobs[i].haps[0].size()), latched));
    return;
  }
}

std::vector<Result> GpuGenotyper::GenotypeMany(const std::vector<GenotypeJob>& jobs, const NameHashFn& name_hash) {
  std::vector<Result> results(jobs.size());
  if (jobs.empty()) return results;
  LatchMidOcc(mCtx, mParams, jobs.data(), jobs.size(), &mLatchedMidOcc);
  mBatch->Pack(jobs.data(), jobs.size(), mLatchedMidOcc);
  Check(mCtx, lgr_genotype_batch(mCtx, &mBatch->In(), &mBatch->Out(), &mStats));
  for (std::size_t g = 0; g < jobs.size(); ++g) results[g] = PackedBatch::BuildResult(jobs[g], mBatch->JobAssign(g), name_hash);
  return results;
}

// ---------------------------------------------------------------------------------------------
// GenotypeBatcher
// ---------------------------------------------------------------------------------------------
static std::uint64_t NowNs() {
  return static_cast<std::uint64_t>(
      std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count());
}

// minimap2's __ac_X31_hash_string over the read name as mm_map sees it (a C string: stops at NUL)
static std::uint32_t X31(std::string_view q) {
  if (q.empty() || q[0] == '\0') return 0;
  std::uint32_t h = static_cast<std::uint32_t>(static_cast<std::int32_t>(static_cast<signed char>(q[0])));
  for (std::size_t i = 1; i < q.size() && q[i] != '\0'; ++i)
    h = (h << 5) - h + static_cast<std::uint32_t>(static_cast<std::int32_t>(static_cast<signed char>(q[i])));
  return h;
}

namespace {
// per-thread scratch of Enqueue: the lgr_group_desc view of one payload (no allocation in steady state)
struct PackScratch {
  std::vector<const std::uint8_t*> hap_seq, read_seq, read_qual;
  std::vector<std::int32_t> hap_len, read_len, var_start, var_len;
  std::vector<std::uint32_t> x31;
  std::vector<std::int8_t> var_allele;
  lgr_pack::Plan last_plan;  // quality dictionary of this thread's previous payload
  bool have_plan = false;
};

void DescribeJob(const GenotypeJob& j, PackScratch& sc, lgr_group_desc* d) {
  sc.hap_seq.resize(j.n_haps), sc.hap_len.resize(j.n_haps);
  for (std::size_t h = 0; h < j.n_haps; ++h) {
    sc.hap_seq[h] = reinterpret_cast<const std::uint8_t*>(j.haps[h].data());
    sc.hap_len[h] = static_cast<std::int32_t>(j.haps[h].size());
  }
  sc.read_seq.resize(j.n_reads), sc.read_qual.resize(j.n_reads), sc.read_len.resize(j.n_reads), sc.x31.resize(j.n_reads);
  for (std::size_t r = 0; r < j.n_reads; ++r) {
    const ReadIn& rd = j.reads[r];
    sc.read_seq[r] = reinterpret_cast<const std::uint8_t*>(rd.seq.data());
    sc.read_qual[r] = rd.qual;
    sc.read_len[r] = static_cast<std::int32_t>(rd.seq.size());
    sc.x31[r] = X31(rd.qname);
  }
  const std::size_t vh = j.n_variants * j.n_haps;
  sc.var_start.assign(vh, -1), sc.var_len.assign(vh, 0), sc.var_allele.assign(vh, -1);
  for (std::size_t v = 0; v < j.n_variants; ++v) {  // ExtractHapBounds (genotyper.cpp:329-352)
    const VariantIn& var = j.variants[v];
    const std::size_t row = v * j.n_haps;
    if (j.n_haps > 0) {
      sc.var_start[row] = static_cast<std::int32_t>(var.local_ref_start0);
      sc.var_len[row] = static_cast<std::int32_t>(var.ref_allele_len);
      sc.var_allele[row] = 0;
    }
    for (std::size_t a = 0; a < var.alts.size(); ++a)
      for (const auto& kv : var.alts[a].hap_start0) {
        const std::size_t h = kv.first;
        if (h == 0 || h >= j.n_haps || sc.var_allele[row + h] >= 0) continue;  // first ALT that lists the haplotype wins
        sc.var_start[row + h] = static_cast<std::int32_t>(kv.second);
        sc.var_len[row + h] = static_cast<std::int32_t>(var.alts[a].seq_len);
        sc.var_allele[row + h] = static_cast<std::int8_t>(a + 1);
      }
  }
  d->n_haps = static_cast<std::int32_t>(j.n_haps), d->n_reads = static_cast<std::int32_t>(j.n_reads);
  d->n_vars = static_cast<std::int32_t>(j.n_variants), d->mid_occ = 0;
  d->hap_seq = sc.hap_seq.data(), d->hap_len = sc.hap_len.data();
  d->read_seq = sc.read_seq.data(), d->read_qual = sc.read_qual.data(), d->read_len = sc.read_len.data();
  d->read_name_hash = sc.x31.data();
  d->var_start = sc.var_start.data(), d->var_len = sc.var_len.data(), d->var_allele = sc.var_allele.data();
}

std::atomic<std::uint64_t> g_latch_uid{1};
// mm_mapopt_update latch of the calling thread, per batcher / dispatcher instance
std::int32_t* ThreadLatch(std::uint64_t uid) {
  thread_local std::unordered_map<std::uint64_t, std::int32_t> latches;
  return &latches[uid];
}
}  // namespace

// per calling thread: device context + pinned staging of the blocking Genotype() path (GenotypeDirect below)
struct GenotypeBatcher::DirectSlot {
  lgr_ctx* ctx = nullptr;
  std::uint8_t* slab = nullptr;
  std::size_t slab_cap = 0;
  lgr_assign* assign = nullptr;  // pinned [assign_cap + 1] followed by one int32 status
  std::size_t assign_cap = 0;
  std::int64_t graph_replayed = 0;  // lgr_graph_counters of ctx after the previous call
  PackScratch sc;
  ~DirectSlot() {
    if (ctx) lgr_destroy(ctx);
    if (slab) lgr_free_pinned(slab);
    if (assign) lgr_free_pinned(assign);
  }
};

// results of one device batch: lives until the last of its payloads has been collected, while the
// staging slab it came from goes back to the pool as soon as the device is done with it (a worker may
// enqueue many windows before it collects the first)
struct GenotypeBatcher::ResultBlock {
  // one pinned block: [lgr_assign x assign_cap][int32 status x max_jobs], (re)allocated at seal time by the
  // batcher thread — never while mMu is held: CUDA's host allocator may wait for the device, and the
  // device's completion callback (OnDeviceDone) needs mMu
  lgr_assign* assign = nullptr;
  std::size_t assign_cap = 0;
  std::int32_t* status = nullptr;      // lgr_batch_out::grp_status
  std::vector<std::int64_t> job_asg;   // [max_jobs] first lgr_assign record of every payload
  std::vector<std::int32_t> job_mid;   // [max_jobs] mid_occ the payload was packed with (for a re-run alone)
  std::uint32_t refs = 0;              // payloads not yet released
  bool done = false;
  int rc = LGR_OK;
  std::string err;
};

struct GenotypeBatcher::Slab {
  std::uint8_t* mem = nullptr;  // pinned: group records, then (at seal time) the directory
  std::size_t cap = 0, used = 0;
  std::vector<lgr_group_dir> dir;      // [max_jobs], entry written by the payload's worker
  std::uint32_t n_jobs = 0;
  std::int64_t pairs = 0, n_assign = 0;
  std::atomic<int> packing{0};         // workers still writing their record
  ResultBlock* res = nullptr;
  lgr_packed_in in{};
  lgr_batch_out out{};
  lgr_ticket ticket = -1;
  std::uint64_t opened_ns = 0;         // when the batcher thread first saw jobs in this slab
};

static void* PinnedOrThrow(std::size_t bytes) {
  void* p = lgr_alloc_pinned(bytes);
  if (!p) throw std::bad_alloc();
  return p;
}

GenotypeBatcher::GenotypeBatcher(const Options& opt, NameHashFn name_hash) : mOpt(opt), mNameHash(std::move(name_hash)) {
  // tuning knobs without a rebuild (tools/bench_batcher.py sweeps them); unset = the Options given
  auto env_int = [](const char* name, long long cur) {
    const char* v = std::getenv(name);
    return v && *v ? std::atoll(v) : cur;
  };
  mOpt.depth = static_cast<int>(env_int("LGR_BATCHER_DEPTH", mOpt.depth));
  mOpt.min_pairs_busy = env_int("LGR_BATCHER_MIN_PAIRS", mOpt.min_pairs_busy);
  mOpt.max_wait_us = static_cast<int>(env_int("LGR_BATCHER_MAX_WAIT_US", mOpt.max_wait_us));
  mOpt.linger_us = static_cast<int>(env_int("LGR_BATCHER_LINGER_US", mOpt.linger_us));
  mOpt.direct_blocking_callers = static_cast<int>(env_int("LGR_BATCHER_DIRECT", mOpt.direct_blocking_callers));
  if (mOpt.depth < 1) mOpt.depth = 1;
  if (mOpt.depth > LGR_MAX_INFLIGHT) mOpt.depth = LGR_MAX_INFLIGHT;
  if (mOpt.max_jobs < 1) mOpt.max_jobs = 1;
  if (mOpt.slab_bytes < (1u << 16)) mOpt.slab_bytes = 1u << 16;
  if (opt.params) mParams = *opt.params;
  else lgr_default_params(&mParams);
  mOpt.params = nullptr;
  mUid = g_latch_uid.fetch_add(1);
  Check(nullptr, lgr_create(mOpt.device, &mParams, &mCtx));
  Check(nullptr, lgr_create(mOpt.device, &mParams, &mAuxCtx));
  Check(mCtx, lgr_set_notify(mCtx, &GenotypeBatcher::OnDeviceDone, this));
  mOpt.arena_reserve_bytes = env_int("LGR_BATCHER_ARENA_MB", mOpt.arena_reserve_bytes >> 20) << 20;
  if (mOpt.arena_reserve_bytes > 0) Check(mCtx, lgr_reserve(mCtx, mOpt.arena_reserve_bytes, mOpt.depth));
  const int n_slabs = mOpt.depth + 2;  // in flight + one filling + one waiting for a device slot
  for (int i = 0; i < n_slabs; ++i) {
    auto s = std::make_unique<Slab>();
    s->cap = mOpt.slab_bytes;
    s->mem = static_cast<std::uint8_t*>(PinnedOrThrow(s->cap));
    s->dir.resize(mOpt.max_jobs);
    mFree.push_back(s.get());
    mSlabs.push_back(std::move(s));
  }
  // result blocks are sized once, generously: growing one means cudaFreeHost + cudaHostAlloc (hundreds of
  // microseconds on the batcher thread, and a device-wide synchronisation) — measured as the bulk of the
  // per-batch submit time when the blocks were sized to each batch
  for (int i = 0; i < n_slabs + 2; ++i) {
    auto r = std::make_unique<ResultBlock>();
    r->job_asg.resize(mOpt.max_jobs), r->job_mid.resize(mOpt.max_jobs);
    r->assign_cap = mOpt.result_records;
    r->assign = static_cast<lgr_assign*>(PinnedOrThrow(r->assign_cap * sizeof(lgr_assign) + sizeof(std::int32_t) * mOpt.max_jobs));
    r->status = reinterpret_cast<std::int32_t*>(r->assign + r->assign_cap);
    mFreeResults.push_back(r.get());
    mResults.push_back(std::move(r));
  }
  mThread = std::thread([this] { Run(); });
}

GenotypeBatcher::~GenotypeBatcher() {
  {
    std::lock_guard<std::mutex> lk(mMu);
    mStop = true;
  }
  mCv.notify_all();
  mFreeCv.notify_all();
  if (mThread.joinable()) mThread.join();
  lgr_destroy(mCtx);
  lgr_destroy(mAuxCtx);
  for (auto& s : mSlabs) lgr_free_pinned(s->mem);
  for (auto& r : mResults) lgr_free_pinned(r->assign);
  mSlabs.clear();
  mResults.clear();
}

void GenotypeBatcher::OnDeviceDone(void* self, lgr_ticket ticket) {  // CUDA-owned thread: no CUDA / library calls here
  auto* b = static_cast<GenotypeBatcher*>(self);
  {
    std::lock_guard<std::mutex> lk(b->mMu);
    b->mDeviceDone |= 1u << ticket;
  }
  b->mCv.notify_all();
}

// an empty slab with room for `need_bytes` of records plus one directory entry
GenotypeBatcher::Slab* GenotypeBatcher::TakeFreeSlabLocked(std::unique_lock<std::mutex>& lk, std::size_t need_bytes) {
  mFreeCv.wait(lk, [&] { return mStop || !mFree.empty(); });
  if (mStop) throw std::runtime_error("lancet_gpu::GenotypeBatcher: shut down");
  Slab* s = mFree.back();
  mFree.pop_back();
  (void)need_bytes;
  if (!s->res) {
    if (mFreeResults.empty()) {
      auto r = std::make_unique<ResultBlock>();
      r->job_asg.resize(mOpt.max_jobs), r->job_mid.resize(mOpt.max_jobs);  // no pinned memory here (mMu is held)
      mFreeResults.push_back(r.get());
      mResults.push_back(std::move(r));
    }
    s->res = mFreeResults.back();
    mFreeResults.pop_back();
  }
  return s;
}

std::int32_t GenotypeBatcher::LatchFor(const GenotypeJob& job) {
  if (mParams.mid_occ > 0) return 0;  // fixed by the option set: nothing to latch
  std::int32_t* latch = job.mid_occ_latch ? job.mid_occ_latch : ThreadLatch(mUid);
  if (*latch > 0 || job.n_haps == 0) return *latch;
  std::lock_guard<std::mutex> lk(mAuxMu);
  Check(mAuxCtx, lgr_hap_mid_occ(mAuxCtx, reinterpret_cast<const std::uint8_t*>(job.haps[0].data()),
                                 static_cast<std::int32_t>(job.haps[0].size()), latch));
  return *latch;
}

GenotypeBatcher::Ticket GenotypeBatcher::Enqueue(const GenotypeJob& job) {
  const std::uint64_t t0 = NowNs();
  thread_local PackScratch sc;
  lgr_group_desc desc;
  DescribeJob(job, sc, &desc);
  const lgr_pack::Plan plan = lgr_pack::plan_group(&desc, sc.have_plan ? &sc.last_plan : nullptr);
  // a payload outside the static caps is refused here, alone: it never joins (and fails) a batch
  if (plan.rc != LGR_OK) throw std::runtime_error(std::string("lancet_gpu::GenotypeBatcher: ") + lgr_strerror(plan.rc) + " (this payload only)");
  if (lgr_check_limits(&mParams, plan.max_hap_len, plan.max_read_len) != LGR_OK)
    throw std::runtime_error("lancet_gpu::GenotypeBatcher: payload beyond the device path's static caps (this payload only)");
  sc.last_plan = plan, sc.have_plan = true;
  desc.mid_occ = LatchFor(job);
  if (plan.bytes + sizeof(lgr_group_dir) + 64 > mOpt.slab_bytes) {
    // a payload larger than a whole staging slab travels alone (no pinned reallocation on this path)
    Ticket big;
    big.job = job;
    big.alone = std::make_shared<std::vector<lgr_assign>>(RunAlone(job, desc.mid_occ));
    return big;
  }
  const std::int64_t pairs = static_cast<std::int64_t>(job.n_reads) * static_cast<std::int64_t>(job.n_haps);
  const std::int64_t n_asg = static_cast<std::int64_t>(job.n_reads) * static_cast<std::int64_t>(job.n_variants);
  Ticket t;
  t.job = job;
  std::size_t off = 0;
  Slab* s = nullptr;
  {
    std::unique_lock<std::mutex> lk(mMu);
    if (mStop) throw std::runtime_error("lancet_gpu::GenotypeBatcher: shut down");
    for (;;) {
      if (!mOpen) {
        Slab* f = TakeFreeSlabLocked(lk, plan.bytes);  // may wait: another worker can open a slab meanwhile
        if (mOpen) mFree.push_back(f), mFreeCv.notify_one();
        else mOpen = f;
      }
      s = mOpen;
      const std::size_t dir_room = sizeof(lgr_group_dir) * (s->n_jobs + 1) + 32;
      const bool fits = s->n_jobs < mOpt.max_jobs && s->used + plan.bytes + dir_room <= s->cap &&
                        (s->n_jobs == 0 || (s->pairs + pairs <= mOpt.max_pairs &&
                                            static_cast<std::size_t>(s->n_assign + n_asg) < mOpt.result_records));
      if (fits) break;
      mSealable.push_back(s);  // full: the batcher thread submits it as soon as a device slot is free
      mOpen = nullptr;
      mCv.notify_all();
    }
    s = mOpen;
    t.res = s->res, t.slot = s->n_jobs++;
    off = s->used, s->used += plan.bytes;
    s->res->job_asg[t.slot] = s->n_assign, s->res->job_mid[t.slot] = desc.mid_occ;
    s->n_assign += n_asg, s->pairs += pairs;
    ++s->res->refs;
    s->packing.fetch_add(1, std::memory_order_relaxed);
  }
  mCv.notify_all();
  const int rc = lgr_pack::pack_group(&desc, plan, s->mem + off, &s->dir[t.slot]);
  s->dir[t.slot].rec_off = off;
  if (rc != LGR_OK) s->dir[t.slot].n_reads = -1;  // the batch will be rejected as a whole (cannot happen: plan checked)
  if (s->packing.fetch_sub(1, std::memory_order_release) == 1) mCv.notify_all();
  const std::uint64_t t1 = NowNs();
  {
    std::lock_guard<std::mutex> lk(mMu);
    mCounters.ns_pack += t1 - t0;
  }
  return t;
}

void GenotypeBatcher::SealAndSubmit(Slab* s) {
  const std::uint64_t t0 = NowNs();
  while (s->packing.load(std::memory_order_acquire) != 0) std::this_thread::yield();  // workers finishing their record
  const std::uint64_t t_packed = NowNs();
  try {
    const std::size_t dir_off = (s->used + 15) & ~static_cast<std::size_t>(15);
    std::memcpy(s->mem + dir_off, s->dir.data(), sizeof(lgr_group_dir) * s->n_jobs);
    s->in = lgr_packed_in{};
    s->in.n_groups = static_cast<std::int32_t>(s->n_jobs);
    s->in.slab = s->mem;
    s->in.slab_bytes = dir_off + sizeof(lgr_group_dir) * s->n_jobs;
    s->in.dir = reinterpret_cast<const lgr_group_dir*>(s->mem + dir_off);
    ResultBlock* r = s->res;
    if (!r->assign || static_cast<std::size_t>(s->n_assign) + 1 > r->assign_cap) {
      lgr_free_pinned(r->assign);
      r->assign = nullptr, r->assign_cap = 0, r->status = nullptr;
      const std::size_t want = std::max<std::size_t>(mOpt.result_records, static_cast<std::size_t>(s->n_assign) + static_cast<std::size_t>(s->n_assign) / 2 + 4096);
      r->assign = static_cast<lgr_assign*>(PinnedOrThrow(want * sizeof(lgr_assign) + sizeof(std::int32_t) * mOpt.max_jobs));
      r->assign_cap = want;
      r->status = reinterpret_cast<std::int32_t*>(r->assign + want);
    }
    s->out = lgr_batch_out{};
    s->out.n_assign = s->n_assign;
    s->out.assign = r->assign;  // aln stays NULL: the adapter only needs the assignments
    s->out.grp_status = r->status;
    Check(mCtx, lgr_submit_packed(mCtx, &s->in, &s->out, &s->ticket));
  } catch (const std::exception& e) {
    s->ticket = -1, s->res->rc = LGR_E_CUDA, s->res->err = e.what();
  }
  const std::uint64_t t1 = NowNs();
  std::lock_guard<std::mutex> lk(mMu);
  mCounters.ns_submit += t1 - t0, mCounters.ns_seal_wait += t_packed - t0;
  mCounters.batches += 1, mCounters.jobs += s->n_jobs, mCounters.pairs += static_cast<std::uint64_t>(s->pairs);
  mCounters.h2d_bytes += s->in.slab_bytes;
  if (s->n_jobs > mCounters.max_jobs_in_batch) mCounters.max_jobs_in_batch = s->n_jobs;
}

void GenotypeBatcher::Complete(Slab* s) {
  const std::uint64_t t0 = NowNs();
  lgr_stats st{};
  ResultBlock* r = s->res;
  if (s->ticket >= 0) {
    r->rc = lgr_wait(mCtx, s->ticket, &st);  // the stream has drained: returns at once (except for the rare overflow pass)
    if (r->rc != LGR_OK) {
      const char* detail = lgr_last_error(mCtx);
      r->err = std::string(lgr_strerror(r->rc)) + (detail && *detail ? std::string(": ") + detail : std::string());
    }
  }
  const std::uint64_t t1 = NowNs();
  {
    std::lock_guard<std::mutex> lk(mMu);
    r->done = true;
    mCounters.ns_wait += t1 - t0;
    mCounters.d2h_bytes += static_cast<std::uint64_t>(st.d2h_bytes);
    // the staging slab is free again; the result block stays with the tickets
    s->used = 0, s->n_jobs = 0, s->pairs = 0, s->n_assign = 0, s->ticket = -1, s->opened_ns = 0, s->res = nullptr;
    mFree.push_back(s);
  }
  mDoneCv.notify_all();
  mFreeCv.notify_all();
}

void GenotypeBatcher::Run() {
  std::unique_lock<std::mutex> lk(mMu);
  for (;;) {
    // batches whose device work has finished (tickets may finish out of order: each has its own stream)
    bool progressed = false;
    for (auto it = mInFlight.begin(); it != mInFlight.end();) {
      Slab* s = *it;
      if (s->ticket < 0 || (mDeviceDone & (1u << s->ticket))) {
        if (s->ticket >= 0) mDeviceDone &= ~(1u << s->ticket);
        it = mInFlight.erase(it);
        lk.unlock();
        Complete(s);
        lk.lock();
        progressed = true;
        break;  // the deque may have changed while unlocked
      }
      ++it;
    }
    if (progressed) continue;
    if (mInFlight.size() < static_cast<std::size_t>(mOpt.depth)) {
      Slab* s = nullptr;
      if (!mSealable.empty()) {
        s = mSealable.front();
        mSealable.pop_front();
      } else if (mOpen && mOpen->n_jobs > 0) {
        // When to launch what has gathered so far.  Idle GPU: after one short linger (other workers get a
        // moment to join).  Busy GPU: a small batch only adds per-launch overhead and leaves the device
        // latency bound, so keep gathering until the slab carries enough pairs to fill the machine or has
        // waited max_wait_us; the batches in flight hide the wait.
        const std::uint64_t now = NowNs();
        if (mOpen->opened_ns == 0) mOpen->opened_ns = now;
        const std::uint64_t age_us = (now - mOpen->opened_ns) / 1000;
        const bool big = mOpen->pairs >= mOpt.min_pairs_busy;
        // the idle-GPU linger only pays while it actually gathers company: after eight batches in a row that left
        // with a single payload (one blocking caller) it is skipped until a batch carries more than one again
        const std::uint64_t linger_us = mLingerCredit > 0 ? static_cast<std::uint64_t>(mOpt.linger_us) : 0;
        const std::uint64_t wait_us = mInFlight.empty() ? linger_us : static_cast<std::uint64_t>(mOpt.max_wait_us);
        if (!mStop && !big && age_us < wait_us) {
          mCv.wait_for(lk, std::chrono::microseconds(wait_us - age_us));
          continue;
        }
        s = mOpen;
        mOpen = nullptr;
      }
      if (s) {
        if (s->n_jobs > 1) mLingerCredit = 8;
        else if (mLingerCredit > 0) --mLingerCredit;
        lk.unlock();
        SealAndSubmit(s);
        lk.lock();
        mInFlight.push_back(s);
        continue;
      }
    }
    if (mStop && mInFlight.empty() && mSealable.empty() && (!mOpen || mOpen->n_jobs == 0)) break;
    mCv.wait(lk);
  }
}

// one payload in a device batch of its own, synchronously (after a device-side cap hit it inside a shared batch)
std::vector<lgr_assign> GenotypeBatcher::RunAlone(const GenotypeJob& job, std::int32_t mid_occ) {
  PackScratch sc;
  lgr_group_desc desc;
  DescribeJob(job, sc, &desc);
  desc.mid_occ = mid_occ;
  const lgr_pack::Plan plan = lgr_pack::plan_group(&desc);
  std::vector<std::uint64_t> buf((plan.bytes + sizeof(lgr_group_dir) + 64) / 8 + 1);
  lgr_group_dir dir{};
  if (lgr_pack::pack_group(&desc, plan, buf.data(), &dir) != LGR_OK) throw std::runtime_error("lancet_gpu::GenotypeBatcher: packing failed");
  dir.rec_off = 0;
  std::vector<lgr_assign> assign(job.n_reads * job.n_variants + 1);
  lgr_packed_in in{};
  in.n_groups = 1, in.slab = buf.data(), in.slab_bytes = plan.bytes, in.dir = &dir;
  lgr_batch_out out{};
  out.n_assign = static_cast<std::int64_t>(job.n_reads * job.n_variants), out.assign = assign.data();
  std::lock_guard<std::mutex> lk(mAuxMu);
  Check(mAuxCtx, lgr_genotype_packed(mAuxCtx, &in, &out, nullptr));
  return assign;
}

const lgr_assign* GenotypeBatcher::WaitAssign(Ticket& t, std::vector<lgr_assign>* retry_storage) {
  ResultBlock* r = t.res;
  if (!r && t.alone) return t.alone->data();
  if (!r) throw std::runtime_error("lancet_gpu::GenotypeBatcher: empty ticket");
  {
    std::unique_lock<std::mutex> lk(mMu);
    mDoneCv.wait(lk, [&] { return r->done; });
  }
  if (r->rc == LGR_OK || (r->rc == LGR_E_PARTIAL && r->status[t.slot] == LGR_OK)) return r->assign + r->job_asg[t.slot];
  if (r->rc == LGR_E_PARTIAL) {  // a device-side cap hit THIS payload inside the shared batch: once more, alone
    {
      std::lock_guard<std::mutex> lk(mMu);
      ++mCounters.retried_alone;
    }
    *retry_storage = RunAlone(t.job, r->job_mid[t.slot]);
    return retry_storage->data();
  }
  throw std::runtime_error("lancet_gpu::GenotypeBatcher: " + r->err);
}

void GenotypeBatcher::Release(Ticket& t) {
  ResultBlock* r = t.res;
  if (!r) return;
  t.res = nullptr;
  std::lock_guard<std::mutex> lk(mMu);
  if (--r->refs == 0) {
    r->done = false, r->rc = LGR_OK, r->err.clear();
    mFreeResults.push_back(r);
  }
}

Result GenotypeBatcher::Collect(Ticket& ticket) {
  struct Guard {
    GenotypeBatcher* b;
    Ticket* t;
    ~Guard() { b->Release(*t); }
  } guard{this, &ticket};
  std::vector<lgr_assign> retry;
  const lgr_assign* assign = WaitAssign(ticket, &retry);  // throws for this payload only
  const std::uint64_t t0 = NowNs();
  // AddToTable on the collecting thread, reading the records in place from the pinned result block
  Result res = PackedBatch::BuildResult(ticket.job, assign, mNameHash);
  const std::uint64_t t1 = NowNs();
  {
    std::lock_guard<std::mutex> lk(mMu);
    mCounters.ns_deliver += t1 - t0;
  }
  return res;
}

// The blocking call shape on a context of its own.  A caller that blocks keeps one window in flight, so there is
// nothing for the batcher to coalesce with unless other threads happen to arrive inside the linger; what the detour
// through the batcher thread did cost was four thread hand-offs per call (worker -> batcher -> CUDA callback ->
// batcher -> worker).  Here the calling thread packs into its own pinned slab and runs lgr_genotype_packed on its
// own lgr_ctx (the reference's model: one Genotyper per worker thread); concurrent callers overlap on the GPU
// through their streams.  An idle context holds < 64 MiB of device memory (tests/test_gpu_packed.py).

GenotypeBatcher::DirectSlot* GenotypeBatcher::DirectFor() {
  thread_local std::unordered_map<std::uint64_t, DirectSlot*> mine;  // per batcher instance
  DirectSlot*& slot = mine[mUid];
  if (!slot) {
    auto s = std::make_unique<DirectSlot>();
    Check(nullptr, lgr_create(mOpt.device, &mParams, &s->ctx));
    if (mOpt.direct_graph) Check(s->ctx, lgr_set_graph_mode(s->ctx, 1));
    std::lock_guard<std::mutex> lk(mDirectMu);
    slot = s.get();
    mDirect.push_back(std::move(s));
  }
  return slot;
}

Result GenotypeBatcher::GenotypeDirect(const GenotypeJob& job) {
  const std::uint64_t t0 = NowNs();
  DirectSlot* ds = DirectFor();
  lgr_group_desc desc;
  DescribeJob(job, ds->sc, &desc);
  const lgr_pack::Plan plan = lgr_pack::plan_group(&desc, ds->sc.have_plan ? &ds->sc.last_plan : nullptr);
  if (plan.rc != LGR_OK) throw std::runtime_error(std::string("lancet_gpu::GenotypeBatcher: ") + lgr_strerror(plan.rc) + " (this payload only)");
  if (lgr_check_limits(&mParams, plan.max_hap_len, plan.max_read_len) != LGR_OK)
    throw std::runtime_error("lancet_gpu::GenotypeBatcher: payload beyond the device path's static caps (this payload only)");
  ds->sc.last_plan = plan, ds->sc.have_plan = true;
  desc.mid_occ = LatchFor(job);
  const std::size_t need = plan.bytes + sizeof(lgr_group_dir) + 64;
  if (need > ds->slab_cap) {
    if (ds->slab) lgr_free_pinned(ds->slab);
    ds->slab = nullptr, ds->slab_cap = 0;
    ds->slab = static_cast<std::uint8_t*>(PinnedOrThrow(need + need / 2));
    ds->slab_cap = need + need / 2;
  }
  const std::size_t n_asg = job.n_reads * job.n_variants;
  if (!ds->assign || n_asg + 1 > ds->assign_cap) {
    if (ds->assign) lgr_free_pinned(ds->assign);
    ds->assign = nullptr, ds->assign_cap = 0;
    const std::size_t want = n_asg + n_asg / 2 + 4096;
    ds->assign = static_cast<lgr_assign*>(PinnedOrThrow(want * sizeof(lgr_assign) + sizeof(std::int32_t)));
    ds->assign_cap = want;
  }
  lgr_group_dir* dir = reinterpret_cast<lgr_group_dir*>(ds->slab + ((plan.bytes + 15) & ~static_cast<std::size_t>(15)));
  if (lgr_pack::pack_group(&desc, plan, ds->slab, dir) != LGR_OK) throw std::runtime_error("lancet_gpu::GenotypeBatcher: packing failed");
  dir->rec_off = 0;
  lgr_packed_in in{};
  in.n_groups = 1, in.slab = ds->slab, in.dir = dir;
  in.slab_bytes = static_cast<std::size_t>(reinterpret_cast<std::uint8_t*>(dir + 1) - ds->slab);
  lgr_batch_out out{};
  out.n_assign = static_cast<std::int64_t>(n_asg), out.assign = ds->assign;
  out.grp_status = reinterpret_cast<std::int32_t*>(ds->assign + ds->assign_cap);
  const std::uint64_t t1 = NowNs();
  Check(ds->ctx, lgr_genotype_packed(ds->ctx, &in, &out, nullptr));  // throws for this payload only
  const std::uint64_t t2 = NowNs();
  Result res = PackedBatch::BuildResult(job, ds->assign, mNameHash);
  const std::uint64_t t3 = NowNs();
  std::int64_t replayed = ds->graph_replayed;
  lgr_graph_counters(ds->ctx, nullptr, nullptr, &replayed);
  const std::uint64_t graph_launches = static_cast<std::uint64_t>(replayed - ds->graph_replayed);
  ds->graph_replayed = replayed;
  std::lock_guard<std::mutex> lk(mMu);
  mCounters.graph_launches += graph_launches;
  mCounters.ns_pack += t1 - t0, mCounters.ns_submit += t2 - t1, mCounters.ns_deliver += t3 - t2;
  mCounters.batches += 1, mCounters.jobs += 1, mCounters.pairs += static_cast<std::uint64_t>(job.n_reads * job.n_haps);
  mCounters.h2d_bytes += in.slab_bytes, mCounters.d2h_bytes += n_asg * sizeof(lgr_assign);
  if (mCounters.max_jobs_in_batch < 1) mCounters.max_jobs_in_batch = 1;
  return res;
}

Result GenotypeBatcher::Genotype(const std::string* haps, std::size_t n_haps, const ReadIn* reads, std::size_t n_reads,
                                 const VariantIn* variants, std::size_t n_variants) {
  return Genotype(GenotypeJob{haps, n_haps, reads, n_reads, variants, n_variants});
}

Result GenotypeBatcher::Genotype(const GenotypeJob& job) {
  struct Inside {
    std::atomic<int>& n;
    int mine;
    explicit Inside(std::atomic<int>& c) : n(c), mine(c.fetch_add(1, std::memory_order_relaxed) + 1) {}
    ~Inside() { n.fetch_sub(1, std::memory_order_relaxed); }
  } inside{mBlockingCallers};
  if (inside.mine <= mOpt.direct_blocking_callers) return GenotypeDirect(job);
  Ticket t = Enqueue(job);
  return Collect(t);
}

GenotypeBatcher::Counters GenotypeBatcher::Stats() {
  std::lock_guard<std::mutex> lk(mMu);
  return mCounters;
}

// ---------------------------------------------------------------------------------------------
// GenotypeDispatcher
// ---------------------------------------------------------------------------------------------
GenotypeDispatcher::GenotypeDispatcher(const std::vector<int>& devices, NameHashFn name_hash, GenotypeBatcher::Options base) {
  if (devices.empty()) throw std::runtime_error("lancet_gpu::GenotypeDispatcher: no devices given (there is no CPU fallback)");
  mUid = g_latch_uid.fetch_add(1);
  mOutstanding = std::make_unique<std::atomic<std::int64_t>[]>(devices.size());
  for (std::size_t i = 0; i < devices.size(); ++i) {
    base.device = devices[i];
    mOutstanding[i].store(0);
    mBatchers.push_back(std::make_unique<GenotypeBatcher>(base, name_hash));
  }
}

std::int64_t GenotypeDispatcher::Cost(const GenotypeJob& job) {
  std::int64_t hap_total = 0;
  for (std::size_t h = 0; h < job.n_haps; ++h) hap_total += static_cast<std::int64_t>(job.haps[h].size());
  return static_cast<std::int64_t>(job.n_reads) * hap_total + 1;
}

GenotypeDispatcher::Ticket GenotypeDispatcher::Enqueue(const GenotypeJob& job_in) {
  // the calling thread's mm_mapopt_update latch belongs to the dispatcher, not to the device a payload
  // happens to be routed to: results do not depend on the routing
  GenotypeJob job = job_in;
  if (!job.mid_occ_latch) job.mid_occ_latch = ThreadLatch(mUid);
  std::size_t best = 0;
  std::int64_t best_load = mOutstanding[0].load(std::memory_order_relaxed);
  for (std::size_t i = 1; i < mBatchers.size(); ++i) {
    const std::int64_t load = mOutstanding[i].load(std::memory_order_relaxed);
    if (load < best_load) best = i, best_load = load;
  }
  Ticket t;
  t.device_slot = best;
  t.cost = Cost(job);
  mOutstanding[best].fetch_add(t.cost, std::memory_order_relaxed);
  try {
    t.inner = mBatchers[best]->Enqueue(job);
  } catch (...) {
    mOutstanding[best].fetch_sub(t.cost, std::memory_order_relaxed);
    throw;
  }
  return t;
}

Result GenotypeDispatcher::Collect(Ticket& ticket) {
  struct Release {
    std::atomic<std::int64_t>& load;
    std::int64_t cost;
    ~Release() { load.fetch_sub(cost, std::memory_order_relaxed); }
  } release{mOutstanding[ticket.device_slot], ticket.cost};
  return mBatchers[ticket.device_slot]->Collect(ticket.inner);
}

Result GenotypeDispatcher::Genotype(const std::string* haps, std::size_t n_haps, const ReadIn* reads, std::size_t n_reads,
                                    const VariantIn* variants, std::size_t n_variants) {
  GenotypeJob job{haps, n_haps, reads, n_reads, variants, n_variants};
  job.mid_occ_latch = ThreadLatch(mUid);
  std::size_t best = 0;
  std::int64_t best_load = mOutstanding[0].load(std::memory_order_relaxed);
  for (std::size_t i = 1; i < mBatchers.size(); ++i) {
    const std::int64_t load = mOutstanding[i].load(std::memory_order_relaxed);
    if (load < best_load) best = i, best_load = load;
  }
  struct Load {
    std::atomic<std::int64_t>& load;
    std::int64_t cost;
    Load(std::atomic<std::int64_t>& l, std::int64_t c) : load(l), cost(c) { load.fetch_add(cost, std::memory_order_relaxed); }
    ~Load() { load.fetch_sub(cost, std::memory_order_relaxed); }
  } held{mOutstanding[best], Cost(job)};
  return mBatchers[best]->Genotype(job);  // blocking: the batcher runs it on the calling thread's own context
}

}  // namespace lancet_gpu
