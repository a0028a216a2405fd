// PacBio read generator (SURVEY.md section 8f rank 3; /root/reference/src/hts_pacbio.{h,cpp}, R/hts_pacbio.R).
// Host side: per-read quantities are computed on the host (O(reads): read length, number of passes, the
// per-pass-count error probabilities and the two quality characters), per-base work on the device
// (O(bases): the insertion / deletion / substitution walk, extraction, reverse complement, the FASTQ record).
#ifndef JLP_PACBIO_H
#define JLP_PACBIO_H

#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <memory>
#include <vector>

#include "jlp_host.h"
#include "jlp_kernels.cuh"

namespace jlp {

struct PbModel {
    double scale = 17922.611306, sigma = 0.200110276521, loc = -10075.4363813, min_read_len = 50;
    std::vector<double> read_probs;           // custom read lengths (alias-sampled) when non-empty
    std::vector<uint64_t> read_lens;
    uint64_t max_passes = 40;
    double chi2_n[3] = {0.00189237136, 2.53944970, 5500};
    double chi2_s[5] = {0.01214, -5.12, 675, 48303.0732881, 1.4691051212330266};
    double sqrt_params[2] = {0.5, 0.2247};
    double norm_params[2] = {0, 0.2};
    double prob_thresh = 0.2, prob_ins = 0.11, prob_del = 0.04, prob_subst = 0.01;
    double min_exp = 0;                       // calc_min_exp(), set by pb_prepare
    mutable std::shared_ptr<std::atomic<double>[]> qchisq_cache;   // outlier threshold per min(read_length, chi2_n[2]), filled on first use (a context keeps it from call to call)
    size_t qchisq_n = 0;
    std::vector<double> len_prob;             // alias tables of the custom read lengths
    std::vector<uint64_t> len_alias;
    // update_probs / trunc_norm: what depends only on the (whole) number of passes, per value 0 .. max_passes + 1
    struct PassTab { double sig, root, thresh, a_bar, p_low; };
    std::vector<PassTab> pass_tab;
};
// PacBioQualityError::calc_min_exp (src/hts_pacbio.cpp) and the tables of the samplers.  Throws on bad input.
void pb_prepare(PbModel& m);

// What the stateful samplers of the reference produce for one read (PacBioReadLenSampler::sample, src/hts_pacbio.cpp;
// PacBioPassSampler::sample, src/hts_pacbio.h:160-200), drawn here from the read's own Philox stream with
// inverse-CDF / Marsaglia-Tsang samplers: same laws, not the same draws (statistical tier).
struct PbSample {
    uint64_t read_length;      // already limited to the chromosome's length
    uint64_t split_pos;
    double passes_left, passes_right;
};
PbSample pb_sample(const PbModel& m, uint64_t seed, uint64_t j, uint64_t chrom_len);
// the same for a duplicate (PacBioOneGenome::re_read): the chain's read length, a new number of passes
PbSample pb_sample_passes(const PbModel& m, uint64_t seed, uint64_t j, uint64_t read_length);
// the draw ReadWriterOneThread::create_reads makes after read j (src/hts.h:264-277): the next read re-reads iff it is < prob_dup
uint64_t pb_dup_draw(uint64_t seed, uint64_t j);

// Per-read input of the kernels: the walk's comparisons as integer thresholds on the 64-bit draws
// (update_probs + fill_quals, src/hts_pacbio.cpp / src/hts_pacbio.h:383-391; exact under replay).
struct PbRead {
    uint64_t thr[2][3];        // [left|right][ins, del, any]: x < thr[.][0] insertion, else < [1] deletion, else < [2] substitution
    uint32_t read_length;
    uint32_t split_pos;
    uint32_t flags;            // bits 0..5: threshold [side][k] is 2^64 (always true); bits 8..15 qual_left, 16..23 qual_right
    uint32_t group;
    // written by k_pb_plan
    const uint8_t* seg;        // first template base
    uint32_t space;            // template bases used (read_chrom_space)
    uint32_t rec_len;          // FASTQ bytes of the record
    uint64_t start;            // read_start
    uint32_t reverse;
    uint32_t pad;              // bases of the sequence line (k_pb_warp<false>)
    uint32_t leader;           // a duplicate: index (in the batch) of the first read of its chain; kPbNoLeader otherwise
    uint32_t del_keep;         // recorded deletions append_pool still sees (a duplicate may have to give some up)
};
static_assert(sizeof(PbRead) == 104, "PbRead layout");
constexpr uint32_t kPbNoLeader = 0xffffffffu;
constexpr uint32_t kPbSerial = 1u << 24;      // PbRead::flags: the read is walked by one lane throughout
void pb_read_model(const PbModel& m, uint64_t seed, uint64_t j, const PbSample& s, PbRead& out);

// The plan of reads [b0, b0 + n) of a job whose reads start at job_lo (b0 - job_lo a whole number of pools of `pool`
// reads).  Chains of duplicates (ReadWriterOneThread::create_reads, src/hts.h:264-277): read j re-reads its chain's first
// read iff pb_dup_draw(seed, j - 1) passes t_dup and j does not open a pool.  A chain's first read takes the group of
// group_off (reads per group, cumulative) that j falls in and a pb_sample of its chromosome; a duplicate takes its
// leader's group and read length and a pb_sample_passes.  out[i] is filled by pb_read_model, with group and leader.
// Worker k of min(max(n_threads, 1), 64) takes reads k, k + nt, ...: first the leaders, then the duplicates.
// samples (may be NULL) receives what was drawn per read.  Returns the sum of the read lengths.
uint64_t pb_plan(const PbModel& m, uint64_t seed, uint64_t b0, uint32_t n, uint64_t job_lo, uint64_t pool, Thr t_dup,
                 const std::vector<uint64_t>& group_off, const GroupDev* groups, uint64_t n_threads, PbRead* out,
                 PbSample* samples);

// plan: walk -> counts -> template span, start, strand, record length; reads: the record itself
cudaError_t launch_pb_plan(PbRead* reads, uint32_t n, uint64_t first_read, uint64_t seed, const GroupDev* groups,
                           uint64_t c_rev, uint32_t* rec_len, cudaStream_t s);
// duplicates take their chain's start; deletions are given up until the template fits (re_read, src/hts_pacbio.cpp)
cudaError_t launch_pb_dups(PbRead* reads, uint32_t n, uint64_t first_read, uint64_t seed, const GroupDev* groups, uint32_t* rec_len,
                           cudaStream_t s);
cudaError_t launch_pb_reads(const PbRead* reads, uint32_t n, uint64_t first_read, uint64_t seed, const GroupDev* groups,
                            const uint8_t* strpool, const uint32_t* rec_local, const uint64_t* block_base, uint8_t* out,
                            cudaStream_t s);

}  // namespace jlp
#endif
