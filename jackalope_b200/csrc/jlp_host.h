// Host-side model preparation for the Illumina kernels: alias tables, integer
// thresholds, fragment-length table, read apportioning; the loop that spreads host
// work over a few threads.  Plain C++ (g++), no
// CUDA.  Each function cites the reference code it stands in for
// (paths relative to /root/reference).
#ifndef JLP_HOST_H
#define JLP_HOST_H

#include <atomic>
#include <cstdint>
#include <exception>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace jlp {

// --- host work over a few threads --------------------------------------------------
// f(i) for every i in [0, n) on n_threads threads, the calling thread one of them; items are handed out one at a time.
// Every item runs even when others throw; then the exception of the lowest failing i is rethrown, as a serial loop would
// report it.  Every thread started is joined before this returns or throws; a thread that cannot be started is reported
// after the items have run on the others.
template <typename F> void parallel_for(uint64_t n, unsigned n_threads, F f) {
    std::atomic<uint64_t> next{0};
    std::mutex mu;
    uint64_t first_bad = n;
    std::exception_ptr err, start_err;
    auto work = [&]() {
        for (uint64_t i; (i = next.fetch_add(1)) < n;) {
            try { f(i); } catch (...) {
                std::lock_guard<std::mutex> g(mu);
                if (i < first_bad) { first_bad = i; err = std::current_exception(); }
            }
        }
    };
    std::vector<std::thread> th;
    try {
        for (unsigned k = 1; k < n_threads; k++) th.emplace_back(work);
    } catch (...) { start_err = std::current_exception(); }
    work();
    for (std::thread& t : th) t.join();
    if (err) std::rethrow_exception(err);
    if (start_err) std::rethrow_exception(start_err);
}

// --- comparison thresholds -------------------------------------------------
// A comparison of u = runif_01(x) against a constant is monotone in x, so it
// equals an integer comparison on x.  `thr` counts the x for which the
// predicate holds from the low end; all == true means every x (count 2^64).
struct Thr {
    uint64_t thr;
    bool all;
};
// #{x : (double)u <  p}   src/alias_sampler.h:57-58, src/hts_illumina.h:251-252, src/hts.h:265-266
Thr thr_double_lt(double p);
// #{x : !((double)u > p)} src/hts_illumina.cpp:132-135
Thr thr_double_le(double p);
// #{x : u < p} (long double compare) src/hts_illumina.cpp:352
Thr thr_ld_lt(double p);
// the same three found by evaluating the reference's x87 expressions at candidate draws (only where long double is
// the x87 format; elsewhere they return the integer forms): the test oracle of the integer restatements
Thr thr_double_lt_x87(double p);
Thr thr_double_le_x87(double p);
Thr thr_ld_lt_x87(double p);

// --- alias tables ------------------------------------------------------------
// AliasSampler::construct, src/alias_sampler.h:68-106
void alias_build(const double* probs, uint64_t n, double* Prob, uint64_t* Alias);

// One read end's quality/error model in the layout the kernels read.
struct EndTables {
    uint64_t L = 0;
    std::vector<uint32_t> meta;     // [4*L]  offset << 8 | n
    std::vector<uint64_t> entry64;  // (q_alias+33) | (q_self+33) << 8 | coin16 << 16 | mis16[q_self] << 32 | mis16[q_alias] << 48
    std::vector<uint64_t> coin;     // full coin threshold per slot (slow path)
    std::vector<uint64_t> mis;      // [256] full mismatch threshold per quality
    uint32_t max_n = 0;
};
// IlluminaQualityError ctor (src/hts_illumina.h:154-189) + IllQualPos ctor (:102-116).
// Throws std::runtime_error with the reference's message on malformed input.
void build_end_tables(uint64_t L, const uint32_t* nq, const double* probs, const uint8_t* quals,
                      EndTables& out);

// --- fragment lengths ----------------------------------------------------------
// Table of P(frag_len <= frag_min + i) * 2^64 for
// frag_len = clamp((uint64)Gamma(shape, scale), frag_min, frag_max)
// (src/hts_illumina.cpp:206-208).  Entry count = hi - frag_min where hi is
// frag_max or the point past which the tail mass is < 2^-64.
std::vector<uint64_t> frag_table(double shape, double scale, uint64_t frag_min, uint64_t frag_max);
// guide[b] = #{i : cdf[i] <= (b << 56)} for b = 0..256 (guide[256] = cdf.size()): the inverse-CDF
// search for a draw x only has to look at cdf[guide[x >> 56] .. guide[(x >> 56) + 1]).
std::vector<uint32_t> frag_guide(const std::vector<uint64_t>& cdf);
// regularised lower incomplete gamma P(a, x)
long double gamma_p(long double a, long double x);

// --- read apportioning ---------------------------------------------------------
// reads_per_group, src/hts.h:58-103 (own engine; statistically equivalent)
std::vector<uint64_t> reads_per_group(uint64_t n_reads, std::vector<double> probs, uint64_t seed);
// split_int, src/util.h:245-258
std::vector<uint64_t> split_int(uint64_t x, uint64_t n);

// --- substitution model (create_haplotypes) -------------------------------------
// P = expm(Q t), 4x4 in T,C,A,G, Q's diagonal taken as minus the off-diagonal row sum; t == 0 gives exactly I
void transition_matrix(const double Q[16], double t, double P[16]);
// a cumulative probability as a draw threshold: floor(c 2^64), 0 for c <= 0, 2^64 - 1 for c >= 1
uint64_t prob_threshold(double c);
// one row of P as the thresholds of a 64-bit draw X: new state = #{j < 3 : X >= thr[j]}; the row is clipped at 0
// and renormalised, thr[j] = prob_threshold(p[0] + ... + p[j])
void row_thresholds(const double* row, uint64_t thr[3]);

// --- gene trees (create_haplotypes along ms output, jlp_gtrees.cpp) ---------------------
struct GeneTree {                       // a tree in preorder, nodes numbered as parse_newick numbers them
    std::vector<int32_t> parent;        // parent[0] = -1, parent[i] < i
    std::vector<double> branch_len;
    std::vector<uint32_t> tip_node;     // [n_tips]: the node of haplotype i
};
struct TreeRegion {                     // sites [start, end) of a chromosome follow trees[tree]
    uint32_t start, end, tree;
};
struct GeneTrees {
    std::vector<GeneTree> trees;
    std::vector<std::vector<TreeRegion>> regions;   // per chromosome, in position order, none empty
};
// ms-format text (DESIGN.md section 10, "Gene trees") -> its trees and each chromosome's regions; tip labels are matched
// to tip_names.  Trees are parsed on up to n_threads threads.  Throws std::runtime_error naming the problem.
void parse_ms(const char* text, uint64_t len, const std::vector<uint64_t>& chrom_len, const char* const* tip_names,
              uint32_t n_tips, uint32_t max_nodes, unsigned n_threads, GeneTrees& out);

// --- insertions and deletions along the tree (create_haplotypes, jlp_indel.cpp) --------
// One insertion or deletion record of a (tip, chromosome) in HapChromHost::packed terms (DESIGN.md section 10).
struct IndelRec {
    uint32_t old_pos, new_pos;
    uint32_t kind;          // kDelRec, kAnchorRec (pool = the tip base at old_pos, then the inserted bases), kLeadRec
    uint32_t pad;
    int64_t size_mod;       // -(deleted columns), or the inserted bases (kLeadRec: minus one)
    uint64_t pool_before;   // pool bytes of the indel records before this one in its (tip, chromosome)
};
constexpr uint32_t kDelRec = 0, kAnchorRec = 1, kLeadRec = 2;
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint64_t indel_pool_len(const IndelRec& r) { return r.kind == kDelRec ? 0 : (uint64_t)(r.size_mod + 1); }

struct IndelModel {
    double rate_ins = 0, rate_del = 0, epsilon = 0;
    uint32_t n_ins = 0;                 // (kind, length) index < n_ins: insertion of index + 1 columns, else deletion
    std::vector<uint64_t> kl_thr;       // the (kind, length) draw's cumulative thresholds (see indel_thresholds)
};
// (kind, length) probabilities (rate_ins / R) (w_ins[u] / sum w_ins) for u = 1..n_ins, then the deletions alike, summed
// in that order into prob_threshold()s (all but the last)
std::vector<uint64_t> indel_thresholds(double rate_ins, const double* w_ins, uint32_t n_ins, double rate_del,
                                       const double* w_del, uint32_t n_del);
// the steps of a branch: max(1, ceil(R t / epsilon)); throws past 2^31
uint32_t indel_steps(double R, double t, double epsilon);

struct IndelTip {                       // one (tip, chromosome)
    std::vector<IndelRec> recs;         // by old_pos
    std::vector<uint32_t> ids;          // the inserted columns of the insertion records, in pool order
    std::vector<uint64_t> ids_off;      // [recs.size() + 1]: record j's columns are ids[ids_off[j] .. ids_off[j + 1])
    uint64_t size = 0;                  // the tip's chromosome length
};
struct IndelChrom {
    std::vector<uint32_t> birth;        // per inserted column (its id): the node at the end of the branch it was born on
    std::vector<IndelTip> tip;          // per tip
    uint64_t insertions = 0, deletions = 0, inserted_bases = 0, steps = 0;
};
// The event pass of one chromosome of `len` reference columns: nodes in preorder (parent[v] < v), each branch cut into
// indel_steps() steps, the events of a step drawn from plane IEV and applied at once.  tip_of[v] = tip index or -1.
// Throws std::runtime_error past the limits (a tip chromosome or the inserted columns at 2^32).
void indel_events(uint64_t seed, uint32_t chrom, uint64_t len, uint32_t n_nodes, const int32_t* parent,
                  const double* branch_len, const int32_t* tip_of, uint32_t n_tips, const IndelModel& m, IndelChrom& out);

}  // namespace jlp
#endif
