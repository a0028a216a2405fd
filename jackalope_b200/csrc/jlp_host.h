// Host-side model preparation for the Illumina kernels: alias tables, integer
// thresholds, fragment-length table, read apportioning.  Plain C++ (g++), no
// CUDA.  Each function cites the reference code it stands in for
// (paths relative to /root/reference).
#ifndef JLP_HOST_H
#define JLP_HOST_H

#include <cstdint>
#include <string>
#include <vector>

namespace jlp {

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

}  // namespace jlp
#endif
