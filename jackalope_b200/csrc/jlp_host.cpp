// Host-side model preparation (see jlp_host.h).  Compiled by g++.
//
// The comparison thresholds restate the reference's floating-point tests on u = runif_01(x) = (x + 1) / 2^64
// (x87 long double, src/pcg.h:99-101) as counts of 64-bit draws, in pure integer arithmetic (SURVEY.md App. A.2):
// they do not need an x87 and give the same numbers on any host.  Where long double has the x87 format the
// reference's own expressions are also evaluated (thr_*_x87) and the tests require both to agree.
#include "jlp_host.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <deque>
#include <numeric>
#include <random>
#include <stdexcept>

namespace jlp {

namespace {

typedef unsigned __int128 u128;

// smallest integer y >= m * 2^s (strict: > m * 2^s); m < 2^55.  Values above 2^64 are returned as 2^64 + 1.
u128 int_at_least(uint64_t m, int s, bool strict) {
    const u128 cap = ((u128)1 << 64) + 1;
    if (m == 0) return strict ? 1 : 0;
    if (s >= 0) {
        if (s > 64) return cap;
        const u128 v = (u128)m << s;
        return std::min<u128>(cap, v + (strict ? 1 : 0));
    }
    const int k = -s;
    if (k >= 64) return 1;                              // 0 < m * 2^s < 1
    const uint64_t q = m >> k, rem = m & ((1ull << k) - 1);
    return rem ? (u128)q + 1 : (u128)q + (strict ? 1 : 0);
}

// p = M * 2^E with 2^52 <= M < 2^53 (p a positive normal double)
void split_double(double p, uint64_t& M, int& E) {
    int ex;
    const double f = std::frexp(p, &ex);                // p = f * 2^ex, 0.5 <= f < 1
    M = (uint64_t)std::ldexp(f, 53);
    E = ex - 53;
}

// y* = the smallest integer y in [0, 2^64 + 1] whose u = y / 2^64, ROUNDED TO DOUBLE (nearest, ties to even), is >= p.
// u rounds to a double >= p exactly when it lies at or above the midpoint between p and the double below it -- above
// it only, if the tie goes to the neighbour (p's mantissa odd).
u128 first_y_double_ge(double p) {
    if (!(p > 0)) return 0;
    if (p > 1) return ((u128)1 << 64) + 1;
    if (p < 1e-300) return 1;
    uint64_t M;
    int E;
    split_double(p, M, E);
    const bool pow2 = M == (1ull << 52);                // the spacing below a power of two is half the one above
    const uint64_t mm = pow2 ? 4 * M - 1 : 2 * M - 1;   // midpoint = mm * 2^(E - 2) or mm * 2^(E - 1)
    return int_at_least(mm, (pow2 ? E - 2 : E - 1) + 64, (M & 1) != 0);
}

Thr count_below(u128 ystar) {                           // #{x in [0, 2^64) : x + 1 < y*}
    if (ystar <= 1) return Thr{0, false};
    if (ystar > ((u128)1 << 64)) return Thr{UINT64_MAX, true};
    return Thr{(uint64_t)(ystar - 1), false};
}

}  // namespace

// #{x : double(u) < p}
Thr thr_double_lt(double p) { return count_below(first_y_double_ge(p)); }
// #{x : !(double(u) > p)} = #{x : double(u) < the double above p}
Thr thr_double_le(double p) {
    if (p < 0) return Thr{0, false};
    return count_below(first_y_double_ge(std::nextafter(p, INFINITY)));
}
// #{x : u < p} in long double: u = y / 2^64 exactly, so y < p * 2^64
Thr thr_ld_lt(double p) {
    if (!(p > 0)) return Thr{0, false};
    if (p > 1) return Thr{UINT64_MAX, true};
    if (p < 1e-300) return Thr{0, false};
    uint64_t M;
    int E;
    split_double(p, M, E);
    return count_below(int_at_least(M, E + 64, false));
}

#if LDBL_MANT_DIG == 64
// ---- the reference's own expressions, evaluated on an x87 (test oracle of the integer forms above)
namespace {
inline long double runif_01(uint64_t x) {
    const long double max64 = static_cast<long double>(UINT64_MAX);
    return (static_cast<long double>(x) + 1) / (max64 + 2);
}
// smallest x for which pred is false, pred being true on a prefix of [0, 2^64)
template <typename F> Thr prefix_count(F pred) {
    if (pred(UINT64_MAX)) return Thr{UINT64_MAX, true};
    if (!pred(0)) return Thr{0, false};
    uint64_t lo = 0, hi = UINT64_MAX;  // pred(lo) true, pred(hi) false
    while (hi - lo > 1) {
        uint64_t mid = lo + (hi - lo) / 2;
        if (pred(mid)) lo = mid; else hi = mid;
    }
    return Thr{hi, false};
}
}  // namespace
Thr thr_double_lt_x87(double p) { return prefix_count([p](uint64_t x) { double u = runif_01(x); return u < p; }); }
Thr thr_double_le_x87(double p) { return prefix_count([p](uint64_t x) { double u = runif_01(x); return !(u > p); }); }
Thr thr_ld_lt_x87(double p) { return prefix_count([p](uint64_t x) { return runif_01(x) < p; }); }
#else
Thr thr_double_lt_x87(double p) { return thr_double_lt(p); }
Thr thr_double_le_x87(double p) { return thr_double_le(p); }
Thr thr_ld_lt_x87(double p) { return thr_ld_lt(p); }
#endif

void alias_build(const double* probs, uint64_t n, double* Prob, uint64_t* Alias) {
    std::vector<double> p(probs, probs + n);
    double total = std::accumulate(p.begin(), p.end(), 0.0);
    for (double& v : p) v /= total;
    for (double& v : p) v *= static_cast<double>(n);
    for (uint64_t i = 0; i < n; i++) { Prob[i] = 0.0; Alias[i] = 0; }
    std::deque<uint64_t> small, large;
    for (uint64_t i = 0; i < n; i++) (p[i] < 1 ? small : large).push_back(i);
    while (!small.empty() && !large.empty()) {
        uint64_t l = small.front(); small.pop_front();
        uint64_t g = large.front(); large.pop_front();
        Prob[l] = p[l];
        Alias[l] = g;
        p[g] = (p[g] + p[l]) - 1;
        (p[g] < 1 ? small : large).push_back(g);
    }
    for (uint64_t g : large) Prob[g] = 1;
    for (uint64_t l : small) Prob[l] = 1;
}

void build_end_tables(uint64_t L, const uint32_t* nq, const double* probs, const uint8_t* quals,
                      EndTables& out) {
    if (L == 0) throw std::runtime_error("read length must be >= 1");
    out = EndTables();
    out.L = L;
    out.meta.resize(4 * L);
    uint64_t tot = 0;
    for (uint64_t i = 0; i < 4 * L; i++) {
        if (nq[i] == 0) throw std::runtime_error("profile position without any quality value");
        if (nq[i] > 255) throw std::runtime_error("more than 255 quality values at one profile position");
        tot += nq[i];
    }
    if (tot >= (1ull << 24)) throw std::runtime_error("profile too large");
    std::vector<uint32_t> entry(tot);          // coin16 | q_self << 16 | q_alias << 24
    out.coin.resize(tot);
    unsigned max_qual = 0;
    std::vector<double> Prob;
    std::vector<uint64_t> Alias;
    uint64_t off = 0;
    for (uint64_t i = 0; i < 4 * L; i++) {
        uint32_t n = nq[i];
        out.meta[i] = static_cast<uint32_t>(off << 8) | n;
        if (n > out.max_n) out.max_n = n;
        Prob.assign(n, 0.0);
        Alias.assign(n, 0);
        alias_build(probs + off, n, Prob.data(), Alias.data());
        for (uint32_t k = 0; k < n; k++) {
            Thr t = thr_double_lt(Prob[k]);             // u < Prob[i], src/alias_sampler.h:58
            uint64_t c = t.thr;                          // never `all`: Prob <= 1 and u == 1 exists
            out.coin[off + k] = c;
            uint32_t q_self = quals[off + k], q_alias = quals[off + Alias[k]];
            entry[off + k] = static_cast<uint32_t>(c >> 48) | (q_self << 16) | (q_alias << 24);
            if (q_self > max_qual) max_qual = q_self;
        }
        off += n;
    }
    // qual_prob_map, src/hts_illumina.h:182-187.  Entries above max_qual do not
    // exist in the reference; they are never indexed.
    out.mis.assign(256, 0);
    std::vector<uint16_t> mis16(256, 0);       // high 16 bits of the mismatch threshold per quality
    for (unsigned q = 0; q <= max_qual; q++) {
        double prob = q == 0 ? 1.0 : std::pow(10, static_cast<double>(q) / -10.0);
        Thr t = thr_double_lt(prob);
        out.mis[q] = t.thr;
        mis16[q] = static_cast<uint16_t>(t.thr >> 48);
    }
    out.entry64.resize(tot);
    for (uint64_t k = 0; k < tot; k++) {
        uint32_t e = entry[k];
        uint32_t qs = (e >> 16) & 0xffu, qa = e >> 24;
        // the quality CHARACTERS (q + '!', modulo 256 as the reference's uint8 arithmetic gives)
        uint32_t lo = ((qa + 33u) & 0xffu) | (((qs + 33u) & 0xffu) << 8) | ((e & 0xffffu) << 16);
        out.entry64[k] = static_cast<uint64_t>(lo) | (static_cast<uint64_t>(mis16[qs]) << 32) |
                         (static_cast<uint64_t>(mis16[qa]) << 48);
    }
}

// ---------------------------------------------------------------------------
// regularised incomplete gamma: series for x < a + 1, Lentz continued fraction
// for the upper tail otherwise.  Returns P in [0, 1]; q_out (if given) gets 1-P
// computed without cancellation.
static long double gamma_pq(long double a, long double x, long double* q_out) {
    if (x <= 0) { if (q_out) *q_out = 1; return 0; }
    const long double lg = lgammal(a);
    const long double pre = expl(a * logl(x) - x - lg);
    if (x < a + 1) {
        long double ap = a, term = 1 / a, sum = term;
        for (int n = 0; n < 1000000; n++) {
            ap += 1;
            term *= x / ap;
            sum += term;
            if (fabsl(term) < fabsl(sum) * 1e-21L) break;
        }
        long double p = sum * pre;
        if (p > 1) p = 1;
        if (q_out) *q_out = 1 - p;
        return p;
    }
    const long double tiny = 1e-4000L;
    long double b = x + 1 - a, c = 1 / tiny, d = 1 / b, h = d;
    for (int i = 1; i < 1000000; i++) {
        long double an = -i * (i - a);
        b += 2;
        d = an * d + b; if (fabsl(d) < tiny) d = tiny;
        c = b + an / c; if (fabsl(c) < tiny) c = tiny;
        d = 1 / d;
        long double del = d * c;
        h *= del;
        if (fabsl(del - 1) < 1e-20L) break;
    }
    long double q = pre * h;
    if (q > 1) q = 1;
    if (q_out) *q_out = q;
    return 1 - q;
}

long double gamma_p(long double a, long double x) { return gamma_pq(a, x, nullptr); }

std::vector<uint64_t> frag_table(double shape, double scale, uint64_t frag_min, uint64_t frag_max) {
    std::vector<uint64_t> cdf;
    if (frag_max <= frag_min) return cdf;
    const long double two64 = 18446744073709551616.0L;
    const uint64_t cap = 1ull << 24;
    uint64_t prev = 0;
    for (uint64_t i = 0; frag_min + i < frag_max && i < cap; i++) {
        // P(len <= frag_min + i) = P(Gamma < frag_min + i + 1)
        long double x = static_cast<long double>(frag_min + i + 1) / scale;
        long double q;
        long double p = gamma_pq(shape, x, &q);
        long double v = (q < 0.25L) ? (two64 - q * two64) : p * two64;
        uint64_t c = v >= two64 ? UINT64_MAX : (v <= 0 ? 0 : static_cast<uint64_t>(v));
        if (c < prev) c = prev;
        if (q * two64 < 0.5L) break;     // the rest of the tail is below one draw value
        cdf.push_back(c);
        prev = c;
    }
    return cdf;
}

std::vector<uint32_t> frag_guide(const std::vector<uint64_t>& cdf) {
    std::vector<uint32_t> g(257);
    for (uint32_t b = 0; b < 256; b++) {
        uint64_t x = static_cast<uint64_t>(b) << 56;
        g[b] = static_cast<uint32_t>(std::upper_bound(cdf.begin(), cdf.end(), x) - cdf.begin());
    }
    g[256] = static_cast<uint32_t>(cdf.size());
    return g;
}

std::vector<uint64_t> reads_per_group(uint64_t n_reads, std::vector<double> probs, uint64_t seed) {
    std::vector<uint64_t> out(probs.size(), 0);
    if (n_reads == 0 || probs.empty()) return out;
    std::mt19937_64 eng(seed ^ 0xA5A5F00DBAADC0DEull);
    double sum_probs = std::accumulate(probs.begin(), probs.end(), 0.0);
    for (double& p : probs) p /= sum_probs;
    std::binomial_distribution<uint64_t> distr(n_reads, 0.5);
    for (size_t i = 0; i + 1 < probs.size(); i++) {
        if (probs[i] >= 1) { out[i] = n_reads; return out; }
        if (probs[i] == 0) continue;
        distr.param(std::binomial_distribution<uint64_t>::param_type(n_reads, probs[i]));
        out[i] = distr(eng);
        n_reads -= out[i];
        if (n_reads == 0) break;
        sum_probs = 1 - probs[i];
        for (size_t j = i + 1; j < probs.size(); j++) probs[j] /= sum_probs;
    }
    out.back() = n_reads;
    return out;
}

std::vector<uint64_t> split_int(uint64_t x, uint64_t n) {
    std::vector<uint64_t> out(n, x / n);
    uint64_t sum = n * (x / n);
    for (uint64_t i = 0; sum < x; i++, sum++) out[i]++;
    return out;
}

// --- substitution model (create_haplotypes) ------------------------------------

void transition_matrix(const double Q[16], double t, double P[16]) {
    for (int i = 0; i < 16; i++) P[i] = (i % 5 == 0) ? 1.0 : 0.0;
    if (t == 0) return;
    // A = Q t with the diagonal made minus the row sum; scaled by 2^-s so that ||A||_1 <= 1, Taylor series to
    // 30 terms (remainder < 1/30!), then squared s times
    double A[16], norm = 0;
    for (int i = 0; i < 4; i++) {
        double row = 0;
        for (int j = 0; j < 4; j++) if (j != i) { A[4 * i + j] = Q[4 * i + j] * t; row += A[4 * i + j]; }
        A[5 * i] = -row;
    }
    for (int j = 0; j < 4; j++) {
        double col = 0;
        for (int i = 0; i < 4; i++) col += std::fabs(A[4 * i + j]);
        norm = std::max(norm, col);
    }
    int s = 0;
    if (norm > 1) s = std::min(1000, (int)std::ceil(std::log2(norm)));
    const double sc = std::ldexp(1.0, -s);
    for (double& a : A) a *= sc;
    double term[16], next[16];
    for (int i = 0; i < 16; i++) term[i] = P[i];
    for (int k = 1; k <= 30; k++) {
        for (int i = 0; i < 4; i++)
            for (int j = 0; j < 4; j++) {
                double acc = 0;
                for (int m = 0; m < 4; m++) acc += term[4 * i + m] * A[4 * m + j];
                next[4 * i + j] = acc / k;
            }
        for (int i = 0; i < 16; i++) { term[i] = next[i]; P[i] += next[i]; }
    }
    for (int r = 0; r < s; r++) {
        for (int i = 0; i < 4; i++)
            for (int j = 0; j < 4; j++) {
                double acc = 0;
                for (int m = 0; m < 4; m++) acc += P[4 * i + m] * P[4 * m + j];
                next[4 * i + j] = acc;
            }
        for (int i = 0; i < 16; i++) P[i] = next[i];
    }
}

uint64_t prob_threshold(double c) {
    if (!(c > 0)) return 0;
    if (c >= 1) return ~0ull;
    return (uint64_t)std::ldexp(c, 64);
}

void row_thresholds(const double* row, uint64_t thr[3]) {
    double p[4], sum = 0;
    for (int j = 0; j < 4; j++) { p[j] = row[j] > 0 ? row[j] : 0.0; sum += p[j]; }
    double c = 0;
    for (int j = 0; j < 3; j++) { c += p[j] / sum; thr[j] = prob_threshold(c); }
}

}  // namespace jlp
