// Host side of the PacBio read generator: see jlp_pacbio.h.
#include "jlp_pacbio.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <stdexcept>

#include "jlp_draws.h"
#include "jlp_host.h"

namespace jlp {

namespace {

// Draw planes of the PacBio generator: counter = (j_lo, j_hi, block, PL_PB | sub << 8), two 64-bit draws per block.
// sub 0 read-level (block 0: truncated normals left / right; block 1: start, strand; blocks 16.. the tail branch's
// rejection loop), sub 1 the walk (position p: block p >> 1, half p & 1), sub 2 the inserted / substituted bases,
// sub 3 the samplers of this file.
constexpr uint32_t PL_PB = 6;
uint64_t pb_draw(uint64_t seed, uint64_t j, uint32_t sub, uint32_t block, uint32_t half) {
    const U4 w = draw_block(seed, j, block, PL_PB, sub);
    return half ? hi64(w) : lo64(w);
}

// runif_01 (src/pcg.h:99-101) in the reference's own type
long double runif_01(uint64_t x) { return ((long double)x + 1) / ((long double)UINT64_MAX + 2); }

// Standard normal distribution function and quantile.  The reference calls R::pnorm5 / R::qnorm5 here
// (src/hts_pacbio.h:349-352); these agree with Rmath to a few ulp: the lower tail through erfc, the quantile by
// Wichura's AS 241 (the algorithm R's qnorm5 uses), the same expressions as oracle/rmath_standin.h.
double pnorm(double x) { return 0.5 * std::erfc(-x * 0.70710678118654752440); }
double qnorm(double p) {
    /* Wichura (1988), Algorithm AS 241, routine PPND16 -- the algorithm R's qnorm5 itself uses: rational approximations
     * in q = p - 1/2 (central part) and in r = std::sqrt(-std::log(min(p, 1 - p))) (the tails), about 16 digits */
    if (!(p > 0.0)) return -INFINITY;
    if (!(p < 1.0)) return INFINITY;
    const double q = p - 0.5;
    if (std::fabs(q) <= 0.425) {
        const double r = 0.180625 - q * q;
        return q * (((((((2.5090809287301226727e+3 * r + 3.3430575583588128105e+4) * r + 6.7265770927008700853e+4) * r +
                        4.5921953931549871457e+4) * r + 1.3731693765509461125e+4) * r + 1.9715909503065514427e+3) * r +
                      1.3314166789178437745e+2) * r + 3.3871328727963666080) /
               (((((((5.2264952788528545610e+3 * r + 2.8729085735721942674e+4) * r + 3.9307895800092710610e+4) * r +
                    2.1213794301586595867e+4) * r + 5.3941960214247511077e+3) * r + 6.8718700749205790830e+2) * r +
                  4.2313330701600911252e+1) * r + 1.0);
    }
    double r = std::sqrt(-std::log(q < 0 ? p : 1.0 - p));
    double v;
    if (r <= 5.0) {
        r -= 1.6;
        v = (((((((7.74545014278341407640e-4 * r + 2.27238449892691845833e-2) * r + 2.41780725177450611770e-1) * r +
                 1.27045825245236838258) * r + 3.64784832476320460504) * r + 5.76949722146069140550) * r +
               4.63033784615654529590) * r + 1.42343711074968357734) /
            (((((((1.05075007164441684324e-9 * r + 5.47593808499534494600e-4) * r + 1.51986665636164571966e-2) * r +
                 1.48103976427480074590e-1) * r + 6.89767334985100004550e-1) * r + 1.67638483018380384940) * r +
               2.05319162663775882187) * r + 1.0);
    } else {
        r -= 5.0;
        v = (((((((2.01033439929228813265e-7 * r + 2.71155556874348757815e-5) * r + 1.24266094738807843860e-3) * r +
                 2.65321895265761230930e-2) * r + 2.96560571828504891230e-1) * r + 1.78482653991729133580) * r +
               5.46378491116411436990) * r + 6.65790464350110377720) /
            (((((((2.04426310338993978564e-15 * r + 1.42151175831644588870e-7) * r + 1.84631831751005468180e-5) * r +
                 7.86869131145613259100e-4) * r + 1.48753612908506148525e-2) * r + 1.36929880922735805310e-1) * r +
               5.99832206555887937690e-1) * r + 1.0);
    }
    return q < 0 ? -v : v;
}

// quantile of the chi-squared distribution (R::qchisq, src/hts_pacbio.h:178) by bisection on gamma_p
double qchisq(double p, double df) {
    const long double a = 0.5L * df;
    double lo = 0.0, hi = df + 10.0 * std::sqrt(2.0 * df) + 50.0;
    while ((double)gamma_p(a, 0.5L * hi) < p) hi *= 2.0;
    for (int i = 0; i < 60; i++) {
        const double mid = 0.5 * (lo + hi);
        if ((double)gamma_p(a, 0.5L * mid) < p) lo = mid; else hi = mid;
    }
    return 0.5 * (lo + hi);
}

double total_prob(const PbModel& m, double e) { return std::pow(m.prob_ins, e) + std::pow(m.prob_del, e) + std::pow(m.prob_subst, e); }

double sigmoid(double x) { return 1 / (1 + std::pow(2, (-2.5 / 3 * x + 6.5 / 3))); }

// a stream of uniforms in (0, 1) for the samplers of one read
struct SampleStream {
    uint64_t seed, j;
    uint32_t k = 0;
    U4 w{};                 // the Philox block draws k and k ^ 1 come from
    double next() {
        if ((k & 1u) == 0u) w = draw_block(seed, j, k >> 1, PL_PB, 3);
        const uint64_t x = (k & 1u) ? hi64(w) : lo64(w);
        k++;
        return ((double)(x >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    }
};

// Gamma(a, 1), Marsaglia and Tsang (2000); a < 1 through Gamma(a + 1) U^(1/a)
double sample_gamma(double a, SampleStream& S) {
    if (a < 1.0) return sample_gamma(a + 1.0, S) * std::pow(S.next(), 1.0 / a);
    const double d = a - 1.0 / 3.0, c = 1.0 / std::sqrt(9.0 * d);
    for (;;) {
        const double z = qnorm(S.next());
        const double v0 = 1.0 + c * z;
        if (v0 <= 0) continue;
        const double v = v0 * v0 * v0, u = S.next();
        if (std::log(u) < 0.5 * z * z + d - d * v + d * std::log(v)) return d * v;
    }
}

}  // namespace

void pb_prepare(PbModel& m) {
    if (!(m.prob_ins >= 0 && m.prob_del >= 0 && m.prob_subst >= 0) || m.prob_ins + m.prob_del + m.prob_subst > 1)
        throw std::runtime_error("\nWhen providing info for the PacBio sequencer, the insertion, deletion, and substitution "
                                 "probabilities cannot sum to > 1.");
    if (m.read_probs.size() != m.read_lens.size())
        throw std::runtime_error("Probability and read lengths vector should be the same length.");   // src/hts_pacbio.h:72-74
    // PacBioQualityError::calc_min_exp
    double min_exp = 1, total = total_prob(m, min_exp), left, right;
    if (total < m.prob_thresh) {
        while (total < m.prob_thresh) { min_exp /= 2; total = total_prob(m, min_exp); }
        left = min_exp; right = min_exp * 2;
    } else {
        while (total > m.prob_thresh) { min_exp *= 2; total = total_prob(m, min_exp); }
        left = min_exp / 2; right = min_exp;
    }
    for (int i = 0; i < 15; i++) {
        const double mid = (left + right) / 2;
        total = total_prob(m, mid);
        if (total == m.prob_thresh) { min_exp = mid; break; }
        else if (total > m.prob_thresh) { left = mid; min_exp = (mid + right) / 2; }
        else { right = mid; min_exp = (left + mid) / 2; }
    }
    m.min_exp = min_exp;
    m.qchisq_n = (size_t)std::max(1.0, std::floor(m.chi2_n[2])) + 2;
    m.qchisq_cache.reset(new std::atomic<double>[m.qchisq_n]);
    for (size_t i = 0; i < m.qchisq_n; i++) m.qchisq_cache.get()[i].store(-1.0, std::memory_order_relaxed);
    // the number of passes of a side is a whole number in [1, max_passes]: everything update_probs and trunc_norm derive
    // from it alone is computed once (the same expressions, so the same doubles)
    m.pass_tab.resize((size_t)std::min<uint64_t>(m.max_passes, 4096) + 2);
    for (size_t i = 0; i < m.pass_tab.size(); i++) {
        PbModel::PassTab& T = m.pass_tab[i];
        const double pass = (double)i;
        T.sig = sigmoid(pass);
        T.root = std::sqrt(pass + m.sqrt_params[0]) - m.sqrt_params[1];
        T.thresh = (m.min_exp - T.root) / T.sig;
        T.a_bar = (T.thresh - m.norm_params[0]) / m.norm_params[1];
        T.p_low = pnorm(T.a_bar);
    }
    if (!m.read_probs.empty()) {
        m.len_prob.resize(m.read_probs.size());
        m.len_alias.resize(m.read_probs.size());
        alias_build(m.read_probs.data(), m.read_probs.size(), m.len_prob.data(), m.len_alias.data());
    }
}

namespace {
// PacBioPassSampler::sample for r.read_length
void pb_passes(const PbModel& m, SampleStream& S, PbSample& r) {
    const double read_length = (double)r.read_length;
    const double lcap = std::min(read_length, m.chi2_n[2]);
    double n = m.chi2_n[0] * lcap + m.chi2_n[1];
    if (n < 0.001) n = 0.001;
    double s;
    if (read_length <= m.chi2_s[2]) {
        s = m.chi2_s[0] * read_length - m.chi2_s[1];
        if (s < 0.001) s = 0.001;
    } else {
        s = m.chi2_s[3] / std::pow(read_length, m.chi2_s[4]);
    }
    // the outlier threshold is a pure function of lcap (an integer): filled on first use; concurrent callers may compute
    // the same value twice
    std::atomic<double>& slot = m.qchisq_cache.get()[(size_t)std::floor(lcap)];
    double thr = slot.load(std::memory_order_relaxed);
    if (thr < 0) { thr = qchisq(0.9925, n); slot.store(thr, std::memory_order_relaxed); }
    double passes = 2.0 * sample_gamma(0.5 * n, S);
    while (passes > thr) passes = 2.0 * sample_gamma(0.5 * n, S);
    passes *= s;
    passes += 1;
    if (passes > (double)m.max_passes) passes = (double)m.max_passes;
    double wholes;
    const double fraction = std::modf(passes, &wholes);
    if (((uint64_t)wholes & 1ull) == 0ull) {
        r.split_pos = (uint64_t)std::round(read_length * fraction);
        r.passes_left = std::ceil(passes);
        r.passes_right = std::floor(passes);
    } else {
        r.split_pos = (uint64_t)std::round(read_length * (1 - fraction));
        r.passes_left = std::floor(passes);
        r.passes_right = std::ceil(passes);
    }
}
}  // namespace

PbSample pb_sample(const PbModel& m, uint64_t seed, uint64_t j, uint64_t chrom_len) {
    SampleStream S{seed, j};
    PbSample r;
    // ---- PacBioReadLenSampler::sample
    if (m.read_probs.empty()) {
        const double mu = std::log(m.scale);
        double min_len = std::ceil(m.min_read_len);
        if (min_len < 1) min_len = 1;
        double rnd = std::exp(mu + m.sigma * qnorm(S.next())) + m.loc;
        for (int it = 0; rnd < min_len && it < 10; it++) rnd = std::exp(mu + m.sigma * qnorm(S.next())) + m.loc;
        if (rnd < min_len) rnd = min_len;
        r.read_length = (uint64_t)rnd;
    } else {
        const uint64_t n = m.read_lens.size();
        uint64_t i = (uint64_t)(S.next() * (double)n);
        if (i >= n) i = n - 1;
        if (!(S.next() < m.len_prob[i])) i = m.len_alias[i];
        r.read_length = m.read_lens[i];
    }
    if (r.read_length >= chrom_len) r.read_length = chrom_len;          // one_read, src/hts_pacbio.cpp
    pb_passes(m, S, r);
    return r;
}

PbSample pb_sample_passes(const PbModel& m, uint64_t seed, uint64_t j, uint64_t read_length) {
    SampleStream S{seed, j};
    PbSample r;
    r.read_length = read_length;
    pb_passes(m, S, r);
    return r;
}

uint64_t pb_dup_draw(uint64_t seed, uint64_t j) { return pb_draw(seed, j, 0, 2, 0); }

namespace {

// PacBioQualityError::trunc_norm (src/hts_pacbio.h:340-370); side 0 = left, 1 = right
double trunc_norm(const PbModel& m, double lower_thresh, double a_bar, double p, uint64_t seed, uint64_t j, uint32_t side) {
    if (lower_thresh < (m.norm_params[0] + 5 * m.norm_params[1])) {
        const long double u = (long double)p + runif_01(pb_draw(seed, j, 0, 0, side)) * ((long double)1 - (long double)p);   // runif_ab
        return qnorm((double)u) * m.norm_params[1] + m.norm_params[0];
    }
    double x_bar;
    for (uint32_t it = 0;; it++) {
        const double u = (double)runif_01(pb_draw(seed, j, 0, 16 + 2 * it, side));
        x_bar = std::sqrt(a_bar * a_bar - 2 * std::log(1 - u));
        const double v = (double)runif_01(pb_draw(seed, j, 0, 17 + 2 * it, side));
        if (!(v > (x_bar / a_bar))) break;
    }
    return m.norm_params[1] * x_bar + m.norm_params[0];
}

}  // namespace

void pb_read_model(const PbModel& m, uint64_t seed, uint64_t j, const PbSample& s, PbRead& out) {
    // ---- update_probs
    const double pass[2] = {s.passes_left, s.passes_right};
    double cum[2][3];
    for (uint32_t side = 0; side < 2; side++) {
        PbModel::PassTab T;
        const size_t pi = pass[side] >= 0 && pass[side] < (double)m.pass_tab.size() ? (size_t)pass[side] : m.pass_tab.size();
        if (pi < m.pass_tab.size() && (double)pi == pass[side]) T = m.pass_tab[pi];
        else {
            T.sig = sigmoid(pass[side]);
            T.root = std::sqrt(pass[side] + m.sqrt_params[0]) - m.sqrt_params[1];
            T.thresh = (m.min_exp - T.root) / T.sig;
            T.a_bar = (T.thresh - m.norm_params[0]) / m.norm_params[1];
            T.p_low = pnorm(T.a_bar);
        }
        const double incr = trunc_norm(m, T.thresh, T.a_bar, T.p_low, seed, j, side);
        double e = incr * T.sig + std::sqrt(pass[side] + m.sqrt_params[0]) - m.sqrt_params[1];
        if (e < 0.6) e = 0.6;
        cum[side][0] = std::pow(m.prob_ins, e);
        cum[side][1] = std::pow(m.prob_del, e) + cum[side][0];
        cum[side][2] = std::pow(m.prob_subst, e) + cum[side][1];
    }
    // ---- fill_quals
    uint32_t flags = 0;
    for (uint32_t side = 0; side < 2; side++) {
        uint64_t q = (uint64_t)std::round(-10.0 * std::log10(cum[side][2]));
        if (q > 93) q = 93;
        flags |= (uint32_t)(q + '!') << (8 + 8 * side);
        // ---- the walk's comparisons on `double u` (src/hts_pacbio.h:300-316): u > cum[2] no event; u < cum[0] insertion;
        //      u < cum[1] deletion; else substitution
        const Thr t[3] = {thr_double_lt(cum[side][0]), thr_double_lt(cum[side][1]), thr_double_le(cum[side][2])};
        for (uint32_t k = 0; k < 3; k++) {
            out.thr[side][k] = t[k].thr;
            if (t[k].all) flags |= 1u << (3 * side + k);
        }
    }
    out.read_length = (uint32_t)s.read_length;
    out.split_pos = (uint32_t)s.split_pos;
    out.flags = flags;
}

uint64_t pb_plan(const PbModel& m, uint64_t seed, uint64_t b0, uint32_t n, uint64_t job_lo, uint64_t pool, Thr t_dup,
                 const std::vector<uint64_t>& group_off, const GroupDev* groups, uint64_t n_threads, PbRead* out,
                 PbSample* samples) {
    const bool dups = t_dup.thr != 0 || t_dup.all;
    std::vector<uint32_t> lead(n, kPbNoLeader);
    if (dups)
        for (uint32_t i = 1; i < n; i++)
            if ((b0 + i - job_lo) % pool != 0 && (t_dup.all || pb_dup_draw(seed, b0 + i - 1) < t_dup.thr))
                lead[i] = lead[i - 1] == kPbNoLeader ? i - 1 : lead[i - 1];
    // the reads are independent given their leaders
    const uint32_t nt = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(n_threads, 1), 64);
    std::vector<uint64_t> len(nt, 0);
    for (int pass = 0; pass < (dups ? 2 : 1); pass++)
        parallel_for(nt, nt, [&](uint64_t k) {
            for (uint32_t i = (uint32_t)k; i < n; i += nt) {
                if ((lead[i] != kPbNoLeader) != (pass == 1)) continue;
                const uint64_t j = b0 + i;
                PbSample s;
                size_t g;
                if (pass == 0) {
                    g = (size_t)(std::upper_bound(group_off.begin(), group_off.end(), j) - group_off.begin()) - 1;
                    s = pb_sample(m, seed, j, groups[g].len);
                } else {
                    g = out[lead[i]].group;
                    s = pb_sample_passes(m, seed, j, out[lead[i]].read_length);
                }
                std::memset(&out[i], 0, sizeof(PbRead));
                pb_read_model(m, seed, j, s, out[i]);
                out[i].group = (uint32_t)g;
                out[i].leader = lead[i];
                if (samples) samples[i] = s;
                len[k] += s.read_length;
            }
        });
    uint64_t total = 0;
    for (uint64_t v : len) total += v;
    return total;
}

}  // namespace jlp
