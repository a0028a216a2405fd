/*
 * TEST INFRASTRUCTURE ONLY -- CPU oracle for the Illumina read-generation path.
 *
 * A plain-C restatement of the reference algorithm (lucasnell/jackalope v1.1.6)
 * for the path illumina_ref_cpp / illumina_hap_cpp -> IlluminaOneGenome /
 * IlluminaHaplotypes.  Every function cites the reference file:line it follows
 * (paths relative to /root/reference).  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this library; the
 * product (jackalope_b200/) never does and has no CPU fallback.
 *
 * Parity status: PINNED.  tests/test_oracle_vs_reference.py drives the
 * unmodified reference (oracle/_ref/libjlp_ref_replay.so, built from the
 * sources under /root/reference by oracle/Makefile) with the draw ledger this
 * oracle emits and requires byte-identical FASTQ; golden vectors made that way
 * are committed under tests/golden/.
 *
 * What is restated literally: every arithmetic use of a uniform draw uses the
 * same C types as the reference (x87 80-bit long double on x86-64, rounded to
 * double exactly where the reference stores into a `double`).  What differs by
 * design (DESIGN.md "draw addressing"): the reference pulls draws sequentially
 * from one pcg64 per thread; here each logical draw X(pair, end, purpose, pos)
 * is a pure function of a Philox4x32-10 counter, so reads are independent of
 * GPU count.  The ledger lists the draws in the order the reference consumes
 * them (SURVEY.md Appendix A.1) so the reference can be replayed.
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#if LDBL_MANT_DIG != 64
#error "oracle assumes x87 80-bit long double, as the reference's runif_01 does on x86-64"
#endif

/* ------------------------------------------------------------------ Philox */

/* Philox4x32-R (Salmon et al., SC'11), standard constants. */
static void philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4], int rounds) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < rounds; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) { philox4x32(ctr, key, out, 10); }
void orc_philox4x32_r(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4], int rounds) { philox4x32(ctr, key, out, rounds); }

/* Draw addressing (DESIGN.md section 4).  counter = (j_lo, j_hi, block, plane | end<<8) */
enum { PL_PAIR = 0, PL_INDEL = 1, PL_QUAL = 2, PL_SLOW = 3 };
enum { PU_INDEL = 0, PU_DIE = 1, PU_COIN = 2, PU_MIS = 3, PU_SUB = 4, PU_INS = 5 };

static void call(uint64_t seed, uint64_t j, uint32_t block, uint32_t plane, uint32_t end, uint32_t w[4]) {
    uint32_t ctr[4] = {(uint32_t)j, (uint32_t)(j >> 32), block, plane | (end << 8)};
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    philox4x32(ctr, key, w, plane == PL_QUAL || plane == PL_INDEL ? 7 : 10);      /* the per-base planes run 7 rounds (jlp_draws.h, kQualRounds) */
}

/* pair-level draws: which = 0 fraglen, 1 start, 2 strand, 3 dup */
uint64_t orc_draw_pair(uint64_t seed, uint64_t j, int which) {
    uint32_t w[4];
    call(seed, j, (uint32_t)(which >> 1), PL_PAIR, 0, w);
    return (which & 1) ? (((uint64_t)w[3] << 32) | w[2]) : (((uint64_t)w[1] << 32) | w[0]);
}

static uint64_t slow64(uint64_t seed, uint64_t j, uint32_t end, uint32_t purpose, uint32_t pos) {
    uint32_t w[4];
    call(seed, j, (pos << 3) | purpose, PL_SLOW, end, w);
    return ((uint64_t)w[1] << 32) | w[0];
}

/* per-end, per-position draws (layout: jackalope_b200/csrc/jlp_draws.h) */
uint64_t orc_draw_pos(uint64_t seed, uint64_t j, uint32_t end, uint32_t purpose, uint32_t pos) {
    uint32_t w[4];
    uint64_t H, s = slow64(seed, j, end, purpose, pos);
    uint32_t hb;
    if (purpose == PU_INS) return s;
    if (purpose == PU_INDEL) {
        call(seed, j, pos >> 3, PL_INDEL, end, w);
        uint32_t f = pos & 7;
        H = (w[f >> 1] >> (16 * (f & 1))) & 0xffffu;
        hb = 16;
    } else {
        call(seed, j, pos >> 1, PL_QUAL, end, w);
        uint32_t h = pos & 1;
        if (purpose == PU_DIE) { H = w[2 * h] >> 8; hb = 24; }
        else if (purpose == PU_SUB) { H = w[2 * h] & 0xffu; hb = 8; }
        else if (purpose == PU_COIN) { H = w[2 * h + 1] >> 16; hb = 16; }
        else { H = w[2 * h + 1] & 0xffffu; hb = 16; }   /* PU_MIS */
    }
    return (H << (64 - hb)) | (s & (~0ull >> hb));
}

/* -------------------------------------------------- reference primitives */

/* runif_01, src/pcg.h:21,99-101 */
static long double runif_01(uint64_t x) {
    const long double max64 = (long double)UINT64_MAX;
    return ((long double)x + 1) / (max64 + 2);
}

/* nt_map, src/hts.h:36-44: T,C,A,G -> 0..3, everything else 4 */
static uint8_t nt_map(unsigned char c) {
    switch (c) { case 'T': return 0; case 'C': return 1; case 'A': return 2; case 'G': return 3; }
    return 4;
}
/* mm_nucleos, src/hts.h:46 */
static const char* const MM[5] = {"CAG", "TAG", "TCG", "TCA", "NNN"};
/* jlp::bases, src/jackalope_types.h:36; std::string::operator[](size()) yields '\0' */
static const char BASES[5] = {'T', 'C', 'A', 'G', '\0'};

/* cmp_map, src/str_manip.h:58-72: A<->T, C<->G, N->N, anything else -> 0 */
static char cmp_map(unsigned char c) {
    switch (c) { case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'N': return 'N'; case 'T': return 'A'; }
    return 0;
}
/* rev_comp, src/str_manip.h:214-229 */
void orc_rev_comp(char* s, uint64_t n) {
    uint64_t half = n / 2;
    for (uint64_t j = 0; j < half; j++) {
        char tmp = cmp_map((unsigned char)s[j]);
        s[j] = cmp_map((unsigned char)s[n - j - 1]);
        s[n - j - 1] = tmp;
    }
    if (n & 1) s[half] = cmp_map((unsigned char)s[half]);
}

/* AliasSampler::construct, src/alias_sampler.h:68-106 (Vose; FIFO Small/Large) */
int orc_alias_build(const double* probs, uint64_t n, double* Prob, uint64_t* Alias) {
    double* p = (double*)malloc(sizeof(double) * (n ? n : 1));
    uint64_t* small = (uint64_t*)malloc(sizeof(uint64_t) * 2 * (n ? n : 1));
    uint64_t* large = (uint64_t*)malloc(sizeof(uint64_t) * 2 * (n ? n : 1));
    if (!p || !small || !large) return -1;
    double sum = 0.0;
    for (uint64_t i = 0; i < n; i++) sum += probs[i];       /* arma::accu -> plain sum */
    for (uint64_t i = 0; i < n; i++) p[i] = probs[i] / sum;
    for (uint64_t i = 0; i < n; i++) p[i] *= (double)n;
    for (uint64_t i = 0; i < n; i++) { Prob[i] = 0.0; Alias[i] = 0; }
    uint64_t sh = 0, st = 0, lh = 0, lt = 0;                /* queue head/tail */
    for (uint64_t i = 0; i < n; i++) { if (p[i] < 1) small[st++] = i; else large[lt++] = i; }
    /* each pop pair pushes one element, so 2n slots suffice */
    while (sh < st && lh < lt) {
        uint64_t l = small[sh++], g = large[lh++];
        Prob[l] = p[l];
        Alias[l] = g;
        p[g] = (p[g] + p[l]) - 1;
        if (p[g] < 1) small[st++] = g; else large[lt++] = g;
    }
    while (lh < lt) Prob[large[lh++]] = 1;
    while (sh < st) Prob[small[sh++]] = 1;
    free(p); free(small); free(large);
    return 0;
}

/* HapChrom::size_modifier, src/hap_classes.h:314-333 */
static int64_t size_modifier(uint64_t i, uint64_t M, const uint64_t* old_pos, const uint64_t* new_pos,
                             uint64_t chrom_size, uint64_t ref_size) {
    int64_t sm;
    if (i < M - 1) sm = (int64_t)(new_pos[i + 1] - old_pos[i + 1]);
    else sm = (int64_t)(chrom_size - ref_size);
    sm += (int64_t)(old_pos[i] - new_pos[i]);
    return sm;
}
/* HapChrom::get_char_, src/hap_classes.h:439-455 */
static char get_char_(uint64_t pos, uint64_t i, const char* ref, uint64_t ref_size, uint64_t M,
                      const uint64_t* old_pos, const uint64_t* new_pos, const uint64_t* nuc_off,
                      const char* pool, uint64_t chrom_size) {
    uint64_t ind = pos - new_pos[i];
    int64_t sm = size_modifier(i, M, old_pos, new_pos, chrom_size, ref_size);
    if ((int64_t)ind > sm) {
        ind += old_pos[i] - (uint64_t)sm;
        return ref[ind];
    }
    return pool[nuc_off[i] + ind];
}
/* HapChrom::get_chrom_full, src/hap_classes.cpp:80-116 */
int orc_materialize(const char* ref, uint64_t ref_size, uint64_t M, const uint64_t* old_pos,
                    const uint64_t* new_pos, const uint64_t* nuc_off, const char* pool,
                    uint64_t chrom_size, char* out) {
    if (M == 0) { memcpy(out, ref, ref_size); return 0; }
    uint64_t mut_i = 0, pos = 0, n = 0;
    while (pos < new_pos[mut_i]) { out[n++] = ref[pos]; ++pos; }
    uint64_t next = mut_i + 1;
    while (next < M) {
        while (pos < new_pos[next]) {
            out[n++] = get_char_(pos, mut_i, ref, ref_size, M, old_pos, new_pos, nuc_off, pool, chrom_size);
            ++pos;
        }
        ++mut_i; ++next;
    }
    while (pos < chrom_size) {
        out[n++] = get_char_(pos, mut_i, ref, ref_size, M, old_pos, new_pos, nuc_off, pool, chrom_size);
        ++pos;
    }
    return 0;
}

/* ---------------------------------------------------------- read generation */

typedef struct {
    uint64_t L;
    double* Prob;        /* alias tables, concatenated in (nt,pos) order */
    uint64_t* Alias;
    const uint8_t* quals;
    uint64_t* off;       /* [4*L+1] */
    double qual_prob_map[256];
} EndModel;

/* IlluminaQualityError ctor, src/hts_illumina.h:154-189; IllQualPos ctor :102-116 */
static int end_model_init(EndModel* m, uint64_t L, const uint32_t* nq, const double* probs, const uint8_t* quals) {
    m->L = L;
    m->off = (uint64_t*)malloc(sizeof(uint64_t) * (4 * L + 1));
    uint64_t tot = 0;
    for (uint64_t i = 0; i < 4 * L; i++) { m->off[i] = tot; tot += nq[i]; }
    m->off[4 * L] = tot;
    m->Prob = (double*)malloc(sizeof(double) * (tot ? tot : 1));
    m->Alias = (uint64_t*)malloc(sizeof(uint64_t) * (tot ? tot : 1));
    m->quals = quals;
    uint8_t max_qual = 0;
    for (uint64_t i = 0; i < 4 * L; i++) {
        if (orc_alias_build(probs + m->off[i], nq[i], m->Prob + m->off[i], m->Alias + m->off[i])) return -1;
        for (uint32_t k = 0; k < nq[i]; k++) if (quals[m->off[i] + k] > max_qual) max_qual = quals[m->off[i] + k];
    }
    m->qual_prob_map[0] = 1;
    for (unsigned q = 1; q <= max_qual; q++) {
        /* std::pow(10, double(q) / -10.0), src/hts_illumina.h:185 */
        m->qual_prob_map[q] = pow(10, (double)q / -10.0);
    }
    return 0;
}
static void end_model_free(EndModel* m) { free(m->off); free(m->Prob); free(m->Alias); }

int orc_qual_prob_map(uint64_t L, const uint32_t* nq, const double* probs, const uint8_t* quals, double* out) {
    EndModel m;
    if (end_model_init(&m, L, nq, probs, quals)) return -1;
    memcpy(out, m.qual_prob_map, sizeof(double) * 256);
    end_model_free(&m);
    return 0;
}

typedef struct {
    uint64_t* data; uint64_t n, cap; int on;
} Ledger;
static void led(Ledger* l, uint64_t x) {
    if (!l->on) return;
    if (l->n < l->cap) l->data[l->n] = x;
    l->n++;
}

typedef struct {
    char* data; uint64_t n, cap;
} Sink;
static void put(Sink* s, const char* p, uint64_t n) {
    if (s->n + n <= s->cap) memcpy(s->data + s->n, p, n);
    s->n += n;
}
static void putc_(Sink* s, char c) { put(s, &c, 1); }

/*
 * One call generates pair instances [lo, hi) of one job.
 *
 *  job_lo/job_hi  : pair-index range of the job (one write_reads_cpp_ call of the
 *                   reference; with sep_files there is one job per haplotype,
 *                   src/hts.h:512-552).  Duplicate chains and pool boundaries are
 *                   relative to job_lo (src/hts.h:254-280).
 *  group_off      : [n_groups+1] pair-index prefix offsets of the (haplotype,
 *                   chromosome) groups, hap-major / chrom-major, i.e. the order
 *                   in which the reference exhausts chrom_reads / n_reads_vc
 *                   (src/hts_illumina.cpp:199-201, :505-528).
 *  frag_cdf       : fragment-length table (DESIGN.md): frag_len = frag_min +
 *                   #{i : X >= frag_cdf[i]}.  Replaces std::gamma_distribution,
 *                   whose draw count is stateful (SURVEY.md A.1) -- "injected".
 *  plan           : optional [4*(hi-lo)] out: group, frag_len, frag_start, leader
 *  ledger         : optional out, draws in reference consumption order;
 *                   ledger_cnt[i] = draws of instance i.
 */
typedef struct {
    uint64_t seed;
    int32_t paired, matepair;
    uint64_t job_lo, job_hi;
    uint64_t pool_pairs;
    double prob_dup;
    uint64_t L;
    double ins_prob[2], del_prob[2];
    const uint32_t* nq[2];
    const double* probs[2];
    const uint8_t* quals[2];
    const uint64_t* frag_cdf; uint64_t frag_cdf_n; uint64_t frag_min;
    uint64_t n_groups;
    const uint64_t* group_off;
    const char* const* group_seq;
    const uint64_t* group_len;
    const char* const* group_genome_name;
    const char* const* group_chrom_name;
    const char* const* group_barcode;
    /* optional out (NULL: not counted), added to: the draws whose high bits alone leave the answer open in k_reads
     * (base_fast / base_rare, jackalope_b200/csrc/jlp_kernels.cu), and those where the exact answer differs from the
     * one the high bits give -- coverage accounting of the kernels' exact-draw fallbacks, never part of the output.
     * [0] ambiguous / [1] flipped alias slot, [2] / [3] N quality, [4] / [5] substitution index. */
    uint64_t* fallback;
} OrcJob;

static uint64_t find_group(const OrcJob* J, uint64_t k) {
    /* last g with group_off[g] <= k (empty groups are skipped) */
    uint64_t lo = 0, hi = J->n_groups;
    while (hi - lo > 1) { uint64_t mid = (lo + hi) / 2; if (J->group_off[mid] <= k) lo = mid; else hi = mid; }
    return lo;
}

/* ReadWriterOneThread::create_reads, src/hts.h:254-280: instance j re-reads the
 * fragment of j-1 iff the draw made after j-1 satisfies `dup < prob_dup`, j is
 * not the first of its job and the pool is not full. */
static uint64_t find_leader(const OrcJob* J, uint64_t j) {
    uint64_t k = j;
    while (k > J->job_lo && ((k - J->job_lo) % J->pool_pairs) != 0) {
        double dup = (double)runif_01(orc_draw_pair(J->seed, k - 1, 3));
        if (!(dup < J->prob_dup)) break;
        k--;
    }
    return k;
}

int orc_generate(const OrcJob* J, uint64_t lo, uint64_t hi,
                 char* out1, uint64_t cap1, uint64_t* len1,
                 char* out2, uint64_t cap2, uint64_t* len2,
                 uint64_t* plan, uint64_t* ledger, uint64_t ledger_cap,
                 uint64_t* ledger_n, uint64_t* ledger_cnt) {
    const uint64_t L = J->L;
    const int n_ends = J->paired ? 2 : 1;
    EndModel em[2];
    for (int e = 0; e < n_ends; e++)
        if (end_model_init(&em[e], L, J->nq[e], J->probs[e], J->quals[e])) return -1;
    Sink sk[2] = {{out1, 0, cap1}, {out2, 0, cap2}};
    Ledger lg = {ledger, 0, ledger_cap, ledger != NULL};
    uint64_t cap_t = 4 * L + 64;
    uint64_t* ins[2]; uint64_t* del[2]; uint64_t n_ins[2], n_del[2];
    for (int e = 0; e < 2; e++) {
        ins[e] = (uint64_t*)malloc(sizeof(uint64_t) * cap_t);
        del[e] = (uint64_t*)malloc(sizeof(uint64_t) * cap_t * 64);
    }
    char* read = (char*)malloc(cap_t * 64 + 2 * L + 64);
    char* qual = (char*)malloc(cap_t + 64);
    int rc = 0;

    for (uint64_t j = lo; j < hi; j++) {
        uint64_t led0 = lg.n;
        /* --- fragment: chrom_indels_frag / indels_frag, src/hts_illumina.cpp:191-265 */
        uint64_t k = find_leader(J, j);
        uint64_t g = find_group(J, k);
        uint64_t chrom_len = J->group_len[g];
        const char* chrom = J->group_seq[g];
        uint64_t xf = orc_draw_pair(J->seed, k, 0);
        uint64_t frag_len = J->frag_min;
        for (uint64_t i = 0; i < J->frag_cdf_n; i++) { if (xf >= J->frag_cdf[i]) frag_len++; else break; }
        uint64_t frag_start;
        if (frag_len >= chrom_len) { frag_len = chrom_len; frag_start = 0; }
        else {
            double u = (double)runif_01(orc_draw_pair(J->seed, k, 1));
            frag_start = (uint64_t)(u * (chrom_len - frag_len + 1));
        }
        if (plan) { uint64_t* p = plan + 4 * (j - lo); p[0] = g; p[1] = frag_len; p[2] = frag_start; p[3] = k; }
        const char* barcode = J->group_barcode[g] ? J->group_barcode[g] : "";
        uint64_t b = strlen(barcode);

        /* --- sample_indels, src/hts_illumina.cpp:116-150 */
        uint64_t space[2];
        for (int r = 0; r < n_ends; r++) {
            uint64_t frag_pos = 0, length_now = 0;
            n_ins[r] = n_del[r] = 0;
            double ins_prob = J->ins_prob[r], del_prob = J->del_prob[r];
            while (length_now < L && frag_pos < frag_len) {
                uint64_t x = orc_draw_pos(J->seed, j, (uint32_t)r, PU_INDEL, (uint32_t)frag_pos);
                led(&lg, x);
                double u = (double)runif_01(x);
                if (u > (ins_prob + del_prob)) length_now++;
                else if (u > ins_prob) {
                    if (n_del[r] >= cap_t * 64) { rc = -2; goto done; }
                    del[r][n_del[r]++] = frag_pos;
                } else {
                    if (length_now == (L - 1)) length_now++;
                    else { ins[r][n_ins[r]++] = frag_pos; length_now += 2; }
                }
                frag_pos++;
            }
            /* adjust_chrom_spaces, src/hts_illumina.cpp:153-184 */
            int64_t indel_effect = (int64_t)n_del[r] - (int64_t)n_ins[r];
            uint64_t S = L + (uint64_t)indel_effect;
            if (S > frag_len) S = frag_len;
            if (S <= b) { rc = -3; goto done; }   /* barcode >= template: UB in the reference */
            space[r] = S - b;
        }

        /* --- append_pools, src/hts_illumina.cpp:337-482 */
        uint64_t xs = orc_draw_pair(J->seed, j, 2);
        led(&lg, xs);
        int reverse = runif_01(xs) < 0.5;
        for (int i = 0; i < n_ends; i++) {
            uint64_t S = space[i] + b;
            uint64_t start;
            if ((!J->matepair && !reverse) || (J->matepair && reverse)) start = frag_start;
            else start = frag_start + frag_len - space[i];
            uint64_t rl = S;
            memset(read, 'N', S);
            if (!reverse) memcpy(read + b, chrom + start, space[i]);   /* fill_read, src/ref_classes.h:102-116; fill_read__, src/hts.h:109-130 */
            else { memcpy(read, chrom + start, space[i]); orc_rev_comp(read, S); }
            memcpy(read, barcode, b);

            /* fill_read_qual, src/hts_illumina.h:202-259 : indels from the back */
            {
                uint64_t ni = n_ins[i], nd = n_del[i];
                uint64_t chrom_pos = rl - 1;
                while (ni > 0 || nd > 0) {
                    if (ni > 0 && chrom_pos == ins[i][ni - 1]) {
                        uint64_t x = orc_draw_pos(J->seed, j, (uint32_t)i, PU_INS, (uint32_t)chrom_pos);
                        led(&lg, x);
                        char c = BASES[(uint64_t)(runif_01(x) * 4.0)];
                        memmove(read + chrom_pos + 2, read + chrom_pos + 1, rl - chrom_pos - 1);
                        read[chrom_pos + 1] = c;
                        rl++; ni--;
                    } else if (nd > 0 && chrom_pos == del[i][nd - 1]) {
                        memmove(read + chrom_pos, read + chrom_pos + 1, rl - chrom_pos - 1);
                        rl--; nd--;
                    }
                    if (chrom_pos == 0) break;
                    chrom_pos--;
                }
            }
            /* mismatches + qualities */
            for (uint64_t pos = 0; pos < rl; pos++) {
                uint8_t nt_ind = nt_map((unsigned char)read[pos]);
                uint8_t qint;
                if (nt_ind > 3) {
                    uint64_t x = orc_draw_pos(J->seed, j, (uint32_t)i, PU_DIE, (uint32_t)pos);
                    led(&lg, x);
                    qint = (uint8_t)(runif_01(x) * 10 + (uint8_t)'!');
                    if (J->fallback) {          /* base_rare: u * 10 + 33 on the draw's high 24 bits */
                        const uint32_t dn = (uint32_t)(x >> 40) << 8;
                        if (dn * 10u + 2560u < 2560u) {
                            J->fallback[2]++;
                            J->fallback[3] += (uint8_t)((uint32_t)(((uint64_t)dn * 10u) >> 32) + 33u) != qint;
                        }
                    }
                    qual[pos] = (char)qint;
                    read[pos] = 'N';
                    continue;
                }
                /* IllQualPos::sample :128-132 ; AliasSampler::sample src/alias_sampler.h:53-60 */
                const EndModel* m = &em[i];
                uint64_t o = m->off[nt_ind * L + pos];
                uint64_t n = m->off[nt_ind * L + pos + 1] - o;
                uint64_t xd = orc_draw_pos(J->seed, j, (uint32_t)i, PU_DIE, (uint32_t)pos);
                led(&lg, xd);
                uint64_t ii = (uint64_t)(runif_01(xd) * n);
                if (ii >= n) ii = n - 1;   /* u == 1.0 (x = 2^64-1) reads past the table in the reference: clamp (DESIGN.md) */
                if (J->fallback) {          /* base_fast / base_rare: the slot from the draw's high 24 bits */
                    const uint32_t dc = (uint32_t)(xd >> 40) << 8, n32 = (uint32_t)n;
                    if (dc * n32 + (n32 << 8) < (n32 << 8)) {
                        J->fallback[0]++;
                        J->fallback[1] += (uint32_t)(((uint64_t)dc * n32) >> 32) != ii;
                    }
                }
                uint64_t xc = orc_draw_pos(J->seed, j, (uint32_t)i, PU_COIN, (uint32_t)pos);
                led(&lg, xc);
                double u = (double)runif_01(xc);
                uint64_t kk = (u < m->Prob[o + ii]) ? ii : m->Alias[o + ii];
                qint = m->quals[o + kk];
                double mis_prob = m->qual_prob_map[qint];
                qint = (uint8_t)(qint + (uint8_t)'!');
                qual[pos] = (char)qint;
                uint64_t xm = orc_draw_pos(J->seed, j, (uint32_t)i, PU_MIS, (uint32_t)pos);
                led(&lg, xm);
                u = (double)runif_01(xm);
                if (u < mis_prob) {
                    uint64_t xsub = orc_draw_pos(J->seed, j, (uint32_t)i, PU_SUB, (uint32_t)pos);
                    led(&lg, xsub);
                    uint64_t si = (uint64_t)(runif_01(xsub) * 3.0);
                    if (si > 2) si = 2;    /* same 2^-64 edge as above */
                    if (J->fallback) {      /* base_rare: u * 3 on the draw's high 8 bits */
                        const uint32_t p3 = (uint32_t)(xsub >> 56) * 3u;
                        if ((p3 & 0xffu) + 3u > 0xffu) {
                            J->fallback[4]++;
                            J->fallback[5] += (p3 >> 8) != si;
                        }
                    }
                    read[pos] = MM[nt_ind][si];
                }
            }
            /* fill_fq_lines, src/hts_illumina.cpp:285-326 */
            {
                char num[32];
                Sink* s = &sk[i];
                putc_(s, '@');
                put(s, J->group_genome_name[g], strlen(J->group_genome_name[g]));
                putc_(s, '-');
                put(s, J->group_chrom_name[g], strlen(J->group_chrom_name[g]));
                putc_(s, '-');
                int nn = snprintf(num, sizeof num, "%llu", (unsigned long long)start);
                put(s, num, (uint64_t)nn);
                putc_(s, '-');
                putc_(s, reverse ? 'R' : 'F');
                if (J->paired) { putc_(s, '/'); putc_(s, (char)('1' + i)); }
                putc_(s, '\n');
                put(s, read, rl); putc_(s, '\n');
                putc_(s, '+'); putc_(s, '\n');
                put(s, qual, rl); putc_(s, '\n');
                reverse = !reverse;
            }
        }
        if (ledger_cnt) ledger_cnt[j - lo] = lg.n - led0;
    }
done:
    *len1 = sk[0].n;
    if (len2) *len2 = sk[1].n;
    if (ledger_n) *ledger_n = lg.n;
    if (rc == 0 && (sk[0].n > cap1 || sk[1].n > cap2)) rc = -4;
    if (rc == 0 && lg.on && lg.n > lg.cap) rc = -5;
    for (int e = 0; e < n_ends; e++) end_model_free(&em[e]);
    for (int e = 0; e < 2; e++) { free(ins[e]); free(del[e]); }
    free(read); free(qual);
    return rc;
}

/* ----------------------------------------------------------- create_genome */

/* draws of the genome generator (layout: jackalope_b200/csrc/jlp_draws.h): which 0 = die, 1 = coin */
uint64_t orc_genome_draw(uint64_t seed, uint32_t chrom, uint64_t b, int which) {
    uint32_t ctr[4] = {(uint32_t)(b >> 2), (uint32_t)((b >> 2) >> 32), chrom, 4u}, key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)}, w[4], v[4];
    orc_philox4x32_10(ctr, key, w);
    uint32_t word = w[b & 3];
    uint32_t c2[4] = {(uint32_t)b, (uint32_t)(b >> 32), chrom, 5u | ((uint32_t)which << 8)};
    orc_philox4x32_10(c2, key, v);
    uint64_t s = ((uint64_t)v[1] << 32) | v[0];
    if (which == 0) return ((uint64_t)(word >> 30) << 62) | (s & (~0ull >> 2));
    return ((uint64_t)((word >> 14) & 0xffffu) << 48) | (s & (~0ull >> 16));
}

/* One chromosome of create_chromosomes_ (src/create_sequences.cpp:129-132): per base
 * k = sampler.sample(engine) (AliasSampler::sample, src/alias_sampler.h:53-60), base = jlp::bases[k].
 * ledger (optional, 2 * len): the draws in the order the reference consumes them. */
int orc_create_chrom(uint64_t seed, uint32_t chrom, uint64_t len, const double* pi_tcag, char* out, uint64_t* ledger) {
    double Prob[4];
    uint64_t Alias[4];
    if (orc_alias_build(pi_tcag, 4, Prob, Alias)) return -1;
    for (uint64_t b = 0; b < len; b++) {
        uint64_t xd = orc_genome_draw(seed, chrom, b, 0), xc = orc_genome_draw(seed, chrom, b, 1);
        if (ledger) { ledger[2 * b] = xd; ledger[2 * b + 1] = xc; }
        uint64_t i = (uint64_t)(runif_01(xd) * 4);
        if (i > 3) i = 3;                       /* u == 1.0 (x = 2^64-1) indexes past the table in the reference: clamp */
        double u = (double)runif_01(xc);
        uint64_t k = (u < Prob[i]) ? i : Alias[i];
        out[b] = BASES[k];
    }
    return 0;
}

/* literal uniform expressions, same numbering as jref_unif_expr in ref_driver.cpp */
uint64_t orc_unif_expr(int kind, uint64_t x, double p, uint64_t n) {
    long double ul = runif_01(x);
    switch (kind) {
    case 0: return (uint64_t)(ul * n);
    case 1: { double u = (double)ul; return u < p; }
    case 2: { double u = (double)ul; return u > p; }
    case 3: return ul < p;
    case 4: { uint8_t q = (uint8_t)(ul * 10 + (uint8_t)'!'); return q; }
    case 5: { double u = (double)ul; return (uint64_t)(u * n); }
    }
    return 0;
}

/* ==================================================================== PacBio ===
 * C restatement of the PacBio read model (SURVEY.md section 8f rank 3; /root/reference/src/hts_pacbio.{h,cpp}):
 * what PacBioOneGenome::one_read does once the two stateful samplers have spoken.  Read length and
 * (split_pos, passes_left, passes_right) are INJECTED per read (std::lognormal_distribution and
 * std::chi_squared_distribution keep cached normals, so their draw counts depend on the history; they are
 * compared statistically), everything after them is restated draw for draw:
 *   PacBioQualityError::calc_min_exp      src/hts_pacbio.cpp
 *   PacBioQualityError::update_probs      src/hts_pacbio.cpp      (trunc_norm: src/hts_pacbio.h:340-370)
 *   PacBioQualityError::fill_quals        src/hts_pacbio.h:383-391
 *   PacBioQualityError::sample (the walk) src/hts_pacbio.h:282-318
 *   read_chrom_space, read_start          src/hts_pacbio.cpp, one_read
 *   PacBioOneGenome::append_pool          src/hts_pacbio.cpp
 * R::pnorm5 / R::qnorm5 are the stand-ins of rmath_standin.h on both sides of the comparison.
 *
 * Draw addressing: counter = (j_lo, j_hi, block, PL_PB | sub << 8), two 64-bit draws per Philox block.
 *   sub 0 (read):  block 0: truncated normal left, right (its usual branch: one draw each);
 *                  block 1: read_start, strand;
 *                  blocks 16 + 2 it / 17 + 2 it: draws (u, v) of iteration `it` of the tail branch's rejection
 *                  loop, left (lo halves) and right (hi halves)
 *   sub 1 (walk):  template position p -> block p >> 1, half p & 1
 *   sub 2 (edit):  the inserted / substituted base drawn at read position p -> block p >> 1, half p & 1 */
#include "rmath_standin.h"

enum { PL_PB = 6 };   /* planes 4 and 5 address the genome generator */

static uint64_t pb_draw(uint64_t seed, uint64_t j, uint32_t sub, uint32_t block, uint32_t half) {
    uint32_t w[4];
    call(seed, j, block, PL_PB, sub, w);
    return half ? (((uint64_t)w[3] << 32) | w[2]) : (((uint64_t)w[1] << 32) | w[0]);
}
uint64_t orc_pb_draw(uint64_t seed, uint64_t j, uint32_t sub, uint32_t block, uint32_t half) { return pb_draw(seed, j, sub, block, half); }

typedef struct {
    double sqrt_params[2], norm_params[2];
    double prob_thresh, prob_ins, prob_del, prob_subst;
    double min_exp;
} PbModel;

static double pb_total(const PbModel* m, double e) { return pow(m->prob_ins, e) + pow(m->prob_del, e) + pow(m->prob_subst, e); }

/* PacBioQualityError::calc_min_exp */
static double pb_calc_min_exp(const PbModel* m) {
    double min_exp = 1, total = pb_total(m, min_exp), left, right;
    if (total < m->prob_thresh) {
        while (total < m->prob_thresh) { min_exp /= 2; total = pb_total(m, min_exp); }
        left = min_exp; right = min_exp * 2;
    } else {
        while (total > m->prob_thresh) { min_exp *= 2; total = pb_total(m, min_exp); }
        left = min_exp / 2; right = min_exp;
    }
    for (int i = 0; i < 15; i++) {
        double mid = (left + right) / 2;
        total = pb_total(m, mid);
        if (total == m->prob_thresh) { min_exp = mid; break; }
        else if (total > m->prob_thresh) { left = mid; min_exp = (mid + right) / 2; }
        else { right = mid; min_exp = (left + mid) / 2; }
    }
    return min_exp;
}
double orc_pb_min_exp(const double* sqrt_params, const double* norm_params, double prob_thresh, double prob_ins,
                      double prob_del, double prob_subst) {
    PbModel m = {{sqrt_params[0], sqrt_params[1]}, {norm_params[0], norm_params[1]}, prob_thresh, prob_ins, prob_del, prob_subst, 0};
    return pb_calc_min_exp(&m);
}

static double pb_sigmoid(double x) { return 1 / (1 + pow(2, (-2.5 / 3 * x + 6.5 / 3))); }

/* PacBioQualityError::trunc_norm; side 0 = left, 1 = right */
static double pb_trunc_norm(const PbModel* m, double lower_thresh, uint64_t seed, uint64_t j, int side, Ledger* lg) {
    double rnd;
    const double a_bar = (lower_thresh - m->norm_params[0]) / m->norm_params[1];
    if (lower_thresh < (m->norm_params[0] + 5 * m->norm_params[1])) {
        const double p = jlp_pnorm(a_bar);
        const uint64_t x = pb_draw(seed, j, 0, 0, (uint32_t)side);
        led(lg, x);
        /* runif_ab(eng, p, 1), src/pcg.h:103-105, in long double; R::qnorm5 takes a double */
        const long double u = (long double)p + runif_01(x) * ((long double)1 - (long double)p);
        const double q = jlp_qnorm((double)u);
        rnd = q * m->norm_params[1] + m->norm_params[0];
    } else {
        double u, x_bar, v;
        for (uint32_t it = 0;; it++) {
            const uint64_t xu = pb_draw(seed, j, 0, 16 + 2 * it, (uint32_t)side), xv = pb_draw(seed, j, 0, 17 + 2 * it, (uint32_t)side);
            led(lg, xu);
            u = (double)runif_01(xu);
            x_bar = sqrt(a_bar * a_bar - 2 * log(1 - u));
            led(lg, xv);
            v = (double)runif_01(xv);
            if (!(v > (x_bar / a_bar))) break;
        }
        rnd = m->norm_params[1] * x_bar + m->norm_params[0];
    }
    return rnd;
}

typedef struct {
    uint64_t seed;
    uint64_t job_lo, job_hi;
    double sqrt_params[2], norm_params[2];
    double prob_thresh, prob_ins, prob_del, prob_subst;
    uint64_t n_groups;
    const uint64_t* group_off;
    const char* const* group_seq;
    const uint64_t* group_len;
    const char* const* group_genome_name;
    const char* const* group_chrom_name;
    /* injected, indexed by j - job_lo */
    const uint64_t* read_len;
    const uint64_t* split_pos;
    const double* passes_left;
    const double* passes_right;
    /* append_pool can step past the template it copied when a deletion the walk drew could not be recorded (no spare
     * chromosome left: reads about as long as their chromosome); the reference then reads whatever an earlier read
     * left in its buffer.  0: the same here (sequential, for the replay against the reference); 1: such a position
     * reads 'N' (the defined behaviour the CUDA path is compared with). */
    int32_t beyond_template_is_n;
    /* duplicates (ReadWriterOneThread::create_reads, src/hts.h:254-280; PacBioOneGenome::re_read, src/hts_pacbio.cpp): read j
     * re-reads the chromosome, read length and read_start of the first read of its chain iff the draw made after read
     * j - 1 (sub 0, block 2, lo half) satisfies `dup < prob_dup` and j is not the first of its pool.  read_len of a
     * duplicate is injected like any other (the caller passes its leader's) */
    double prob_dup;
    uint64_t pool_reads;
} OrcPbJob;

static uint64_t pb_group_of(const OrcPbJob* J, uint64_t j) {
    uint64_t glo = 0, ghi = J->n_groups;
    while (ghi - glo > 1) { uint64_t mid = (glo + ghi) / 2; if (J->group_off[mid] <= j) glo = mid; else ghi = mid; }
    return glo;
}
static uint64_t pb_leader_of(const OrcPbJob* J, uint64_t j) {
    uint64_t k = j;
    if (!(J->prob_dup > 0) || J->pool_reads == 0) return k;
    while (k > J->job_lo && ((k - J->job_lo) % J->pool_reads) != 0) {
        const double dup = (double)runif_01(pb_draw(J->seed, k - 1, 0, 2, 0));
        if (!(dup < J->prob_dup)) break;
        k--;
    }
    return k;
}
static void pb_cum_probs(const PbModel* m, double passes_left, double passes_right, uint64_t seed, uint64_t j, Ledger* lg,
                         double* cum_left, double* cum_right) {
    const double left_thresh = (m->min_exp - (sqrt(passes_left + m->sqrt_params[0]) - m->sqrt_params[1])) / pb_sigmoid(passes_left);
    const double right_thresh = (m->min_exp - (sqrt(passes_right + m->sqrt_params[0]) - m->sqrt_params[1])) / pb_sigmoid(passes_right);
    const double incr_l = pb_trunc_norm(m, left_thresh, seed, j, 0, lg);
    const double incr_r = pb_trunc_norm(m, right_thresh, seed, j, 1, lg);
    double exp_l = incr_l * pb_sigmoid(passes_left) + sqrt(passes_left + m->sqrt_params[0]) - m->sqrt_params[1];
    double exp_r = incr_r * pb_sigmoid(passes_right) + sqrt(passes_right + m->sqrt_params[0]) - m->sqrt_params[1];
    if (exp_l < 0.6) exp_l = 0.6;
    if (exp_r < 0.6) exp_r = 0.6;
    cum_left[0] = pow(m->prob_ins, exp_l);
    cum_left[1] = pow(m->prob_del, exp_l) + cum_left[0];
    cum_left[2] = pow(m->prob_subst, exp_l) + cum_left[1];
    cum_right[0] = pow(m->prob_ins, exp_r);
    cum_right[1] = pow(m->prob_del, exp_r) + cum_right[0];
    cum_right[2] = pow(m->prob_subst, exp_r) + cum_right[1];
}
/* read_start of a chain's first read k: its own model, walk (counts only) and start draw, nothing emitted */
static uint64_t pb_leader_start(const OrcPbJob* J, const PbModel* m, uint64_t k, uint64_t chrom_len) {
    uint64_t read_length = J->read_len[k - J->job_lo];
    if (read_length >= chrom_len) read_length = chrom_len;
    const uint64_t split_pos = J->split_pos[k - J->job_lo];
    double cum_left[3], cum_right[3];
    Ledger off = {NULL, 0, 0, 0};
    pb_cum_probs(m, J->passes_left[k - J->job_lo], J->passes_right[k - J->job_lo], J->seed, k, &off, cum_left, cum_right);
    uint64_t current_length = 0, chrom_pos = 0, extra_space = chrom_len - read_length, n_ins = 0, n_del = 0;
    const double* cum = cum_left;
    while (current_length < read_length) {
        if (current_length == split_pos) cum = cum_right;
        const double u = (double)runif_01(pb_draw(J->seed, k, 1, (uint32_t)(chrom_pos >> 1), (uint32_t)(chrom_pos & 1)));
        if (u > cum[2]) current_length++;
        else if (u < cum[0]) {
            if (current_length < (read_length - 1)) { n_ins++; current_length++; extra_space++; if (current_length == split_pos) cum = cum_right; }
            current_length++;
        } else if (u < cum[1]) { if (extra_space > 0) { n_del++; extra_space--; } }
        else current_length++;
        chrom_pos++;
    }
    const uint64_t space = read_length + n_del - n_ins;
    if (!(space < chrom_len)) return 0;
    const double u = (double)runif_01(pb_draw(J->seed, k, 0, 1, 0));
    return (uint64_t)(u * (double)(chrom_len - space + 1));
}

/* Reads [lo, hi) of the job.  plan (optional): [4 * (hi - lo)] group, read_length, read_start, read_chrom_space. */
int orc_pacbio_generate(const OrcPbJob* J, uint64_t lo, uint64_t hi, char* out, uint64_t cap, uint64_t* len,
                        uint64_t* plan, uint64_t* ledger, uint64_t ledger_cap, uint64_t* ledger_n, uint64_t* ledger_cnt) {
    PbModel m = {{J->sqrt_params[0], J->sqrt_params[1]}, {J->norm_params[0], J->norm_params[1]},
                 J->prob_thresh, J->prob_ins, J->prob_del, J->prob_subst, 0};
    m.min_exp = pb_calc_min_exp(&m);
    Sink S = {out, 0, cap};
    Ledger lg = {ledger, 0, ledger_cap, ledger != NULL};
    char* read = NULL;
    uint64_t read_cap = 0;
    uint64_t *ins = NULL, *del = NULL, *sub = NULL;
    uint64_t ev_cap = 0;
    int rc = 0;
    for (uint64_t j = lo; j < hi; j++) {
        const uint64_t led0 = lg.n;
        /* the group: first (haplotype, chromosome) with reads left, one_read */
        const uint64_t leader = pb_leader_of(J, j);
        const int is_dup = leader != j;
        const uint64_t g = pb_group_of(J, leader);
        const char* chrom = J->group_seq[g];
        const uint64_t chrom_len = J->group_len[g];
        uint64_t read_length = J->read_len[j - J->job_lo];
        if (read_length >= chrom_len) read_length = chrom_len;
        const uint64_t split_pos = J->split_pos[j - J->job_lo];
        const double passes_left = J->passes_left[j - J->job_lo], passes_right = J->passes_right[j - J->job_lo];

        /* ---- update_probs */
        double cum_left[3], cum_right[3];
        pb_cum_probs(&m, passes_left, passes_right, J->seed, j, &lg, cum_left, cum_right);
        /* ---- fill_quals */
        char qual_left, qual_right;
        {
            uint64_t tl = (uint64_t)round(-10.0 * log10(cum_left[2])), tr = (uint64_t)round(-10.0 * log10(cum_right[2]));
            if (tl > 93) tl = 93;
            if (tr > 93) tr = 93;
            qual_left = (char)(tl + '!');
            qual_right = (char)(tr + '!');
        }
        /* ---- the walk (PacBioQualityError::sample) */
        if (2 * read_length + 16 > ev_cap) {
            ev_cap = 2 * read_length + 16;
            ins = (uint64_t*)realloc(ins, ev_cap * 8); del = (uint64_t*)realloc(del, ev_cap * 8); sub = (uint64_t*)realloc(sub, ev_cap * 8);
            if (!ins || !del || !sub) { rc = -2; break; }
        }
        uint64_t n_ins = 0, n_del = 0, n_sub = 0;
        {
            uint64_t current_length = 0, chrom_pos = 0, extra_space = chrom_len - read_length;
            const double* cum = cum_left;
            while (current_length < read_length) {
                if (current_length == split_pos) cum = cum_right;
                const uint64_t x = pb_draw(J->seed, j, 1, (uint32_t)(chrom_pos >> 1), (uint32_t)(chrom_pos & 1));
                led(&lg, x);
                const double u = (double)runif_01(x);     /* `double u` in the reference */
                if (u > cum[2]) {
                    current_length++;
                } else if (u < cum[0]) {
                    if (current_length < (read_length - 1)) {
                        if (n_ins < ev_cap) ins[n_ins] = chrom_pos;
                        n_ins++;
                        current_length++;
                        extra_space++;
                        if (current_length == split_pos) cum = cum_right;
                    }
                    current_length++;
                } else if (u < cum[1]) {
                    if (extra_space > 0) {
                        if (n_del < ev_cap) del[n_del] = chrom_pos;
                        n_del++;
                        extra_space--;
                    }
                } else {
                    if (n_sub < ev_cap) sub[n_sub] = chrom_pos;
                    n_sub++;
                    current_length++;
                }
                chrom_pos++;
                if (chrom_pos >= ev_cap + 4 * read_length + (1u << 20)) { rc = -3; break; }   /* cannot happen: guards the loop */
            }
            if (rc) break;
        }
        /* ---- read_chrom_space, read_start */
        uint64_t space = read_length + n_del - n_ins;
        uint64_t read_start = 0;
        if (is_dup) {
            /* re_read: the chain's read_start; deletions are given up from the back until the template fits, and a read
             * that still does not fit is not written */
            read_start = pb_leader_start(J, &m, leader, chrom_len);
            while (space + read_start > chrom_len) {
                if (n_del == 0) break;
                n_del--;
                space--;
            }
            if (space + read_start > chrom_len) {
                if (plan) { uint64_t* p = plan + 4 * (j - lo); p[0] = g; p[1] = read_length; p[2] = read_start; p[3] = ~0ull; }
                if (ledger_cnt) ledger_cnt[j - lo] = lg.n - led0;
                continue;
            }
        } else if (space < chrom_len) {
            const uint64_t x = pb_draw(J->seed, j, 0, 1, 0);
            led(&lg, x);
            const double u = (double)runif_01(x);
            read_start = (uint64_t)(u * (double)(chrom_len - space + 1));
        } else if (space > chrom_len) { rc = -4; break; }
        /* ---- append_pool */
        {
            const uint64_t x = pb_draw(J->seed, j, 0, 1, 1);
            led(&lg, x);
            const int reverse = runif_01(x) < 0.5;
            char num[24];
            putc_(&S, '@');
            put(&S, J->group_genome_name[g], strlen(J->group_genome_name[g]));
            putc_(&S, '-');
            put(&S, J->group_chrom_name[g], strlen(J->group_chrom_name[g]));
            putc_(&S, '-');
            int nd = snprintf(num, sizeof num, "%llu", (unsigned long long)read_start);
            put(&S, num, (uint64_t)nd);
            putc_(&S, '-');
            putc_(&S, reverse ? 'R' : 'F');
            putc_(&S, '\n');
            if (space + read_length + 16 > read_cap) {
                const uint64_t old = read_cap;
                read_cap = space + read_length + 16;
                read = (char*)realloc(read, read_cap);
                if (!read) { rc = -2; break; }
                memset(read + old, old ? 0 : 'N', read_cap - old);      /* std::string(1000, 'N'), then resize() appends '\0' */
            }
            memcpy(read, chrom + read_start, space);
            if (reverse) orc_rev_comp(read, space);
            uint64_t read_pos = 0, current_length = 0, ii = 0, di = 0, si = 0;
            while (current_length < read_length) {
                if (J->beyond_template_is_n && read_pos >= space) read[read_pos] = 'N';
                if (ii < n_ins && read_pos == ins[ii]) {
                    const uint64_t xe = pb_draw(J->seed, j, 2, (uint32_t)(read_pos >> 1), (uint32_t)(read_pos & 1));
                    led(&lg, xe);
                    const uint64_t rndi = (uint64_t)(runif_01(xe) * 4);
                    putc_(&S, read[read_pos]);
                    putc_(&S, BASES[rndi]);
                    ii++;
                    current_length += 2;
                } else if (di < n_del && read_pos == del[di]) {
                    di++;
                } else if (si < n_sub && read_pos == sub[si]) {
                    const uint64_t xe = pb_draw(J->seed, j, 2, (uint32_t)(read_pos >> 1), (uint32_t)(read_pos & 1));
                    led(&lg, xe);
                    const uint64_t rndi = (uint64_t)(runif_01(xe) * 3);
                    putc_(&S, MM[nt_map((unsigned char)read[read_pos])][rndi]);
                    si++;
                    current_length++;
                } else {
                    putc_(&S, read[read_pos]);
                    current_length++;
                }
                read_pos++;
            }
            putc_(&S, '\n'); putc_(&S, '+'); putc_(&S, '\n');
            for (uint64_t i = 0; i < split_pos; i++) putc_(&S, qual_left);
            for (uint64_t i = split_pos; i < read_length; i++) putc_(&S, qual_right);
            putc_(&S, '\n');
        }
        if (plan) { uint64_t* p = plan + 4 * (j - lo); p[0] = g; p[1] = read_length; p[2] = read_start; p[3] = space; }
        if (ledger_cnt) ledger_cnt[j - lo] = lg.n - led0;
    }
    free(read); free(ins); free(del); free(sub);
    *len = S.n;
    if (ledger_n) *ledger_n = lg.n;
    return rc;
}
