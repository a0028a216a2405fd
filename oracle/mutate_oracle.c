/*
 * TEST INFRASTRUCTURE ONLY -- CPU oracle for create_haplotypes (DESIGN.md section 10).
 *
 * A plain-C restatement of the per-site walk jlp_create_haplotypes performs on the GPU, with its own Philox
 * addressing and full 64-bit comparisons (the kernels decide on the high words and fetch the low words only on
 * ties).  Built on demand by oracle/harness_mutate.py; the product (jackalope_b200/) never loads it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static const char BASES[4] = {'T', 'C', 'A', 'G'};

/* Philox4x32-10 (Salmon et al., SC'11), standard constants. */
static void philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
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

/* X(chrom, site b, node v) of the haplotype mutator (layout: jackalope_b200/csrc/jlp_draws.h, planes 7 and 8):
 * high word = word b&3 of the block (b>>2, chrom, 7 | v<<8), low word = w0 of the block (b, chrom, 8 | v<<8) */
uint64_t orc_mut_draw(uint64_t seed, uint32_t chrom, uint64_t b, uint32_t node) {
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)}, w[4], v[4];
    uint32_t c1[4] = {(uint32_t)(b >> 2), (uint32_t)((b >> 2) >> 32), chrom, 7u | (node << 8)};
    uint32_t c2[4] = {(uint32_t)b, (uint32_t)(b >> 32), chrom, 8u | (node << 8)};
    philox4x32_10(c1, key, w);
    philox4x32_10(c2, key, v);
    return ((uint64_t)w[b & 3] << 32) | v[0];
}

/* a cumulative probability as a threshold on X: floor(c 2^64), 0 for c <= 0, 2^64 - 1 for c >= 1 */
static uint64_t mut_thr(double c) {
    if (!(c > 0)) return 0;
    if (c >= 1) return UINT64_MAX;
    return (uint64_t)ldexp(c, 64);
}

struct mut_recs { uint64_t n, cap; uint64_t* pos; char* nuc; };

/* The per-site walk of jlp_create_haplotypes: every T/C/A/G site draws its category (node 0's draw: invariant with
 * probability `invariant`, else one of n_cat equally likely categories), then, nodes in the given preorder, the
 * state of node v is #{j : X(c, b, v) >= t_j} over the cumulative thresholds of row `parent state` of
 * P[v][category] (clipped at 0, renormalised).  Records of tip i (node tip_node[i]) are the sites whose tip state
 * differs from the reference, written tip-major, then by chromosome, then by position: counts[i * n_chroms + c],
 * positions into pos[], new bases into nuc[].  Returns -2 (counts filled) when cap is too small. */
int orc_mutate(uint64_t seed, const char* bases, const uint64_t* chrom_off, uint64_t n_chroms, uint32_t n_nodes,
               const int32_t* parent, uint32_t n_cat, double invariant, const double* P, uint32_t n_tips,
               const uint32_t* tip_node, uint64_t* counts, uint64_t* pos, char* nuc, uint64_t cap) {
    uint64_t* thr = malloc(sizeof(uint64_t) * 12 * (size_t)n_nodes * n_cat);
    uint64_t* cat_thr = malloc(sizeof(uint64_t) * n_cat);
    uint8_t* st = malloc(n_nodes);
    int32_t* tip_of = malloc(sizeof(int32_t) * n_nodes);
    struct mut_recs* R = calloc(n_tips, sizeof(struct mut_recs));
    int rc = 0;
    if (!thr || !cat_thr || !st || !tip_of || !R) { rc = -1; goto done; }
    for (uint32_t v = 0; v < n_nodes; v++) tip_of[v] = -1;
    for (uint32_t t = 0; t < n_tips; t++) tip_of[tip_node[t]] = (int32_t)t;
    for (uint64_t r = 0; r < (uint64_t)n_nodes * n_cat * 4; r++) {
        const double* row = P + (r / 4) * 16 + (r % 4) * 4;
        double p[4], sum = 0, cum = 0;
        for (int j = 0; j < 4; j++) { p[j] = row[j] > 0 ? row[j] : 0.0; sum += p[j]; }
        for (int j = 0; j < 3; j++) { cum += p[j] / sum; thr[3 * r + j] = mut_thr(cum); }
    }
    cat_thr[0] = mut_thr(invariant);
    for (uint32_t j = 1; j < n_cat; j++) cat_thr[j] = mut_thr(invariant + j * (1 - invariant) / n_cat);
    for (uint64_t c = 0; c < n_chroms && rc == 0; c++) {
        const char* seq = bases + chrom_off[c];
        const uint64_t len = chrom_off[c + 1] - chrom_off[c];
        for (uint32_t t = 0; t < n_tips; t++) counts[t * n_chroms + c] = R[t].n;     /* start; made a count below */
        for (uint64_t b = 0; b < len && rc == 0; b++) {
            const char ch = seq[b];
            const int code = ch == 'T' ? 0 : ch == 'C' ? 1 : ch == 'A' ? 2 : ch == 'G' ? 3 : -1;
            if (code < 0) continue;
            const uint64_t xc = orc_mut_draw(seed, (uint32_t)c, b, 0);
            uint32_t idx = 0;
            for (uint32_t j = 0; j < n_cat; j++) idx += xc >= cat_thr[j];
            if (idx == 0) continue;                                  /* invariant site */
            const uint32_t cat = idx - 1;
            st[0] = (uint8_t)code;
            for (uint32_t v = 1; v < n_nodes; v++) {
                const uint64_t x = orc_mut_draw(seed, (uint32_t)c, b, v);
                const uint64_t* t3 = thr + 3 * (((uint64_t)v * n_cat + cat) * 4 + st[parent[v]]);
                st[v] = (uint8_t)((x >= t3[0]) + (x >= t3[1]) + (x >= t3[2]));
                const int32_t tip = tip_of[v];
                if (tip >= 0 && st[v] != code) {
                    struct mut_recs* m = &R[tip];
                    if (m->n == m->cap) {
                        m->cap = m->cap ? 2 * m->cap : 1024;
                        uint64_t* np_ = realloc(m->pos, m->cap * sizeof(uint64_t));
                        char* nn = np_ ? realloc(m->nuc, m->cap) : NULL;
                        if (np_) m->pos = np_;
                        if (nn) m->nuc = nn;
                        if (!np_ || !nn) { rc = -1; break; }
                    }
                    m->pos[m->n] = b;
                    m->nuc[m->n] = BASES[st[v]];
                    m->n++;
                }
            }
        }
        for (uint32_t t = 0; t < n_tips; t++) counts[t * n_chroms + c] = R[t].n - counts[t * n_chroms + c];
    }
    if (rc == 0) {
        uint64_t total = 0;
        for (uint32_t t = 0; t < n_tips; t++) total += R[t].n;
        if (total > cap) rc = -2;
    }
    if (rc == 0) {
        uint64_t k = 0;
        for (uint32_t t = 0; t < n_tips; t++) {      /* per tip the records are already in (chromosome, position) order */
            if (R[t].n) { memcpy(pos + k, R[t].pos, R[t].n * sizeof(uint64_t)); memcpy(nuc + k, R[t].nuc, R[t].n); }
            k += R[t].n;
        }
    }
done:
    if (R) for (uint32_t t = 0; t < n_tips; t++) { free(R[t].pos); free(R[t].nuc); }
    free(R); free(thr); free(cat_thr); free(st); free(tip_of);
    return rc;
}
