/*
 * TEST INFRASTRUCTURE ONLY -- CPU oracle for create_haplotypes with insertions and deletions (DESIGN.md section 10).
 *
 * Built on demand by oracle/harness_indels.py; the product (jackalope_b200/) never loads it.  It includes
 * mutate_oracle.c so that reference columns are drawn and decided by the very code of orc_mutate (orc_mut_draw,
 * mut_thr, the Philox block) rather than a copy of it.
 */
#include "mutate_oracle.c"

/* ---- insertions and deletions along the tree (DESIGN.md section 10) ----------------------------------------------
 * orc_indels: every node's column list is materialised explicitly (a column is a reference site b >= 0 or inserted
 * column -(id + 1)), each branch is cut into max(1, ceil(R t / epsilon)) steps and the events of a step, drawn with
 * the library's addressing (planes 9 to 12, jackalope_b200/csrc/jlp_draws.h) or taken from a given list, are applied
 * position by position.  States: a reference column evolves exactly as in orc_mutate; an inserted column draws its
 * category and its state at the end of its birth branch (from pi) from plane 10 and evolves below from planes 11/12.
 * The tips' sequences and canonical records are built here on their own.  Built with -ffp-contract=off, like the
 * library's host code. */

static void orc_block(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t out[4]) {
    uint32_t ctr[4] = {c0, c1, c2, c3}, key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    philox4x32_10(ctr, key, out);
}

/* the clipped, renormalised cumulative thresholds of a 4-row (row_thresholds) */
static void orc_row_thr(const double* row, uint64_t t[3]) {
    double p[4], sum = 0, cum = 0;
    for (int j = 0; j < 4; j++) { p[j] = row[j] > 0 ? row[j] : 0.0; sum += p[j]; }
    for (int j = 0; j < 3; j++) { cum += p[j] / sum; t[j] = mut_thr(cum); }
}

typedef struct {
    uint64_t* seq_off;      /* [n_tips * n_chroms + 1], tip-major: the tip sequences in seq */
    char* seq;
    uint64_t* rec_off;      /* [n_tips * n_chroms + 1]: records */
    uint64_t *old_pos, *new_pos, *nuc_off;
    int64_t* size_mod;
    uint64_t* pool_off;     /* [n_tips * n_chroms + 1]: pools */
    char* pool;
    uint64_t n_steps;       /* rows (chrom, node, step, L, events) */
    uint64_t* steps;
    uint64_t n_events;      /* rows (chrom, node, step, pos, insertion (1) / deletion (0), length) */
    uint64_t* events;
} orc_indel_result;

typedef struct { void* p; uint64_t n, cap; size_t sz; } vec;
static int vpush(vec* v, const void* x) {
    if (v->n == v->cap) {
        uint64_t nc = v->cap ? 2 * v->cap : 256;
        void* q = realloc(v->p, nc * v->sz);
        if (!q) return -1;
        v->p = q; v->cap = nc;
    }
    memcpy((char*)v->p + v->n * v->sz, x, v->sz);
    v->n++;
    return 0;
}

void orc_indel_free(orc_indel_result* r) {
    if (!r) return;
    free(r->seq_off); free(r->seq); free(r->rec_off); free(r->old_pos); free(r->new_pos); free(r->nuc_off);
    free(r->size_mod); free(r->pool_off); free(r->pool); free(r->steps); free(r->events); free(r);
}

typedef struct { int64_t col; uint8_t st; } ocol;       /* st: 0..3, or 255 for a non-T/C/A/G reference byte */

/* given: NULL, or n_given rows (chrom, node, step, pos, insertion 1 / deletion 0, length) in that order */
orc_indel_result* orc_indels(uint64_t seed, const char* bases, const uint64_t* chrom_off, uint64_t n_chroms,
                             uint32_t n_nodes, const int32_t* parent, const double* branch_len, uint32_t n_cat,
                             double invariant, const double* P, const double* pi, double rate_ins, const double* w_ins,
                             uint32_t n_ins, double rate_del, const double* w_del, uint32_t n_del, double epsilon,
                             uint32_t n_tips, const uint32_t* tip_node, const int64_t* given, uint64_t n_given) {
    orc_indel_result* res = calloc(1, sizeof(orc_indel_result));
    const uint64_t n_items = (uint64_t)n_tips * n_chroms;
    const double R = rate_ins + rate_del;
    if (rate_ins == 0) n_ins = 0;
    if (rate_del == 0) n_del = 0;
    uint64_t* thr = malloc(sizeof(uint64_t) * 12 * (size_t)n_nodes * n_cat);
    uint64_t* cat_thr = malloc(sizeof(uint64_t) * n_cat);
    uint64_t* kl = malloc(sizeof(uint64_t) * (n_ins + n_del + 1));
    uint64_t pi_thr[3];
    int32_t* tip_of = malloc(sizeof(int32_t) * n_nodes);
    ocol** node_cols = calloc(n_nodes, sizeof(ocol*));
    uint64_t* node_len = calloc(n_nodes, sizeof(uint64_t));
    vec steps = {0, 0, 0, 40}, evs = {0, 0, 0, 48};
    /* per (tip, chrom) results are produced chromosome by chromosome; kept per item, then laid out tip-major */
    vec* iseq = calloc(n_items, sizeof(vec));
    vec* irec = calloc(n_items, sizeof(vec));        /* rows (old, new, nuc_off, sm) */
    vec* ipool = calloc(n_items, sizeof(vec));
    if (!res || !thr || !cat_thr || !kl || !tip_of || !node_cols || !node_len || !iseq || !irec || !ipool)
        goto fail;
    for (uint64_t i = 0; i < n_items; i++) {
        iseq[i].sz = 1; irec[i].sz = 32; ipool[i].sz = 1;
    }
    for (uint64_t r = 0; r < (uint64_t)n_nodes * n_cat * 4; r++) orc_row_thr(P + (r / 4) * 16 + (r % 4) * 4, thr + 3 * r);
    cat_thr[0] = mut_thr(invariant);
    for (uint32_t j = 1; j < n_cat; j++) cat_thr[j] = mut_thr(invariant + j * (1 - invariant) / n_cat);
    orc_row_thr(pi, pi_thr);
    {
        double W_ins = 0, W_del = 0, cum = 0;
        for (uint32_t u = 0; u < n_ins; u++) W_ins += w_ins[u];
        for (uint32_t u = 0; u < n_del; u++) W_del += w_del[u];
        for (uint32_t j = 0; j + 1 < n_ins + n_del; j++) {
            cum += j < n_ins ? (rate_ins / R) * (w_ins[j] / W_ins) : (rate_del / R) * (w_del[j - n_ins] / W_del);
            kl[j] = mut_thr(cum);
        }
    }
    for (uint32_t v = 0; v < n_nodes; v++) tip_of[v] = -1;
    for (uint32_t t = 0; t < n_tips; t++) tip_of[tip_node[t]] = (int32_t)t;

    for (uint64_t c = 0; c < n_chroms; c++) {
        const char* ref = bases + chrom_off[c];
        const uint64_t len = chrom_off[c + 1] - chrom_off[c];
        uint64_t next_id = 0;
        node_cols[0] = malloc(sizeof(ocol) * (len ? len : 1));
        node_len[0] = len;
        for (uint64_t b = 0; b < len; b++) {
            const char ch = ref[b];
            node_cols[0][b].col = (int64_t)b;
            node_cols[0][b].st = ch == 'T' ? 0 : ch == 'C' ? 1 : ch == 'A' ? 2 : ch == 'G' ? 3 : 255;
        }
        for (uint32_t v = 1; v < n_nodes; v++) {
            const uint32_t u = (uint32_t)parent[v];
            uint64_t L = node_len[u];
            ocol* cur = malloc(sizeof(ocol) * (L ? L : 1));
            memcpy(cur, node_cols[u], sizeof(ocol) * L);
            const uint64_t first_new = next_id;
            const double t = branch_len[v];
            double mm = ceil(R * t / epsilon);
            const uint32_t m = mm < 1 ? 1u : (uint32_t)mm;
            const double p = -expm1(-R * (t / m));
            const double lp = log1p(-p);
            for (uint32_t s = 0; s < m; s++) {
                /* the step's events: (pos, ins, len) */
                uint64_t ne = 0, cap = 16;
                uint64_t* e = malloc(cap * 3 * 8);
                if (given) {
                    for (uint64_t g = 0; g < n_given; g++) {
                        const int64_t* row = given + 6 * g;
                        if ((uint64_t)row[0] != c || row[1] != v || row[2] != s || (uint64_t)row[3] >= L) continue;
                        if (ne == cap) { cap *= 2; e = realloc(e, cap * 3 * 8); }
                        e[3 * ne] = (uint64_t)row[3]; e[3 * ne + 1] = (uint64_t)row[4]; e[3 * ne + 2] = (uint64_t)row[5];
                        ne++;
                    }
                } else if (L && p > 0) {
                    uint64_t pos = 0;
                    for (uint32_t k = 0; pos < L; k++) {
                        uint32_t w[4];
                        orc_block(k, s, (uint32_t)c, 9u | (v << 8), seed, w);
                        const uint64_t x = ((uint64_t)w[1] << 32) | w[0], y = ((uint64_t)w[3] << 32) | w[2];
                        const double U = (double)((x >> 11) + 1) * 0x1p-53;
                        const double g = floor(log(U) / lp);
                        if (!(g < (double)(L - pos))) break;
                        const uint64_t i = pos + (uint64_t)g;
                        uint32_t idx = 0;
                        for (uint32_t j = 0; j + 1 < n_ins + n_del; j++) idx += y >= kl[j];
                        if (ne == cap) { cap *= 2; e = realloc(e, cap * 3 * 8); }
                        e[3 * ne] = i;
                        e[3 * ne + 1] = idx < n_ins;
                        e[3 * ne + 2] = idx < n_ins ? idx + 1 : idx - n_ins + 1;
                        ne++;
                        pos = i + 1;
                    }
                }
                uint64_t srow[5] = {c, v, s, L, ne};
                vpush(&steps, srow);
                for (uint64_t q = 0; q < ne; q++) {
                    uint64_t erow[6] = {c, v, s, e[3 * q], e[3 * q + 1], e[3 * q + 2]};
                    vpush(&evs, erow);
                }
                if (ne) {
                    uint8_t* del = calloc(L ? L : 1, 1);
                    uint64_t add = 0;
                    for (uint64_t q = 0; q < ne; q++) {
                        if (e[3 * q + 1]) { add += e[3 * q + 2]; continue; }
                        for (uint64_t i = e[3 * q]; i < e[3 * q] + e[3 * q + 2] && i < L; i++) del[i] = 1;
                    }
                    ocol* nx = malloc(sizeof(ocol) * (L + add + 1));
                    uint64_t nl = 0, q = 0;
                    for (uint64_t i = 0; i < L; i++) {
                        if (!del[i]) nx[nl++] = cur[i];
                        if (q < ne && e[3 * q] == i) {
                            if (e[3 * q + 1])
                                for (uint64_t k = 0; k < e[3 * q + 2]; k++) { nx[nl].col = -(int64_t)(next_id++) - 1; nx[nl].st = 0; nl++; }
                            q++;
                        }
                    }
                    free(del); free(cur);
                    cur = nx; L = nl;
                }
                free(e);
            }
            /* states at v */
            for (uint64_t i = 0; i < L; i++) {
                ocol* x = &cur[i];
                if (x->col < 0) {
                    const uint64_t id = (uint64_t)(-x->col - 1);
                    uint32_t w[4];
                    orc_block((uint32_t)id, 0, (uint32_t)c, 10u, seed, w);
                    const uint64_t xc = ((uint64_t)w[1] << 32) | w[0], xs = ((uint64_t)w[3] << 32) | w[2];
                    if (id >= first_new) { x->st = (uint8_t)((xs >= pi_thr[0]) + (xs >= pi_thr[1]) + (xs >= pi_thr[2])); continue; }
                    uint32_t idx = 0;
                    for (uint32_t j = 0; j < n_cat; j++) idx += xc >= cat_thr[j];
                    if (!idx) continue;
                    uint32_t h[4], lo[4];
                    orc_block((uint32_t)(id >> 2), (uint32_t)((id >> 2) >> 32), (uint32_t)c, 11u | (v << 8), seed, h);
                    orc_block((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)c, 12u | (v << 8), seed, lo);
                    const uint64_t X = ((uint64_t)h[id & 3] << 32) | lo[0];
                    const uint64_t* t3 = thr + 3 * (((uint64_t)v * n_cat + idx - 1) * 4 + x->st);
                    x->st = (uint8_t)((X >= t3[0]) + (X >= t3[1]) + (X >= t3[2]));
                } else if (x->st != 255) {
                    const uint64_t b = (uint64_t)x->col;
                    uint32_t idx = 0;
                    const uint64_t xc = orc_mut_draw(seed, (uint32_t)c, b, 0);
                    for (uint32_t j = 0; j < n_cat; j++) idx += xc >= cat_thr[j];
                    if (!idx) continue;
                    const uint64_t X = orc_mut_draw(seed, (uint32_t)c, b, v);
                    const uint64_t* t3 = thr + 3 * (((uint64_t)v * n_cat + idx - 1) * 4 + x->st);
                    x->st = (uint8_t)((X >= t3[0]) + (X >= t3[1]) + (X >= t3[2]));
                }
            }
            node_cols[v] = cur;
            node_len[v] = L;
            if (tip_of[v] < 0) continue;
            /* the tip: its sequence and its canonical records */
            const uint64_t item = (uint64_t)tip_of[v] * n_chroms + c;
            vec* S = &iseq[item];
            vec* RR = &irec[item];
            vec* PP = &ipool[item];
            for (uint64_t i = 0; i < L; i++) {
                const char ch = cur[i].st == 255 ? ref[cur[i].col] : BASES[cur[i].st];
                vpush(S, &ch);
            }
            const char* tipseq = (const char*)S->p;
            int64_t last = -1;              /* tip index of the last live reference column */
            uint64_t expect = 0;            /* the next reference column */
            for (uint64_t i = 0; i <= L; i++) {
                if (i < L && cur[i].col < 0) continue;
                /* close the gap before column i (i == L: the end) */
                const uint64_t r_next = i < L ? (uint64_t)cur[i].col : len;
                const uint64_t D = r_next - expect;
                const uint64_t gs = last < 0 ? 0 : (uint64_t)last + 1, I = i - gs;
                if (last < 0) {
                    if (I == 0) {
                        if (D) { int64_t row[4] = {0, 0, (int64_t)PP->n, -(int64_t)D}; vpush(RR, row); }
                    } else {
                        int64_t row[4] = {0, 0, (int64_t)PP->n, (int64_t)I - 1};
                        vpush(RR, row);
                        for (uint64_t k = 0; k < I; k++) vpush(PP, &tipseq[k]);
                        if (D > 1) { int64_t d[4] = {1, (int64_t)I, (int64_t)PP->n, -(int64_t)(D - 1)}; vpush(RR, d); }
                    }
                } else {
                    const uint64_t r = (uint64_t)cur[last].col;
                    if (I) {
                        int64_t row[4] = {(int64_t)r, last, (int64_t)PP->n, (int64_t)I};
                        vpush(RR, row);
                        for (uint64_t k = 0; k <= I; k++) vpush(PP, &tipseq[last + k]);
                    } else if (tipseq[last] != ref[r]) {
                        int64_t row[4] = {(int64_t)r, last, (int64_t)PP->n, 0};
                        vpush(RR, row);
                        vpush(PP, &tipseq[last]);
                    }
                    if (D) { int64_t d[4] = {(int64_t)r + 1, last + 1 + (int64_t)I, (int64_t)PP->n, -(int64_t)D}; vpush(RR, d); }
                }
                if (i < L) { last = (int64_t)i; expect = r_next + 1; }
            }
        }
        for (uint32_t v = 0; v < n_nodes; v++) { free(node_cols[v]); node_cols[v] = NULL; }
    }
    /* tip-major layout */
    res->seq_off = calloc(n_items + 1, 8); res->rec_off = calloc(n_items + 1, 8); res->pool_off = calloc(n_items + 1, 8);
    for (uint64_t i = 0; i < n_items; i++) {
        res->seq_off[i + 1] = res->seq_off[i] + iseq[i].n;
        res->rec_off[i + 1] = res->rec_off[i] + irec[i].n;
        res->pool_off[i + 1] = res->pool_off[i] + ipool[i].n;
    }
    res->seq = malloc(res->seq_off[n_items] + 1);
    res->pool = malloc(res->pool_off[n_items] + 1);
    const uint64_t NR = res->rec_off[n_items];
    res->old_pos = malloc(8 * NR + 8); res->new_pos = malloc(8 * NR + 8); res->nuc_off = malloc(8 * NR + 8);
    res->size_mod = malloc(8 * NR + 8);
    for (uint64_t i = 0; i < n_items; i++) {
        if (iseq[i].n) memcpy(res->seq + res->seq_off[i], iseq[i].p, iseq[i].n);
        if (ipool[i].n) memcpy(res->pool + res->pool_off[i], ipool[i].p, ipool[i].n);
        const int64_t* rows = (const int64_t*)irec[i].p;
        for (uint64_t k = 0; k < irec[i].n; k++) {
            const uint64_t o = res->rec_off[i] + k;
            res->old_pos[o] = (uint64_t)rows[4 * k]; res->new_pos[o] = (uint64_t)rows[4 * k + 1];
            res->nuc_off[o] = (uint64_t)rows[4 * k + 2]; res->size_mod[o] = rows[4 * k + 3];
        }
        free(iseq[i].p); free(irec[i].p); free(ipool[i].p);
    }
    res->n_steps = steps.n; res->steps = steps.p;
    res->n_events = evs.n; res->events = evs.p;
    free(iseq); free(irec); free(ipool);
    free(thr); free(cat_thr); free(kl); free(tip_of); free(node_cols); free(node_len);
    return res;
fail:
    orc_indel_free(res);
    return NULL;
}
