/*
 * TEST INFRASTRUCTURE ONLY -- CPU oracle for create_haplotypes along gene trees (DESIGN.md section 10, "Gene trees").
 *
 * Every site walks the tree of its region with the draws, thresholds and full 64-bit comparisons of orc_mutate.
 * Built on demand by oracle/harness_gtrees.py; the product (jackalope_b200/) never loads it.  It includes
 * oracle/mutate_oracle.c, so the Philox addressing and the thresholds are that oracle's own.
 */
#include "mutate_oracle.c"

/* The per-site walk along gene trees: the sites [reg_start[r], reg_end[r]) of chromosome c (regions reg_off[c] ..
 * reg_off[c + 1] - 1, in position order) walk tree reg_tree[r] exactly as orc_mutate walks its one tree, the draws
 * X(c, b, v) addressed by the absolute site b and the node's index v in that tree.  Tree i has the nodes
 * node_off[i] .. node_off[i + 1] - 1 of `parent` (indices within the tree), its tip t at node tip_node[i * n_tips + t],
 * and P[((node_off[i] + v) * n_cat + k) * 16 ..] for node v, category k.  Output as orc_mutate. */
int orc_mutate_gtrees(uint64_t seed, const char* bases, const uint64_t* chrom_off, uint64_t n_chroms,
                      const uint64_t* reg_off, const uint64_t* reg_start, const uint64_t* reg_end,
                      const uint32_t* reg_tree, uint32_t n_trees, const uint64_t* node_off, const int32_t* parent,
                      const uint32_t* tip_node, uint32_t n_cat, double invariant, const double* P, uint32_t n_tips,
                      uint64_t* counts, uint64_t* pos, char* nuc, uint64_t cap) {
    const uint64_t nn_all = node_off[n_trees];
    uint64_t* thr = malloc(sizeof(uint64_t) * 12 * (size_t)(nn_all ? nn_all : 1) * n_cat);
    uint64_t* cat_thr = malloc(sizeof(uint64_t) * n_cat);
    int32_t* tip_of = malloc(sizeof(int32_t) * (size_t)(nn_all ? nn_all : 1));
    struct mut_recs* R = calloc(n_tips, sizeof(struct mut_recs));
    uint32_t max_nodes = 1;
    for (uint32_t i = 0; i < n_trees; i++)
        if (node_off[i + 1] - node_off[i] > max_nodes) max_nodes = (uint32_t)(node_off[i + 1] - node_off[i]);
    uint8_t* st = malloc(max_nodes);
    int rc = 0;
    if (!thr || !cat_thr || !st || !tip_of || !R) { rc = -1; goto done; }
    for (uint64_t v = 0; v < nn_all; v++) tip_of[v] = -1;
    for (uint32_t i = 0; i < n_trees; i++)
        for (uint32_t t = 0; t < n_tips; t++) tip_of[node_off[i] + tip_node[(size_t)i * n_tips + t]] = (int32_t)t;
    for (uint64_t r = 0; r < nn_all * n_cat * 4; r++) {
        const double* row = P + (r / 4) * 16 + (r % 4) * 4;
        double p[4], sum = 0, cum = 0;
        for (int j = 0; j < 4; j++) { p[j] = row[j] > 0 ? row[j] : 0.0; sum += p[j]; }
        for (int j = 0; j < 3; j++) { cum += p[j] / sum; thr[3 * r + j] = mut_thr(cum); }
    }
    cat_thr[0] = mut_thr(invariant);
    for (uint32_t j = 1; j < n_cat; j++) cat_thr[j] = mut_thr(invariant + j * (1 - invariant) / n_cat);
    for (uint64_t c = 0; c < n_chroms && rc == 0; c++) {
        const char* seq = bases + chrom_off[c];
        for (uint32_t t = 0; t < n_tips; t++) counts[t * n_chroms + c] = R[t].n;
        for (uint64_t g = reg_off[c]; g < reg_off[c + 1] && rc == 0; g++) {
            const uint64_t n0 = node_off[reg_tree[g]];
            const uint32_t nn = (uint32_t)(node_off[reg_tree[g] + 1] - n0);
            const int32_t* par = parent + n0;
            for (uint64_t b = reg_start[g]; b < reg_end[g] && rc == 0; b++) {
                const char ch = seq[b];
                const int code = ch == 'T' ? 0 : ch == 'C' ? 1 : ch == 'A' ? 2 : ch == 'G' ? 3 : -1;
                if (code < 0) continue;
                const uint64_t xc = orc_mut_draw(seed, (uint32_t)c, b, 0);
                uint32_t idx = 0;
                for (uint32_t j = 0; j < n_cat; j++) idx += xc >= cat_thr[j];
                if (idx == 0) continue;
                const uint32_t cat = idx - 1;
                st[0] = (uint8_t)code;
                for (uint32_t v = 1; v < nn; v++) {
                    const uint64_t x = orc_mut_draw(seed, (uint32_t)c, b, v);
                    const uint64_t* t3 = thr + 3 * (((n0 + v) * n_cat + cat) * 4 + st[par[v]]);
                    st[v] = (uint8_t)((x >= t3[0]) + (x >= t3[1]) + (x >= t3[2]));
                    const int32_t tip = tip_of[n0 + v];
                    if (tip >= 0 && st[v] != code) {
                        struct mut_recs* m = &R[tip];
                        if (m->n == m->cap) {
                            m->cap = m->cap ? 2 * m->cap : 1024;
                            uint64_t* np_ = realloc(m->pos, m->cap * sizeof(uint64_t));
                            char* nw = np_ ? realloc(m->nuc, m->cap) : NULL;
                            if (np_) m->pos = np_;
                            if (nw) m->nuc = nw;
                            if (!np_ || !nw) { rc = -1; break; }
                        }
                        m->pos[m->n] = b;
                        m->nuc[m->n] = BASES[st[v]];
                        m->n++;
                    }
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
        for (uint32_t t = 0; t < n_tips; t++) {
            if (R[t].n) { memcpy(pos + k, R[t].pos, R[t].n * sizeof(uint64_t)); memcpy(nuc + k, R[t].nuc, R[t].n); }
            k += R[t].n;
        }
    }
done:
    if (R) for (uint32_t t = 0; t < n_tips; t++) { free(R[t].pos); free(R[t].nuc); }
    free(R); free(thr); free(cat_thr); free(st); free(tip_of);
    return rc;
}
