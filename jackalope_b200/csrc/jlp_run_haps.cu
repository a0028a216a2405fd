// The create_haplotypes driver (jlp_create_haplotypes*, DESIGN.md section 10): substitutions, insertions and
// deletions along one tree, or substitutions along gene trees, on the first device of the context.
#include "jlp_ctx.h"

#include <cmath>
#include <cstring>

using namespace jlp;

namespace {

// The visiting order of one tree and the node-state slots (k_mutate): preorder with the child of fewer tips first, a
// parent's slot freed when its last child is visited (before that child takes one), so at most about log2(tips) + 2
// slots are live.  Childless nodes that are not tips are left out.  tab: the node's first row after the tree's.
std::vector<MutNode> mut_schedule(const GeneTree& T, uint32_t n_cat, uint32_t& max_slots) {
    const uint32_t n = (uint32_t)T.parent.size();
    std::vector<int32_t> tip_of(n, -1);
    for (uint32_t t = 0; t < T.tip_node.size(); t++) tip_of[T.tip_node[t]] = (int32_t)t;
    std::vector<std::vector<uint32_t>> kids(n);
    for (uint32_t i = 1; i < n; i++) kids[T.parent[i]].push_back(i);
    std::vector<uint64_t> tips(n, 0);
    for (uint32_t i = n; i-- > 0;) {
        if (kids[i].empty()) tips[i] = tip_of[i] >= 0 ? 1 : 0;
        if (i) tips[T.parent[i]] += tips[i];
    }
    for (auto& k : kids) std::stable_sort(k.begin(), k.end(), [&](uint32_t a, uint32_t b) { return tips[a] < tips[b]; });
    std::vector<uint32_t> left(n), slot(n, 0), free_slots;
    for (uint32_t i = 0; i < n; i++) left[i] = (uint32_t)kids[i].size();
    for (uint32_t s = kMutSlots; s-- > 1;) free_slots.push_back((uint32_t)s);
    max_slots = 1;
    std::vector<MutNode> out;
    std::vector<uint32_t> stack(kids[0].rbegin(), kids[0].rend());
    while (!stack.empty()) {
        const uint32_t v = stack.back();
        stack.pop_back();
        const uint32_t par = (uint32_t)T.parent[v];
        MutNode m;
        m.node = v;
        m.tab = v * n_cat * 4;
        m.tip = tip_of[v];
        m.pslot = (uint16_t)slot[par];
        m.slot = 0;
        if (--left[par] == 0) free_slots.push_back(slot[par]);
        if (!kids[v].empty()) {
            if (free_slots.empty()) throw ArgErr("tree too deep for the node-state slots");
            slot[v] = free_slots.back();
            free_slots.pop_back();
            m.slot = (uint16_t)slot[v];
            max_slots = std::max<uint32_t>(max_slots, kMutSlots - (uint32_t)free_slots.size());
            for (auto it = kids[v].rbegin(); it != kids[v].rend(); ++it) stack.push_back(*it);
        }
        if (!kids[v].empty() || m.tip >= 0) out.push_back(m);
    }
    return out;
}

struct EventSet {
    cudaEvent_t e[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    EventSet() { for (cudaEvent_t& x : e) CK(cudaEventCreate(&x)); }
    ~EventSet() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
};

constexpr uint64_t kTableBudget = 1ull << 30;       // default bytes of threshold tables per window

// Device buffers of the threshold tables: the items of a window, the flagged items, the tables.
struct TableBufs {
    DevBuf<TabItem> items;
    DevBuf<uint32_t> flag;
    std::vector<uint32_t> h_flag;
    std::vector<uint4> h_rows;
};

// The tables of `items` built on the device (k_mut_tables); the items it flags are recomputed here with the host's
// transition_matrix + row_thresholds and copied over theirs (and over P_out's, when given).  Returns their count.
uint64_t device_tables(cudaStream_t s, const double Q[16], const std::vector<TabItem>& items, TableBufs& B, uint4* hi,
                       uint4* lo, double* P_out) {
    if (items.empty()) return 0;
    if (items.size() >> 32) throw ArgErr("2^32 or more transition matrices in one window");
    TabQ q;
    std::memcpy(q.q, Q, sizeof q.q);
    B.items.upload(items, s);
    B.flag.ensure(items.size() + 1);
    CK(cudaMemsetAsync(B.flag.p, 0, 4, s));
    CK(launch_mut_tables(B.items.p, (uint32_t)items.size(), q, hi, lo, P_out, B.flag.p, B.flag.p + 1, s));
    uint32_t nf = 0;
    CK(cudaMemcpyAsync(&nf, B.flag.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (nf == 0) return 0;
    B.h_flag.resize(nf);
    CK(cudaMemcpyAsync(B.h_flag.data(), B.flag.p + 1, (size_t)nf * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    B.h_rows.resize((size_t)nf * 8);
    std::vector<double> Ps(P_out ? (size_t)nf * 16 : 0);
    for (uint32_t f = 0; f < nf; f++) {
        const TabItem& it = items[B.h_flag[f]];
        double P[16];
        transition_matrix(Q, it.t, P);
        if (P_out) std::memcpy(&Ps[16 * (size_t)f], P, sizeof P);
        for (uint32_t a = 0; a < 4; a++) {
            uint64_t t[3];
            row_thresholds(P + 4 * a, t);
            B.h_rows[8 * (size_t)f + a] = make_uint4((uint32_t)(t[0] >> 32), (uint32_t)(t[1] >> 32), (uint32_t)(t[2] >> 32), 0);
            B.h_rows[8 * (size_t)f + 4 + a] = make_uint4((uint32_t)t[0], (uint32_t)t[1], (uint32_t)t[2], 0);
        }
        CK(cudaMemcpyAsync(hi + it.row, &B.h_rows[8 * (size_t)f], 4 * sizeof(uint4), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(lo + it.row, &B.h_rows[8 * (size_t)f + 4], 4 * sizeof(uint4), cudaMemcpyHostToDevice, s));
        if (P_out)
            CK(cudaMemcpyAsync(P_out + 16 * (size_t)B.h_flag[f], &Ps[16 * (size_t)f], 16 * sizeof(double),
                               cudaMemcpyHostToDevice, s));
    }
    CK(cudaStreamSynchronize(s));
    return nf;
}

void check_model(const jlp_ctx* c, const jlp_mutation_params* p) {
    if (c->chrom_off.size() < 2) throw ArgErr("set the reference genome first");
    for (int i = 0; i < 16; i++)
        if (i % 5 && !(std::isfinite(p->Q[i]) && p->Q[i] >= 0)) throw ArgErr("the off-diagonal rates of Q must be finite and >= 0");
    if (!(p->invariant >= 0 && p->invariant < 1)) throw ArgErr("invariant must be >= 0 and < 1");
    if (p->n_rates < 1 || p->n_rates > 255 || !p->rates) throw ArgErr("n_rates must be 1..255 (rates not NULL)");
    for (uint32_t k = 0; k < p->n_rates; k++)
        if (!(std::isfinite(p->rates[k]) && p->rates[k] >= 0)) throw ArgErr("category rates must be finite and >= 0");
    if (p->n_tips < 1 || p->n_tips > kMutMaxTips)
        throw ArgErr("a tree of " + std::to_string(p->n_tips) + " tips: 1 to " + std::to_string(kMutMaxTips) + " tips are supported");
    if (!p->tip_names) throw ArgErr("tip_node / tip_names is NULL");
    for (uint32_t t = 0; t < p->n_tips; t++)
        if (!p->tip_names[t]) throw ArgErr("tip name is NULL");
}

// the tree of p as the one tree of the genome: one region per (non-empty) chromosome
GeneTrees one_tree(const jlp_ctx* c, const jlp_mutation_params* p) {
    const uint32_t n = p->n_nodes;
    if (n < 2 || n > kMutMaxNodes || !p->parent || !p->branch_len)
        throw ArgErr("the tree needs 2 to " + std::to_string(kMutMaxNodes) + " nodes (parent / branch_len not NULL)");
    if (p->parent[0] != -1) throw ArgErr("parent[0] must be -1 (the root comes first)");
    std::vector<char> has_kid(n, 0);
    for (uint32_t i = 1; i < n; i++) {
        if (p->parent[i] < 0 || (uint32_t)p->parent[i] >= i) throw ArgErr("the tree must be in preorder: 0 <= parent[i] < i");
        if (!(std::isfinite(p->branch_len[i]) && p->branch_len[i] >= 0)) throw ArgErr("branch lengths must be finite and >= 0");
        has_kid[p->parent[i]] = 1;
    }
    if (!p->tip_node) throw ArgErr("tip_node / tip_names is NULL");
    std::vector<char> is_tip(n, 0);
    for (uint32_t t = 0; t < p->n_tips; t++) {
        const uint32_t v = p->tip_node[t];
        if (v >= n || has_kid[v] || is_tip[v]) throw ArgErr("tip_node must list distinct childless nodes");
        is_tip[v] = 1;
    }
    GeneTrees g;
    g.trees.resize(1);
    g.trees[0].parent.assign(p->parent, p->parent + n);
    g.trees[0].branch_len.assign(p->branch_len, p->branch_len + n);
    g.trees[0].tip_node.assign(p->tip_node, p->tip_node + p->n_tips);
    const std::vector<uint64_t> len = chrom_lengths(c);
    g.regions.resize(len.size());
    for (uint64_t ci = 0; ci < len.size(); ci++)
        if (len[ci]) g.regions[ci].push_back(TreeRegion{0, (uint32_t)len[ci], 0});
    return g;
}

// A window: contiguous tiles [t0, t1) whose trees' tables (rows in all) fit the budget together.
struct Window { uint32_t t0, t1; uint64_t rows; std::vector<uint32_t> trees; };

// What the plan stages (on the host) hand to the device passes.
struct MutPlan {
    std::vector<MutNode> sched;           // the used trees' schedules, one after the other
    std::vector<uint64_t> sched0;         // [trees + 1] each tree's first entry in sched
    uint32_t max_slots = 0;
    std::vector<uint32_t> tile0;          // [chromosomes + 1] each chromosome's first tile
    std::vector<MutTile> tiles;
    std::vector<Window> win;
    uint64_t max_win_rows = 0, table_bytes = 0;
    // indels only: the event pass's chromosomes, the tips' records, each tile's first record, the inserted columns
    std::vector<IndelChrom> ich;
    std::vector<IndelRec> irec;
    std::vector<uint64_t> ir_start;
    std::vector<uint32_t> icur;
    std::vector<InsCol> cols;
    std::vector<InsEnt> ents;
    double event_ms = 0;
};

// the trees' schedules, one after the other (trees no region uses get none)
void plan_trees(const GeneTrees& G, uint32_t K, MutPlan& P) {
    const uint64_t n_trees = G.trees.size();
    std::vector<char> used(n_trees, 0);
    for (const auto& rs : G.regions)
        for (const TreeRegion& r : rs) used[r.tree] = 1;
    std::vector<std::vector<MutNode>> scheds(n_trees);
    std::vector<uint32_t> slots(n_trees, 0);
    parallel_for(n_trees, host_threads(n_trees / 64 + 1), [&](uint64_t i) {
        if (used[i]) scheds[i] = mut_schedule(G.trees[i], K, slots[i]);
    });
    P.sched0.assign(n_trees + 1, 0);
    for (uint64_t i = 0; i < n_trees; i++) P.sched0[i + 1] = P.sched0[i] + scheds[i].size();
    if (P.sched0[n_trees] >> 32) throw ArgErr("2^32 or more tree nodes in all");
    P.sched.resize(P.sched0[n_trees]);
    for (uint64_t i = 0; i < n_trees; i++) std::copy(scheds[i].begin(), scheds[i].end(), P.sched.begin() + P.sched0[i]);
    P.max_slots = n_trees ? *std::max_element(slots.begin(), slots.end()) : 0;
}

// tiles: per region from its start rounded down to a multiple of 4, kMutTile sites apart.  Returns each tile's tree.
std::vector<uint32_t> plan_tiles(const GeneTrees& G, uint64_t nc, MutPlan& P) {
    std::vector<uint32_t> tile_tree;
    P.tile0.assign(nc + 1, 0);
    for (uint64_t ci = 0; ci < nc; ci++) {
        P.tile0[ci] = (uint32_t)P.tiles.size();
        for (const TreeRegion& r : G.regions[ci])
            for (uint64_t f = r.start & ~3u; f < r.end; f += kMutTile) {
                P.tiles.push_back(MutTile{(uint32_t)ci, (uint32_t)f, r.start, r.end, (uint32_t)P.sched0[r.tree],
                                          (uint32_t)(P.sched0[r.tree + 1] - P.sched0[r.tree]), 0, 0});
                tile_tree.push_back(r.tree);
            }
        if (P.tiles.size() >> 32) throw ArgErr("genome too large");
    }
    P.tile0[nc] = (uint32_t)P.tiles.size();
    return tile_tree;
}

// windows: contiguous tile ranges whose trees' tables fit the budget (a window holds at least one tree); every tile's
// tab0 is its tree's first row in the window's tables
void plan_windows(const GeneTrees& G, uint32_t K, uint64_t table_budget, const std::vector<uint32_t>& tile_tree, MutPlan& P) {
    const uint64_t n_trees = G.trees.size();
    const uint32_t n_tiles = (uint32_t)P.tiles.size();
    std::vector<Window>& win = P.win;
    const uint64_t budget = table_budget ? table_budget : kTableBudget;
    const uint64_t max_rows = std::min<uint64_t>(budget / (2 * sizeof(uint4)), 1ull << 31);
    std::vector<uint64_t> stamp(n_trees, UINT64_MAX), base(n_trees, 0);
    for (uint32_t tl = 0; tl < n_tiles; tl++) {
        const uint32_t tr = tile_tree[tl];
        if (win.empty() || stamp[tr] != win.size() - 1) {
            const uint64_t rows = (uint64_t)G.trees[tr].parent.size() * K * 4;
            if (win.empty() || (win.back().rows && win.back().rows + rows > max_rows)) {
                if (!win.empty()) win.back().t1 = tl;
                win.push_back(Window{tl, tl, 0, {}});
            }
            stamp[tr] = win.size() - 1;
            base[tr] = win.back().rows;
            win.back().rows += rows;
            win.back().trees.push_back(tr);
        }
        P.tiles[tl].tab0 = (uint32_t)base[tr];
    }
    if (!win.empty()) win.back().t1 = n_tiles;
    for (const Window& w : win) {
        P.max_win_rows = std::max(P.max_win_rows, w.rows);
        P.table_bytes += w.rows * 2 * sizeof(uint4);
    }
}

// indels (one tree): the event pass, chromosomes on up to 16 host threads; then the tips' records in one array (region
// tip * nc + chromosome), each tile's first record, and the inserted columns with their places in the pools
void plan_indels(const jlp_ctx* c, const jlp_mutation_params* p, const IndelModel& im, MutPlan& P) {
    const uint32_t n = p->n_nodes, n_tips = p->n_tips;
    const uint64_t nc = c->chrom_off.size() - 1;
    const size_t n_items = (size_t)n_tips * nc;
    const uint32_t n_tiles = P.tile0[nc];
    std::vector<IndelChrom>& ich = P.ich;
    std::vector<IndelRec>& irec = P.irec;
    std::vector<uint64_t>& ir_start = P.ir_start;
    ich.resize(nc);
    std::vector<int32_t> tip_of(n, -1);
    for (uint32_t t = 0; t < n_tips; t++) tip_of[p->tip_node[t]] = (int32_t)t;
    const auto te = std::chrono::steady_clock::now();
    parallel_for(nc, host_threads(nc), [&](uint64_t ci) {
        indel_events(p->seed, (uint32_t)ci, c->chrom_off[ci + 1] - c->chrom_off[ci], n, p->parent, p->branch_len,
                     tip_of.data(), n_tips, im, ich[ci]);
    });
    ir_start.resize(n_items + 1);
    for (size_t r = 0; r < n_items; r++) {
        ir_start[r] = irec.size();
        const std::vector<IndelRec>& v = ich[r % nc].tip[r / nc].recs;
        irec.insert(irec.end(), v.begin(), v.end());
    }
    ir_start[n_items] = irec.size();
    if (irec.size() >> 32) throw ArgErr("2^32 or more insertion and deletion records are not supported");
    P.icur.resize((size_t)n_tips * n_tiles);
    for (size_t r = 0; r < n_items; r++) {
        const uint64_t ci = r % nc;
        uint64_t j = ir_start[r];
        for (uint32_t tl = P.tile0[ci]; tl < P.tile0[ci + 1]; tl++) {
            while (j < ir_start[r + 1] && irec[j].old_pos < P.tiles[tl].first) j++;
            P.icur[(r / nc) * n_tiles + tl] = (uint32_t)j;
        }
    }
    P.event_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - te).count();

    // the inserted columns: birth node -> its schedule index and the end of its subtree's interval; per column the
    // (tip, record, byte) it fills, tips in schedule order
    const std::vector<MutNode>& sched = P.sched;
    std::vector<InsCol>& cols = P.cols;
    std::vector<InsEnt>& ents = P.ents;
    std::vector<int64_t> spos(n, -1);
    std::vector<uint32_t> scount(n, 0);
    for (size_t i = 0; i < sched.size(); i++) spos[sched[i].node] = (int64_t)i;
    for (uint32_t i = n; i-- > 1;) {
        scount[i] += spos[i] >= 0;
        scount[p->parent[i]] += scount[i];
    }
    std::vector<uint64_t> col_base(nc + 1, 0);
    for (uint64_t ci = 0; ci < nc; ci++) col_base[ci + 1] = col_base[ci] + ich[ci].birth.size();
    if (col_base[nc] >> 32) throw ArgErr("2^32 or more inserted columns are not supported");
    cols.resize(col_base[nc]);
    std::vector<uint64_t> ecount(cols.size() + 1, 0);
    for (int pass = 0; pass < 2; pass++) {
        for (size_t si = 0; si < sched.size(); si++) {
            if (sched[si].tip < 0) continue;
            const uint32_t t = (uint32_t)sched[si].tip;
            for (uint64_t ci = 0; ci < nc; ci++) {
                const IndelTip& T = ich[ci].tip[t];
                const size_t r = (size_t)t * nc + ci;
                for (size_t j = 0; j < T.recs.size(); j++)
                    for (uint64_t q = T.ids_off[j]; q < T.ids_off[j + 1]; q++) {
                        const uint64_t g = col_base[ci] + T.ids[q];
                        if (pass == 0) { ecount[g + 1]++; continue; }
                        const uint32_t k = (uint32_t)(q - T.ids_off[j]) + (T.recs[j].kind == kAnchorRec);
                        ents[cols[g].e1++] = InsEnt{(uint32_t)si, k, r, ir_start[r] + j};
                    }
            }
        }
        if (pass == 0) {
            for (size_t g = 0; g < cols.size(); g++) ecount[g + 1] += ecount[g];
            ents.resize(ecount.back());
            for (uint64_t ci = 0; ci < nc; ci++)
                for (uint32_t id = 0; id < ich[ci].birth.size(); id++) {
                    const uint64_t g = col_base[ci] + id;
                    const uint32_t u = ich[ci].birth[id];
                    InsCol& col = cols[g];
                    col.chrom = (uint32_t)ci; col.id = id;
                    col.n0 = spos[u] >= 0 ? (uint32_t)spos[u] : 0;
                    col.n1 = spos[u] >= 0 ? (uint32_t)spos[u] + scount[u] : 0;
                    col.e0 = col.e1 = ecount[g];
                }
        }
    }
}

// What the device passes leave: their buffers (freed with it, once the stores are filled), the records' regions (count,
// pool bytes and first word per (tip, chromosome)) and the timings.
struct MutPasses {
    DevBuf<uint64_t> d_off, d_cat, d_region, d_region_n, d_out, d_ir_start, d_ir_nuc;
    DevBuf<uint32_t> d_tile0, d_cnt, d_icur;
    DevBuf<MutTile> d_tiles;
    DevBuf<IndelRec> d_irec;
    DevBuf<InsCol> d_cols;
    DevBuf<InsEnt> d_ents;
    DevBuf<MutNode> d_sched;
    DevBuf<uint4> d_hi, d_lo;
    TableBufs tb;
    std::vector<uint64_t> region_n, region, pool;
    uint64_t words = 0, records = 0;
    float count_ms = 0, scan_ms = 0, write_ms = 0;
    double table_ms = 0;
    bool all_smem = true;
};

// On the first device: pass 1 (k_mutate counts records per tip and tile) window by window, k_mut_scan, the regions'
// offsets, pass 2 (k_mutate writes the records at their final places) window by window, and with indels the inserted
// columns' walk.  gtrees: gene trees (k_mutate's variant for several trees).
void run_passes(jlp_ctx* c, const jlp_mutation_params* p, const GeneTrees& G, const MutPlan& P, const IndelModel* im,
                const double* ins_pi, bool gtrees, MutPasses& R) {
    const uint64_t nc = c->chrom_off.size() - 1;
    const uint32_t K = p->n_rates, n_tips = p->n_tips;
    const uint32_t n_tiles = P.tile0[nc];
    const std::vector<Window>& win = P.win;
    std::vector<uint64_t> cat_thr(K);
    cat_thr[0] = prob_threshold(p->invariant);
    for (uint32_t j = 1; j < K; j++) cat_thr[j] = prob_threshold(p->invariant + j * (1 - p->invariant) / K);

    Device& d = device0(c);
    finish_upload(c, d);
    cudaStream_t s = d.s_compute;
    R.d_off.upload(c->chrom_off, s);
    R.d_tile0.upload(P.tile0, s);
    R.d_tiles.upload(P.tiles, s);
    R.d_sched.upload(P.sched, s);
    R.d_cat.upload(cat_thr, s);
    R.d_hi.ensure(P.max_win_rows);
    R.d_lo.ensure(P.max_win_rows);
    if (P.max_win_rows) {                    // rows no node uses (the root's) are staged too: defined, never read
        CK(cudaMemsetAsync(R.d_hi.p, 0, P.max_win_rows * sizeof(uint4), s));
        CK(cudaMemsetAsync(R.d_lo.p, 0, P.max_win_rows * sizeof(uint4), s));
    }
    const size_t n_cnt = (size_t)n_tips * n_tiles;
    R.d_cnt.ensure(n_cnt);
    if (n_cnt) CK(cudaMemsetAsync(R.d_cnt.p, 0, n_cnt * 4, s));
    R.d_region_n.ensure((size_t)n_tips * nc);
    MutParams mp{};
    mp.seed = p->seed;
    mp.genome = d.genome.p + kPad;
    mp.chrom_off = R.d_off.p;
    mp.tile0 = R.d_tile0.p;
    mp.tiles = R.d_tiles.p;
    mp.n_chroms = (uint32_t)nc; mp.n_tiles = n_tiles; mp.n_tips = n_tips; mp.n_sched = (uint32_t)P.sched.size();
    mp.sched = R.d_sched.p;
    mp.n_cat = K;
    mp.cat_thr = R.d_cat.p;
    mp.thr_hi = R.d_hi.p; mp.thr_lo = R.d_lo.p;
    mp.cnt = R.d_cnt.p;
    if (im) {
        R.d_irec.upload(P.irec, s);
        R.d_ir_start.upload(P.ir_start, s);
        R.d_icur.upload(P.icur, s);
        R.d_ir_nuc.ensure(P.irec.size());
        mp.irec = R.d_irec.p; mp.ir_start = R.d_ir_start.p; mp.icur = R.d_icur.p; mp.ir_nuc = R.d_ir_nuc.p;
    }

    // a window's tables: one item per (tree, scheduled node, category)
    std::vector<TabItem> titems;
    auto build_tables = [&](const Window& w) {
        const auto tt = std::chrono::steady_clock::now();
        titems.clear();
        uint64_t base = 0;
        for (uint32_t tr : w.trees) {
            const double* bl = G.trees[tr].branch_len.data();
            for (uint64_t i = P.sched0[tr]; i < P.sched0[tr + 1]; i++)
                for (uint32_t k = 0; k < K; k++)
                    titems.push_back(TabItem{p->rates[k] * bl[P.sched[i].node], (uint32_t)(base + P.sched[i].tab + 4ull * k), 0});
            base += (uint64_t)G.trees[tr].parent.size() * K * 4;
        }
        device_tables(s, p->Q, titems, R.tb, R.d_hi.p, R.d_lo.p, nullptr);
        R.table_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tt).count();
    };
    auto set_window = [&](const Window& w) {
        mp.tile_begin = w.t0; mp.tile_end = w.t1;
        mp.tab_rows = (uint32_t)w.rows;
        mp.tab_smem = w.trees.size() == 1 && mut_smem_bytes((uint32_t)w.rows) <= (64u << 10);
        R.all_smem &= mp.tab_smem != 0;
    };
    EventSet ev;
    for (const Window& w : win) {
        build_tables(w);
        set_window(w);
        CK(cudaEventRecord(ev.e[0], s));
        CK(launch_mutate(mp, false, im != nullptr, gtrees, s));
        CK(cudaEventRecord(ev.e[1], s));
        CK(cudaEventSynchronize(ev.e[1]));
        R.count_ms += elapsed_ms(ev.e[0], ev.e[1]);
    }
    CK(cudaEventRecord(ev.e[1], s));
    CK(launch_mut_scan(mp, R.d_region_n.p, s));
    CK(cudaEventRecord(ev.e[2], s));
    std::vector<uint64_t>& region_n = R.region_n;
    std::vector<uint64_t>& region = R.region;
    region_n.resize((size_t)n_tips * nc);
    region.resize((size_t)n_tips * nc);
    CK(cudaMemcpyAsync(region_n.data(), R.d_region_n.p, region_n.size() * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    R.scan_ms = elapsed_ms(ev.e[1], ev.e[2]);
    // with indels region_n becomes substitution + indel records, pool the substitutions' bytes + the indel records'
    std::vector<uint64_t>& pool = R.pool;
    pool = region_n;
    if (im)
        for (size_t r = 0; r < region.size(); r++) {
            const uint64_t a = P.ir_start[r], b = P.ir_start[r + 1];
            region_n[r] += b - a;
            if (b > a) pool[r] += P.irec[b - 1].pool_before + indel_pool_len(P.irec[b - 1]);
        }
    for (size_t r = 0; r < region.size(); r++) {
        region[r] = R.words;
        R.words += 4 * region_n[r] + (pool[r] + 7) / 8;
        R.records += region_n[r];
    }
    R.d_region.upload(region, s);
    if (im) {
        R.d_region_n.upload(region_n, s);
        R.d_icur.upload(P.icur, s);
    }
    mp.region = R.d_region.p;
    mp.region_n = R.d_region_n.p;            // k_mut_scan left the totals there
    R.d_out.ensure(R.words);
    if (R.words) CK(cudaMemsetAsync(R.d_out.p, 0, R.words * 8, s));
    mp.out = R.d_out.p;
    if (R.records)
        for (const Window& w : win) {
            if (win.size() > 1) build_tables(w);
            set_window(w);
            CK(cudaEventRecord(ev.e[3], s));
            CK(launch_mutate(mp, true, im != nullptr, gtrees, s));
            CK(cudaEventRecord(ev.e[4], s));
            CK(cudaEventSynchronize(ev.e[4]));
            R.write_ms += elapsed_ms(ev.e[3], ev.e[4]);
        }
    const std::vector<InsCol>& cols = P.cols;
    if (im && !cols.empty()) {               // one tree: one window, whose tables are still in place
        R.d_cols.upload(cols, s);
        R.d_ents.upload(P.ents, s);
        InsParams ip{};
        ip.seed = p->seed;
        if (cols.size() >> 32) throw ArgErr("2^32 or more inserted columns are not supported");
        ip.n_cols = (uint32_t)cols.size();
        ip.n_cat = K;
        ip.cols = R.d_cols.p; ip.ent = R.d_ents.p; ip.sched = R.d_sched.p; ip.cat_thr = R.d_cat.p;
        row_thresholds(ins_pi, ip.pi_thr);
        ip.thr_hi = R.d_hi.p; ip.thr_lo = R.d_lo.p;
        ip.out = R.d_out.p; ip.region = R.d_region.p; ip.region_n = R.d_region_n.p; ip.ir_nuc = R.d_ir_nuc.p;
        CK(cudaEventRecord(ev.e[3], s));
        CK(launch_ins_walk(ip, s));
        CK(cudaEventRecord(ev.e[4], s));
        CK(cudaEventSynchronize(ev.e[4]));
        R.write_ms += elapsed_ms(ev.e[3], ev.e[4]);
    }
    CK(cudaStreamSynchronize(s));
}

// the tips' records as regions of the passes' output, for store_haps
HapRegions tip_regions(const jlp_ctx* c, const jlp_mutation_params* p, const IndelModel* im, const MutPlan& P,
                       const MutPasses& R) {
    const uint64_t nc = c->chrom_off.size() - 1;
    const size_t n_items = (size_t)p->n_tips * nc;
    HapRegions G;
    G.names.assign(p->tip_names, p->tip_names + p->n_tips);
    G.src.resize(n_items);
    G.size.resize(n_items);
    for (size_t r = 0; r < n_items; r++) {
        G.src[r] = R.d_out.p + R.region[r];
        G.size[r] = im ? P.ich[r % nc].tip[r / nc].size : c->chrom_off[r % nc + 1] - c->chrom_off[r % nc];
    }
    G.n = R.region_n;
    G.pool = R.pool;
    return G;
}

// The whole call: the trees and every chromosome's regions (one tree for the genome: one region per chromosome);
// im == nullptr: substitutions only, otherwise the indel model (ins_pi: the inserted columns' birth distribution) and
// its stats (one tree only).  table_budget: bytes of threshold tables per window (0: the default).
void create_haps(jlp_ctx* c, const jlp_mutation_params* p, const GeneTrees& G, uint64_t table_budget, const IndelModel* im,
                 const double* ins_pi, jlp_mutation_stats* stats, jlp_indel_stats* istats, jlp_gtree_stats* gstats) {
    const auto t0 = std::chrono::steady_clock::now();
    MutPlan P;
    plan_trees(G, p->n_rates, P);
    const std::vector<uint32_t> tile_tree = plan_tiles(G, c->chrom_off.size() - 1, P);
    plan_windows(G, p->n_rates, table_budget, tile_tree, P);
    if (im) plan_indels(c, p, *im, P);
    MutPasses R;
    run_passes(c, p, G, P, im, ins_pi, gstats != nullptr, R);
    const auto t_gen = std::chrono::steady_clock::now();
    store_haps(c, tip_regions(c, p, im, P, R), host_threads((uint64_t)p->n_tips * (c->chrom_off.size() - 1)));

    if (stats) {
        const auto t1 = std::chrono::steady_clock::now();
        stats->count_ms = R.count_ms;
        stats->scan_ms = R.scan_ms;
        stats->write_ms = R.write_ms;
        stats->store_ms = std::chrono::duration<double, std::milli>(t1 - t_gen).count();
        stats->total_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
        stats->records = R.records;
        stats->d2h_bytes = R.words * 8;
        stats->table_bytes = P.table_bytes;
        stats->table_in_smem = (int)(R.all_smem && !P.win.empty());
        stats->max_slots = P.max_slots;
    }
    if (istats) {
        *istats = jlp_indel_stats{};
        for (const IndelChrom& x : P.ich) {
            istats->insertions += x.insertions;
            istats->deletions += x.deletions;
            istats->inserted_bases += x.inserted_bases;
            istats->steps += x.steps;
        }
        istats->indel_records = P.irec.size();
        istats->event_ms = P.event_ms;
    }
    if (gstats) {
        gstats->n_trees = G.trees.size();
        gstats->n_regions = 0;
        for (const auto& rs : G.regions) gstats->n_regions += rs.size();
        gstats->windows = P.win.size();
        gstats->table_ms = R.table_ms;
    }
}

// substitutions along the tree of p (jlp_create_haplotypes, and jlp_create_haplotypes_indels with indel rates of 0)
void create_subst(jlp_ctx* c, const jlp_mutation_params* p, jlp_mutation_stats* stats) {
    check_model(c, p);
    create_haps(c, p, one_tree(c, p), 0, nullptr, nullptr, stats, nullptr, nullptr);
}

}  // namespace

extern "C" {

int jlp_create_haplotypes(jlp_ctx* c, const jlp_mutation_params* p, jlp_mutation_stats* stats) {
    if (!c || !p) return JLP_ERR_ARG;
    return guarded(c, [&]() { create_subst(c, p, stats); });
}

int jlp_create_haplotypes_indels(jlp_ctx* c, const jlp_mutation_params* p, const jlp_indel_params* ip,
                                 jlp_mutation_stats* stats, jlp_indel_stats* istats) {
    if (!c || !p || !ip) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        auto rate_ok = [](double x) { return std::isfinite(x) && x >= 0; };
        if (!rate_ok(ip->rate_ins) || !rate_ok(ip->rate_del)) throw ArgErr("indel rates must be finite and >= 0");
        const double R = ip->rate_ins + ip->rate_del;
        if (R == 0) {
            create_subst(c, p, stats);
            if (istats) *istats = jlp_indel_stats{};
            return;
        }
        if (!(std::isfinite(ip->epsilon) && ip->epsilon > 0))
            throw ArgErr("epsilon must be > 0 when an indel rate is > 0");
        auto weights_ok = [&](double rate, uint32_t nw, const double* w) {
            if (rate == 0) return;
            if (nw < 1 || !w) throw ArgErr("an indel kind with a rate > 0 needs length weights (n >= 1, not NULL)");
            double sum = 0;
            for (uint32_t u = 0; u < nw; u++) {
                if (!rate_ok(w[u])) throw ArgErr("indel length weights must be finite and >= 0");
                sum += w[u];
            }
            if (!(sum > 0)) throw ArgErr("indel length weights need one weight > 0");
        };
        weights_ok(ip->rate_ins, ip->n_ins, ip->w_ins);
        weights_ok(ip->rate_del, ip->n_del, ip->w_del);
        double pis = 0;
        for (double x : ip->pi) {
            if (!rate_ok(x)) throw ArgErr("pi must be finite and >= 0");
            pis += x;
        }
        if (!(pis > 0)) throw ArgErr("pi needs one value > 0");
        // a kind of rate 0 has no lengths
        const uint32_t n_ins = ip->rate_ins > 0 ? ip->n_ins : 0, n_del = ip->rate_del > 0 ? ip->n_del : 0;
        IndelModel im;
        im.rate_ins = ip->rate_ins; im.rate_del = ip->rate_del; im.epsilon = ip->epsilon;
        im.n_ins = n_ins;
        im.kl_thr = indel_thresholds(ip->rate_ins, ip->w_ins, n_ins, ip->rate_del, ip->w_del, n_del);
        check_model(c, p);
        create_haps(c, p, one_tree(c, p), 0, &im, ip->pi, stats, istats, nullptr);
    });
}

int jlp_create_haplotypes_gtrees(jlp_ctx* c, const jlp_mutation_params* p, const jlp_gtree_params* g,
                                 jlp_mutation_stats* stats, jlp_gtree_stats* gstats) {
    if (!c || !p || !g) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        check_model(c, p);
        if (p->n_nodes || p->parent || p->branch_len || p->tip_node)
            throw ArgErr("with gene trees the trees come from the ms text: n_nodes, parent, branch_len and tip_node must be 0 / NULL");
        if (!g->text && g->text_len) throw ArgErr("the ms text is NULL");
        const std::vector<uint64_t> len = chrom_lengths(c);
        const auto t0 = std::chrono::steady_clock::now();
        GeneTrees G;
        parse_ms(g->text, g->text_len, len, p->tip_names, p->n_tips, kMutMaxNodes,
                 std::max(1u, std::thread::hardware_concurrency()), G);
        const double parse_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        jlp_gtree_stats gs{};
        create_haps(c, p, G, g->table_budget, nullptr, nullptr, stats, nullptr, &gs);
        gs.parse_ms = parse_ms;
        if (stats) stats->total_ms += parse_ms;
        if (gstats) *gstats = gs;
    });
}

int jlp_ms_regions(const char* text, uint64_t text_len, const uint64_t* chrom_len, uint64_t n_chroms,
                   const char* const* tip_names, uint32_t n_tips, uint64_t* reg, uint64_t cap, uint64_t* n_regions,
                   uint64_t* n_trees, char* err, uint64_t err_cap) {
    try {
        if ((!text && text_len) || (!chrom_len && n_chroms) || (!tip_names && n_tips)) throw ArgErr("NULL argument");
        GeneTrees G;
        parse_ms(text, text_len, std::vector<uint64_t>(chrom_len, chrom_len + n_chroms), tip_names, n_tips, kMutMaxNodes,
                 std::max(1u, std::thread::hardware_concurrency()), G);
        uint64_t k = 0;
        for (uint64_t ci = 0; ci < n_chroms; ci++)
            for (const TreeRegion& r : G.regions[ci]) {
                if (reg && k < cap) { reg[4 * k] = ci; reg[4 * k + 1] = r.start; reg[4 * k + 2] = r.end; reg[4 * k + 3] = r.tree; }
                k++;
            }
        if (n_regions) *n_regions = k;
        if (n_trees) *n_trees = G.trees.size();
        return JLP_OK;
    } catch (const std::exception& e) {
        if (err && err_cap) { std::strncpy(err, e.what(), err_cap - 1); err[err_cap - 1] = 0; }
        return JLP_ERR_ARG;
    }
}

int jlp_transition_tables(jlp_ctx* c, const double Q[16], const double* t, uint64_t n, double* P, uint64_t* thr,
                          uint64_t* n_host) {
    if (!c || !Q || (n && (!t || !P || !thr))) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (n >> 28) throw ArgErr("n must be below 2^28");
        std::vector<TabItem> items(n);
        for (uint64_t i = 0; i < n; i++) items[i] = TabItem{t[i], (uint32_t)(4 * i), 0};
        Device& d = device0(c);
        cudaStream_t s = d.s_compute;
        DevBuf<uint4> hi, lo;
        DevBuf<double> dP;
        TableBufs tb;
        hi.ensure(4 * n); lo.ensure(4 * n); dP.ensure(16 * n);
        const uint64_t nh = device_tables(s, Q, items, tb, hi.p, lo.p, dP.p);
        std::vector<uint4> h(4 * n), l(4 * n);
        if (n) {
            CK(cudaMemcpyAsync(h.data(), hi.p, 4 * n * sizeof(uint4), cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(l.data(), lo.p, 4 * n * sizeof(uint4), cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(P, dP.p, 16 * n * sizeof(double), cudaMemcpyDeviceToHost, s));
        }
        CK(cudaStreamSynchronize(s));
        for (uint64_t r = 0; r < 4 * n; r++) {
            thr[3 * r] = (uint64_t)h[r].x << 32 | l[r].x;
            thr[3 * r + 1] = (uint64_t)h[r].y << 32 | l[r].y;
            thr[3 * r + 2] = (uint64_t)h[r].z << 32 | l[r].z;
        }
        if (n_host) *n_host = nh;
    });
}

}  // extern "C"
