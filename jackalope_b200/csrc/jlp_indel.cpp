// create_haplotypes: the host event pass of insertions and deletions along the tree (DESIGN.md section 10).  No CUDA.
//
// Per chromosome the nodes are visited in preorder.  A node's sequence is an ordered list of segments (runs of
// reference columns, runs of inserted column ids); a branch is cut into steps, and the events of a step, drawn in
// increasing position order, are applied in one linear merge pass over the parent's list.  The work is proportional to
// the events, not to the sites: the per-site walk (substitutions, the states of the inserted columns) stays on the
// device.  Built without floating-point contraction (build.py): log / log1p feed integer decisions that the oracle
// restates.
#include <cmath>
#include <stdexcept>
#include <string>

#include "jlp_draws.h"
#include "jlp_host.h"

namespace jlp {

std::vector<uint64_t> indel_thresholds(double rate_ins, const double* w_ins, uint32_t n_ins, double rate_del,
                                       const double* w_del, uint32_t n_del) {
    const double R = rate_ins + rate_del;
    double W_ins = 0, W_del = 0;
    for (uint32_t u = 0; u < n_ins; u++) W_ins += w_ins[u];
    for (uint32_t u = 0; u < n_del; u++) W_del += w_del[u];
    std::vector<uint64_t> thr;
    double cum = 0;
    for (uint32_t j = 0; j + 1 < n_ins + n_del; j++) {
        cum += j < n_ins ? (rate_ins / R) * (w_ins[j] / W_ins) : (rate_del / R) * (w_del[j - n_ins] / W_del);
        thr.push_back(prob_threshold(cum));
    }
    return thr;
}

uint32_t indel_steps(double R, double t, double epsilon) {
    const double m = std::ceil(R * t / epsilon);
    if (!(m < 2147483648.0)) throw std::runtime_error("more than 2^31 indel steps on one branch (R * t / epsilon)");
    return m < 1 ? 1u : (uint32_t)m;
}

namespace {

struct Seg {
    uint32_t a, n;      // columns a .. a + n - 1
    uint32_t ins;       // 1: inserted column ids, 0: reference columns
};

void push(std::vector<Seg>& d, uint32_t ins, uint32_t a, uint32_t n) {
    if (!d.empty() && d.back().ins == ins && d.back().a + d.back().n == a) d.back().n += n;
    else d.push_back(Seg{a, n, ins});
}

// copies positions [a, b) of src (a never below the last call's b) into dst
struct Reader {
    const std::vector<Seg>& src;
    size_t si = 0;
    uint64_t base = 0;      // position of src[si]
    void copy(uint64_t a, uint64_t b, std::vector<Seg>& dst) {
        while (a < b) {
            while (base + src[si].n <= a) base += src[si++].n;
            const uint64_t take = std::min<uint64_t>(b, base + src[si].n) - a;
            push(dst, src[si].ins, src[si].a + (uint32_t)(a - base), (uint32_t)take);
            a += take;
        }
    }
};

struct Event { uint64_t pos; uint32_t len; uint32_t ins; };

// the records of one tip (see DESIGN.md section 10, "Records")
void tip_records(const std::vector<Seg>& segs, uint64_t len, IndelTip& T) {
    uint64_t pos = 0, expect = 0, pos_last = 0;
    int64_t last = -1;                          // the last live reference column
    std::vector<uint32_t> gap;                  // inserted columns since it
    uint64_t pool = 0;
    auto rec = [&](uint32_t kind, uint64_t old_pos, uint64_t new_pos, int64_t sm, const uint32_t* ids, size_t n) {
        IndelRec r{(uint32_t)old_pos, (uint32_t)new_pos, kind, 0, sm, pool};
        pool += indel_pool_len(r);
        T.recs.push_back(r);
        T.ids.insert(T.ids.end(), ids, ids + n);
        T.ids_off.push_back(T.ids.size());
    };
    auto close_gap = [&](uint64_t D) {
        const uint64_t I = gap.size();
        if (last < 0) {
            if (I == 0) {
                if (D) rec(kDelRec, 0, 0, -(int64_t)D, nullptr, 0);
            } else {                            // D >= 1: nothing is inserted before the first column of the root
                rec(kLeadRec, 0, 0, (int64_t)I - 1, gap.data(), I);
                if (D > 1) rec(kDelRec, 1, I, -(int64_t)(D - 1), nullptr, 0);
            }
        } else {
            if (I) rec(kAnchorRec, (uint64_t)last, pos_last, (int64_t)I, gap.data(), I);
            if (D) rec(kDelRec, (uint64_t)last + 1, pos_last + 1 + I, -(int64_t)D, nullptr, 0);
        }
        gap.clear();
    };
    T.ids_off.assign(1, 0);
    for (const Seg& s : segs) {
        if (s.ins) {
            for (uint32_t i = 0; i < s.n; i++) gap.push_back(s.a + i);
            pos += s.n;
        } else {
            close_gap(s.a - expect);
            last = (int64_t)s.a + s.n - 1;
            pos += s.n;
            pos_last = pos - 1;
            expect = (uint64_t)s.a + s.n;
        }
    }
    close_gap(len - expect);
    if (pos >> 32) throw std::runtime_error("a tip chromosome of 2^32 bases or more is not supported");
    T.size = pos;
}

}  // namespace

void indel_events(uint64_t seed, uint32_t chrom, uint64_t len, uint32_t n_nodes, const int32_t* parent,
                  const double* branch_len, const int32_t* tip_of, uint32_t n_tips, const IndelModel& m, IndelChrom& out) {
    const double R = m.rate_ins + m.rate_del;
    std::vector<uint32_t> left(n_nodes, 0);
    for (uint32_t v = 1; v < n_nodes; v++) left[parent[v]]++;
    std::vector<std::vector<Seg>> seq(n_nodes);
    if (len) seq[0].push_back(Seg{0, (uint32_t)len, 0});
    out.tip.assign(n_tips, IndelTip{});
    uint64_t next_id = 0;
    std::vector<Event> ev;
    for (uint32_t v = 1; v < n_nodes; v++) {
        const uint32_t u = (uint32_t)parent[v];
        std::vector<Seg> cur = --left[u] == 0 ? std::move(seq[u]) : seq[u];
        if (left[u] == 0) std::vector<Seg>().swap(seq[u]);
        uint64_t L = 0;
        for (const Seg& s : cur) L += s.n;
        const double t = branch_len[v];
        const uint32_t steps = indel_steps(R, t, m.epsilon);
        out.steps += steps;
        const double p = -std::expm1(-R * (t / steps));
        const double lp = std::log1p(-p);
        for (uint32_t s = 0; s < steps && L && p > 0; s++) {
            ev.clear();
            uint64_t pos = 0;
            for (uint32_t k = 0; pos < L; k++) {
                const U4 w = indel_event_block(seed, chrom, v, s, k);
                const double U = (double)((lo64(w) >> 11) + 1) * 0x1p-53;
                const double g = std::floor(std::log(U) / lp);
                if (!(g < (double)(L - pos))) break;
                const uint64_t i = pos + (uint64_t)g;
                const uint64_t x = hi64(w);
                uint32_t idx = 0;
                for (uint64_t th : m.kl_thr) idx += x >= th;
                ev.push_back(idx < m.n_ins ? Event{i, idx + 1, 1} : Event{i, idx - m.n_ins + 1, 0});
                pos = i + 1;
            }
            if (ev.empty()) continue;
            std::vector<Seg> nxt;
            nxt.reserve(cur.size() + 2 * ev.size());
            Reader rd{cur};
            uint64_t done = 0, dz = 0;          // positions below `done` are handled; below `dz` deleted
            for (const Event& e : ev) {
                const uint64_t lo = std::max(done, dz);
                if (lo < e.pos) rd.copy(lo, e.pos, nxt);
                if (!e.ins) {
                    dz = std::max(dz, std::min<uint64_t>(L, e.pos + e.len));
                    out.deletions++;
                } else {
                    if (e.pos >= dz) rd.copy(e.pos, e.pos + 1, nxt);
                    if (next_id + e.len > 0xffffffffull)
                        throw std::runtime_error("2^32 or more inserted columns on one chromosome are not supported");
                    push(nxt, 1, (uint32_t)next_id, e.len);
                    out.birth.insert(out.birth.end(), e.len, v);
                    next_id += e.len;
                    out.insertions++;
                    out.inserted_bases += e.len;
                }
                done = e.pos + 1;
            }
            const uint64_t lo = std::max(done, dz);
            if (lo < L) rd.copy(lo, L, nxt);
            cur.swap(nxt);
            L = 0;
            for (const Seg& x : cur) L += x.n;
            if (L >> 32) throw std::runtime_error("a chromosome of 2^32 bases or more along the tree is not supported");
        }
        if (tip_of[v] >= 0) tip_records(cur, len, out.tip[tip_of[v]]);
        if (left[v]) seq[v] = std::move(cur);
    }
}

}  // namespace jlp
