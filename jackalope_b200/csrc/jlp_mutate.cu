// create_haplotypes on the device: substitutions along a tree, or along gene trees, one per region of a chromosome
// (DESIGN.md section 10).
//
// Every T/C/A/G site of the reference walks down its region's tree in the schedule the host prepared (preorder, the child
// with fewer tips first, so at most log2(tips) + 2 internal nodes are live at once).  Per (site, node) it is one
// decision on a 64-bit draw X(chromosome, site, node) (jlp_draws.h, planes MUT / MSLOW) against the cumulative
// thresholds of row `parent state` of P(node, category); the decision is taken on the high 32 bits and the low word
// is fetched only when the high word equals a threshold's, so it always equals the full 64-bit comparison.
//
// With gene trees (k_mutate<., ., true>) a tile's chromosome, first site, region and schedule come from its MutTile.
// The threshold tables are built on the device (k_mut_tables) for a window of tiles at a time; both passes run window
// by window (one tree: one window).
//
// Two passes over the same draws, no atomics:
//   k_mutate<false>  records per (tip, tile) into cnt (a tile is owned by one warp, its lane 0 adds)
//   k_mut_scan       exclusive scan of every (tip, chromosome) run of cnt: each tile's first record in its region
//   k_mutate<true>   the records again, written at their final places in HapChromHost::packed layout
//                    (old_pos | new_pos | nuc_off | size_modifier (0) | pool), sorted by position
#include <cuda_runtime.h>
#include <stdint.h>

#include "jlp_draws.h"
#include "jlp_host.h"
#include "jlp_kernels.cuh"

namespace jlp {

namespace {

__device__ __forceinline__ uint32_t base_code(uint32_t c) {
    return c == 'T' ? 0u : c == 'C' ? 1u : c == 'A' ? 2u : c == 'G' ? 3u : 4u;
}

// #{j : X >= t[j]} for the three thresholds of a row, X = H:low; the low word only on a tie of the high words
__device__ __forceinline__ uint32_t decide(uint32_t H, const uint4& th, const uint4* __restrict__ lo_tab, uint32_t row,
                                           uint64_t seed, uint32_t chrom, uint64_t site, uint32_t node) {
    uint32_t b = (uint32_t)(H > th.x) + (uint32_t)(H > th.y) + (uint32_t)(H > th.z);
    if (H == th.x || H == th.y || H == th.z) {
        const uint4 tl = lo_tab[row];
        const uint32_t L = mut_low(seed, chrom, site, node);
        b = (uint32_t)(H > th.x || (H == th.x && L >= tl.x)) + (uint32_t)(H > th.y || (H == th.y && L >= tl.y)) +
            (uint32_t)(H > th.z || (H == th.z && L >= tl.z));
    }
    return b;
}

__device__ __forceinline__ uint8_t base_char(uint32_t states, uint32_t k) {
    return (uint8_t)(__byte_perm(0x47414354u, 0u, (states >> (2 * k)) & 3u) & 0xffu);
}

// At tip `tip`, the indel instantiation: the step's sites against the tip's indel records.  A site is dead (covered by a
// deletion, or column 0 under a leading insertion) or an anchor (its base is pool[0] of an insertion record): neither
// gives a substitution record.  A substitution record at site b goes to index (substitutions before b) + (indel records
// before b), new_pos = b + the shift after those records; an indel record of the step goes to index j + (substitutions
// before its old_pos), written by the lane that owns that site.
template <bool WRITE>
__device__ __forceinline__ void indel_tip(const MutParams& p, uint32_t tip, uint32_t c, uint32_t tile, uint64_t step0,
                                          uint64_t s0, const uint8_t* seq, uint32_t ev, uint32_t ref, uint32_t ns,
                                          uint32_t lane) {
    const size_t r = (size_t)tip * p.n_chroms + c;
    const uint64_t rs = p.ir_start[r], re = p.ir_start[r + 1];
    uint32_t* cur = p.icur + (size_t)tip * p.n_tiles + tile;
    uint32_t* cp = p.cnt + (size_t)tip * p.n_tiles + tile;
    const uint32_t j0 = *cur;
    uint32_t j1 = j0;
    while (j1 < re && p.irec[j1].old_pos < step0 + 128) j1++;
    int64_t sh = 0;                                      // new_pos - old_pos after the records passed
    uint64_t ix = 0, pb = 0, dend = 0;                   // records passed, their pool bytes, end of the dead run
    auto pass = [&](uint32_t j) {
        const IndelRec q = p.irec[j];
        sh = (int64_t)q.new_pos - (int64_t)q.old_pos + q.size_mod;
        ix = j - rs + 1;
        pb = q.pool_before + indel_pool_len(q);
        dend = q.kind == kDelRec ? q.old_pos - q.size_mod : q.kind == kLeadRec ? 1 : 0;
    };
    if (j0 > rs) pass(j0 - 1);
    uint32_t skip = 0, jj = j0;
    int64_t shk[4];
    uint64_t ixk[4], pbk[4];
#pragma unroll
    for (uint32_t k = 0; k < 4; k++) {
        const uint64_t b = s0 + k;
        while (jj < j1 && p.irec[jj].old_pos <= b) {
            if (p.irec[jj].old_pos == b && p.irec[jj].kind == kAnchorRec) skip |= 1u << k;
            pass(jj++);
        }
        if (b < dend) skip |= 1u << k;
        shk[k] = sh; ixk[k] = ix; pbk[k] = pb;
    }
    uint32_t dm = 0;
#pragma unroll
    for (uint32_t k = 0; k < 4; k++)
        if (((ev >> k) & 1u) && (((ns ^ ref) >> (2 * k)) & 3u) && !((skip >> k) & 1u)) dm |= 1u << k;
    if (!WRITE) {
        const uint32_t tot = __reduce_add_sync(~0u, (uint32_t)__popc(dm));
        if (lane == 0) { if (tot) *cp += tot; if (j1 != j0) *cur = j1; }
        return;
    }
    if (j1 == j0 && __ballot_sync(~0u, dm) == 0) return;
    const uint32_t mine = (uint32_t)__popc(dm);
    uint32_t incl = mine;
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(~0u, incl, d);
        if (lane >= d) incl += v;
    }
    uint32_t base = lane == 0 ? *cp : 0u;
    base = __shfl_sync(~0u, base, 0);
    const uint32_t tot = __shfl_sync(~0u, incl, 31);
    const uint32_t excl = base + incl - mine;            // substitution records before the lane's first site
    uint64_t* R = p.out + p.region[r];
    const uint64_t N = p.region_n[r];
    uint8_t* pool = reinterpret_cast<uint8_t*>(R + 4 * N);
    uint64_t before = excl;
#pragma unroll
    for (uint32_t k = 0; k < 4; k++) {
        if (!((dm >> k) & 1u)) continue;
        const uint64_t b = s0 + k, i = before + ixk[k], off = before + pbk[k];
        R[i] = b;
        R[N + i] = (uint64_t)((int64_t)b + shk[k]);
        R[2 * N + i] = off;                              // size_modifier, R[3N + i], stays 0
        pool[off] = base_char(ns, k);
        before++;
    }
    for (uint32_t j = j0; j < j1; j++) {
        const IndelRec q = p.irec[j];
        const uint32_t l = (uint32_t)((q.old_pos - step0) >> 2), kk = q.old_pos & 3u;
        const uint32_t sb = __shfl_sync(~0u, excl + (uint32_t)__popc(dm & ((1u << kk) - 1u)), l);
        if (lane == l) {
            const uint64_t i = sb + (j - rs), off = sb + q.pool_before;
            R[i] = q.old_pos;
            R[N + i] = q.new_pos;
            R[2 * N + i] = off;
            R[3 * N + i] = (uint64_t)q.size_mod;
            p.ir_nuc[j] = off;
            if (q.kind == kAnchorRec) pool[off] = ((ev >> kk) & 1u) ? base_char(ns, kk) : seq[q.old_pos];
        }
    }
    __syncwarp();
    if (lane == 0) { *cp = base + tot; *cur = j1; }
}

// GT = false: one tree for the genome (jlp_create_haplotypes and _indels); the tile's chromosome from tile0 and the
// schedule and tables from the parameters, as before gene trees.  GT = true: the tile's region, schedule and table rows from its
// MutTile.  The two are kept apart so that the one-tree passes keep their speed (DESIGN.md section 10, "Gene trees").
template <bool WRITE, bool INDEL, bool GT>
__global__ void __launch_bounds__(kMutWarps * 32)
k_mutate(const __grid_constant__ MutParams p) {
    __shared__ uint8_t st[kMutSlots][kMutWarps * 32];     // node states: 2 bits per site, one byte per (slot, thread)
    extern __shared__ uint4 tab_s[];
    const uint4* thi = p.thr_hi;
    if (p.tab_smem) {
        for (uint32_t i = threadIdx.x; i < p.tab_rows; i += blockDim.x) tab_s[i] = p.thr_hi[i];
        __syncthreads();
        thi = tab_s;
    }
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    const uint32_t tile = (GT ? p.tile_begin : 0u) + blockIdx.x * kMutWarps + (tid >> 5);
    if (tile >= (GT ? p.tile_end : p.n_tiles)) return;     // one tree: one window of every tile
    uint32_t c;
    const uint8_t* seq;
    uint64_t first, lo = 0, hi;                           // the tile's first site; the sites it decides, [lo, hi)
    uint32_t n_begin = 0, n_end = p.n_sched;              // its tree's schedule entries
    const uint4* tlo = p.thr_lo;
    if (GT) {
        const MutTile T = p.tiles[tile];
        c = T.chrom; first = T.first; lo = T.lo; hi = T.hi;
        seq = p.genome + p.chrom_off[c];
        n_begin = T.sched0; n_end = T.sched0 + T.n_sched;
        thi += T.tab0;                                    // tab0 is 0 when the table is staged (one tree)
        tlo += T.tab0;
    } else {
        uint32_t a = 0, b = p.n_chroms;                   // the last chromosome whose first tile is <= tile
        while (b - a > 1) {
            const uint32_t mid = (a + b) >> 1;
            if (p.tile0[mid] <= tile) a = mid; else b = mid;
        }
        c = a;
        const uint64_t off = p.chrom_off[c];
        seq = p.genome + off;
        hi = p.chrom_off[c + 1] - off;
        first = (uint64_t)(tile - p.tile0[c]) * kMutTile;
    }
    const uint64_t seed = p.seed;
    uint32_t* cnt = p.cnt + tile;

    for (uint32_t step = 0; step < kMutSteps; step++) {
        const uint64_t s0 = first + step * 128u + lane * 4u;
        if (first + step * 128u >= hi) break;
        uint32_t ref = 0, cand = 0, ev = 0, cats = 0;      // 2 bits per site; T/C/A/G sites; evolving sites; 8 bits per site
#pragma unroll
        for (uint32_t k = 0; k < 4; k++)
            if ((!GT || s0 + k >= lo) && s0 + k < hi) {
                const uint32_t code = base_code(seq[s0 + k]);
                if (code < 4) { ref |= code << (2 * k); cand |= 1u << k; }
            }
        if (cand) {
            const U4 w = mut_block(seed, c, s0 >> 2, 0);
#pragma unroll
            for (uint32_t k = 0; k < 4; k++) {
                if (!((cand >> k) & 1u)) continue;
                const uint32_t H = genome_word(w, k);
                uint32_t idx = 0;
                bool tie = false;
                for (uint32_t j = 0; j < p.n_cat; j++) {
                    const uint32_t th = (uint32_t)(__ldg(p.cat_thr + j) >> 32);
                    idx += (uint32_t)(H > th);
                    tie |= H == th;
                }
                if (tie) {
                    const uint64_t X = ((uint64_t)H << 32) | mut_low(seed, c, s0 + k, 0);
                    idx = 0;
                    for (uint32_t j = 0; j < p.n_cat; j++) idx += (uint32_t)(X >= __ldg(p.cat_thr + j));
                }
                if (idx) { ev |= 1u << k; cats |= (idx - 1) << (8 * k); }
            }
        }
        if (!INDEL && __ballot_sync(~0u, ev) == 0) continue;      // with indels the tips' records still need the step
        st[0][tid] = (uint8_t)ref;
        for (uint32_t n = n_begin; n < (GT ? n_end : p.n_sched); n++) {
            const MutNode nd = p.sched[n];
            const uint32_t ps = st[nd.pslot][tid];
            uint32_t ns = ps;
            if (ev) {
                const U4 w = mut_block(seed, c, s0 >> 2, nd.node);
#pragma unroll
                for (uint32_t k = 0; k < 4; k++) {
                    if (!((ev >> k) & 1u)) continue;
                    const uint32_t a = (ps >> (2 * k)) & 3u, row = nd.tab + 4u * ((cats >> (8 * k)) & 0xffu) + a;
                    const uint32_t b = decide(genome_word(w, k), thi[row], GT ? tlo : p.thr_lo, row, seed, c, s0 + k, nd.node);
                    ns = (ns & ~(3u << (2 * k))) | (b << (2 * k));
                }
            }
            if (nd.tip < 0) { st[nd.slot][tid] = (uint8_t)ns; continue; }
            if (INDEL) {
                indel_tip<WRITE>(p, (uint32_t)nd.tip, c, tile, first + step * 128u, s0, seq, ev, ref, ns, lane);
                continue;
            }
            uint32_t dm = 0;                                 // sites where the tip differs from the reference
#pragma unroll
            for (uint32_t k = 0; k < 4; k++)
                if (((ev >> k) & 1u) && (((ns ^ ref) >> (2 * k)) & 3u)) dm |= 1u << k;
            uint32_t* cp = cnt + (size_t)nd.tip * p.n_tiles;
            if (!WRITE) {
                const uint32_t tot = __reduce_add_sync(~0u, (uint32_t)__popc(dm));
                if (lane == 0 && tot) *cp += tot;
                continue;
            }
            if (__ballot_sync(~0u, dm) == 0) continue;
            const uint32_t mine = (uint32_t)__popc(dm);
            uint32_t incl = mine;
#pragma unroll
            for (uint32_t d = 1; d < 32; d <<= 1) {
                const uint32_t v = __shfl_up_sync(~0u, incl, d);
                if (lane >= d) incl += v;
            }
            uint32_t base = lane == 0 ? *cp : 0u;
            base = __shfl_sync(~0u, base, 0);
            const uint32_t tot = __shfl_sync(~0u, incl, 31);
            if (lane == 0) *cp = base + tot;
            if (!dm) continue;
            const size_t r = (size_t)nd.tip * p.n_chroms + c;
            uint64_t* R = p.out + p.region[r];
            const uint64_t N = p.region_n[r];
            uint8_t* pool = reinterpret_cast<uint8_t*>(R + 4 * N);
            uint64_t i = base + incl - mine;
#pragma unroll
            for (uint32_t k = 0; k < 4; k++) {
                if (!((dm >> k) & 1u)) continue;
                const uint64_t pos = s0 + k;
                R[i] = pos;
                R[N + i] = pos;
                R[2 * N + i] = i;                        // size_modifier, R[3N + i], stays 0
                pool[i] = base_char(ns, k);
                i++;
            }
        }
    }
}

// one CTA per (tip, chromosome): exclusive scan of the chromosome's tiles, 1024 at a time
__global__ void __launch_bounds__(1024) k_mut_scan(const __grid_constant__ MutParams p, uint64_t* region_n) {
    __shared__ uint32_t wsum[32];
    const uint32_t r = blockIdx.x, tip = r / p.n_chroms, c = r % p.n_chroms;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t* a = p.cnt + (size_t)tip * p.n_tiles + p.tile0[c];
    const uint32_t n = p.tile0[c + 1] - p.tile0[c];
    uint32_t carry = 0;
    for (uint32_t b0 = 0; b0 < n; b0 += 1024) {
        const uint32_t i = b0 + threadIdx.x;
        const uint32_t v = i < n ? a[i] : 0u;
        uint32_t x = v;
#pragma unroll
        for (uint32_t d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(~0u, x, d);
            if (lane >= d) x += y;
        }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t y = wsum[lane];
#pragma unroll
            for (uint32_t d = 1; d < 32; d <<= 1) {
                const uint32_t z = __shfl_up_sync(~0u, y, d);
                if (lane >= d) y += z;
            }
            wsum[lane] = y;
        }
        __syncthreads();
        if (i < n) a[i] = carry + (warp ? wsum[warp - 1] : 0u) + x - v;
        carry += wsum[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) region_n[r] = carry;
}

// one thread per inserted column: its category and birth state (plane ICOL), then the nodes of its birth node's subtree
// in schedule order (planes IMUT / IMSLOW), node states in shared memory as in k_mutate; at a tip the state goes to
// every entry of that tip (the column's byte in an insertion record's pool)
__global__ void __launch_bounds__(256) k_ins_walk(const __grid_constant__ InsParams p) {
    __shared__ uint8_t st[kMutSlots][256];
    const uint32_t tid = threadIdx.x, g = blockIdx.x * 256u + tid;
    if (g >= p.n_cols) return;
    const InsCol col = p.cols[g];
    if (col.e0 == col.e1) return;
    const U4 w = ins_col_block(p.seed, col.chrom, col.id);
    const uint64_t xc = lo64(w), xs = hi64(w);
    uint32_t idx = 0;
    for (uint32_t j = 0; j < p.n_cat; j++) idx += (uint32_t)(xc >= p.cat_thr[j]);
    uint32_t s = (uint32_t)(xs >= p.pi_thr[0]) + (uint32_t)(xs >= p.pi_thr[1]) + (uint32_t)(xs >= p.pi_thr[2]);
    uint64_t e = col.e0;
    auto put = [&](uint32_t sched, uint32_t state) {
        for (; e < col.e1 && p.ent[e].sched == sched; e++) {
            const InsEnt E = p.ent[e];
            uint64_t* R = p.out + p.region[E.region];
            uint8_t* pool = reinterpret_cast<uint8_t*>(R + 4 * p.region_n[E.region]);
            pool[p.ir_nuc[E.ir] + E.k] = base_char(state, 0);
        }
    };
    put(col.n0, s);
    if (col.n0 + 1 >= col.n1) return;
    st[p.sched[col.n0].slot][tid] = (uint8_t)s;
    for (uint32_t n = col.n0 + 1; n < col.n1 && e < col.e1; n++) {
        const MutNode nd = p.sched[n];
        uint32_t ns = st[nd.pslot][tid];
        if (idx) {
            const uint32_t row = nd.tab + 4u * (idx - 1) + ns;
            const uint32_t H = genome_word(imut_block(p.seed, col.chrom, col.id >> 2, nd.node), col.id & 3u);
            const uint4 th = p.thr_hi[row];
            if (H == th.x || H == th.y || H == th.z) {
                const uint4 tl = p.thr_lo[row];
                const uint32_t L = imut_low(p.seed, col.chrom, col.id, nd.node);
                ns = (uint32_t)(H > th.x || (H == th.x && L >= tl.x)) + (uint32_t)(H > th.y || (H == th.y && L >= tl.y)) +
                     (uint32_t)(H > th.z || (H == th.z && L >= tl.z));
            } else {
                ns = (uint32_t)(H > th.x) + (uint32_t)(H > th.y) + (uint32_t)(H > th.z);
            }
        }
        if (nd.tip < 0) st[nd.slot][tid] = (uint8_t)ns;
        else put(n, ns);
    }
}

// One thread per (tree, node, category) item: P = expm(Q t) and its four rows' thresholds, restating
// transition_matrix + row_thresholds (jlp_host.cpp) operation for operation: every product and sum rounded on its own
// (__dmul_rn / __dadd_rn, no contraction), IEEE division, in the host's order; fabs, max, ldexp and the truncating
// conversion are exact on both sides.  The one libm step is the host's s = ceil(log2(norm)).  Here s comes from frexp:
// norm = m 2^e, m in [0.5, 1), so s = e - 1 when m = 0.5 and e otherwise.  glibc's log2 is within an ulp of the exact
// value; the result's ulp is at most 2^-42 for norms below 2^1024, and log2(2^(e-1) (1 + d)) exceeds e - 1 by about
// 1.44 d, so the host's ceil can only differ when 0 < d <= 2^-40, i.e. 0.5 < m <= 0.5 + 2^-41.  Those items, and a
// norm that is not finite, are listed in `flag` and recomputed on the host by the caller.
__global__ void __launch_bounds__(128) k_mut_tables(const TabItem* __restrict__ items, uint32_t n, const TabQ Q,
                                                   uint4* __restrict__ thr_hi, uint4* __restrict__ thr_lo,
                                                   double* __restrict__ P_out, uint32_t* n_flag, uint32_t* flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const TabItem it = items[i];
    const double t = it.t;
    double P[16];
#pragma unroll
    for (int k = 0; k < 16; k++) P[k] = (k % 5 == 0) ? 1.0 : 0.0;
    if (t != 0) {
        double A[16], norm = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            double row = 0;
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (j != r) { A[4 * r + j] = __dmul_rn(Q.q[4 * r + j], t); row = __dadd_rn(row, A[4 * r + j]); }
            A[5 * r] = -row;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            double col = 0;
#pragma unroll
            for (int r = 0; r < 4; r++) col = __dadd_rn(col, fabs(A[4 * r + j]));
            norm = norm < col ? col : norm;                 // std::max(norm, col)
        }
        int s = 0;
        if (!isfinite(norm)) {
            s = 0;
            flag[atomicAdd(n_flag, 1u)] = i;
        } else if (norm > 1) {
            int e;
            const double m = frexp(norm, &e);
            s = min(1000, m == 0.5 ? e - 1 : e);
            if (m > 0.5 && m <= 0.5 + 0x1p-41) flag[atomicAdd(n_flag, 1u)] = i;
        }
        const double sc = ldexp(1.0, -s);
#pragma unroll
        for (int k = 0; k < 16; k++) A[k] = __dmul_rn(A[k], sc);
        double term[16];
#pragma unroll
        for (int k = 0; k < 16; k++) term[k] = P[k];
        for (int k = 1; k <= 30; k++) {
            const double dk = (double)k;
#pragma unroll
            for (int r = 0; r < 4; r++) {                    // row r of the next term needs row r of this one only
                double nx[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    double acc = 0;
#pragma unroll
                    for (int m = 0; m < 4; m++) acc = __dadd_rn(acc, __dmul_rn(term[4 * r + m], A[4 * m + j]));
                    nx[j] = __ddiv_rn(acc, dk);
                }
#pragma unroll
                for (int j = 0; j < 4; j++) { term[4 * r + j] = nx[j]; P[4 * r + j] = __dadd_rn(P[4 * r + j], nx[j]); }
            }
        }
        for (int q = 0; q < s; q++) {
            double nx[16];
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    double acc = 0;
#pragma unroll
                    for (int m = 0; m < 4; m++) acc = __dadd_rn(acc, __dmul_rn(P[4 * r + m], P[4 * m + j]));
                    nx[4 * r + j] = acc;
                }
#pragma unroll
            for (int k = 0; k < 16; k++) P[k] = nx[k];
        }
    }
    if (P_out) {
#pragma unroll
        for (int k = 0; k < 16; k++) P_out[16 * (size_t)i + k] = P[k];
    }
#pragma unroll
    for (int a = 0; a < 4; a++) {
        double p[4], sum = 0, cum = 0;
        uint64_t th[3];
#pragma unroll
        for (int j = 0; j < 4; j++) { p[j] = P[4 * a + j] > 0 ? P[4 * a + j] : 0.0; sum = __dadd_rn(sum, p[j]); }
#pragma unroll
        for (int j = 0; j < 3; j++) {
            cum = __dadd_rn(cum, __ddiv_rn(p[j], sum));
            th[j] = !(cum > 0) ? 0ull : cum >= 1 ? ~0ull : __double2ull_rz(ldexp(cum, 64));   // prob_threshold
        }
        thr_hi[it.row + a] = make_uint4((uint32_t)(th[0] >> 32), (uint32_t)(th[1] >> 32), (uint32_t)(th[2] >> 32), 0);
        thr_lo[it.row + a] = make_uint4((uint32_t)th[0], (uint32_t)th[1], (uint32_t)th[2], 0);
    }
}

}  // namespace

cudaError_t launch_mut_tables(const TabItem* items, uint32_t n, const TabQ& Q, uint4* hi, uint4* lo, double* P_out,
                              uint32_t* n_flag, uint32_t* flag, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    k_mut_tables<<<(n + 127) / 128, 128, 0, s>>>(items, n, Q, hi, lo, P_out, n_flag, flag);
    return cudaGetLastError();
}

size_t mut_smem_bytes(uint32_t tab_rows) { return (size_t)tab_rows * sizeof(uint4); }

template <bool WRITE, bool INDEL, bool GT>
cudaError_t launch_mutate_t(const MutParams& p, cudaStream_t s) {
    const size_t smem = p.tab_smem ? mut_smem_bytes(p.tab_rows) : 0;
    const unsigned grid = (p.tile_end - p.tile_begin + kMutWarps - 1) / kMutWarps;
    cudaError_t e = cudaFuncSetAttribute(k_mutate<WRITE, INDEL, GT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_mutate<WRITE, INDEL, GT><<<grid, kMutWarps * 32, smem, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_mutate(const MutParams& p, bool write, bool indels, bool gtrees, cudaStream_t s) {
    if (p.tile_end <= p.tile_begin) return cudaSuccess;
    if (gtrees) return write ? launch_mutate_t<true, false, true>(p, s) : launch_mutate_t<false, false, true>(p, s);
    if (indels) return write ? launch_mutate_t<true, true, false>(p, s) : launch_mutate_t<false, true, false>(p, s);
    return write ? launch_mutate_t<true, false, false>(p, s) : launch_mutate_t<false, false, false>(p, s);
}

cudaError_t launch_ins_walk(const InsParams& p, cudaStream_t s) {
    if (p.n_cols == 0) return cudaSuccess;
    k_ins_walk<<<(p.n_cols + 255) / 256, 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_mut_scan(const MutParams& p, uint64_t* region_n, cudaStream_t s) {
    const uint64_t n = (uint64_t)p.n_tips * p.n_chroms;
    if (n == 0) return cudaSuccess;
    k_mut_scan<<<(unsigned)n, 1024, 0, s>>>(p, region_n);
    return cudaGetLastError();
}

}  // namespace jlp
