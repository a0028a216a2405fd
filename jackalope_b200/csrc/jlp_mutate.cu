// create_haplotypes on the device: substitutions along a tree (DESIGN.md section 10).
//
// Every T/C/A/G site of the reference walks down the tree in the schedule the host prepared (preorder, the child
// with fewer tips first, so at most log2(tips) + 2 internal nodes are live at once).  Per (site, node) it is one
// decision on a 64-bit draw X(chromosome, site, node) (jlp_draws.h, planes MUT / MSLOW) against the cumulative
// thresholds of row `parent state` of P(node, category); the decision is taken on the high 32 bits and the low word
// is fetched only when the high word equals a threshold's, so it always equals the full 64-bit comparison.
//
// Two passes over the same draws, no atomics:
//   k_mutate<false>  records per (tip, tile) into cnt (a tile is owned by one warp, its lane 0 adds)
//   k_mut_scan       exclusive scan of every (tip, chromosome) run of cnt: each tile's first record in its region
//   k_mutate<true>   the records again, written at their final places in HapChromHost::packed layout
//                    (old_pos | new_pos | nuc_off | size_modifier (0) | pool), sorted by position
#include <cuda_runtime.h>
#include <stdint.h>

#include "jlp_draws.h"
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

template <bool WRITE>
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
    const uint32_t tile = blockIdx.x * kMutWarps + (tid >> 5);
    if (tile >= p.n_tiles) return;
    uint32_t lo = 0, hi = p.n_chroms;                     // the last chromosome whose first tile is <= tile
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (p.tile0[mid] <= tile) lo = mid; else hi = mid;
    }
    const uint32_t c = lo;
    const uint64_t off = p.chrom_off[c], len = p.chrom_off[c + 1] - off;
    const uint8_t* seq = p.genome + off;
    const uint64_t first = (uint64_t)(tile - p.tile0[c]) * kMutTile;
    const uint64_t seed = p.seed;
    uint32_t* cnt = p.cnt + tile;

    for (uint32_t step = 0; step < kMutSteps; step++) {
        const uint64_t s0 = first + step * 128u + lane * 4u;
        if (first + step * 128u >= len) break;
        uint32_t ref = 0, cand = 0, ev = 0, cats = 0;      // 2 bits per site; T/C/A/G sites; evolving sites; 8 bits per site
#pragma unroll
        for (uint32_t k = 0; k < 4; k++)
            if (s0 + k < len) {
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
        if (__ballot_sync(~0u, ev) == 0) continue;
        st[0][tid] = (uint8_t)ref;
        for (uint32_t n = 0; n < p.n_sched; n++) {
            const MutNode nd = p.sched[n];
            const uint32_t ps = st[nd.pslot][tid];
            uint32_t ns = ps;
            if (ev) {
                const U4 w = mut_block(seed, c, s0 >> 2, nd.node);
#pragma unroll
                for (uint32_t k = 0; k < 4; k++) {
                    if (!((ev >> k) & 1u)) continue;
                    const uint32_t a = (ps >> (2 * k)) & 3u, row = nd.tab + 4u * ((cats >> (8 * k)) & 0xffu) + a;
                    const uint32_t b = decide(genome_word(w, k), thi[row], p.thr_lo, row, seed, c, s0 + k, nd.node);
                    ns = (ns & ~(3u << (2 * k))) | (b << (2 * k));
                }
            }
            if (nd.tip < 0) { st[nd.slot][tid] = (uint8_t)ns; continue; }
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
                pool[i] = (uint8_t)(__byte_perm(0x47414354u, 0u, (ns >> (2 * k)) & 3u) & 0xffu);
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

}  // namespace

size_t mut_smem_bytes(uint32_t tab_rows) { return (size_t)tab_rows * sizeof(uint4); }

cudaError_t launch_mutate(const MutParams& p, bool write, cudaStream_t s) {
    if (p.n_tiles == 0) return cudaSuccess;
    const size_t smem = p.tab_smem ? mut_smem_bytes(p.tab_rows) : 0;
    const unsigned grid = (p.n_tiles + kMutWarps - 1) / kMutWarps;
    if (write) {
        cudaError_t e = cudaFuncSetAttribute(k_mutate<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        k_mutate<true><<<grid, kMutWarps * 32, smem, s>>>(p);
    } else {
        cudaError_t e = cudaFuncSetAttribute(k_mutate<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        k_mutate<false><<<grid, kMutWarps * 32, smem, s>>>(p);
    }
    return cudaGetLastError();
}

cudaError_t launch_mut_scan(const MutParams& p, uint64_t* region_n, cudaStream_t s) {
    const uint64_t n = (uint64_t)p.n_tips * p.n_chroms;
    if (n == 0) return cudaSuccess;
    k_mut_scan<<<(unsigned)n, 1024, 0, s>>>(p, region_n);
    return cudaGetLastError();
}

}  // namespace jlp
