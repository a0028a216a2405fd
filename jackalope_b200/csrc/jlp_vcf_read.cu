// haps_vcf on the device (DESIGN.md section 12): a batch of whole VCF lines parsed into alleles and non-REF calls, and a
// chromosome's calls walked into records.  One thread per line for the fixed columns and the alleles; one warp per line
// for the sample columns (field starts from ballots over the line's bytes, one lane per GT field), counted, scanned and
// written so that the calls come out line-major; CUB's stable radix sort then groups a chromosome's calls by haplotype
// slot in file order, and one thread per slot applies the overlap rule and writes the records.  No kernel reads outside
// its batch's lines whatever the bytes are; a malformed line is reported through the status word, never by a trap.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>

#include "jlp_kernels.cuh"

namespace jlp {

namespace {

constexpr unsigned kFull = 0xffffffffu;

unsigned grid_of(uint64_t n) { return (unsigned)std::max<uint64_t>(1, (n + 255) / 256); }

uint32_t bits_of(uint64_t x) {
    uint32_t b = 1;
    while (b < 64 && (x >> b)) b++;
    return b;
}

__device__ __forceinline__ uint8_t up(uint8_t c) { return c >= 'a' && c <= 'z' ? (uint8_t)(c - 32) : c; }
__device__ __forceinline__ bool letter(uint8_t c) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z'); }
__device__ __forceinline__ bool digit(uint8_t c) { return c >= '0' && c <= '9'; }

__device__ __forceinline__ void report(const VrBatch& b, uint32_t i, uint32_t reason) {
    atomicMin(b.status, (unsigned long long)((b.line0 + i) << 8 | reason));
}

// [a, e) of line i: its newline and a CR before it excluded
__device__ __forceinline__ void line_span(const VrBatch& b, uint32_t i, uint32_t& a, uint32_t& e) {
    a = i ? b.nl[i - 1] + 1 : 0;
    e = b.nl[i];
    if (e > a && b.text[e - 1] == '\r') e--;
}

struct IsNewline {
    const uint8_t* t;
    __device__ __forceinline__ bool operator()(uint32_t i) const { return t[i] == '\n'; }
};

// bytewise comparison of t[0, n) with name k of the sorted table
__device__ int cmp_name(const VrBatch& b, const uint8_t* t, uint32_t n, uint32_t k) {
    const uint8_t* s = b.names + b.name_off[k];
    const uint32_t m = b.name_off[k + 1] - b.name_off[k];
    for (uint32_t j = 0; j < n && j < m; j++)
        if (t[j] != s[j]) return t[j] < s[j] ? -1 : 1;
    return n < m ? -1 : (n > m ? 1 : 0);
}

__device__ bool same_key(const uint8_t* t, uint32_t n, const char* k, uint32_t kn) {
    if (n != kn) return false;
    for (uint32_t j = 0; j < n; j++)
        if (t[j] != (uint8_t)k[j]) return false;
    return true;
}

// one ALT entry: its kind, or kVrNone if it is malformed
__device__ uint32_t alt_kind(const uint8_t* t, uint32_t n, bool sv_info) {
    if (n == 0) return kVrNone;
    bool all = true, brk = false;
    for (uint32_t j = 0; j < n; j++) {
        all &= letter(t[j]);
        brk |= t[j] == '[' || t[j] == ']';
    }
    if (all) return VR_SEQ;
    if (n == 1 && t[0] == '*') return VR_STAR;
    if (same_key(t, n, "<DEL>", 5)) return sv_info ? VR_SYM : VR_SEQ;
    if ((n >= 3 && t[0] == '<' && t[n - 1] == '>') || brk) return VR_SYM;
    return kVrNone;
}

// The fixed columns of one line per thread.  A line with fewer than 10 columns is left to k_vr_gt, which counts them.
__global__ void k_vr_fixed(VrBatch b) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b.n_lines) return;
    const uint8_t* t = b.text;
    uint32_t a, e;
    line_span(b, i, a, e);
    VrLine L{kVrNone, 0, 0, 0, 0, 0, 0, 0};
    uint32_t fs[10];
    fs[0] = a;
    uint32_t nf = 1;
    for (uint32_t p = a; p < e && nf < 10; p++)
        if (t[p] == '\t') fs[nf++] = p + 1;
    uint32_t reason = 0;
    uint32_t c = kVrNone;
    do {
        if (nf < 10) break;
        // CHROM: lower bound in the sorted names
        {
            const uint32_t n = fs[1] - 1 - fs[0];
            uint32_t lo = 0, hi = b.n_chroms;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) / 2;
                if (cmp_name(b, t + fs[0], n, mid) > 0) lo = mid + 1; else hi = mid;
            }
            if (lo == b.n_chroms || cmp_name(b, t + fs[0], n, lo) != 0) { reason = VR_CHROM; break; }
            c = b.name_idx[lo];
        }
        // POS
        const uint32_t pn = fs[2] - 1 - fs[1];
        uint64_t pos = 0;
        bool ok = pn >= 1 && pn <= 10;
        for (uint32_t j = 0; ok && j < pn; j++) {
            ok = digit(t[fs[1] + j]);
            pos = pos * 10 + (t[fs[1] + j] - '0');
        }
        if (!ok || pos < 1 || pos >= (1ull << 32)) { reason = VR_POS; break; }
        // REF
        const uint32_t m = fs[4] - 1 - fs[3];
        ok = m >= 1;
        for (uint32_t j = 0; ok && j < m; j++) ok = letter(t[fs[3] + j]);
        if (!ok) { reason = VR_REF_LETTERS; break; }
        const uint64_t Lc = b.chrom_off[c + 1] - b.chrom_off[c];
        if (pos - 1 + m > Lc) { reason = VR_REF_RANGE; break; }
        const uint8_t* R = b.genome + b.chrom_off[c] + pos - 1;
        for (uint32_t j = 0; ok && j < m; j++) ok = up(t[fs[3] + j]) == up(R[j]);
        if (!ok) { reason = VR_REF_DIFF; break; }
        // INFO keys END / SVLEN
        bool sv = false;
        for (uint32_t k0 = fs[7], p = fs[7]; p <= fs[8] - 1; p++)
            if (p == fs[8] - 1 || t[p] == ';') {
                uint32_t k1 = k0;
                while (k1 < p && t[k1] != '=') k1++;
                sv |= same_key(t + k0, k1 - k0, "END", 3) || same_key(t + k0, k1 - k0, "SVLEN", 5);
                k0 = p + 1;
            }
        // ALT
        const uint32_t an = fs[5] - 1 - fs[4];
        uint32_t n_alt = 0;
        if (!(an == 1 && t[fs[4]] == '.')) {
            for (uint32_t k0 = fs[4], p = fs[4]; ok && p <= fs[5] - 1; p++)
                if (p == fs[5] - 1 || t[p] == ',') {
                    ok = alt_kind(t + k0, p - k0, sv) != kVrNone;
                    n_alt++;
                    k0 = p + 1;
                }
            if (!ok) { reason = VR_ALT; break; }
        }
        // FORMAT
        const uint32_t fn = fs[9] - 1 - fs[8];
        if (!(fn >= 2 && t[fs[8]] == 'G' && t[fs[8] + 1] == 'T' && (fn == 2 || t[fs[8] + 2] == ':'))) { reason = VR_FORMAT; break; }
        L = VrLine{c, (uint32_t)(pos - 1), m, fs[4], an, fs[9], n_alt, sv ? 1u : 0u};
    } while (0);
    if (reason) report(b, i, reason);
    b.line[i] = L;
    b.n_alt[i] = L.chrom == kVrNone ? 0 : L.n_alt;
    b.alt_len[i] = L.chrom == kVrNone ? 0 : L.alt_len;
}

// The alleles of one line per thread: kinds, their text copied out of the batch, and the size of their encoding.
__global__ void k_vr_alleles(VrBatch b) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b.n_lines) return;
    const VrLine L = b.line[i];
    if (L.chrom == kVrNone || L.n_alt == 0) return;
    const uint8_t* t = b.text + L.alt_at;
    uint8_t* dst = b.alt_text + b.text0[i];
    for (uint32_t j = 0; j < L.alt_len; j++) dst[j] = t[j];
    const uint8_t* R = b.genome + b.chrom_off[L.chrom] + L.s;
    uint32_t k = b.alt0[i];
    for (uint32_t k0 = 0, p = 0; p <= L.alt_len; p++) {
        if (p < L.alt_len && t[p] != ',') continue;
        VrAllele A;
        A.s = L.s; A.m = L.m;
        A.kind = alt_kind(t + k0, p - k0, L.sv_info != 0);
        A.n = A.kind == VR_SEQ && t[k0] != '<' ? p - k0 : 0;
        A.text = b.text0[i] + k0;
        A.nrec = 0; A.pool = 0;
        if (A.kind == VR_SEQ) {
            const uint32_t m = A.m, n = A.n;
            const uint32_t lim = n > m ? m - 1 : min(m, n);
            for (uint32_t j = 0; j < lim; j++)
                if (up(t[k0 + j]) != up(R[j])) { A.nrec++; A.pool++; }
            if (n > m) { A.nrec++; A.pool += n - m + 1; }
            else if (m > n) A.nrec++;
        }
        b.allele[k++] = A;
        k0 = p + 1;
    }
}

// One GT field at t[q..e): its alleles (kVrNone for '.'), at most kVrMaxPloidy; returns the count or 0 with *reason set.
__device__ __forceinline__ uint32_t parse_gt(const uint8_t* t, uint32_t q, uint32_t e, uint32_t* al, uint32_t& reason) {
    uint32_t na = 0;
    while (true) {
        uint32_t v;
        if (q < e && t[q] == '.') {
            v = kVrNone;
            q++;
        } else {
            uint32_t nd = 0;
            v = 0;
            while (q < e && digit(t[q])) {
                v = min(v * 10 + (t[q] - '0'), 0x7fffffffu);
                nd++;
                q++;
            }
            if (nd == 0) { reason = VR_GT; return 0; }
        }
        if (na < kVrMaxPloidy) al[na] = v;
        na++;
        const uint8_t c = q < e ? t[q] : '\t';
        if (c == '|' || c == '/') { q++; continue; }
        if (c == ':' || c == '\t') break;
        reason = VR_GT;
        return 0;
    }
    if (na > kVrMaxPloidy) { reason = VR_PLOIDY; return 0; }
    return na;
}

// The sample columns, one warp per line.  Count pass: the column count, the GT fields' checks, the largest allele count
// per sample, missing and symbolic calls, and the line's non-REF calls.  Write pass: the calls at call0[line] on, as
// (slot, allele) pairs.
template <bool kWrite> __global__ void k_vr_gt(VrBatch b) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_warps = gridDim.x * (blockDim.x / 32);
    const uint8_t* t = b.text;
    for (uint32_t i = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; i < b.n_lines; i += n_warps) {
        uint32_t a, e;
        line_span(b, i, a, e);
        const VrLine L = b.line[i];
        const bool valid = L.chrom != kVrNone;
        const uint32_t alt0 = valid && L.n_alt ? b.alt0[i] : 0;
        uint32_t field = 0, out = kWrite ? b.call0[i] : 0, reason = 0, calls = 0;
        unsigned long long missing = 0, symbolic = 0;
        for (uint32_t base = a; base <= e; base += 32) {
            const uint32_t p = base + lane;
            const bool st = p <= e && (p == a || t[p - 1] == '\t');
            const unsigned m = __ballot_sync(kFull, st);
            const uint32_t f = field + __popc(m & ((1u << lane) - 1));
            field += __popc(m);
            uint32_t nc = 0, sl[kVrMaxPloidy], av[kVrMaxPloidy];
            if (st && valid && f >= 9 && f - 9 < b.n_samples) {
                uint32_t al[kVrMaxPloidy], why = 0;
                const uint32_t na = parse_gt(t, p, e, al, why);
                if (why) reason = reason ? min(reason, why) : why;
                if (!kWrite && na) atomicMax(b.ploidy + (f - 9), na);
                for (uint32_t k = 0; k < na; k++) {
                    if (al[k] == kVrNone) { missing++; continue; }
                    if (al[k] == 0) continue;
                    if (al[k] > L.n_alt) { reason = reason ? min(reason, (uint32_t)VR_INDEX) : VR_INDEX; continue; }
                    const uint32_t kind = b.allele[alt0 + al[k] - 1].kind;
                    if (kind == VR_SYM) symbolic++;
                    if (kind != VR_SEQ) continue;
                    sl[nc] = (f - 9) * kVrMaxPloidy + k;
                    av[nc] = alt0 + al[k] - 1;
                    nc++;
                }
            }
            if (kWrite) {
                uint32_t x = nc;
                for (uint32_t d = 1; d < 32; d <<= 1) {
                    const uint32_t y = __shfl_up_sync(kFull, x, d);
                    if (lane >= d) x += y;
                }
                const uint32_t total = __shfl_sync(kFull, x, 31);
                for (uint32_t k = 0; k < nc; k++) {
                    b.call_slot[out + x - nc + k] = sl[k];
                    b.call_allele[out + x - nc + k] = av[k];
                }
                out += total;
            } else {
                calls += nc;
            }
        }
        if (kWrite) continue;
        if (field != b.n_cols) reason = VR_COLUMNS;
        for (uint32_t d = 16; d; d >>= 1) {
            calls += __shfl_xor_sync(kFull, calls, d);
            missing += __shfl_xor_sync(kFull, missing, d);
            symbolic += __shfl_xor_sync(kFull, symbolic, d);
            const uint32_t r = __shfl_xor_sync(kFull, reason, d);
            if (r && (!reason || r < reason)) reason = r;
        }
        if (lane == 0) {
            b.n_calls[i] = calls;
            if (missing) atomicAdd(b.counts, missing);
            if (symbolic) atomicAdd(b.counts + 1, symbolic);
            if (reason) report(b, i, reason);
        }
    }
}

// POS against the line before in the same chromosome; where the chromosome changes a run of lines starts
__global__ void k_vr_order(VrBatch b) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b.n_lines) return;
    const VrLine L = b.line[i];
    uint32_t pc = b.prev_chrom, ps = b.prev_s;
    if (i) { const VrLine P = b.line[i - 1]; pc = P.chrom; ps = P.s; }
    if (L.chrom != kVrNone && L.chrom == pc && L.s < ps) report(b, i, VR_ORDER);
    b.run_flag[i] = L.chrom != pc || (i == 0 && pc == kVrNone);
    b.run_key[i] = (uint64_t)i << 32 | L.chrom;
}

__global__ void k_vr_append(VrBatch b, uint32_t a0, uint32_t a1, uint32_t c0, uint32_t c1, uint32_t t0, uint64_t n_alleles,
                            uint64_t n_calls, uint64_t text_bytes, VrAllele* allele, uint32_t* slot, uint32_t* val) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < a1 - a0) {
        VrAllele A = b.allele[a0 + j];
        A.text = A.text - t0 + text_bytes;
        allele[n_alleles + j] = A;
    }
    if (j < c1 - c0) {
        slot[n_calls + j] = b.call_slot[c0 + j];
        val[n_calls + j] = (uint32_t)(b.call_allele[c0 + j] - a0 + n_alleles);
    }
}

__global__ void k_vr_bounds(VrChrom v) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= v.n_calls) return;
    const uint32_t k = v.slot2[i];
    if (i == 0 || v.slot2[i - 1] != k) v.seg[2 * (uint64_t)k] = i;
    if (i + 1 == v.n_calls || v.slot2[i + 1] != k) v.seg[2 * (uint64_t)k + 1] = i + 1;
}

// One thread per haplotype slot: its calls in file order, a call skipped when its line starts before the end of the last
// applied line.  Count pass: records, pool bytes, size change, applied and skipped calls.  Write pass: the records
// (old_pos | new_pos | nuc_off | size_modifier | pool) at region[slot].
template <bool kWrite> __global__ void k_vr_walk(VrChrom v) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= v.n_slots) return;
    const uint64_t lo = v.seg[2 * (uint64_t)q], hi = v.seg[2 * (uint64_t)q + 1];
    uint32_t end = 0;
    VrSlot S{0, 0, 0, 0, 0};
    uint64_t M = 0, *w = nullptr;
    if (kWrite) {
        M = v.out_slot[q].nrec;
        if (M == 0) return;
        w = v.out + v.region[q];
    }
    uint8_t* pool = reinterpret_cast<uint8_t*>(w + 4 * M);
    uint64_t k = 0, pb = 0;
    int64_t shift = 0;
    auto emit = [&](uint64_t p, int64_t d, const uint8_t* x, uint32_t nx, const uint8_t* first) {
        w[k] = p;
        w[M + k] = (uint64_t)((int64_t)p + shift);
        w[2 * M + k] = pb;
        reinterpret_cast<int64_t*>(w + 3 * M)[k] = d;
        for (uint32_t j = 0; j < nx; j++) pool[pb + j] = j == 0 && first ? *first : x[j];
        pb += nx;
        shift += d;
        k++;
    };
    for (uint64_t j = lo; j < hi; j++) {
        const VrAllele A = v.allele[v.val2[j]];
        if (A.s < end) { S.skipped++; continue; }
        end = A.s + A.m;
        S.applied++;
        if (!kWrite) {
            S.nrec += A.nrec;
            S.pool += A.pool;
            S.delta += (long long)A.n - (long long)A.m;
            continue;
        }
        const uint8_t* x = v.text + A.text;
        const uint8_t* R = v.ref + A.s;
        const uint32_t m = A.m, n = A.n;
        const uint32_t lim = n > m ? m - 1 : min(m, n);
        for (uint32_t i = 0; i < lim; i++)
            if (up(x[i]) != up(R[i])) emit(A.s + i, 0, x + i, 1, nullptr);
        if (n > m) emit(A.s + m - 1, (int64_t)(n - m), x + m - 1, n - m + 1, up(x[m - 1]) == up(R[m - 1]) ? R + m - 1 : nullptr);
        else if (m > n) emit(A.s + n, -(int64_t)(m - n), nullptr, 0, nullptr);
    }
    if (!kWrite) v.out_slot[q] = S;
}

}  // namespace

size_t vr_cub_bytes(uint64_t n) {
    size_t a = 0, b = 0, c = 0, d = 0;
    cub::DeviceSelect::If(nullptr, a, thrust::counting_iterator<uint32_t>(0), (uint32_t*)nullptr, (uint32_t*)nullptr,
                          (int64_t)n, IsNewline{nullptr});
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int64_t)n);
    cub::DeviceSelect::Flagged(nullptr, c, (const uint64_t*)nullptr, (const uint8_t*)nullptr, (uint64_t*)nullptr,
                               (uint32_t*)nullptr, (int64_t)n);
    cub::DeviceRadixSort::SortPairs(nullptr, d, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int64_t)n);
    return std::max(std::max(a, b), std::max(c, d));
}

cudaError_t launch_vr_parse(const VrBatch& b, int stage, uint8_t* tmp, size_t tmp_bytes, cudaStream_t s) {
    size_t tb = tmp_bytes;
    cudaError_t e = cudaSuccess;
    const int64_t n1 = (int64_t)b.n_lines + 1;
    if (stage == 0)
        return cub::DeviceSelect::If(tmp, tb, thrust::counting_iterator<uint32_t>(0), b.nl, b.n_sel, (int64_t)b.n_bytes,
                                     IsNewline{b.text}, s);
    if (stage == 1) {
        // the last entries stay 0, so the exclusive prefixes end with the batch's totals
        if ((e = cudaMemsetAsync(b.n_alt, 0, n1 * 4, s)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(b.alt_len, 0, n1 * 4, s)) != cudaSuccess) return e;
        k_vr_fixed<<<grid_of(b.n_lines), 256, 0, s>>>(b);
        if ((e = cub::DeviceScan::ExclusiveSum(tmp, tb, b.n_alt, b.alt0, n1, s)) != cudaSuccess) return e;
        tb = tmp_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(tmp, tb, b.alt_len, b.text0, n1, s)) != cudaSuccess) return e;
        return cudaGetLastError();
    }
    const unsigned gt_blocks = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((b.n_lines + 7) / 8, 148u * 16));
    if (stage == 2) {
        if ((e = cudaMemsetAsync(b.n_calls, 0, n1 * 4, s)) != cudaSuccess) return e;
        k_vr_alleles<<<grid_of(b.n_lines), 256, 0, s>>>(b);
        k_vr_gt<false><<<gt_blocks, 256, 0, s>>>(b);
        if ((e = cub::DeviceScan::ExclusiveSum(tmp, tb, b.n_calls, b.call0, n1, s)) != cudaSuccess) return e;
        return cudaGetLastError();
    }
    k_vr_gt<true><<<gt_blocks, 256, 0, s>>>(b);
    k_vr_order<<<grid_of(b.n_lines), 256, 0, s>>>(b);
    if ((e = cub::DeviceSelect::Flagged(tmp, tb, b.run_key, b.run_flag, b.runs, b.n_sel, (int64_t)b.n_lines, s)) != cudaSuccess)
        return e;
    return cudaGetLastError();
}

cudaError_t launch_vr_append(const VrBatch& b, uint32_t a0, uint32_t a1, uint32_t c0, uint32_t c1, uint32_t t0,
                             uint64_t n_alleles, uint64_t n_calls, uint64_t text_bytes, VrAllele* allele, uint32_t* slot,
                             uint32_t* val, cudaStream_t s) {
    const uint64_t n = std::max<uint64_t>(a1 - a0, c1 - c0);
    if (n == 0) return cudaSuccess;
    k_vr_append<<<grid_of(n), 256, 0, s>>>(b, a0, a1, c0, c1, t0, n_alleles, n_calls, text_bytes, allele, slot, val);
    return cudaGetLastError();
}

cudaError_t launch_vr_count(const VrChrom& v, uint8_t* tmp, size_t tmp_bytes, cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(v.seg, 0, 2 * (size_t)v.n_slots * 8, s);
    if (e != cudaSuccess) return e;
    if (v.n_calls) {
        size_t tb = tmp_bytes;
        e = cub::DeviceRadixSort::SortPairs(tmp, tb, v.slot, v.slot2, v.val, v.val2, (int64_t)v.n_calls, 0, bits_of(v.n_slots), s);
        if (e != cudaSuccess) return e;
        k_vr_bounds<<<grid_of(v.n_calls), 256, 0, s>>>(v);
    }
    k_vr_walk<false><<<grid_of(v.n_slots), 256, 0, s>>>(v);
    return cudaGetLastError();
}

cudaError_t launch_vr_write(const VrChrom& v, cudaStream_t s) {
    k_vr_walk<true><<<grid_of(v.n_slots), 256, 0, s>>>(v);
    return cudaGetLastError();
}

}  // namespace jlp
