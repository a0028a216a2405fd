// write_vcf on the device (DESIGN.md section 11): the spans of a chromosome's records, their lines, and the lines' text.
// The work follows the records and the lines: one thread per record for the spans, CUB sorts and scans to group them
// into lines, then one warp per line to build its alleles and, in a second pass, to write its text at its final offset.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda/functional>

#include <algorithm>

#include "jlp_kernels.cuh"

namespace jlp {

namespace {

constexpr uint32_t kNone = 0xffffffffu;

__device__ __forceinline__ uint32_t ndigits(uint64_t v) {
    uint32_t n = 1;
    while (v >= 10) { v /= 10; n++; }
    return n;
}
__device__ __forceinline__ void put_uint(uint8_t* dst, uint64_t v, uint32_t n) {
    for (uint32_t k = n; k-- > 0;) { dst[k] = (uint8_t)('0' + v % 10); v /= 10; }
}
__device__ __forceinline__ void warp_copy(uint8_t* dst, const uint8_t* src, uint64_t n, uint32_t lane) {
    for (uint64_t t = lane; t < n; t += 32) dst[t] = src[t];
}

struct HapView {
    const uint64_t *op, *np, *no;
    const int64_t* sm;
    const uint8_t* pool;
};
__device__ __forceinline__ HapView hap_view(const VcfChrom& v, uint32_t u) {
    const VcfHap H = v.hap[u];
    const uint64_t* w = v.recs + H.woff;
    return HapView{w, w + H.n, w + 2 * (uint64_t)H.n, reinterpret_cast<const int64_t*>(w + 3 * (uint64_t)H.n),
                   reinterpret_cast<const uint8_t*>(w + 4 * (uint64_t)H.n)};
}

// Byte t of a carrier's allele: k_materialize's rule (jlp_kernels.cu) over the carrier's records of the line, at the
// haplotype position new_s + t.  car == NULL: the reference allele.
__device__ uint8_t allele_byte(const VcfChrom& v, const VcfCar* car, uint64_t s, uint64_t t) {
    if (!car) return v.ref[s + t];
    const HapView h = hap_view(v, car->u);
    const uint64_t p = car->new_s + t;
    int64_t lo = (int64_t)car->i0 - 1, hi = (int64_t)car->i1 + 1;      // np[lo] <= p < np[hi]
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) / 2;
        if (h.np[mid] <= p) lo = mid; else hi = mid;
    }
    if (lo < (int64_t)car->i0) return v.ref[s + t];
    const uint64_t ind = p - h.np[lo];
    const int64_t sm = h.sm[lo];
    return (int64_t)ind > sm ? v.ref[ind + h.op[lo] - (uint64_t)sm] : h.pool[h.no[lo] + ind];
}

// the first min(len, 8) bytes of an allele, packed: with len <= 8, (len, key) identifies the allele
__device__ uint64_t allele_key(const VcfChrom& v, const VcfCar* car, uint64_t s, uint64_t len) {
    uint64_t k = 0;
    for (uint64_t t = 0; t < len && t < 8; t++) k |= (uint64_t)allele_byte(v, car, s, t) << (8 * t);
    return k;
}

// whole-warp comparison of two alleles of equal length
__device__ bool warp_equal(const VcfChrom& v, const VcfCar* a, const VcfCar* b, uint64_t s, uint64_t len, uint32_t lane) {
    for (uint64_t t0 = 0; t0 < len; t0 += 32) {
        const uint64_t t = t0 + lane;
        const bool diff = t < len && allele_byte(v, a, s, t) != allele_byte(v, b, s, t);
        if (__any_sync(0xffffffffu, diff)) return false;
    }
    return true;
}

__global__ void __launch_bounds__(256) k_vcf_span(const VcfChrom v) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= v.n_rec) return;
    uint32_t lo = 0, hi = v.n_hap;                // the haplotype whose records hold j: rec0[lo] <= j < rec0[lo + 1]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) / 2;
        if (v.hap[mid].rec0 <= j) lo = mid; else hi = mid;
    }
    const HapView h = hap_view(v, lo);
    const uint32_t i = (uint32_t)j - v.hap[lo].rec0;
    const uint64_t op = h.op[i];
    const int64_t sm = h.sm[i];
    uint64_t s = op, e = op + (sm < 0 ? (uint64_t)(-sm) : 1);
    if (sm < 0) {                                   // a deletion takes the base before it (or after it at position 0)
        if (op > 0) s = op - 1;
        else e = min(v.L, (uint64_t)(1 - sm));
    }
    v.start[j] = s;
    v.end[j] = e;
    v.rec_hap[j] = lo;
    v.val[j] = (uint32_t)j;
}

__global__ void __launch_bounds__(256) k_vcf_gather_end(const VcfChrom v) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < v.n_rec) v.end_sorted[k] = v.end[v.order[k]];
}

// record k of the sorted order starts a line when no span before it reaches past its start
__global__ void __launch_bounds__(256) k_vcf_flag(const VcfChrom v) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < v.n_rec) v.flag[k] = k == 0 || v.start_sorted[k] >= v.maxend[k - 1];
}

__global__ void __launch_bounds__(256) k_vcf_group(const VcfChrom v) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= v.n_rec) return;
    const uint32_t l = v.lid[k] - 1;
    if (v.flag[k]) { v.line_first[l] = (uint32_t)k; v.line_s[l] = v.start_sorted[k]; }
    if (k + 1 == v.n_rec || v.flag[k + 1]) v.line_e[l] = v.maxend[k];
    if (k + 1 == v.n_rec) v.line_first[l + 1] = v.n_rec;
    v.key2[k] = (uint64_t)l << 32 | v.order[k];    // second sort: by line, then by record (haplotype-major)
}

__device__ __forceinline__ uint32_t rec_at(const VcfChrom& v, uint64_t k) { return (uint32_t)v.key2_sorted[k]; }

// One warp per line.  Sizing pass (WRITE = false): the line's carriers (haplotypes with records in it, in haplotype
// order), their alleles' classes (REF, or one per distinct allele), the ALTs in order of their first slot of the sample
// matrix, each carrier's allele index, and the line's text length (0 when every allele is REF).  Text pass: the text
// of lines [l0, l1) at line_off[l] - line_off[l0] + out_skip of `out`.
template <bool WRITE>
__global__ void __launch_bounds__(256) k_vcf_lines(const VcfChrom v, uint32_t l0, uint32_t l1, uint8_t* out, uint64_t out_skip) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    uint32_t* hidx = v.hidx + warp * v.n_hap;
    const uint64_t base = WRITE && l0 ? v.line_end[l0 - 1] : 0;
    for (uint64_t l = l0 + warp; l < l1; l += n_warps) {
        const uint32_t f = v.line_first[l], g = v.line_first[l + 1];
        const uint64_t s = v.line_s[l], e = v.line_e[l], ref_len = e - s;
        if (!WRITE) {
            // ---- carriers: where the haplotype changes along the line's records
            uint32_t n_c = 0;
            for (uint32_t k0 = f; k0 < g; k0 += 32) {
                const uint32_t k = k0 + lane;
                const bool first = k < g && (k == f || v.rec_hap[rec_at(v, k)] != v.rec_hap[rec_at(v, k - 1)]);
                const uint32_t m = __ballot_sync(0xffffffffu, first);
                if (first) v.car_pos[f + n_c + __popc(m & ((1u << lane) - 1))] = k;
                n_c += __popc(m);
            }
            __syncwarp();
            for (uint32_t c = lane; c < n_c; c += 32) {
                const uint32_t k = v.car_pos[f + c], kend = c + 1 < n_c ? v.car_pos[f + c + 1] : g;
                const uint32_t j0 = rec_at(v, k), j1 = rec_at(v, kend - 1), u = v.rec_hap[j0];
                const HapView h = hap_view(v, u);
                VcfCar C;
                C.u = u; C.i0 = j0 - v.hap[u].rec0; C.i1 = j1 - v.hap[u].rec0;
                const uint64_t d0 = h.np[C.i0] - h.op[C.i0], d1 = h.np[C.i1] - h.op[C.i1] + (uint64_t)h.sm[C.i1];
                C.new_s = s + d0;
                C.len = ref_len + d1 - d0;
                C.key = allele_key(v, &C, s, C.len);
                C.idx = 0;
                v.car[f + c] = C;
            }
            // ---- classes: class 0 is REF; the others in order of discovery, each with its first slot
            const uint64_t ref_key = allele_key(v, nullptr, s, ref_len);
            uint32_t n_cls = 1;
            __syncwarp();
            for (uint32_t c = 0; c < n_c; c++) {
                const VcfCar C = v.car[f + c];
                uint32_t match = kNone;
                if (C.len == ref_len && C.key == ref_key && (C.len <= 8 || warp_equal(v, &C, nullptr, s, C.len, lane))) match = 0;
                for (uint32_t q0 = 1; q0 < n_cls && match == kNone; q0 += 32) {
                    const uint32_t q = q0 + lane;
                    bool cand = false;
                    if (q < n_cls) {
                        const VcfCar& R = v.car[f + v.cls_car[f + q]];
                        cand = R.len == C.len && R.key == C.key;
                    }
                    uint32_t m = __ballot_sync(0xffffffffu, cand);
                    while (m && match == kNone) {
                        const uint32_t q1 = q0 + __ffs(m) - 1;
                        m &= m - 1;
                        if (C.len <= 8 || warp_equal(v, &C, &v.car[f + v.cls_car[f + q1]], s, C.len, lane)) match = q1;
                    }
                }
                const uint32_t slot = v.first_slot[C.u];
                if (lane == 0) {
                    if (match == kNone) { v.cls_car[f + n_cls] = c; v.cls_slot[f + n_cls] = slot; }
                    else if (match > 0 && slot < v.cls_slot[f + match]) v.cls_slot[f + match] = slot;
                    v.car[f + c].idx = match == kNone ? n_cls : match;
                }
                if (match == kNone) n_cls++;
                __syncwarp();
            }
            // ---- ALT k is the class with the k-th smallest first slot (slots of different classes differ)
            const uint32_t n_alt = n_cls - 1;
            for (uint32_t q = 1 + lane; q < n_cls; q += 32) {
                const uint32_t sq = v.cls_slot[f + q];
                uint32_t r = 1;
                for (uint32_t q2 = 1; q2 < n_cls; q2++) r += v.cls_slot[f + q2] < sq;
                v.cls_rank[f + q] = r;
                v.alt_car[f + r - 1] = v.cls_car[f + q];
            }
            __syncwarp();
            uint64_t extra = 0, alt_bytes = 0;
            for (uint32_t c = lane; c < n_c; c += 32) {
                const uint32_t cls = v.car[f + c].idx, idx = cls ? v.cls_rank[f + cls] : 0;
                v.car[f + c].idx = idx;
                if (idx >= 10) extra += (uint64_t)v.n_slots[v.car[f + c].u] * (ndigits(idx) - 1);
            }
            for (uint32_t a = lane; a < n_alt; a += 32) {
                const uint64_t n = v.car[f + v.alt_car[f + a]].len;
                alt_bytes += n ? n : 5;                                          // "<DEL>"
            }
            for (int o = 16; o; o >>= 1) {
                extra += __shfl_xor_sync(0xffffffffu, extra, o);
                alt_bytes += __shfl_xor_sync(0xffffffffu, alt_bytes, o);
            }
            if (lane == 0) {
                v.n_car[l] = n_c;
                v.n_alt[l] = n_alt;
                v.line_len[l] = n_alt == 0 ? 0 : v.name_len + ndigits(s + 1) + ref_len + alt_bytes + (n_alt - 1) + 18 +
                                                 2ull * v.ploidy * v.n_samples + extra;
            }
        } else {
            const uint32_t n_alt = v.n_alt[l], n_c = v.n_car[l];
            if (n_alt == 0) continue;
            uint8_t* o = out + out_skip + (l ? v.line_end[l - 1] : 0) - base;
            warp_copy(o, v.name, v.name_len, lane);
            o += v.name_len;
            const uint32_t dp = ndigits(s + 1);
            if (lane == 0) { o[0] = '\t'; put_uint(o + 1, s + 1, dp); o[dp + 1] = '\t'; o[dp + 2] = '.'; o[dp + 3] = '\t'; }
            o += dp + 4;
            warp_copy(o, v.ref + s, ref_len, lane);
            o += ref_len;
            if (lane == 0) *o = '\t';
            o++;
            for (uint32_t a = 0; a < n_alt; a++) {
                if (a) { if (lane == 0) *o = ','; o++; }
                const VcfCar C = v.car[f + v.alt_car[f + a]];
                if (C.len == 0) {
                    if (lane < 5) o[lane] = "<DEL>"[lane];
                    o += 5;
                    continue;
                }
                // k_materialize's rule, segment by segment: before the first record the reference; from record i to
                // the next, its pool bytes and then the reference after its consumed bases
                const HapView h = hap_view(v, C.u);
                const uint64_t p_end = C.new_s + C.len;
                uint64_t p = C.new_s;
                const uint64_t pre = min(h.np[C.i0], p_end) - p;
                warp_copy(o, v.ref + s, pre, lane);
                o += pre; p += pre;
                for (uint32_t i = C.i0; i <= C.i1 && p < p_end; i++) {
                    const uint64_t seg_end = i < C.i1 ? min(h.np[i + 1], p_end) : p_end;
                    if (seg_end <= p) continue;
                    const int64_t sm = h.sm[i];
                    const uint64_t ind0 = p - h.np[i], n = seg_end - p;
                    const uint64_t n_pool = (int64_t)ind0 > sm ? 0 : min(n, (uint64_t)(sm + 1) - ind0);
                    warp_copy(o, h.pool + h.no[i] + ind0, n_pool, lane);
                    warp_copy(o + n_pool, v.ref + (ind0 + n_pool + h.op[i] - (uint64_t)sm), n - n_pool, lane);
                    o += n; p = seg_end;
                }
            }
            if (lane == 0) for (int k = 0; k < 12; k++) o[k] = "\t.\tPASS\t.\tGT"[k];
            o += 12;
            // ---- genotypes: the carriers' indices in the warp's table (every other included haplotype is 0)
            for (uint32_t c = lane; c < n_c; c += 32) hidx[v.car[f + c].u] = v.car[f + c].idx;
            __syncwarp();
            for (uint32_t s0 = 0; s0 < v.n_samples; s0 += 32) {
                const uint32_t smp = s0 + lane;
                uint32_t n = 0;
                if (smp < v.n_samples)
                    for (uint32_t k = 0; k < v.ploidy; k++) n += 1 + ndigits(hidx[v.slot_hap[(uint64_t)smp * v.ploidy + k]]);
                uint32_t incl = n;
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= (uint32_t)d) incl += y;
                }
                if (smp < v.n_samples) {
                    uint8_t* q = o + incl - n;
                    for (uint32_t k = 0; k < v.ploidy; k++) {
                        const uint32_t idx = hidx[v.slot_hap[(uint64_t)smp * v.ploidy + k]], nd = ndigits(idx);
                        *q++ = k ? '|' : '\t';
                        put_uint(q, idx, nd);
                        q += nd;
                    }
                }
                o += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (lane == 0) *o = '\n';
            __syncwarp();
            for (uint32_t c = lane; c < n_c; c += 32) hidx[v.car[f + c].u] = 0;
            __syncwarp();
        }
    }
}

unsigned grid_of(uint64_t n) { return (unsigned)((n + 255) / 256); }

uint32_t bits_of(uint64_t x) {
    uint32_t b = 1;
    while (b < 64 && (x >> b)) b++;
    return b;
}

}  // namespace

size_t vcf_cub_bytes(uint32_t n_rec) {
    size_t a = 0, b = 0, c = 0, d = 0, e = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, n_rec);
    cub::DeviceScan::InclusiveScan(nullptr, b, (const uint64_t*)nullptr, (uint64_t*)nullptr, cuda::maximum<>{}, n_rec);
    cub::DeviceScan::InclusiveSum(nullptr, c, (const uint32_t*)nullptr, (uint32_t*)nullptr, n_rec);
    cub::DeviceRadixSort::SortKeys(nullptr, d, (const uint64_t*)nullptr, (uint64_t*)nullptr, n_rec);
    cub::DeviceScan::InclusiveSum(nullptr, e, (const uint64_t*)nullptr, (uint64_t*)nullptr, n_rec);
    return std::max(std::max(std::max(a, b), std::max(c, d)), e);
}

cudaError_t launch_vcf_spans(const VcfChrom& v, cudaStream_t s) {
    if (v.n_rec == 0) return cudaSuccess;
    size_t tb = v.cub_bytes;
    k_vcf_span<<<grid_of(v.n_rec), 256, 0, s>>>(v);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(v.cub_tmp, tb, v.start, v.start_sorted, v.val, v.order, v.n_rec, 0,
                                                    bits_of(v.L), s);
    if (e != cudaSuccess) return e;
    k_vcf_gather_end<<<grid_of(v.n_rec), 256, 0, s>>>(v);
    tb = v.cub_bytes;
    e = cub::DeviceScan::InclusiveScan(v.cub_tmp, tb, v.end_sorted, v.maxend, cuda::maximum<>{}, v.n_rec, s);
    if (e != cudaSuccess) return e;
    k_vcf_flag<<<grid_of(v.n_rec), 256, 0, s>>>(v);
    tb = v.cub_bytes;
    e = cub::DeviceScan::InclusiveSum(v.cub_tmp, tb, v.flag, v.lid, v.n_rec, s);
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

cudaError_t launch_vcf_size(const VcfChrom& v, uint32_t n_lines, int n_sm, cudaStream_t s) {
    if (n_lines == 0) return cudaSuccess;
    k_vcf_group<<<grid_of(v.n_rec), 256, 0, s>>>(v);
    size_t tb = v.cub_bytes;
    cudaError_t e = cub::DeviceRadixSort::SortKeys(v.cub_tmp, tb, v.key2, v.key2_sorted, v.n_rec, 0, 32 + bits_of(n_lines), s);
    if (e != cudaSuccess) return e;
    k_vcf_lines<false><<<vcf_line_blocks(n_lines, n_sm), 256, 0, s>>>(v, 0, n_lines, nullptr, 0);
    tb = v.cub_bytes;
    e = cub::DeviceScan::InclusiveSum(v.cub_tmp, tb, v.line_len, v.line_end, n_lines, s);
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

cudaError_t launch_vcf_text(const VcfChrom& v, uint32_t l0, uint32_t l1, uint8_t* out, uint64_t out_skip, int n_sm,
                            cudaStream_t s) {
    if (l1 <= l0) return cudaSuccess;
    k_vcf_lines<true><<<vcf_line_blocks(l1 - l0, n_sm), 256, 0, s>>>(v, l0, l1, out, out_skip);
    return cudaGetLastError();
}

unsigned vcf_line_blocks(uint64_t n_lines, int n_sm) {
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n_lines + 7) / 8, (uint64_t)n_sm * 8));
}

}  // namespace jlp
