// Draw addressing and exact uniform arithmetic, shared by host and device code.
//
// The reference consumes one pcg64 output per uniform draw, sequentially, and
// turns it into u = (x+1)/2^64 with x87 long-double arithmetic
// (/root/reference/src/pcg.h:21,99-101).  Here every logical draw
// X(pair instance j, end, purpose, position) is a pure function of a
// Philox4x32 counter (10 rounds; 7 in the per-base QUAL and INDEL planes), so a read does not depend on which GPU, CTA or thread
// produced it (DESIGN.md section 4):
//
//   counter = (j_lo, j_hi, block, plane | end << 8),  key = (seed_lo, seed_hi)
//   plane PAIR : block 0 -> X_fraglen = w1:w0, X_start = w3:w2
//                block 1 -> X_strand  = w1:w0, X_dup   = w3:w2
//   plane INDEL: block t>>3, 16-bit field t&7      -> high 16 bits of X_indel(t)
//   plane QUAL : block p>>1, base h = p&1:
//                die  = w[2h] >> 8  (high 24 bits of X_die), sub = w[2h] & 0xff (high 8 bits of X_sub)
//                coin = w[2h+1] >> 16, mis = w[2h+1] & 0xffff   (high 16 bits)
//   plane SLOW : block pos<<3 | purpose, S = w1:w0 -> the low bits of X: 48 (INDEL, COIN, MIS),
//                40 (DIE), 56 (SUB); the whole of X for INS
//   X = H << (64 - hbits) | (S & (2^(64 - hbits) - 1))
//
// A kernel decides on the high bits alone whenever that is provably enough
// and fetches the SLOW plane only for the (rare) ambiguous cases, so the result
// always equals the one a full 64-bit draw gives.
//
// The integer forms below reproduce the reference's floating-point expressions
// bit for bit, including the x87 round-to-64-bit-mantissa step (tests/
// test_exact_arith.py checks them against the compiled reference expressions).
#ifndef JLP_DRAWS_H
#define JLP_DRAWS_H

#include <stdint.h>

#if defined(__CUDACC__)
#define JLP_HD __host__ __device__ __forceinline__
#else
#define JLP_HD inline
#endif

namespace jlp {

// plane 6 is the oracle's PacBio plane
enum Plane : uint32_t { PL_PAIR = 0, PL_INDEL = 1, PL_QUAL = 2, PL_SLOW = 3, PL_GENOME = 4, PL_GSLOW = 5, PL_MUT = 7, PL_MSLOW = 8,
                        PL_IEV = 9, PL_ICOL = 10, PL_IMUT = 11, PL_IMSLOW = 12 };
enum Purpose : uint32_t { PU_INDEL = 0, PU_DIE = 1, PU_COIN = 2, PU_MIS = 3, PU_SUB = 4, PU_INS = 5 };

struct U4 { uint32_t w0, w1, w2, w3; };

JLP_HD void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umulhi(a, b);
#else
    uint64_t p = (uint64_t)a * b;
    lo = (uint32_t)p;
    hi = (uint32_t)(p >> 32);
#endif
}

// Philox4x32-R, Salmon et al. SC'11, standard multipliers and Weyl constants.  R = 10 everywhere except the QUAL and INDEL
// planes (the per-base draws: nine tenths of all the blocks a run draws), which use R = 7: the fewest rounds at which Philox4x32 passes
// BigCrush in that paper (their "Crush-resistant" column; 10 is its safety margin).
constexpr int kQualRounds = 7;
template <int R>
JLP_HD U4 philox4x32_r(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < R; r++) {
        uint32_t h0, l0, h1, l1;
        mulhilo(0xD2511F53u, c0, h0, l0);
        mulhilo(0xCD9E8D57u, c2, h1, l1);
        c0 = h1 ^ c1 ^ k0;
        c2 = h0 ^ c3 ^ k1;
        c1 = l1;
        c3 = l0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    U4 o = {c0, c1, c2, c3};
    return o;
}
JLP_HD U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    return philox4x32_r<10>(c0, c1, c2, c3, k0, k1);
}

// The same block with the round keys precomputed (rk[2r] = k0 + r * 0x9E3779B9,
// rk[2r+1] = k1 + r * 0xBB67AE85): in a kernel they sit in the constant bank and feed the
// XORs directly.
template <int R>
JLP_HD U4 philox4x32_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const uint32_t* rk) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < R; r++) {
        uint32_t h0, l0, h1, l1;
        mulhilo(0xD2511F53u, c0, h0, l0);
        mulhilo(0xCD9E8D57u, c2, h1, l1);
        c0 = h1 ^ c1 ^ rk[2 * r];
        c2 = h0 ^ c3 ^ rk[2 * r + 1];
        c1 = l1;
        c3 = l0;
    }
    U4 o = {c0, c1, c2, c3};
    return o;
}
inline void philox_round_keys(uint64_t seed, uint32_t rk[20]) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; r++) { rk[2 * r] = k0; rk[2 * r + 1] = k1; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
}

JLP_HD U4 draw_block(uint64_t seed, uint64_t j, uint32_t block, uint32_t plane, uint32_t end) {
    if (plane == PL_QUAL || plane == PL_INDEL)
        return philox4x32_r<kQualRounds>((uint32_t)j, (uint32_t)(j >> 32), block, plane | (end << 8), (uint32_t)seed, (uint32_t)(seed >> 32));
    return philox4x32_10((uint32_t)j, (uint32_t)(j >> 32), block, plane | (end << 8),
                         (uint32_t)seed, (uint32_t)(seed >> 32));
}

JLP_HD uint64_t lo64(const U4& w) { return ((uint64_t)w.w1 << 32) | w.w0; }
JLP_HD uint64_t hi64(const U4& w) { return ((uint64_t)w.w3 << 32) | w.w2; }

JLP_HD uint64_t slow64(uint64_t seed, uint64_t j, uint32_t end, uint32_t purpose, uint32_t pos) {
    return lo64(draw_block(seed, j, (pos << 3) | purpose, PL_SLOW, end));
}
// number of high bits of a draw that live outside the SLOW plane
JLP_HD uint32_t high_bits(uint32_t purpose) {
    return purpose == PU_DIE ? 24u : purpose == PU_SUB ? 8u : purpose == PU_INS ? 0u : 16u;
}
JLP_HD uint64_t full_draw(uint32_t H, uint64_t seed, uint64_t j, uint32_t end, uint32_t purpose, uint32_t pos) {
    const uint32_t hb = high_bits(purpose);
    const uint64_t s = slow64(seed, j, end, purpose, pos);
    if (hb == 0) return s;
    return ((uint64_t)H << (64u - hb)) | (s & (~0ull >> hb));
}
// the high bits of draw (purpose, pos) out of its QUAL / INDEL block
JLP_HD uint32_t high_of(const U4& w, uint32_t purpose, uint32_t pos) {
    if (purpose == PU_INDEL) {
        const uint32_t f = pos & 7u;
        const uint32_t v = (f >> 1) == 0 ? w.w0 : (f >> 1) == 1 ? w.w1 : (f >> 1) == 2 ? w.w2 : w.w3;
        return (f & 1u) ? (v >> 16) : (v & 0xffffu);
    }
    const uint32_t a = (pos & 1u) ? w.w2 : w.w0, b = (pos & 1u) ? w.w3 : w.w1;
    return purpose == PU_DIE ? (a >> 8) : purpose == PU_SUB ? (a & 0xffu) : purpose == PU_COIN ? (b >> 16) : (b & 0xffffu);
}

// ---- draws of the genome generator (create_genome): chromosome c, base b ----
//   plane GENOME: counter (b>>2 lo, b>>2 hi, c, PL_GENOME), word b&3:
//                 bits 31..30 = high 2 bits of X_die(b), bits 29..14 = high 16 bits of X_coin(b)
//   plane GSLOW : counter (b lo, b hi, c, PL_GSLOW | which<<8), S = w1:w0 -> the low 62 (die, which 0)
//                 or 48 (coin, which 1) bits
JLP_HD U4 genome_block(uint64_t seed, uint32_t chrom, uint64_t block) {
    return philox4x32_10((uint32_t)block, (uint32_t)(block >> 32), chrom, PL_GENOME, (uint32_t)seed, (uint32_t)(seed >> 32));
}
JLP_HD uint64_t genome_slow(uint64_t seed, uint32_t chrom, uint64_t b, uint32_t which) {
    return lo64(philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), chrom, PL_GSLOW | (which << 8), (uint32_t)seed, (uint32_t)(seed >> 32)));
}
JLP_HD uint32_t genome_word(const U4& w, uint32_t k) { return k == 0 ? w.w0 : k == 1 ? w.w1 : k == 2 ? w.w2 : w.w3; }
JLP_HD uint64_t genome_draw(uint64_t seed, uint32_t chrom, uint64_t b, uint32_t which) {
    const uint32_t w = genome_word(genome_block(seed, chrom, b >> 2), (uint32_t)b & 3u);
    const uint64_t s = genome_slow(seed, chrom, b, which);
    if (which == 0) return ((uint64_t)(w >> 30) << 62) | (s & (~0ull >> 2));
    return ((uint64_t)((w >> 14) & 0xffffu) << 48) | (s & (~0ull >> 16));
}

// ---- draws of the haplotype mutator (create_haplotypes): chromosome c, site b, tree node v ----
//   X(c, b, v) is one 64-bit draw; node 0 (the root, which has no branch) gives the site's rate-category draw,
//   node v >= 1 the transition draw of the branch above v.  v < 2^24.
//   plane MUT  : counter (b>>2 lo, b>>2 hi, c, PL_MUT | v<<8), word b&3 = high 32 bits of X(c, b, v)
//   plane MSLOW: counter (b lo, b hi, c, PL_MSLOW | v<<8), w0 = low 32 bits of X(c, b, v)
//   Decisions compare the high word with the thresholds' high words and fetch the MSLOW block only on equality.
JLP_HD U4 mut_block(uint64_t seed, uint32_t chrom, uint64_t b4, uint32_t node) {
    return philox4x32_10((uint32_t)b4, (uint32_t)(b4 >> 32), chrom, PL_MUT | (node << 8), (uint32_t)seed, (uint32_t)(seed >> 32));
}
JLP_HD uint32_t mut_low(uint64_t seed, uint32_t chrom, uint64_t b, uint32_t node) {
    return philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), chrom, PL_MSLOW | (node << 8), (uint32_t)seed, (uint32_t)(seed >> 32)).w0;
}
JLP_HD uint64_t mut_draw(uint64_t seed, uint32_t chrom, uint64_t b, uint32_t node) {
    const uint32_t h = genome_word(mut_block(seed, chrom, b >> 2, node), (uint32_t)b & 3u);
    return ((uint64_t)h << 32) | mut_low(seed, chrom, b, node);
}

// ---- draws of insertions and deletions along the tree (create_haplotypes with indels) ----
//   plane IEV  : counter (k, step, c, PL_IEV | v<<8): event k of step `step` on the branch above node v;
//                w1:w0 = the gap draw (the k-th event is 1 + floor(log(U) / log1p(-p)) positions after the one before,
//                U = ((X >> 11) + 1) 2^-53), w3:w2 = the (kind, length) draw
//   plane ICOL : counter (id, 0, c, PL_ICOL): inserted column `id` of chromosome c; w1:w0 = its rate-category draw,
//                w3:w2 = its state at the end of the branch where it was born (against the thresholds of pi)
//   plane IMUT / IMSLOW: the transition draws of inserted column `id` at node v, laid out as MUT / MSLOW with id in
//                place of the site
JLP_HD U4 indel_event_block(uint64_t seed, uint32_t chrom, uint32_t node, uint32_t step, uint32_t k) {
    return philox4x32_10(k, step, chrom, PL_IEV | (node << 8), (uint32_t)seed, (uint32_t)(seed >> 32));
}
JLP_HD U4 ins_col_block(uint64_t seed, uint32_t chrom, uint32_t id) {
    return philox4x32_10(id, 0u, chrom, PL_ICOL, (uint32_t)seed, (uint32_t)(seed >> 32));
}
JLP_HD U4 imut_block(uint64_t seed, uint32_t chrom, uint64_t id4, uint32_t node) {
    return philox4x32_10((uint32_t)id4, (uint32_t)(id4 >> 32), chrom, PL_IMUT | (node << 8), (uint32_t)seed, (uint32_t)(seed >> 32));
}
JLP_HD uint32_t imut_low(uint64_t seed, uint32_t chrom, uint64_t id, uint32_t node) {
    return philox4x32_10((uint32_t)id, (uint32_t)(id >> 32), chrom, PL_IMSLOW | (node << 8), (uint32_t)seed, (uint32_t)(seed >> 32)).w0;
}

// ---- exact restatements of the reference's uses of u = runif_01(x) ----

// bit length of a 128-bit value (hi:lo)
JLP_HD int bitlen128(uint64_t hi, uint64_t lo) {
#if defined(__CUDA_ARCH__)
    return hi ? 128 - __clzll((long long)hi) : (lo ? 64 - __clzll((long long)lo) : 0);
#else
    return hi ? 128 - __builtin_clzll(hi) : (lo ? 64 - __builtin_clzll(lo) : 0);
#endif
}

// Round the 128-bit integer (hi:lo) to 64 significant bits, ties to even -- what
// an x87 multiply/add does to an exact result.  Returns the rounded value as
// (hi:lo) again (it may gain one bit).
JLP_HD void round64(uint64_t& hi, uint64_t& lo) {
    int B = bitlen128(hi, lo);
    if (B <= 64) return;
    int d = B - 64;                      // low bits to drop; operands here keep d <= 40
    uint64_t q = (hi << (64 - d)) | (lo >> d);
    uint64_t rem = lo & ((1ull << d) - 1);
    uint64_t half = 1ull << (d - 1);
    if (rem > half || (rem == half && (q & 1))) {
        q++;
        if (q == 0) {                    // mantissa overflowed: value is 2^(64+d)
            hi = 1ull << d;
            lo = 0;
            return;
        }
    }
    hi = q >> (64 - d);
    lo = q << d;
}

// (uint64)(runif_01(x) * n) with the product formed in 80-bit long double
// (src/alias_sampler.h:55 die roll; src/hts_illumina.h:216 n=4, :254 n=3).
// y = x + 1 <= 2^64; product y*n/2^64 rounded to a 64-bit mantissa, then truncated.
JLP_HD uint64_t mul_floor_x87(uint64_t x, uint64_t n) {
    // P = (x + 1) * n as 128 bits
    uint64_t hi, lo;
#if defined(__CUDA_ARCH__)
    lo = x * n;
    hi = __umul64hi(x, n);
#else
    unsigned __int128 p = (unsigned __int128)x * n;
    lo = (uint64_t)p;
    hi = (uint64_t)(p >> 64);
#endif
    uint64_t lo2 = lo + n;
    hi += (lo2 < lo);
    lo = lo2;
    round64(hi, lo);
    return hi;                           // floor(P' / 2^64)
}

// (uint8)(runif_01(x) * 10 + 33)  (src/hts_illumina.h:238): two x87 roundings.
JLP_HD uint32_t nqual_x87(uint64_t x) {
    uint64_t hi, lo;
#if defined(__CUDA_ARCH__)
    lo = x * 10ull;
    hi = __umul64hi(x, 10ull);
#else
    unsigned __int128 p = (unsigned __int128)x * 10u;
    lo = (uint64_t)p;
    hi = (uint64_t)(p >> 64);
#endif
    uint64_t lo2 = lo + 10ull;
    hi += (lo2 < lo);
    lo = lo2;
    round64(hi, lo);                     // u * 10
    hi += 33;                            // + '!' (exact), then rounded again
    round64(hi, lo);
    return (uint32_t)(hi & 0xff);
}

// bases[(uint64)(runif_01(x) * 4.0)] index (src/hts_illumina.h:216): exact, 0..4
JLP_HD uint32_t ins_base_index(uint64_t x) {
    return x == ~0ull ? 4u : (uint32_t)((x + 1) >> 62);
}

}  // namespace jlp
#endif
