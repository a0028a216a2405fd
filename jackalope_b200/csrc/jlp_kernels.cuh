// Device-side data layout and kernel launchers (sm_100a).
#ifndef JLP_KERNELS_CUH
#define JLP_KERNELS_CUH

#include <cuda_runtime.h>
#include <stdint.h>

namespace jlp {

// One (haplotype, chromosome) group: the unit the reference exhausts read
// quotas by (src/hts_illumina.cpp:199-201, :505-528).
struct GroupDev {
    const uint8_t* seq;    // chromosome bases in HBM (byte per base)
    uint64_t len;
    uint32_t prefix_off;   // "@<genome>-<chrom>-" in the string pool
    uint32_t prefix_len;
    uint32_t bc_off;       // barcode in the string pool
    uint32_t bc_len;
};

// Everything scalar about one read end, written by the placement kernel (one
// thread per end), read by the read kernel (one warp per run of consecutive pairs).
struct EndPlan {
    const uint8_t* seg;    // first template base in HBM (chromosome + start)
    uint32_t S;            // template positions consumed, barcode included (adjust_chrom_spaces)
    uint16_t len;          // final read length
    uint8_t flags;         // bit 0 reverse strand, 1 insertions/deletions, 2 barcode, 3 ID line longer than 255 bytes, 4 > 2 indels
    uint8_t idlen;         // bytes of the ID line, '\n' included (when <= 255)
    uint32_t rec_len;      // FASTQ bytes of the record
    uint32_t group;
    uint32_t ev[2];        // the first two insertions / deletions of the read: template position | type << 16 (1 deletion,
                           // 2 insertion), ascending; 0xffffffff = none
};
static_assert(sizeof(EndPlan) == 32, "EndPlan layout");
constexpr uint32_t kPlanReverse = 1, kPlanIndels = 2, kPlanBarcode = 4, kPlanLongId = 8, kPlanManyEv = 16;   // ManyEv: more than two
constexpr uint32_t kPlanChunk = 8;      // pairs whose plans one bulk copy stages into shared memory

struct EndDev {
    const uint32_t* meta;    // [4*L] offset << 8 | n
    const uint64_t* entry64; // low word: (q_alias + 33) | (q_self + 33) << 8 | coin16 << 16; high word: mis16[q_self] | mis16[q_alias] << 16
    const uint64_t* coin;    // full thresholds (slow path)
    const uint64_t* mis;     // [256] full mismatch thresholds (slow path)
    uint32_t entry_n;
    uint32_t hA;             // high-16 gate of the indel draw: a field > hA is a plain base (0x10000 = never)
    uint64_t tA, tI;         // x >= tA: plain base; else x >= tI: deletion; else insertion
    uint32_t tA_all, tI_all; // threshold is 2^64 (never reached)
};

struct GenParams {
    uint64_t seed;
    uint32_t rk[20];         // Philox round keys of `seed`
    uint64_t job_lo, job_hi;
    uint64_t pool_pairs;
    uint64_t batch_lo;
    uint32_t batch_pairs;
    uint32_t n_ends;
    uint32_t L;
    uint32_t matepair;
    uint32_t dup_never;      // prob_dup threshold is 0
    uint32_t rec_buf;        // bytes of shared memory per (warp, end) output buffer: 16 + the longest record, rounded to 16
    uint32_t tpl_buf;        // bytes of shared memory per staged template window (multiple of 16)
    uint32_t cod_buf;        // bytes of shared memory per (warp, end) base-code line (multiple of 16)
    uint64_t c_dup;          // x < c_dup: duplicate of the previous fragment
    uint64_t c_rev;          // x < c_rev: reverse strand first
    EndDev end[2];
    const uint64_t* frag_cdf;
    const uint32_t* frag_guide;  // [257]
    uint32_t frag_n;
    uint32_t n_groups;
    uint64_t frag_min;
    const uint64_t* group_off;   // [n_groups + 1] pair-index prefix offsets
    const GroupDev* groups;
    const uint8_t* strpool;
    EndPlan* plan;               // [records]
    uint32_t* rec_len;           // [records] FASTQ bytes of each record (scan input)
    const uint32_t* rec_local;   // [records] exclusive prefix inside the scan block
    const uint64_t* block_base;  // [n_ends][n_scan_blocks] exclusive prefix of block totals
    uint32_t n_scan_blocks;
    uint8_t* out[2];             // FASTQ output of the batch, per file
    uint32_t* status;            // device error bits (1: barcode >= template)
};

// haplotype materialisation (HapChrom::get_chrom_full)
cudaError_t launch_materialize(const uint8_t* ref, uint64_t ref_size, uint64_t n_muts,
                               const uint64_t* old_pos, const uint64_t* new_pos,
                               const int64_t* size_mod, const uint64_t* nuc_off,
                               const uint8_t* pool, uint64_t chrom_size, uint8_t* out,
                               cudaStream_t s);

// create_genome: alias-sampled nucleotides of one chromosome, written straight into HBM
struct GenomeTables {
    uint32_t thr16[4];      // high 16 bits of the alias coin threshold per slot
    uint64_t thr[4];        // full thresholds
    uint32_t alias[4];
};
cudaError_t launch_create_chrom(uint8_t* out, uint64_t len, uint32_t chrom, uint64_t seed, const GenomeTables& t,
                                cudaStream_t s);

// create_haplotypes: substitutions along a tree (jlp_mutate.cu).  A warp owns a tile of kMutTile consecutive sites
// of one chromosome, a lane 4 consecutive sites per 128-site step; the states of the live internal nodes sit in
// shared memory, 2 bits per site, one byte per (slot, lane).
constexpr uint32_t kMutWarps = 8;                  // warps per CTA
constexpr uint32_t kMutSteps = 64;                 // 128-site steps per tile
constexpr uint32_t kMutTile = 128 * kMutSteps;     // sites per tile
constexpr uint32_t kMutSlots = 32;                 // node-state slots per lane
constexpr uint32_t kMutMaxTips = 4096;
constexpr uint32_t kMutMaxNodes = 65536;

struct MutNode {          // a non-root node in visiting order
    uint32_t node;        // index in the caller's preorder: addresses the draws
    uint32_t tab;         // its first threshold row: row = tab + 4 * category + parent state
    int32_t tip;          // tip index, or -1 for an internal node
    uint16_t pslot;       // slot holding the parent's states
    uint16_t slot;        // slot receiving this node's states (internal nodes)
};

struct MutParams {
    uint64_t seed;
    const uint8_t* genome;       // reference bases; chromosome c at chrom_off[c]
    const uint64_t* chrom_off;   // [n_chroms + 1]
    const uint32_t* tile0;       // [n_chroms + 1] first tile of each chromosome
    uint32_t n_chroms, n_tiles, n_tips, n_sched;
    const MutNode* sched;        // [n_sched]
    uint32_t n_cat;              // rate categories of the variable sites
    const uint64_t* cat_thr;     // [n_cat]: index = #{j : X_cat >= cat_thr[j]}; 0 = invariant, k = category k - 1
    const uint4* thr_hi;         // [rows] high words of the three thresholds of a row (.w unused)
    const uint4* thr_lo;         // [rows] low words
    uint32_t tab_rows;
    uint32_t tab_smem;           // 1: stage thr_hi in shared memory (thr_lo, read only on ties, stays in global memory)
    uint32_t* cnt;               // [n_tips][n_tiles]: pass 1 counts; after k_mut_scan each tile's first record in its region
    uint64_t* out;               // pass 2: the packed regions (HapChromHost::packed layout)
    const uint64_t* region;      // [n_tips][n_chroms] word offset of the region in `out`
    const uint64_t* region_n;    // [n_tips][n_chroms] records of the region
};
// pass 1 (write = false): records per (tip, tile) added into cnt; pass 2 (write = true): records written
cudaError_t launch_mutate(const MutParams& p, bool write, cudaStream_t s);
// exclusive scan of every (tip, chromosome) run of cnt in place; region_n receives the totals
cudaError_t launch_mut_scan(const MutParams& p, uint64_t* region_n, cudaStream_t s);
size_t mut_smem_bytes(uint32_t tab_rows);

// fragment placement + indel summary + record lengths, one thread per read end
cudaError_t launch_place(const GenParams& p, cudaStream_t s);

// record-offset scan: local exclusive prefixes + per-block totals, then the
// exclusive prefix of the totals (and the grand total per file in totals_out)
cudaError_t launch_scan(const uint32_t* rec_len, uint32_t n_records, uint32_t n_ends,
                        uint32_t* rec_local, uint64_t* block_tot, uint64_t* block_base,
                        uint64_t* totals_out, cudaStream_t s);

// template gather + quality/error model + FASTQ record assembly, one warp per pair;
// n_sm sizes the persistent grid
cudaError_t launch_reads(const GenParams& p, int n_sm, cudaStream_t s);
// false: the records of this read length do not fit the shared memory of an SM (rec_buf / tpl_buf must be set)
bool reads_fits(const GenParams& p);

constexpr uint32_t kScanBlock = 1024;

// BGZF on the device (jlp_bgzf.cu).  totals[0..1] hold the FASTQ bytes of the two files of a batch (device
// memory, as launch_scan leaves them); the compressed sizes come back in totals[2..3].  Block b of a file is
// compressed into slots + b * kBgzfSlot, then gathered to out + (sum of the sizes before it).  nblk_max sizes
// the grids: an upper bound of the blocks of either file.  `matches`: also look for length/distance pairs (a line's
// common prefix with the line four lines earlier); smaller output, more kernel time.  `codes`: kBgzfCodeBytes of
// device scratch of this launch's own (the Huffman codes of the two files, built from their first blocks).
constexpr uint32_t kBgzfIn = 0xff00;     // input bytes per block, htslib's BGZF_BLOCK_SIZE
constexpr uint32_t kBgzfSlot = 65536;    // a BGZF block never exceeds 64 KiB
constexpr uint32_t kBgzfCodeBytes = 4096;
constexpr int kBgzfLaunches = 5;         // kernels per launch_bgzf
cudaError_t bgzf_init();
cudaError_t launch_bgzf(const uint8_t* in0, const uint8_t* in1, uint64_t* totals, uint32_t nblk_max, bool matches, uint8_t* slots0,
                        uint8_t* slots1, uint32_t* zlen0, uint32_t* zlen1, uint64_t* zoff0, uint64_t* zoff1, uint8_t* out0,
                        uint8_t* out1, uint8_t* codes, cudaStream_t s);

}  // namespace jlp
#endif
