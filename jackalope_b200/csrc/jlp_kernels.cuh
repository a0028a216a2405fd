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

struct IndelRec;          // jlp_host.h

struct MutNode {          // a non-root node in visiting order
    uint32_t node;        // index in its tree's preorder: addresses the draws
    uint32_t tab;         // its first threshold row after the tree's: row = tab0 + tab + 4 * category + parent state
    int32_t tip;          // tip index, or -1 for an internal node
    uint16_t pslot;       // slot holding the parent's states
    uint16_t slot;        // slot receiving this node's states (internal nodes)
};

// A tile lies in one region (a run of sites that follows one tree): it starts at a multiple of 4 (one Philox block per
// lane and step) and decides only the sites in [lo, hi), the region.  A chromosome's tiles are contiguous and in
// position order.
struct MutTile {
    uint32_t chrom, first;       // chromosome, first site (a multiple of 4)
    uint32_t lo, hi;             // the region
    uint32_t sched0, n_sched;    // the region's tree: its schedule entries
    uint32_t tab0;               // the tree's first threshold row in its window's tables
    uint32_t pad;
};

struct MutParams {
    uint64_t seed;
    const uint8_t* genome;       // reference bases; chromosome c at chrom_off[c]
    const uint64_t* chrom_off;   // [n_chroms + 1]
    const uint32_t* tile0;       // [n_chroms + 1] first tile of each chromosome
    const MutTile* tiles;        // [n_tiles] (gene trees)
    uint32_t n_chroms, n_tiles, n_tips;
    uint32_t n_sched;            // one tree: its schedule entries
    uint32_t tile_begin, tile_end;   // the window: the tiles a launch covers
    const MutNode* sched;        // every tree's schedule, one after the other
    uint32_t n_cat;              // rate categories of the variable sites
    const uint64_t* cat_thr;     // [n_cat]: index = #{j : X_cat >= cat_thr[j]}; 0 = invariant, k = category k - 1
    const uint4* thr_hi;         // [rows] the window's tables: high words of the three thresholds of a row (.w unused)
    const uint4* thr_lo;         // [rows] low words
    uint32_t tab_rows;
    uint32_t tab_smem;           // 1: stage thr_hi in shared memory (thr_lo, read only on ties, stays in global memory)
    uint32_t* cnt;               // [n_tips][n_tiles]: pass 1 counts; after k_mut_scan each tile's first record in its region
    uint64_t* out;               // pass 2: the packed regions (HapChromHost::packed layout)
    const uint64_t* region;      // [n_tips][n_chroms] word offset of the region in `out`
    const uint64_t* region_n;    // [n_tips][n_chroms] records of the region
    // with indels only: cnt then counts the substitution records alone
    const IndelRec* irec;        // the indel records of every (tip, chromosome), by old_pos
    const uint64_t* ir_start;    // [n_tips * n_chroms + 1] first record of each (tip, chromosome)
    uint32_t* icur;              // [n_tips][n_tiles] the first record not yet passed by the tile's warp
    uint64_t* ir_nuc;            // pass 2: each indel record's nuc_off (where k_ins_walk puts its inserted bases)
};
// pass 1 (write = false): records per (tip, tile) added into cnt; pass 2 (write = true): records written.
// indels: the tips' records follow p.irec (substitutions at live, non-anchor columns; the indel records themselves)
// gtrees: each tile's region, schedule and table rows from p.tiles; otherwise one tree, one region per chromosome
cudaError_t launch_mutate(const MutParams& p, bool write, bool indels, bool gtrees, cudaStream_t s);

// The inserted columns' walk: one thread per column from its birth node through the schedule interval of its subtree
// (state at birth drawn from pi, then the same P rows as a reference site); its tip states go into the insertion
// records' pools.
struct InsCol {
    uint32_t chrom, id;
    uint32_t n0, n1;             // schedule index of the birth node, end of its subtree's interval (n0 == n1: no tip below)
    uint64_t e0, e1;             // its entries
};
struct InsEnt {                  // the column is live at the tip of schedule entry `sched`, byte k of indel record ir
    uint32_t sched, k;
    uint64_t region;             // tip * n_chroms + chromosome
    uint64_t ir;
};
struct InsParams {
    uint64_t seed;
    uint32_t n_cols, n_cat;
    const InsCol* cols;
    const InsEnt* ent;
    const MutNode* sched;
    const uint64_t* cat_thr;
    uint64_t pi_thr[3];
    const uint4* thr_hi;
    const uint4* thr_lo;
    uint64_t* out;
    const uint64_t* region;
    const uint64_t* region_n;
    const uint64_t* ir_nuc;
};
cudaError_t launch_ins_walk(const InsParams& p, cudaStream_t s);
// exclusive scan of every (tip, chromosome) run of cnt in place; region_n receives the totals
cudaError_t launch_mut_scan(const MutParams& p, uint64_t* region_n, cudaStream_t s);
size_t mut_smem_bytes(uint32_t tab_rows);

// The threshold tables on the device (k_mut_tables): per item P = expm(Q t) and the thresholds of its four rows into
// rows row .. row + 3 of hi / lo, bit for bit what transition_matrix + row_thresholds give on the host, except for the
// items the kernel lists in flag[0 .. *n_flag) (the scaling exponent the host's log2 might round differently, or a
// norm that is not finite), which the caller recomputes on the host.  P_out (may be NULL): P of item i at 16 i.
struct TabItem {
    double t;
    uint32_t row, pad;
};
struct TabQ {
    double q[16];
};
cudaError_t launch_mut_tables(const TabItem* items, uint32_t n, const TabQ& Q, uint4* hi, uint4* lo, double* P_out,
                              uint32_t* n_flag, uint32_t* flag, cudaStream_t s);

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

// write_vcf (jlp_vcf.cu, DESIGN.md section 11), one chromosome at a time.  The records of the included haplotypes are
// numbered haplotype-major; their packed arrays (HapChromHost::packed layout) sit in `recs`.
struct VcfHap {
    uint64_t woff;               // word offset of the haplotype's packed records in recs
    uint32_t n, rec0;            // its records, and the number of its first one
};
struct VcfCar {                  // a haplotype with records in a line (a carrier)
    uint64_t new_s, len;         // where its allele starts in the haplotype, and its length
    uint64_t key;                // the allele's first min(len, 8) bytes
    uint32_t u, i0, i1;          // included haplotype; its first and last record of the line
    uint32_t idx;                // its allele index (0: REF)
};
struct VcfChrom {
    const uint64_t* recs;
    const VcfHap* hap;           // [n_hap + 1] included haplotypes (rec0 of the last entry = n_rec)
    uint32_t n_hap, n_rec;
    const uint8_t* ref;          // the chromosome's reference bases
    uint64_t L;
    const uint8_t* name;         // the chromosome's name
    uint32_t name_len;
    uint32_t ploidy, n_samples;
    const uint32_t* slot_hap;    // [n_samples * ploidy] included haplotype of each slot of the sample matrix
    const uint32_t* first_slot;  // [n_hap] its first slot
    const uint32_t* n_slots;     // [n_hap] the slots it fills
    // [n_rec] per record, in record order and in sorted order
    uint64_t *start, *end, *start_sorted, *end_sorted, *maxend, *key2, *key2_sorted;
    uint32_t *rec_hap, *val, *order, *flag, *lid;
    // [n_rec] per position of the line-sorted order: the line's carriers, alleles classes and ALTs start at line_first
    VcfCar* car;
    uint32_t *car_pos, *cls_car, *cls_slot, *cls_rank, *alt_car;
    // [n_rec + 1] per line
    uint32_t *line_first, *n_car, *n_alt;
    uint64_t *line_s, *line_e, *line_len, *line_end;   // line_end: inclusive prefix of line_len
    uint32_t* hidx;              // [warps of the line kernels][n_hap], zero between lines
    uint8_t* cub_tmp;
    size_t cub_bytes;
};
size_t vcf_cub_bytes(uint32_t n_rec);
unsigned vcf_line_blocks(uint64_t n_lines, int n_sm);     // CTAs of 8 warps of the line kernels
// spans, sort by start, running maximum of the ends, line flags and their inclusive prefix (lid[n_rec - 1] = lines)
cudaError_t launch_vcf_spans(const VcfChrom& v, cudaStream_t s);
// line extents, the line-major sort, k_vcf_lines<false> (carriers, alleles, text lengths) and line_end
cudaError_t launch_vcf_size(const VcfChrom& v, uint32_t n_lines, int n_sm, cudaStream_t s);
// the text of lines [l0, l1) into out + out_skip
cudaError_t launch_vcf_text(const VcfChrom& v, uint32_t l0, uint32_t l1, uint8_t* out, uint64_t out_skip, int n_sm,
                            cudaStream_t s);

// haps_vcf: haplotypes read from a VCF file (jlp_vcf_read.cu, DESIGN.md section 12).  A batch of whole lines is parsed
// on the device; its lines' alleles and non-REF calls go to the chromosome they belong to, and once a chromosome's lines
// are all seen its calls are sorted by haplotype slot (sample * kVrMaxPloidy + copy) and walked into records.
constexpr uint32_t kVrMaxPloidy = 8;
constexpr uint32_t kVrNone = 0xffffffffu;
// the reasons a line is rejected, in the order its checks are made; the status word keeps min(line << 8 | reason)
enum VrReason : uint32_t {
    VR_COLUMNS = 1, VR_CHROM, VR_POS, VR_REF_LETTERS, VR_REF_RANGE, VR_REF_DIFF, VR_ALT, VR_FORMAT, VR_GT, VR_PLOIDY,
    VR_INDEX, VR_CONTIG, VR_ORDER
};
enum VrKind : uint32_t { VR_SEQ = 0, VR_STAR = 1, VR_SYM = 2 };
struct VrLine {
    uint32_t chrom;              // kVrNone: a fixed column is malformed
    uint32_t s, m;               // POS - 1, len(REF)
    uint32_t alt_at, alt_len;    // the ALT field in the batch
    uint32_t gt_at;              // the first sample field in the batch
    uint32_t n_alt;
    uint32_t sv_info;            // INFO has an END or SVLEN key
};
struct VrAllele {                // one ALT entry of a line
    uint32_t s, m, n;            // the span it replaces and its length
    uint32_t kind;
    uint64_t text;               // its bytes in the batch's (then the chromosome's) allele text
    uint32_t nrec, pool;         // records and pool bytes of its encoding
};
struct VrSlot {                  // one haplotype slot of a chromosome, from the walk
    unsigned long long nrec, pool, applied, skipped;
    long long delta;
};
struct VrBatch {
    const uint8_t* text;
    uint32_t n_bytes, n_lines;   // the batch ends with '\n'
    uint64_t line0;              // data-line index of its first line
    const uint8_t* genome;       // the resident reference and its chromosomes' offsets
    const uint64_t* chrom_off;
    const uint8_t* names;        // reference chromosome names, sorted bytewise: name_off[k]..name_off[k+1], index name_idx[k]
    const uint32_t* name_off;
    const uint32_t* name_idx;
    uint32_t n_chroms, n_cols, n_samples;
    uint32_t prev_chrom, prev_s; // the line before the batch (prev_chrom kVrNone: none)
    uint32_t* nl;                // [n_lines] newline positions
    VrLine* line;
    uint32_t *n_alt, *alt0, *alt_len, *text0, *n_calls, *call0;   // per line, and their exclusive prefixes
    VrAllele* allele;
    uint8_t* alt_text;
    uint32_t *call_slot, *call_allele;
    uint32_t* ploidy;            // [n_samples] largest allele count of a GT, over the file
    unsigned long long* counts;  // missing, symbolic calls
    unsigned long long* status;  // min(data line << 8 | reason)
    uint8_t* run_flag;
    uint64_t *run_key, *runs;    // line << 32 | chromosome where a line's chromosome differs from the line's before
    uint32_t* n_sel;             // DeviceSelect's count
};
// CUB scratch for any of the calls below over n items
size_t vr_cub_bytes(uint64_t n);
// stage 0: newline positions (n_lines in *n_sel).  1: the fixed columns and the prefixes alt0 / text0 ([n_lines + 1]).
// 2: the alleles and their text, the GT count pass and call0.  3: the calls, and the runs of lines of one chromosome
// (their count in *n_sel).  The host sizes the buffers of a stage from the totals of the one before.
cudaError_t launch_vr_parse(const VrBatch& b, int stage, uint8_t* tmp, size_t tmp_bytes, cudaStream_t s);
// the alleles [a0, a1) and calls [c0, c1) of a batch (lines [l0, l1) with t0 = text0[l0]) appended to a chromosome that
// holds n_alleles alleles and text_bytes of allele text; the text itself is copied by the caller
cudaError_t launch_vr_append(const VrBatch& b, uint32_t a0, uint32_t a1, uint32_t c0, uint32_t c1, uint32_t t0,
                             uint64_t n_alleles, uint64_t n_calls, uint64_t text_bytes, VrAllele* allele, uint32_t* slot,
                             uint32_t* val, cudaStream_t s);
struct VrChrom {
    const VrAllele* allele;
    const uint8_t* text;
    const uint8_t* ref;          // the chromosome's reference bases
    uint32_t *slot, *val, *slot2, *val2;    // [n_calls] line-major, then sorted by slot
    uint64_t n_calls;
    uint32_t n_slots;
    uint64_t* seg;               // [2 * n_slots] each slot's calls in the sorted order
    VrSlot* out_slot;
    const uint64_t* region;      // [n_slots] word offset of each slot's records in out
    uint64_t* out;
};
// the calls sorted by slot (stable: file order within a slot) and each slot's range, then the walk's count pass
cudaError_t launch_vr_count(const VrChrom& v, uint8_t* tmp, size_t tmp_bytes, cudaStream_t s);
cudaError_t launch_vr_write(const VrChrom& v, cudaStream_t s);

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
