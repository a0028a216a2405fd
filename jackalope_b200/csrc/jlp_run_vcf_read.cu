// The VCF reader (jlp_create_haplotypes_vcf, DESIGN.md section 12), on the first device of the context.
#include "jlp_ctx.h"

#include <zlib.h>

#include <sys/stat.h>

#include <cstdio>
#include <cstring>
#include <future>

using namespace jlp;

namespace {

constexpr uint64_t kDefaultBatch = 256ull << 20;
constexpr uint64_t kMaxBatch = (1ull << 31) - (1ull << 20);   // batch offsets are 32 bits wide, and CUB's counts signed
constexpr uint64_t kMaxHaps = 1ull << 16;

const char* const kReason[] = {
    "", "the number of columns differs from the #CHROM line", "CHROM is not a reference chromosome",
    "POS is not an integer >= 1", "REF is not letters", "REF reaches past the end of the chromosome",
    "REF differs from the reference", "ALT is not '.' or a list of letters, '*', or symbolic or breakend alleles",
    "FORMAT does not start with GT", "GT is not alleles separated by '|' or '/'", "GT has more than 8 alleles",
    "an allele index is above the ALT count", "the lines of a chromosome are not contiguous", "POS decreases",
};

[[noreturn]] void bad_line(uint64_t line, const char* reason) {
    throw ArgErr("line " + std::to_string(line) + ": " + reason);
}

// The file's text in order: plain bytes, one gzip stream (members one after the other), or BGZF, whose members are
// inflated on n_threads threads at once.
class Source {
  public:
    Source(const char* path, unsigned n_threads) : threads_(n_threads) {
        f_ = std::fopen(path, "rb");
        if (!f_) throw IoErr(std::string("cannot open ") + path);
        struct stat st;
        if (fstat(fileno(f_), &st) == 0 && S_ISREG(st.st_mode)) size_ = (uint64_t)st.st_size;
        more(18);
        if (in_.size() >= 2 && in_[0] == 0x1f && in_[1] == 0x8b) {
            kind_ = member_size(0) ? BGZF : GZIP;
            if (kind_ == GZIP) {
                std::memset(&z_, 0, sizeof z_);
                if (inflateInit2(&z_, 15 + 16) != Z_OK) throw IoErr("zlib cannot be initialised");
                z_live_ = true;
            }
        }
    }
    ~Source() {
        if (z_live_) inflateEnd(&z_);
        if (f_) std::fclose(f_);
    }
    bool eof() const { return done_; }
    // the file's size when it is plain text, else 0
    uint64_t plain_size() const { return kind_ == PLAIN ? size_ : 0; }

    // up to cap bytes of text into dst (BGZF: whole members only, so fewer when the next one does not fit)
    uint64_t fill(uint8_t* dst, uint64_t cap) {
        if (done_) return 0;
        if (kind_ == PLAIN) {
            uint64_t n = std::min<uint64_t>(cap, in_.size() - pos_);
            std::memcpy(dst, in_.data() + pos_, n);
            pos_ += n;
            if (n < cap) n += std::fread(dst + n, 1, cap - n, f_);
            if (n < cap) {
                if (std::ferror(f_)) throw IoErr("the file cannot be read");
                done_ = true;
            }
            return n;
        }
        return kind_ == GZIP ? fill_gzip(dst, cap) : fill_bgzf(dst, cap);
    }

  private:
    enum Kind { PLAIN, GZIP, BGZF };
    FILE* f_ = nullptr;
    Kind kind_ = PLAIN;
    unsigned threads_;
    std::vector<uint8_t> in_;     // compressed bytes read, from pos_ on not used yet
    size_t pos_ = 0;
    bool file_end_ = false, done_ = false;
    uint64_t size_ = 0;
    z_stream z_;
    bool z_live_ = false;

    // at least `want` unused bytes in in_ unless the file ends
    void more(size_t want) {
        if (in_.size() - pos_ >= want || file_end_) return;
        in_.erase(in_.begin(), in_.begin() + pos_);
        pos_ = 0;
        const size_t have = in_.size(), get = std::max<size_t>(want - have, 1 << 20);
        in_.resize(have + get);
        const size_t n = std::fread(in_.data() + have, 1, get, f_);
        if (n < get && std::ferror(f_)) throw IoErr("the file cannot be read");
        in_.resize(have + n);
        if (n < get) file_end_ = true;
    }
    // the size of the BGZF member at pos_ + at (its header holds BSIZE), 0 if the bytes there are not one
    size_t member_size(size_t at) const {
        const uint8_t* h = in_.data() + pos_ + at;
        if (in_.size() - pos_ - at < 18 || h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return 0;
        const size_t xlen = h[10] | h[11] << 8;
        if (in_.size() - pos_ - at < 12 + xlen) return 0;
        for (size_t k = 12; k + 4 <= 12 + xlen;) {
            const size_t slen = h[k + 2] | h[k + 3] << 8;
            if (h[k] == 'B' && h[k + 1] == 'C' && slen == 2 && k + 6 <= 12 + xlen) return (size_t)(h[k + 4] | h[k + 5] << 8) + 1;
            k += 4 + slen;
        }
        return 0;
    }
    uint64_t fill_gzip(uint8_t* dst, uint64_t cap) {
        z_.next_out = dst;
        z_.avail_out = (uInt)std::min<uint64_t>(cap, 1u << 30);
        const uint64_t want = z_.avail_out;
        while (z_.avail_out) {
            more(1);
            if (pos_ == in_.size()) {
                if (z_live_ && z_.total_in) throw IoErr("the gzip stream is truncated");
                done_ = true;
                break;
            }
            z_.next_in = in_.data() + pos_;
            z_.avail_in = (uInt)(in_.size() - pos_);
            const int r = inflate(&z_, Z_NO_FLUSH);
            pos_ = in_.size() - z_.avail_in;
            if (r == Z_STREAM_END) {
                inflateReset(&z_);          // another member may follow
                z_.total_in = 0;
                more(1);
                if (pos_ == in_.size()) { done_ = true; break; }
            } else if (r != Z_OK && r != Z_BUF_ERROR) {
                throw IoErr("the gzip stream cannot be inflated");
            }
        }
        return want - z_.avail_out;
    }
    uint64_t fill_bgzf(uint8_t* dst, uint64_t cap) {
        struct Member { size_t at, len; uint64_t out; uint32_t isize; };
        std::vector<Member> ms;
        uint64_t total = 0;
        size_t at = 0;
        while (true) {
            more(at + 18);
            if (pos_ + at == in_.size()) break;
            const size_t len = member_size(at);
            if (!len) throw IoErr("the BGZF file has a damaged member");
            more(at + len);
            if (in_.size() - pos_ - at < len) throw IoErr("the BGZF file is truncated");
            const uint8_t* t = in_.data() + pos_ + at + len - 4;
            const uint32_t isize = t[0] | t[1] << 8 | t[2] << 16 | (uint32_t)t[3] << 24;
            if (isize > (1u << 16)) throw IoErr("the BGZF file has a damaged member");
            if (total + isize > cap) break;
            ms.push_back(Member{at, len, total, isize});
            total += isize;
            at += len;
            if (ms.size() >= 4096) break;
        }
        const uint8_t* base = in_.data() + pos_;
        parallel_for(ms.size(), std::min<unsigned>(threads_, (unsigned)ms.size()), [&](uint64_t k) {
            const Member& m = ms[k];
            const uint8_t* h = base + m.at;
            const size_t hl = 12 + (h[10] | h[11] << 8);
            if (m.len < hl + 8) throw IoErr("the BGZF file has a damaged member");
            z_stream z;
            std::memset(&z, 0, sizeof z);
            if (inflateInit2(&z, -15) != Z_OK) throw IoErr("zlib cannot be initialised");
            z.next_in = const_cast<uint8_t*>(h + hl);
            z.avail_in = (uInt)(m.len - hl - 8);
            z.next_out = dst + m.out;
            z.avail_out = m.isize;
            const int r = inflate(&z, Z_FINISH);
            const bool ok = r == Z_STREAM_END && z.avail_out == 0;
            inflateEnd(&z);
            const uint8_t* t = h + m.len - 8;
            const uint32_t crc = t[0] | t[1] << 8 | t[2] << 16 | (uint32_t)t[3] << 24;
            if (!ok || crc32(0, dst + m.out, m.isize) != crc) throw IoErr("a BGZF member cannot be inflated");
        });
        pos_ += at;
        if (ms.empty() && pos_ == in_.size()) done_ = true;
        return total;
    }
};

// Batches of whole lines, each in a pinned buffer: the text after the last newline waits for the next batch, a line
// longer than the batch grows the buffer, and the last line of the file gets a newline when it has none.
class Feed {
  public:
    // a plain file smaller than a batch gets buffers of its own size
    Feed(Source& src, uint64_t batch) : src_(src), batch_(src.plain_size() ? std::min(batch, src.plain_size()) : batch) {}
    double inflate_ms = 0;
    uint64_t text_bytes = 0;

    uint64_t next(PinBuf<uint8_t>& buf) {
        const auto t0 = std::chrono::steady_clock::now();
        const uint64_t n = cut(buf);
        inflate_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        return n;
    }

  private:
    Source& src_;
    uint64_t batch_;
    std::vector<uint8_t> carry_;

    uint64_t cut(PinBuf<uint8_t>& buf) {
        uint64_t want = batch_;
        while (true) {
            // room for the text carried over (a long line's start can be longer than a batch), a batch, one BGZF member
            // and a final newline
            const uint64_t need = std::max<uint64_t>(want, carry_.size()) + (1u << 16) + 1;
            if (buf.n < need) {
                PinBuf<uint8_t> x;
                x.ensure(need);
                std::swap(buf.p, x.p);
                std::swap(buf.n, x.n);
            }
            const uint64_t lim = std::min<uint64_t>(buf.n - 1, kMaxBatch - 1);   // room for a final newline
            uint64_t n = carry_.size();
            std::memcpy(buf.p, carry_.data(), n);
            while (n < want && !src_.eof()) {
                uint64_t got = src_.fill(buf.p + n, want - n);
                if (!got && !src_.eof()) got = src_.fill(buf.p + n, lim - n);     // a BGZF member longer than the rest
                text_bytes += got;
                n += got;
                if (!got && !src_.eof()) break;         // the next BGZF member does not fit at all
            }
            uint64_t j = n;
            while (j > 0 && buf.p[j - 1] != '\n') j--;
            if (j > 0 && !(src_.eof() && j < n)) {
                carry_.assign(buf.p + j, buf.p + n);
                return j;
            }
            if (src_.eof()) {
                carry_.clear();
                if (n && buf.p[n - 1] != '\n') buf.p[n++] = '\n';
                return n;
            }
            // no newline yet: the line is longer than the batch
            if (n >= kMaxBatch - 1) throw ArgErr("a line of 2 GiB or more");
            carry_.assign(buf.p, buf.p + n);
            want = std::min(std::max(want * 2, n + (1u << 20)), kMaxBatch - 1);
        }
    }
};

// a device array that keeps its first `used` elements when it grows
template <typename T> void grow(DevBuf<T>& b, uint64_t used, uint64_t need, cudaStream_t s) {
    if (need <= b.n) return;
    DevBuf<T> x;
    x.ensure(std::max<uint64_t>(need, b.n * 2));
    if (used) CK(cudaMemcpyAsync(x.p, b.p, used * sizeof(T), cudaMemcpyDeviceToDevice, s));
    CK(cudaStreamSynchronize(s));
    std::swap(b.p, x.p);
    std::swap(b.n, x.n);
}

// n values from the device, in the order of stream s: the context's streams do not synchronise with the legacy stream
template <typename T> void read_back(T* out, const T* p, uint64_t n, cudaStream_t s) {
    if (!n) return;
    CK(cudaMemcpyAsync(out, p, n * sizeof(T), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
}

struct EventPair {
    cudaEvent_t a = nullptr, b = nullptr;
    EventPair() { CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b)); }
    ~EventPair() { cudaEventDestroy(a); cudaEventDestroy(b); }
};

// What the reader keeps across batches.
struct Reader {
    jlp_ctx* c;
    Device& d;
    cudaStream_t s;
    uint64_t nc;
    std::vector<uint64_t> len;
    uint32_t n_cols = 0, n_samples = 0;
    std::vector<std::string> samples;
    uint64_t header_lines = 0;
    // the batch's device buffers
    DevBuf<uint8_t> text[2], alt_text, tmp, run_flag, names;
    DevBuf<uint32_t> nl, n_alt, alt0, alt_len, text0, n_calls, call0, call_slot, call_allele, ploidy, n_sel, name_off, name_idx;
    DevBuf<uint64_t> run_key, runs, chrom_off;
    DevBuf<VrLine> line;
    DevBuf<VrAllele> allele;
    DevBuf<unsigned long long> counts, status;   // missing, symbolic; status
    // the open chromosome's alleles, text and calls
    uint32_t open = kVrNone;
    uint64_t open_lines = 0, acc_alleles = 0, acc_text = 0, acc_calls = 0;
    DevBuf<VrAllele> acc_allele;
    DevBuf<uint8_t> acc_txt;
    DevBuf<uint32_t> acc_slot, acc_val, slot2, val2;
    DevBuf<uint64_t> seg, region;
    DevBuf<VrSlot> slots;
    std::vector<char> done;
    // per built chromosome: its records and each slot's figures and region
    std::vector<std::unique_ptr<DevBuf<uint64_t>>> out;
    std::vector<std::vector<VrSlot>> chrom_slot;
    std::vector<std::vector<uint64_t>> chrom_region;
    uint32_t prev_chrom = kVrNone, prev_s = 0;
    uint64_t lines = 0;
    // the parsed batch hand() takes next
    struct Seg { uint32_t l0, l1, chrom; };
    std::vector<Seg> segs_;
    VrBatch view_{};
    float parse_ms = 0, build_ms = 0;
    EventPair ev;

    Reader(jlp_ctx* c_, Device& d_) : c(c_), d(d_), s(d_.s_compute) {}

    template <typename T> T read_one(const T* p) {
        T v;
        read_back(&v, p, 1, s);
        return v;
    }

    void tmp_for(uint64_t n) {
        const size_t b = vr_cub_bytes(n);
        if (tmp.n < b) tmp.ensure(b);
    }

    // the ## lines and the #CHROM line at the start of the file; returns the bytes of t[0, n) they take (all of them when
    // the header goes on in the next batch)
    uint64_t header(const uint8_t* t, uint64_t n, bool& found) {
        uint64_t a = 0;
        while (a < n) {
            uint64_t e = a;
            while (t[e] != '\n') e++;
            header_lines++;
            const std::string ln(reinterpret_cast<const char*>(t + a), e - a - (e > a && t[e - 1] == '\r'));
            a = e + 1;
            if (ln.compare(0, 2, "##") == 0) continue;
            if (ln.compare(0, 6, "#CHROM") != 0) bad_line(header_lines, "no #CHROM line before the data");
            std::vector<std::string> col;
            for (size_t p = 0;;) {
                const size_t q = ln.find('\t', p);
                col.push_back(ln.substr(p, q == std::string::npos ? std::string::npos : q - p));
                if (q == std::string::npos) break;
                p = q + 1;
            }
            if (col.size() < 10 || col[8] != "FORMAT") bad_line(header_lines, "the #CHROM line needs 10 or more columns, FORMAT the 9th");
            samples.assign(col.begin() + 9, col.end());
            std::vector<std::string> sorted = samples;
            std::sort(sorted.begin(), sorted.end());
            bool ok = std::adjacent_find(sorted.begin(), sorted.end()) == sorted.end();
            for (const std::string& x : samples) ok &= !x.empty() && x.find_first_of(" \t\r\n\v\f") == std::string::npos;
            if (!ok) bad_line(header_lines, "sample names must be unique and contain no whitespace");
            if (samples.size() > kMaxHaps) bad_line(header_lines, "more than 65536 haplotypes");
            n_cols = (uint32_t)col.size();
            n_samples = (uint32_t)samples.size();
            found = true;
            return a;
        }
        return n;
    }

    void start() {
        nc = len.size();
        done.assign(nc, 0);
        out.resize(nc);
        chrom_slot.resize(nc);
        chrom_region.resize(nc);
        std::vector<uint32_t> idx(nc);
        for (uint32_t k = 0; k < nc; k++) idx[k] = k;
        std::sort(idx.begin(), idx.end(), [&](uint32_t x, uint32_t y) { return c->chrom_names[x] < c->chrom_names[y]; });
        std::vector<uint8_t> nb;
        std::vector<uint32_t> off{0};
        for (uint32_t k : idx) {
            nb.insert(nb.end(), c->chrom_names[k].begin(), c->chrom_names[k].end());
            off.push_back((uint32_t)nb.size());
        }
        names.upload(nb, s);
        name_off.upload(off, s);
        name_idx.upload(idx, s);
        chrom_off.upload(c->chrom_off, s);
        ploidy.ensure(n_samples);
        counts.ensure(2);
        status.ensure(1);
        n_sel.ensure(1);
        if (n_samples) CK(cudaMemsetAsync(ploidy.p, 0, n_samples * 4, s));
        CK(cudaMemsetAsync(counts.p, 0, 16, s));
        CK(cudaMemsetAsync(status.p, 0xff, 8, s));
        CK(cudaStreamSynchronize(s));
    }

    VrBatch batch_view(const uint8_t* dtext, uint32_t n_bytes, uint32_t n_lines) {
        VrBatch b{};
        b.text = dtext; b.n_bytes = n_bytes; b.n_lines = n_lines; b.line0 = lines;
        b.genome = d.genome.p + kPad; b.chrom_off = chrom_off.p;
        b.names = names.p; b.name_off = name_off.p; b.name_idx = name_idx.p;
        b.n_chroms = (uint32_t)nc; b.n_cols = n_cols; b.n_samples = n_samples;
        b.prev_chrom = prev_chrom; b.prev_s = prev_s;
        b.nl = nl.p; b.line = line.p;
        b.n_alt = n_alt.p; b.alt0 = alt0.p; b.alt_len = alt_len.p; b.text0 = text0.p; b.n_calls = n_calls.p; b.call0 = call0.p;
        b.allele = allele.p; b.alt_text = alt_text.p; b.call_slot = call_slot.p; b.call_allele = call_allele.p;
        b.ploidy = ploidy.p; b.counts = counts.p; b.status = status.p;
        b.run_flag = run_flag.p; b.run_key = run_key.p; b.runs = runs.p; b.n_sel = n_sel.p;
        return b;
    }

    // one batch of data lines, resident at dtext: parsed and checked; false if it has no lines.  hand() then gives its
    // lines to their chromosomes.
    bool parse(const uint8_t* dtext, uint32_t n_bytes) {
        tmp_for((uint64_t)n_bytes + 1);
        nl.ensure(n_bytes);
        VrBatch b = batch_view(dtext, n_bytes, 0);
        CK(cudaEventRecord(ev.a, s));
        CK(launch_vr_parse(b, 0, tmp.p, tmp.n, s));
        const uint32_t n_lines = read_one(n_sel.p);
        if (n_lines == 0) return false;
        const uint64_t n1 = (uint64_t)n_lines + 1;
        line.ensure(n1); n_alt.ensure(n1); alt0.ensure(n1); alt_len.ensure(n1); text0.ensure(n1); n_calls.ensure(n1);
        call0.ensure(n1); run_flag.ensure(n1); run_key.ensure(n1); runs.ensure(n1);
        b = batch_view(dtext, n_bytes, n_lines);
        CK(launch_vr_parse(b, 1, tmp.p, tmp.n, s));
        const uint32_t n_all = read_one(alt0.p + n_lines), n_txt = read_one(text0.p + n_lines);
        allele.ensure(n_all); alt_text.ensure(n_txt);
        b = batch_view(dtext, n_bytes, n_lines);
        CK(launch_vr_parse(b, 2, tmp.p, tmp.n, s));
        const uint32_t n_cl = read_one(call0.p + n_lines);
        call_slot.ensure(n_cl); call_allele.ensure(n_cl);
        b = batch_view(dtext, n_bytes, n_lines);
        CK(launch_vr_parse(b, 3, tmp.p, tmp.n, s));
        CK(cudaEventRecord(ev.b, s));
        CK(cudaStreamSynchronize(s));
        parse_ms += elapsed_ms(ev.a, ev.b);
        const uint32_t n_runs = read_one(n_sel.p);
        std::vector<uint64_t> run(n_runs);
        read_back(run.data(), runs.p, n_runs, s);
        // the runs of lines of one chromosome: the first continues the chromosome before the batch when it starts later
        std::vector<Seg>& segs = segs_;
        segs.clear();
        if (n_runs == 0 || (run[0] >> 32) != 0) segs.push_back(Seg{0, n_runs ? (uint32_t)(run[0] >> 32) : n_lines, prev_chrom});
        for (uint32_t k = 0; k < n_runs; k++)
            segs.push_back(Seg{(uint32_t)(run[k] >> 32), k + 1 < n_runs ? (uint32_t)(run[k + 1] >> 32) : n_lines, (uint32_t)run[k]});
        // the first malformed line: the device's, or a chromosome whose lines resume after another's
        uint64_t bad = read_one(status.p);
        uint32_t cur = open;
        std::vector<char> seen = done;
        for (const Seg& g : segs) {
            if (g.chrom == kVrNone || g.chrom == cur) continue;
            if (cur != kVrNone) seen[cur] = 1;
            if (seen[g.chrom]) {
                bad = std::min<uint64_t>(bad, (lines + g.l0) << 8 | VR_CONTIG);
                break;
            }
            cur = g.chrom;
        }
        if (bad != ~0ull) bad_line(header_lines + (bad >> 8) + 1, kReason[std::min<uint64_t>(bad & 0xff, VR_ORDER)]);
        view_ = b;
        return true;
    }

    void hand() {
        for (const Seg& g : segs_) append(view_, g.l0, g.l1, g.chrom);
        const VrLine last = read_one(line.p + view_.n_lines - 1);
        prev_chrom = last.chrom;
        prev_s = last.s;
        lines += view_.n_lines;
    }

    void append(const VrBatch& b, uint32_t l0, uint32_t l1, uint32_t chrom) {
        if (l1 <= l0) return;
        if (chrom != open) {
            if (open != kVrNone) build();
            open = chrom;
            open_lines = 0;
        }
        open_lines += l1 - l0;
        if (open_lines >> 32) throw ArgErr("2^32 or more lines of one chromosome");
        const uint32_t a0 = read_one(alt0.p + l0), a1 = read_one(alt0.p + l1);
        const uint32_t t0 = read_one(text0.p + l0), t1 = read_one(text0.p + l1);
        const uint32_t c0 = read_one(call0.p + l0), c1 = read_one(call0.p + l1);
        if (acc_alleles + (a1 - a0) >= (1ull << 32)) throw ArgErr("2^32 or more alleles of one chromosome");
        grow(acc_allele, acc_alleles, acc_alleles + (a1 - a0), s);
        grow(acc_txt, acc_text, acc_text + (t1 - t0), s);
        grow(acc_slot, acc_calls, acc_calls + (c1 - c0), s);
        grow(acc_val, acc_calls, acc_calls + (c1 - c0), s);
        if (t1 > t0) CK(cudaMemcpyAsync(acc_txt.p + acc_text, alt_text.p + t0, t1 - t0, cudaMemcpyDeviceToDevice, s));
        CK(launch_vr_append(b, a0, a1, c0, c1, t0, acc_alleles, acc_calls, acc_text, acc_allele.p, acc_slot.p, acc_val.p, s));
        acc_alleles += a1 - a0;
        acc_text += t1 - t0;
        acc_calls += c1 - c0;
    }

    // the open chromosome's records: calls sorted by slot, the walk's count pass, the regions, the write pass
    void build() {
        const uint32_t ch = open;
        const uint32_t n_slots = n_samples * kVrMaxPloidy;
        slot2.ensure(acc_calls); val2.ensure(acc_calls);
        seg.ensure(2 * (uint64_t)n_slots); slots.ensure(n_slots); region.ensure(n_slots);
        tmp_for(acc_calls);
        VrChrom v{};
        v.allele = acc_allele.p; v.text = acc_txt.p; v.ref = d.genome.p + kPad + c->chrom_off[ch];
        v.slot = acc_slot.p; v.val = acc_val.p; v.slot2 = slot2.p; v.val2 = val2.p;
        v.n_calls = acc_calls; v.n_slots = n_slots; v.seg = seg.p; v.out_slot = slots.p; v.region = region.p;
        CK(cudaEventRecord(ev.a, s));
        CK(launch_vr_count(v, tmp.p, tmp.n, s));
        CK(cudaEventRecord(ev.b, s));
        std::vector<VrSlot>& S = chrom_slot[ch];
        S.resize(n_slots);
        CK(cudaMemcpyAsync(S.data(), slots.p, n_slots * sizeof(VrSlot), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        build_ms += elapsed_ms(ev.a, ev.b);
        std::vector<uint64_t>& R = chrom_region[ch];
        R.assign(n_slots, 0);
        uint64_t words = 0;
        for (uint32_t q = 0; q < n_slots; q++) {
            R[q] = words;
            if (S[q].nrec) words += 4 * S[q].nrec + (S[q].pool + 7) / 8;
        }
        out[ch].reset(new DevBuf<uint64_t>());
        if (words) {
            out[ch]->ensure(words);
            CK(cudaMemsetAsync(out[ch]->p, 0, words * 8, s));
            region.upload(R, s);
            v.region = region.p;
            v.out = out[ch]->p;
            CK(cudaEventRecord(ev.a, s));
            CK(launch_vr_write(v, s));
            CK(cudaEventRecord(ev.b, s));
            CK(cudaStreamSynchronize(s));
            build_ms += elapsed_ms(ev.a, ev.b);
        }
        done[ch] = 1;
        acc_alleles = acc_text = acc_calls = 0;
    }
};

void read_vcf(jlp_ctx* c, const jlp_vcf_read_params* P, jlp_vcf_read_stats* stats) {
    const auto t_call = std::chrono::steady_clock::now();
    if (!P) throw ArgErr("params is NULL");
    if (!P->path || !*P->path) throw ArgErr("path is empty");
    if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
    if (P->n_threads < 1 || P->n_threads > 64) throw ArgErr("n_threads must be in 1..64");
    const uint64_t batch = P->batch_bytes ? P->batch_bytes : kDefaultBatch;
    if (batch > kMaxBatch) throw ArgErr("batch_bytes must be below 2 GiB");
    Device& d = device0(c);
    finish_upload(c, d);
    Reader Rd(c, d);
    Rd.len = chrom_lengths(c);
    Source src(P->path, (unsigned)P->n_threads);
    Feed feed(src, batch);
    PinBuf<uint8_t> pin[2];
    EventPair up;                                // the copies into text[0] / text[1]
    // no copy may still read a pinned buffer when the call ends by an exception
    struct Drain { cudaStream_t s; ~Drain() { cudaStreamSynchronize(s); } } drain{d.s_upload};
    uint64_t n_batches = 0;
    bool have_header = false;
    // batch k's text to text[k & 1] on the upload stream, after any header lines it holds are parsed on the host;
    // returns the data bytes copied
    auto stage = [&](uint64_t k, uint64_t n) -> uint64_t {
        uint64_t off = 0;
        if (!have_header) {
            off = Rd.header(pin[k & 1].p, n, have_header);
            if (have_header) Rd.start();
        }
        if (!have_header || off == n) return 0;
        DevBuf<uint8_t>& dt = Rd.text[k & 1];
        dt.ensure(n - off);
        CK(cudaMemcpyAsync(dt.p, pin[k & 1].p + off, n - off, cudaMemcpyHostToDevice, d.s_upload));
        CK(cudaEventRecord(k & 1 ? up.b : up.a, d.s_upload));
        return n - off;
    };
    // While batch k is parsed, batch k + 1 is read and inflated into pin[(k + 1) & 1] on another thread (that buffer
    // held batch k - 1, whose copy ended before its kernels ran); batch k + 1's copy then runs while batch k's lines
    // are appended to their chromosomes and built.
    uint64_t n = feed.next(pin[0]), k = 0;
    uint64_t cur = n ? stage(0, n) : 0;
    while (n) {
        std::future<uint64_t> nxt = std::async(std::launch::async, [&, k]() { return feed.next(pin[(k + 1) & 1]); });
        uint64_t next = 0;
        try {
            bool parsed = false;
            if (cur) {
                CK(cudaStreamWaitEvent(Rd.s, k & 1 ? up.b : up.a, 0));
                parsed = Rd.parse(Rd.text[k & 1].p, (uint32_t)cur);
                n_batches++;
            }
            n = nxt.get();
            if (n) next = stage(k + 1, n);
            if (parsed) Rd.hand();
        } catch (...) {
            if (nxt.valid()) nxt.wait();
            throw;
        }
        cur = next;
        k++;
    }
    if (!have_header) bad_line(Rd.header_lines + 1, "no #CHROM line before the data");
    if (Rd.open != kVrNone) Rd.build();

    // the haplotypes: (sample, copy) for copy < P_s
    std::vector<uint32_t> ploidy(Rd.n_samples);
    read_back(ploidy.data(), Rd.ploidy.p, Rd.n_samples, Rd.s);
    unsigned long long cnt[2] = {0, 0};
    if (have_header) read_back(cnt, Rd.counts.p, 2, Rd.s);
    HapRegions G;
    std::vector<uint32_t> slot_of;
    for (uint32_t si = 0; si < Rd.n_samples; si++) {
        const uint32_t P_s = std::max(1u, ploidy[si]);
        for (uint32_t k2 = 0; k2 < P_s; k2++) {
            G.names.push_back(P_s == 1 ? Rd.samples[si] : Rd.samples[si] + "__" + std::to_string(k2 + 1));
            slot_of.push_back(si * kVrMaxPloidy + k2);
        }
    }
    if (G.names.size() > kMaxHaps) throw ArgErr("more than 65536 haplotypes");
    const uint64_t nc = Rd.nc, n_items = G.names.size() * nc;
    G.src.assign(n_items, nullptr);
    G.n.assign(n_items, 0);
    G.pool.assign(n_items, 0);
    G.size.assign(n_items, 0);
    jlp_vcf_read_stats st{};
    for (size_t h = 0; h < G.names.size(); h++)
        for (uint64_t ci = 0; ci < nc; ci++) {
            const size_t r = h * nc + ci;
            G.size[r] = Rd.len[ci];
            if (!Rd.done[ci]) continue;
            const VrSlot& S = Rd.chrom_slot[ci][slot_of[h]];
            G.n[r] = S.nrec;
            G.pool[r] = S.pool;
            G.size[r] = (uint64_t)((long long)Rd.len[ci] + S.delta);
            if (S.nrec) G.src[r] = Rd.out[ci]->p + Rd.chrom_region[ci][slot_of[h]];
            st.calls += S.applied;
            st.overlaps_skipped += S.skipped;
            st.records += S.nrec;
        }
    const auto t_store = std::chrono::steady_clock::now();
    store_haps(c, G, (unsigned)std::min<uint64_t>(P->n_threads, std::max<uint64_t>(n_items, 1)));
    const auto t1 = std::chrono::steady_clock::now();
    if (stats) {
        st.lines = Rd.lines;
        st.samples = Rd.n_samples;
        st.haplotypes = G.names.size();
        st.missing_calls = cnt[0];
        st.symbolic_calls = cnt[1];
        st.text_bytes = feed.text_bytes;
        st.batches = n_batches;
        st.inflate_ms = feed.inflate_ms;
        st.parse_ms = Rd.parse_ms;
        st.build_ms = Rd.build_ms;
        st.store_ms = std::chrono::duration<double, std::milli>(t1 - t_store).count();
        st.total_ms = std::chrono::duration<double, std::milli>(t1 - t_call).count();
        *stats = st;
    }
}

}  // namespace

extern "C" {

int jlp_create_haplotypes_vcf(jlp_ctx* c, const jlp_vcf_read_params* p, jlp_vcf_read_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { read_vcf(c, p, stats); });
}

int jlp_haplotype_name(jlp_ctx* c, uint64_t h, char* out, uint64_t cap, uint64_t* len) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (h >= c->haps.size()) throw ArgErr("haplotype index out of range");
        const std::string& n = c->haps[h]->name;
        if (len) *len = n.size();
        if (n.size() > cap) throw ArgErr("output buffer too small");
        if (!n.empty()) std::memcpy(out, n.data(), n.size());
    });
}

}  // extern "C"
