#include "jlp_output.h"

#include <fcntl.h>
#include <sys/statvfs.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cstring>

#include "jlp_deflate.h"

namespace jlp {

std::string pwrite_all(int fd, const uint8_t* p, uint64_t n, uint64_t off) {
    while (n) {
        ssize_t w = ::pwrite(fd, p, n > (1u << 30) ? (1u << 30) : n, (off_t)off);
        if (w < 0) { if (errno == EINTR) continue; return std::strerror(errno); }
        p += w; n -= (uint64_t)w; off += (uint64_t)w;
    }
    return std::string();
}

bool map_range(int fd, uint64_t off, uint64_t n, Mapping& m, bool read_only) {
    static const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE);
    const uint64_t a0 = off / page * page;
    void* p = ::mmap(nullptr, (size_t)(off + n - a0), read_only ? PROT_READ : PROT_READ | PROT_WRITE, MAP_SHARED, fd, (off_t)a0);
    if (p == MAP_FAILED) return false;
    m.base = p; m.len = (size_t)(off + n - a0); m.at = static_cast<uint8_t*>(p) + (off - a0);
    return true;
}

std::string copy_range(int out_fd, uint64_t out_off, int in_fd, uint64_t in_off, uint64_t n) {
    std::vector<uint8_t> buf;
    bool use_cfr = true;
    while (n) {
        if (use_cfr) {
            off_t oi = (off_t)in_off, oo = (off_t)out_off;
            const ssize_t w = ::copy_file_range(in_fd, &oi, out_fd, &oo, (size_t)std::min<uint64_t>(n, 1ull << 30), 0);
            if (w > 0) { n -= (uint64_t)w; in_off += (uint64_t)w; out_off += (uint64_t)w; continue; }
            if (w < 0 && errno == EINTR) continue;
            if (w == 0) return "unexpected end of a part file";
            if (errno != EXDEV && errno != EINVAL && errno != ENOSYS && errno != EOPNOTSUPP) return std::strerror(errno);
            use_cfr = false;                                  // file systems without copy_file_range: read + write
        }
        buf.resize(8u << 20);
        const ssize_t r = ::pread(in_fd, buf.data(), (size_t)std::min<uint64_t>(n, buf.size()), (off_t)in_off);
        if (r < 0) { if (errno == EINTR) continue; return std::strerror(errno); }
        if (r == 0) return "unexpected end of a part file";
        const std::string w = pwrite_all(out_fd, buf.data(), (uint64_t)r, out_off);
        if (!w.empty()) return w;
        n -= (uint64_t)r; in_off += (uint64_t)r; out_off += (uint64_t)r;
    }
    return std::string();
}

void Output::begin(const Compression& z, int level, uint64_t n_threads, WriterPool& pool) {
    z_ = z; level_ = level; n_threads_ = n_threads; pool_ = &pool;
    if (kind == SINK_FILES) pool.start((size_t)std::min<uint64_t>(std::max<uint64_t>(n_threads, 1), 64));
}

void Output::open_job(const std::string names[2], int n_ends, const uint64_t base[2], bool shared_files) {
    if (kind == SINK_MEMORY && base)
        for (int e = 0; e < n_ends; e++) len[e] = base[e];
    if (kind != SINK_FILES) return;
    close_files();
    for (int e = 0; e < n_ends; e++) {
        names_[e] = names[e];
        pos_[e] = done_[e] = base ? base[e] : 0;
        own_size_[e] = !shared_files;
        fd_[e] = ::open(names_[e].c_str(), shared_files ? O_RDWR : (O_RDWR | O_CREAT | O_TRUNC), 0644);
        if (fd_[e] < 0) throw IoErr("Unable to open file " + names_[e] + ".\n");  // src/io.h:288-290
    }
}

void Output::deliver(HostBatch& b, const uint8_t* const data[2], const uint64_t n[2], uint64_t job_index, int n_ends) {
    if (z_.zmethod >= 0 && z_pending_) settle(*z_pending_);   // files stay in batch order
    for (int e = 0; e < n_ends; e++) {
        b.file_end[e] = 0;
        if (kind == SINK_FILES && z_.zmethod < 0) {
            // With several writer threads the file is extended and the batch's range mapped; ONE task per file
            // reserves the range's pages (posix_fallocate: a full file system is an error in that task, not a
            // SIGBUS later) and then hands the 8 MiB slices to the pool, which copies them into the mapping.
            // Page allocation is what the kernel serialises per file and it costs more than the copy, so it
            // must neither sit on the driver thread nor be fought over by all the writers (tools/fill_probe.cpp,
            // tools/files_probe.py; tmpfs, 16 threads: reserved by the driver thread 11.1 GB/s, by every writer
            // for its own slice 8.5, by page faults in the copies 9.2, this way 13.3).  Where posix_fallocate is
            // not supported the reservation reserves nothing, so a range is mapped only with room to spare on the
            // file system.  With one thread, or when the range cannot be mapped, plain pwrite.
            const int fd = fd_[e];
            const uint64_t ne = n[e];
            struct statvfs vfs;
            bool mapped = n_threads_ > 1 && ne > 0 && ::fstatvfs(fd, &vfs) == 0 &&
                          (uint64_t)vfs.f_bavail * vfs.f_frsize > 2 * ne + (64ull << 20);
            if (mapped) {
                if (own_size_[e]) mapped = ::ftruncate(fd, (off_t)(pos_[e] + ne)) == 0;
                mapped = mapped && map_range(fd, pos_[e], ne, b.map[e]);
            }
            const uint64_t slice = 8ull << 20;
            if (mapped) {
                pool_->submit(&b.writes, [fd, src0 = data[e], dst0 = b.map[e].at, off0 = pos_[e], ne, slice, pool = pool_, pend = &b.writes]() {
                    const int rc = ::posix_fallocate(fd, (off_t)off0, (off_t)ne);
                    if (rc != 0 && rc != EOPNOTSUPP && rc != EINVAL) return std::string(std::strerror(rc));
                    for (uint64_t o = 0; o < ne; o += slice) {
                        uint8_t* dst = dst0 + o;
                        const uint8_t* src = src0 + o;
                        const uint64_t nb = std::min(slice, ne - o);
                        pool->submit(pend, [dst, src, nb]() { std::memcpy(dst, src, nb); return std::string(); });
                    }
                    return std::string();
                });
            } else {
                for (uint64_t o = 0; o < ne; o += slice) {
                    const uint8_t* src = data[e] + o;
                    const uint64_t nb = std::min(slice, ne - o), off = pos_[e] + o;
                    pool_->submit(&b.writes, [fd, src, nb, off]() { return pwrite_all(fd, src, nb, off); });
                }
            }
            pos_[e] += ne;
            b.file_end[e] = pos_[e];
        } else if (kind == SINK_FILES) {
            // compressed: the writer threads deflate slices of whole members; their output is
            // written in order once the batch is done (settle)
            const int zmethod = z_.zmethod, lvl = level_;
            const uint64_t unit = zmethod == DEFLATE_BGZF ? 0xff00ull : (1ull << 20);
            const uint64_t slice = unit * (zmethod == DEFLATE_BGZF ? 64 : 4);
            const size_t n_slices = (size_t)((n[e] + slice - 1) / slice);
            b.zout[e].assign(n_slices, std::vector<uint8_t>());
            for (size_t k = 0; k < n_slices; k++) {
                const uint8_t* src = data[e] + k * slice;
                const uint64_t nb = std::min<uint64_t>(slice, n[e] - k * slice);
                std::vector<uint8_t>* dst = &b.zout[e][k];
                pool_->submit(&b.writes, [zmethod, lvl, src, nb, dst]() { return deflate_members(zmethod, lvl, src, nb, *dst); });
            }
            z_pending_ = &b;
        } else if (kind == SINK_STREAM) {
            if (chunk_cb(chunk_user, job_index, e, reinterpret_cast<const char*>(data[e]), n[e]))
                throw IoErr("the chunk callback reported an error");
        } else if (kind == SINK_MEMORY) {
            if (len[e] + n[e] <= cap[e]) std::memcpy(mem[e] + len[e], data[e], n[e]);
            len[e] += n[e];
        }
    }
}

void Output::settle(HostBatch& b) {
    if (kind != SINK_FILES) return;
    if (z_pending_ == &b) z_pending_ = nullptr;
    std::string e = pool_->wait(b.writes);
    for (Mapping& m : b.map) m.unmap();
    if (!e.empty()) {
        pool_->clear_error();
        throw IoErr("Error writing to file " + names_[0] + (names_[1].empty() ? "" : " / " + names_[1]) + ": " + e);
    }
    // compressed slices of the batch go to the files in order
    for (int k = 0; k < 2; k++) {
        for (std::vector<uint8_t>& v : b.zout[k]) {
            std::string w = pwrite_all(fd_[k], v.data(), v.size(), pos_[k]);
            if (!w.empty()) throw IoErr("Error writing to file " + names_[k] + ": " + w);
            pos_[k] += v.size();
        }
        b.zout[k].clear();
        if (b.file_end[k] > done_[k]) done_[k] = b.file_end[k];
        if (z_.zmethod >= 0) done_[k] = pos_[k];
    }
}

void Output::end_job(uint64_t job_index, int n_ends, bool eof_block) {
    if (eof_block && z_.dev_z && kind != SINK_FILES) {     // the device coder's output into memory or a stream ends with it too
        HostBatch eof;
        const uint8_t* const data[2] = {kBgzfEof, kBgzfEof};
        const uint64_t n[2] = {sizeof kBgzfEof, sizeof kBgzfEof};
        deliver(eof, data, n, job_index, n_ends);
    }
    if (eof_block && kind == SINK_FILES && (z_.dev_z || z_.zmethod == DEFLATE_BGZF))
        for (int e = 0; e < n_ends; e++) {   // bgzf_close appends the empty end-of-file block
            std::string w = pwrite_all(fd_[e], kBgzfEof, sizeof kBgzfEof, pos_[e]);
            if (!w.empty()) throw IoErr("Error writing to file " + names_[e] + ": " + w);
            pos_[e] += sizeof kBgzfEof;
            done_[e] = pos_[e];
        }
    close_files();
}

void Output::abandon(HostBatch* const* batches, size_t k) {
    for (size_t i = 0; i < k; i++) {
        pool_->wait(batches[i]->writes);
        for (Mapping& m : batches[i]->map) m.unmap();
        batches[i]->zout[0].clear(); batches[i]->zout[1].clear();
    }
    z_pending_ = nullptr;
    pool_->clear_error();
    for (int e = 0; e < 2; e++)
        if (fd_[e] >= 0 && own_size_[e] && ::ftruncate(fd_[e], (off_t)done_[e]) != 0) { /* best effort */ }
}

void Output::close_files() {
    for (int e = 0; e < 2; e++) if (fd_[e] >= 0) { ::close(fd_[e]); fd_[e] = -1; }
}

}  // namespace jlp
