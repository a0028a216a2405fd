// Delivery of generated batches to their sink: plain or zlib-compressed files, the caller's memory, or a chunk
// callback.  Host code only (no CUDA), shared by the Illumina, PacBio and VCF drivers.
#ifndef JLP_OUTPUT_H
#define JLP_OUTPUT_H

#include <sys/mman.h>

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <functional>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/jlp_b200.h"

namespace jlp {

// the library's errors; the C ABI maps each to its JLP_ERR_* code
struct CudaErr : std::runtime_error {
    explicit CudaErr(const std::string& m) : std::runtime_error(m) {}
};
struct ArgErr : std::runtime_error {
    explicit ArgErr(const std::string& m) : std::runtime_error(m) {}
};
struct IoErr : std::runtime_error {
    explicit IoErr(const std::string& m) : std::runtime_error(m) {}
};
struct Unsupported : std::runtime_error {
    explicit Unsupported(const std::string& m) : std::runtime_error(m) {}
};
struct Aborted : std::runtime_error {
    Aborted() : std::runtime_error("aborted by user") {}
};

// Host writer threads: the FASTQ of a batch sits in a pinned buffer; its slices are written
// with pwrite() at their final file offsets while the GPU generates and copies the next
// batch (the reference's threads serialise on one omp critical per pool instead,
// src/hts.h:401-416).
class WriterPool {
public:
    // a task returns an error text (empty = fine); `pending` counts the tasks of one batch slot
    struct Task { std::function<std::string()> run; std::atomic<int>* pending; };
    ~WriterPool() { stop(); }
    void start(size_t n_threads) {
        if (th.size() == n_threads) return;
        stop();
        quit = false;
        for (size_t i = 0; i < n_threads; i++) th.emplace_back([this]() { loop(); });
    }
    void stop() {
        { std::lock_guard<std::mutex> l(m); quit = true; }
        cv.notify_all();
        for (std::thread& t : th) t.join();
        th.clear();
    }
    void submit(std::atomic<int>* pending, std::function<std::string()> f) {
        pending->fetch_add(1);
        { std::lock_guard<std::mutex> l(m); q.push_back(Task{std::move(f), pending}); }
        cv.notify_one();
    }
    // wait until every task counted by `pending` is done; returns the first error text (empty = none)
    std::string wait(std::atomic<int>& pending) {
        std::unique_lock<std::mutex> l(m);
        cv_done.wait(l, [&]() { return pending.load() == 0; });
        return err;
    }
    void clear_error() { std::lock_guard<std::mutex> l(m); err.clear(); }
private:
    void loop() {
        for (;;) {
            Task t;
            {
                std::unique_lock<std::mutex> l(m);
                cv.wait(l, [&]() { return quit || !q.empty(); });
                if (q.empty()) return;
                t = std::move(q.front()); q.pop_front();
            }
            std::string e = t.run();
            {
                std::lock_guard<std::mutex> l(m);
                if (!e.empty() && err.empty()) err = e;
                t.pending->fetch_sub(1);
            }
            cv_done.notify_all();
        }
    }
    std::vector<std::thread> th;
    std::mutex m;
    std::condition_variable cv, cv_done;
    std::deque<Task> q;
    std::string err;
    bool quit = false;
};

std::string pwrite_all(int fd, const uint8_t* p, uint64_t n, uint64_t off);

// Files are also written through shared mappings: the main thread extends the file by a batch and maps the new
// range once, the writer threads copy their slices into the mapping (page-cache pages are allocated and filled by
// the copying thread, so the threads do not queue on the inode lock that serialises write() calls on one file;
// measured on the B200 box's tmpfs: 7.4 GB/s with pwrite from any number of threads, 14 GB/s with 16 threads
// copying into mappings, tools/write_probe.cpp), and the range is unmapped when the batch's slices are done --
// one munmap per batch and file, not one TLB shoot-down per slice.
struct Mapping {
    void* base = nullptr;
    size_t len = 0;
    uint8_t* at = nullptr;      // where the batch's first byte goes
    void unmap() { if (base) ::munmap(base, len); base = nullptr; len = 0; at = nullptr; }
};
bool map_range(int fd, uint64_t off, uint64_t n, Mapping& m, bool read_only = false);

// n bytes from in_fd at in_off to out_fd at out_off (both files on any file system)
std::string copy_range(int out_fd, uint64_t out_off, int in_fd, uint64_t in_off, uint64_t n);

enum SinkKind { SINK_FILES, SINK_MEMORY, SINK_STREAM, SINK_NONE };

// How a run's output is compressed; each driver decides it from its own parameters.
struct Compression {
    bool dev_z = false;       // BGZF on the device (the batches arrive compressed)
    int zmethod = -1;         // host zlib: DEFLATE_BGZF / DEFLATE_GZIP; -1 = none
    bool want_gz = false;     // file names get ".gz"
};

// The host side of one batch on its way into the files.
struct HostBatch {
    std::atomic<int> writes{0};   // slices still being written to / compressed for the files
    std::vector<std::vector<uint8_t>> zout[2];   // compressed slices of the batch, in file order
    Mapping map[2];               // the file ranges this batch is being copied into
    uint64_t file_end[2] = {0, 0};  // where this batch ends in the files (plain FASTQ)
};

// One run's sink.  Batches are delivered in file order; a batch's host buffers may be reused once settle() has
// returned for it.  Files stay in batch order: R1 and R2 receive the same batches, so they stay record-aligned.
class Output {
public:
    SinkKind kind = SINK_NONE;
    // memory
    char* mem[2] = {nullptr, nullptr};
    uint64_t cap[2] = {0, 0}, len[2] = {0, 0};
    // stream
    jlp_chunk_cb chunk_cb = nullptr;
    void* chunk_user = nullptr;

    explicit Output(SinkKind k = SINK_NONE) : kind(k) {}
    ~Output() { close_files(); }
    // files: start the writer threads (n_threads, at most 64) that copy and compress the batches
    void begin(const Compression& z, int level, uint64_t n_threads, WriterPool& pool);
    // files: open names[e] for writing at base[e] (NULL: at 0; truncated unless shared_files, a file created and sized by
    // the caller); memory: the job's bytes start at base[e] (NULL: behind the previous job's)
    void open_job(const std::string names[2], int n_ends, const uint64_t base[2], bool shared_files);
    void deliver(HostBatch& b, const uint8_t* const data[2], const uint64_t n[2], uint64_t job_index, int n_ends);
    // wait until the batch is in the files (its host buffers are free again); throws IoErr on a write error
    void settle(HostBatch& b);
    // after every batch of the job is settled: the BGZF end-of-file block (eof_block), files closed
    void end_job(uint64_t job_index, int n_ends, bool eof_block);
    // on an error: wait for the batches' writes, and cut the files this call sized itself back to the last complete batch
    void abandon(HostBatch* const* batches, size_t k);
    void close_files();

private:
    Compression z_;
    int level_ = 0;
    uint64_t n_threads_ = 1;
    WriterPool* pool_ = nullptr;
    HostBatch* z_pending_ = nullptr;   // the batch whose compressed slices are not in the files yet
    int fd_[2] = {-1, -1};
    uint64_t pos_[2] = {0, 0};         // where the next batch goes
    uint64_t done_[2] = {0, 0};        // end of the last batch known to be completely written (abandon truncates back to it)
    bool own_size_[2] = {false, false};   // this call extends the file itself (not a pre-sized file shared with other devices)
    std::string names_[2];
};

}  // namespace jlp
#endif
