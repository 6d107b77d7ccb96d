// The fetch -> decode -> filter -> join -> count pipeline and the C ABI of libbamsignals_cuda.so.
//
// Host side (this file + plan.cpp + bamio.cpp): BAI query -> fetch segments -> worker pool inflates BGZF blocks into
// pinned staging slots and walks the block_size chain to emit record offsets -> H2D on a copy stream overlapping the
// decode kernel of the previous batch on the compute stream.  Device side (kernels.cu): K1..K5.
// No CPU fallback: every entry point needs a CUDA device.
#include <algorithm>
#include <atomic>
#include <climits>
#include <cstddef>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <unistd.h>

#include "bamio.h"
#include "common.h"
#include "kernels.cuh"
#include "hostsimd.h"
#include "plan.h"
#include "pool.h"

// A run-length result (bsg_coverage_runs, bsg_profile_runs): lengths[n] and values[n] in device memory on `dev`.
struct bsg_runs {
    int dev = -1;
    int32_t* lengths = nullptr;
    int32_t* values = nullptr;
    int64_t n = 0;
    bool live = false;                          // false once bsg_shutdown() has freed the arrays
    void release() {
        if (lengths || values) { cudaSetDevice(dev); cudaFree(lengths); cudaFree(values); cudaGetLastError(); }
        lengths = values = nullptr;
        live = false;
    }
    ~bsg_runs() { release(); }
};

namespace bsg {
void write_sam_as_bam_and_index(const char* sampath, const char* bampath);      // bamwrite.cpp
namespace {

thread_local std::string g_err;
thread_local bsg_timings g_tm;

// NVTX range of one pipeline stage on the calling thread (header-only nvtx3: a no-op unless a profiler is attached)
struct Nvtx {
    explicit Nvtx(const char* name) { nvtxRangePushA(name); }
    ~Nvtx() { nvtxRangePop(); }
    Nvtx(const Nvtx&) = delete;
};


constexpr int kSlots = 4;                       // staging ring depth
constexpr int64_t kDefaultBatch = 64ll << 20;   // uncompressed bytes per batch (host inflate)
constexpr int64_t kDefaultGpuBatch = 2048ll << 20;   // byte cap of a device-inflate batch (the block-count "wave" is the working limit)
constexpr size_t kCompChunk = 16u << 20;        // compressed bytes per pinned upload chunk (GPU inflate)
constexpr uint64_t kSegCBytes = 1ull << 20;     // compressed bytes per fetch segment (parallel walk granularity)
constexpr uint64_t kSpanGap = 160u << 10;       // file gaps up to this many bytes are uploaded rather than skipped
constexpr uint64_t kSmallJobBytes = 16u << 20;   // inflated bytes up to which the default path inflates on the host
constexpr int kMinRecord = 36;                  // block_size + 32-byte fixed part: smallest possible record
constexpr int64_t kD2HChunk = 32ll << 20;       // bytes per pinned result-staging buffer
constexpr int64_t kPackMinInts = 1ll << 16;     // result portions from this size on cross PCIe as bytes (opts.result_pack)
constexpr int kOutSlots = 3;                    // pinned result-staging ring
constexpr int kUp = 4;                          // GPU-inflate path: upload ring (compressed bytes + descriptors); raw buffers: 2
// Staged pileup calls take the fused step when its join would examine at most this share of the resident rows
// (opts.resident_scheme 0).  Placed from tools/resident_ab.py's sweep on one B200 (profiles/resident_ab_c2_sweep.jsonl):
// the fused step is 1.62x / 1.27x / 0.98x / 0.99x the table step at shares 0.13 / 0.23 / 0.34 / 0.43.
constexpr double kFusedShare = 0.3;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    void ensure(size_t bytes) {
        if (bytes <= cap) return;
        if (p) BSG_CUDA(cudaFree(p));
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        BSG_CUDA(cudaMalloc(&p, want));
        cap = want;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    void ensure(size_t bytes) {
        if (bytes <= cap) return;
        if (p) BSG_CUDA(cudaFreeHost(p));
        p = nullptr; cap = 0;
        BSG_CUDA(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
        cap = bytes;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

// Everything cached per device across calls (released by bsg_shutdown).
struct DeviceCtx {
    int dev = 0;
    int n_sm = 148;
    bool init = false;
    cudaStream_t s_copy = nullptr, s_comp = nullptr, s_aux = nullptr, s_walk = nullptr, s_walk2 = nullptr, s_d2h = nullptr, s_hi = nullptr;
    DevBuf d_raw[kSlots], d_offs[kSlots];
    PinBuf h_raw[kSlots], h_offs[kSlots];
    cudaEvent_t ev_h2d[kSlots] = {}, ev_free[kSlots] = {};
    DevBuf tab[2], c0, c1, tiles_i32, tiles_i64, out, scalars;
    DevBuf runs_i32, runs_i64;                  // run-length results: per-tile and per-list scratch (RunTiles, run_off)
    uint64_t tiles_gen = 0;                     // bumped whenever a Session uploads tiles: a staged Session's cached tiles are
                                                // only valid while no other call has replaced them on this device
    // GPU inflate: an upload ring of kUp slots (compressed bytes, descriptors, walk scratch) and two raw / offsets buffers
    DevBuf g_comp[kUp], g_blocks[kUp], g_crc[kUp], g_walkers[kUp], g_counts[kUp], g_base[kUp], g_wscr[kUp], g_spec[kUp], g_raw[2], g_offs[2], g_total;
    PinBuf h_total, h_desc[kUp];
    cudaEvent_t ev_pin[kSlots] = {}, ev_up[kUp] = {}, ev_total[kUp] = {}, ev_inflated[kUp] = {}, ev_crc[kUp] = {}, ev_gfree[2] = {};
    PinBuf h_scalars, h_out[kOutSlots], h_tiles, h_front, h_ovf[kOutSlots], h_pack_cnt, h_runs;
    DevBuf g_pack[kOutSlots], g_pack_cnt;       // result narrowing (opts.result_pack): packed bytes per ring slot, overflow counters
    cudaEvent_t ev_d2h[kOutSlots] = {}, ev_front[2] = {}, ev_order = nullptr;
    cudaEvent_t ev_caller = nullptr;            // device-output calls: the caller's stream at entry
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_next = 0;

    void ensure_init(int device) {
        if (init && dev == device) { BSG_CUDA(cudaSetDevice(dev)); return; }
        dev = device;
        BSG_CUDA(cudaSetDevice(dev));
        BSG_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
        BSG_CUDA(cudaStreamCreateWithFlags(&s_copy, cudaStreamNonBlocking));
        BSG_CUDA(cudaStreamCreateWithFlags(&s_comp, cudaStreamNonBlocking));
        BSG_CUDA(cudaStreamCreateWithFlags(&s_aux, cudaStreamNonBlocking));
        BSG_CUDA(cudaStreamCreateWithFlags(&s_walk, cudaStreamNonBlocking));
        BSG_CUDA(cudaStreamCreateWithFlags(&s_walk2, cudaStreamNonBlocking));
        BSG_CUDA(cudaStreamCreateWithFlags(&s_d2h, cudaStreamNonBlocking));
        {   // decode + count kernels of finished batches overtake the inflate of the next one
            int lo_p = 0, hi_p = 0;
            BSG_CUDA(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
            BSG_CUDA(cudaStreamCreateWithPriority(&s_hi, cudaStreamNonBlocking, hi_p));
        }
        BSG_CUDA(cudaEventCreateWithFlags(&ev_order, cudaEventDisableTiming));
        BSG_CUDA(cudaEventCreateWithFlags(&ev_caller, cudaEventDisableTiming));
        for (int i = 0; i < kSlots; ++i) {
            BSG_CUDA(cudaEventCreateWithFlags(&ev_h2d[i], cudaEventDisableTiming));
            BSG_CUDA(cudaEventCreateWithFlags(&ev_free[i], cudaEventDisableTiming));
        }
        for (int i = 0; i < kOutSlots; ++i) BSG_CUDA(cudaEventCreateWithFlags(&ev_d2h[i], cudaEventDisableTiming));
        h_front.ensure(64);
        for (int i = 0; i < 2; ++i) {
            BSG_CUDA(cudaEventCreateWithFlags(&ev_front[i], cudaEventDisableTiming));
            BSG_CUDA(cudaEventCreateWithFlags(&ev_gfree[i], cudaEventDisableTiming));
        }
        for (int i = 0; i < kUp; ++i) {
            BSG_CUDA(cudaEventCreateWithFlags(&ev_up[i], cudaEventDisableTiming));
            BSG_CUDA(cudaEventCreateWithFlags(&ev_total[i], cudaEventDisableTiming));
            BSG_CUDA(cudaEventCreateWithFlags(&ev_inflated[i], cudaEventDisableTiming));
            BSG_CUDA(cudaEventCreateWithFlags(&ev_crc[i], cudaEventDisableTiming));
        }
        for (int i = 0; i < kSlots; ++i) BSG_CUDA(cudaEventCreateWithFlags(&ev_pin[i], cudaEventDisableTiming));
        h_total.ensure(64 + 4 * kUp);
        g_total.ensure(64 + 4 * kUp);
        h_scalars.ensure(sizeof(DeviceScalars));
        init = true;
    }
    cudaEvent_t timing_event() {
        if (ev_next == ev_pool.size()) {
            cudaEvent_t e;
            BSG_CUDA(cudaEventCreate(&e));
            ev_pool.push_back(e);
        }
        return ev_pool[ev_next++];
    }
    void release() {
        if (!init) return;
        cudaSetDevice(dev);
        cudaDeviceSynchronize();
        for (int i = 0; i < kSlots; ++i) {
            d_raw[i].release(); d_offs[i].release(); h_raw[i].release(); h_offs[i].release();
            cudaEventDestroy(ev_h2d[i]); cudaEventDestroy(ev_free[i]);
        }
        for (auto& b : tab) b.release();
        c0.release(); c1.release(); tiles_i32.release(); tiles_i64.release(); out.release(); scalars.release();
        runs_i32.release(); runs_i64.release(); h_runs.release();
        h_scalars.release();
        for (int i = 0; i < kOutSlots; ++i) { h_out[i].release(); h_ovf[i].release(); g_pack[i].release(); cudaEventDestroy(ev_d2h[i]); }
        h_pack_cnt.release(); g_pack_cnt.release();
        h_tiles.release(); h_front.release();
        cudaEventDestroy(ev_front[0]); cudaEventDestroy(ev_front[1]);
        for (int i = 0; i < 2; ++i) { g_raw[i].release(); g_offs[i].release(); cudaEventDestroy(ev_gfree[i]); }
        for (int i = 0; i < kUp; ++i) {
            g_comp[i].release(); g_blocks[i].release(); g_crc[i].release(); g_walkers[i].release();
            g_counts[i].release(); g_base[i].release(); g_wscr[i].release(); g_spec[i].release(); h_desc[i].release();
            cudaEventDestroy(ev_up[i]); cudaEventDestroy(ev_total[i]); cudaEventDestroy(ev_inflated[i]); cudaEventDestroy(ev_crc[i]);
        }
        for (int i = 0; i < kSlots; ++i) cudaEventDestroy(ev_pin[i]);
        g_total.release(); h_total.release();
        for (auto e : ev_pool) cudaEventDestroy(e);
        ev_pool.clear(); ev_next = 0;
        cudaStreamDestroy(s_copy); cudaStreamDestroy(s_comp); cudaStreamDestroy(s_aux); cudaStreamDestroy(s_walk); cudaStreamDestroy(s_walk2); cudaStreamDestroy(s_d2h); cudaStreamDestroy(s_hi); cudaEventDestroy(ev_order);
        cudaEventDestroy(ev_caller);
        init = false;
    }
};

std::mutex g_mu;                                // one call at a time per process (re-entrancy is not required)
DeviceCtx g_ctx[16];
std::unique_ptr<Pool> g_pool;

// Open BAM files (mmap + parsed header + parsed index) are kept across calls: the reference re-opens the file and
// re-loads the index on every call (src/bamsignals.cpp:449,479); here a call on an unchanged file (same size and
// mtime) reuses them.  Released by bsg_shutdown().
std::vector<std::shared_ptr<BamFile>> g_bams;

// ---- direct DMA from the page cache -------------------------------------------------------------------------------------
// The compressed bytes of a call live in the BAM's file mapping.  Staging them through pinned buffers costs a CPU memcpy
// of every byte and a worker pool that is busy for the whole upload.  Instead, 128 MB windows of the mapping are
// page-locked (cudaHostRegister, read-only, portable) and the copy engine reads the page cache itself: 55 GB/s, no CPU
// (profiles/r2d_pin_probe_*.txt).  Page-locking costs ~15 ms per window, so it is kept off the calls: the FIRST call that
// touches a window stages it as before and only marks it; a background thread locks the marked windows once the call has
// returned; every later call that needs them finds them locked.  They stay locked while the handle is cached.  Where the
// platform refuses, the staging path remains.
constexpr uint64_t kPinWindow = 128ull << 20;
enum : uint8_t { PIN_NONE = 0, PIN_LOCKED = 1, PIN_WANTED = 2, PIN_BUSY = 3 };
struct PinnedMapping {
    std::vector<uint8_t> state;                 // per window
    bool unsupported = false;
};
std::mutex g_pin_mu;
std::condition_variable g_pin_cv;
std::unordered_map<const BamFile*, PinnedMapping> g_pins;
std::deque<std::shared_ptr<BamFile>> g_pin_jobs;   // mappings with PIN_WANTED windows
std::thread g_pin_thread;
bool g_pin_stop = false;
int g_pin_dev = 0;

// true when [off, off + len) of the mapping is page-locked; windows that are not are marked for the background thread
bool ensure_pinned(const BamFile& bam, uint64_t off, uint64_t len) {
    if (len == 0) return true;
    std::lock_guard<std::mutex> g(g_pin_mu);
    PinnedMapping& pm = g_pins[&bam];
    if (pm.unsupported) return false;
    const uint64_t nwin = (bam.size() + kPinWindow - 1) / kPinWindow;
    if (pm.state.size() != nwin) pm.state.assign(nwin, PIN_NONE);
    bool all = true;
    for (uint64_t w = off / kPinWindow; w <= (off + len - 1) / kPinWindow && w < nwin; ++w) {
        if (pm.state[w] == PIN_LOCKED) continue;
        all = false;
        if (pm.state[w] == PIN_NONE) pm.state[w] = PIN_WANTED;
    }
    return all;
}

void pin_thread_main() {
    cudaSetDevice(g_pin_dev);
    nvtxNameOsThreadA(uint32_t(syscall(SYS_gettid)), "bsg page-lock");
    for (;;) {
        std::shared_ptr<BamFile> bam;
        {
            std::unique_lock<std::mutex> lk(g_pin_mu);
            g_pin_cv.wait(lk, [] { return g_pin_stop || !g_pin_jobs.empty(); });
            if (g_pin_stop) return;
            bam = g_pin_jobs.front();
            g_pin_jobs.pop_front();
        }
        for (;;) {
            uint64_t w = 0;
            bool found = false;
            {
                std::lock_guard<std::mutex> g(g_pin_mu);
                if (g_pin_stop) break;
                auto it = g_pins.find(bam.get());
                if (it == g_pins.end() || it->second.unsupported) break;
                for (; w < it->second.state.size(); ++w)
                    if (it->second.state[w] == PIN_WANTED) { it->second.state[w] = PIN_BUSY; found = true; break; }
            }
            if (!found) break;
            const uint64_t beg = w * kPinWindow;
            const uint64_t bytes = ((std::min(bam->size(), beg + kPinWindow) - beg) + 4095) & ~4095ull;   // whole pages of the mapping
            nvtxRangePushA("bsg:cudaHostRegister window");
            const cudaError_t e = cudaHostRegister(const_cast<uint8_t*>(bam->data()) + beg, bytes,
                                                   cudaHostRegisterPortable | cudaHostRegisterReadOnly);
            nvtxRangePop();
            std::lock_guard<std::mutex> g(g_pin_mu);
            auto it = g_pins.find(bam.get());
            if (it == g_pins.end()) { if (e == cudaSuccess) cudaHostUnregister(const_cast<uint8_t*>(bam->data()) + beg); break; }
            if (e == cudaSuccess) it->second.state[w] = PIN_LOCKED;
            else {
                cudaGetLastError();
                it->second.state[w] = PIN_NONE;
                it->second.unsupported = true;
                if (getenv("BSG_DEBUG")) fprintf(stderr, "[bsg] cudaHostRegister of the BAM mapping refused (%s): staging through pinned chunks\n", cudaGetErrorString(e));
            }
        }
        bam.reset();                             // may run the handle's deleter (unpin_mapping): no lock is held here
    }
}

// after a call: hand the mapping to the background thread if the call marked windows
void kick_pinning(const std::shared_ptr<BamFile>& bam, int dev) {
    std::lock_guard<std::mutex> g(g_pin_mu);
    auto it = g_pins.find(bam.get());
    if (it == g_pins.end() || it->second.unsupported) return;
    bool wanted = false;
    for (uint8_t st : it->second.state) wanted = wanted || st == PIN_WANTED;
    if (!wanted) return;
    for (auto& j : g_pin_jobs) if (j.get() == bam.get()) return;
    g_pin_jobs.push_back(bam);
    if (!g_pin_thread.joinable()) { g_pin_stop = false; g_pin_dev = dev; g_pin_thread = std::thread(pin_thread_main); }
    g_pin_cv.notify_all();
}

void stop_pin_thread() {
    {
        std::lock_guard<std::mutex> g(g_pin_mu);
        g_pin_stop = true;
    }
    g_pin_cv.notify_all();
    if (g_pin_thread.joinable()) g_pin_thread.join();
    std::deque<std::shared_ptr<BamFile>> drop;
    {
        std::lock_guard<std::mutex> g(g_pin_mu);
        drop.swap(g_pin_jobs);
        g_pin_stop = false;
    }
}

// joins the background thread before the globals above are destroyed at process exit (it is defined after them)
struct PinThreadGuard { ~PinThreadGuard() { stop_pin_thread(); g_bams.clear(); } } g_pin_guard;

void unpin_mapping(const BamFile* bam) {
    std::lock_guard<std::mutex> g(g_pin_mu);
    auto it = g_pins.find(bam);
    if (it == g_pins.end()) return;
    for (size_t w = 0; w < it->second.state.size(); ++w)
        if (it->second.state[w] == PIN_LOCKED) cudaHostUnregister(const_cast<uint8_t*>(bam->data()) + w * kPinWindow);
    cudaGetLastError();
    g_pins.erase(it);
}

std::shared_ptr<BamFile> open_bam(const char* path) {
    const std::string p = path ? path : "";
    struct stat st;
    if (!p.empty() && ::stat(p.c_str(), &st) == 0) {
        const uint64_t mt = uint64_t(st.st_mtim.tv_sec) * 1000000000ull + uint64_t(st.st_mtim.tv_nsec);
        for (auto it = g_bams.begin(); it != g_bams.end(); ++it)
            if ((*it)->path() == p) {
                if ((*it)->size() == uint64_t(st.st_size) && (*it)->mtime_ns() == mt && (*it)->index_unchanged()) return *it;
                g_bams.erase(it);
                break;
            }
    }
    std::shared_ptr<BamFile> b(new BamFile(p), [](BamFile* f) { unpin_mapping(f); delete f; });    // unpin before munmap
    if (g_bams.size() >= 4) g_bams.erase(g_bams.begin());
    g_bams.push_back(b);
    return b;
}

Pool& get_pool(int want) {
    int n = want > 0 ? want : int(std::thread::hardware_concurrency());
    if (n < 1) n = 1;
    if (!g_pool || g_pool->size() != n) g_pool.reset(new Pool(n));
    return *g_pool;
}

// The caller's options, whatever version of the struct it was compiled against: the first struct_size bytes are taken,
// the rest are defaults (all zero).  verify_crc: 0 = default = on, -1 = off.
bsg_opts effective_opts(const bsg_opts* opts) {
    bsg_opts o;
    memset(&o, 0, sizeof o);
    if (opts) {
        if (opts->struct_size < int32_t(sizeof(int32_t)) || opts->struct_size > (1 << 16))
            fail(BSG_EARG, "bsg_opts.struct_size must be set to sizeof(bsg_opts)");
        memcpy(&o, opts, std::min<size_t>(size_t(opts->struct_size), sizeof o));
    }
    o.struct_size = int32_t(sizeof o);
    o.verify_crc = o.verify_crc < 0 ? 0 : 1;
    return o;
}

struct Span { cudaEvent_t a, b; };
struct KernelTimes {
    std::vector<Span> decode, filter, join, count, all;
    int64_t launches = 0;
};

double sum_ms(const std::vector<Span>& v) {
    double t = 0;
    for (auto& s : v) { float ms = 0; cudaEventElapsedTime(&ms, s.a, s.b); t += ms; }
    return t;
}

struct Batch {
    size_t seg_first = 0, seg_last = 0;         // [first, last)
    uint64_t bytes = 0;                         // staged bytes (sum of segment usize)
    int64_t n_records = 0;                      // filled by the walk
    // runtime state
    std::vector<uint64_t> seg_base;             // byte offset of each segment in the staging buffer
    std::vector<uint64_t> seg_off_base;         // first slot of each segment in the (sparse) offsets array
    std::vector<int64_t> seg_count;
    std::unique_ptr<std::atomic<int>[]> seg_blocks_left;
    std::atomic<int> segs_left{0};
    std::mutex m;
    std::condition_variable cv;
    bool ready = false;
    Error err{0, ""};
};

struct ResidentIndexHost {
    int64_t n = 0;                          // resident rows
    uint32_t status = 0;                    // STATUS_* bits of the resident records
    int64_t reach = 0;                      // max(pos + span)
    uint32_t long_span = ~0u;               // T: rows with span > T are on the long list
    int64_t short_max = 0, long_max = 0;    // largest span at most T / above T
    int64_t n_keys = 0, n_long = 0;         // sampled keys (device), long-list rows (device)
};

struct ResidentBatch { uint64_t raw_base; int64_t offs_base; int64_t n; };

// The records a Session fetched.  A staged session (keep_raw) keeps their raw bytes, offsets, batch table and record
// index resident; its views (bsg_stage_view) hold the same StagedRecords, so the device memory is released with the
// last handle that shares it, whichever that is.
struct StagedRecords {
    int dev = 0;
    bool keep_raw = false;
    std::vector<ResidentBatch> batches;
    DevBuf raw_all, offs_all, batch_table;
    int64_t rows_cap = 0, n_rows = 0;
    int64_t staged_ext = 0;
    int chunks = 0;
    // the fused pileup step of staged sessions (build_resident_index, prepare_resident_pileup)
    ResidentIndexHost idx;
    DevBuf idx_keys, idx_long_key, idx_long_row, idx_scal;
    // the fetch plan's merged index queries, (rid, beg) order: every record overlapping one of them is resident
    std::vector<QueryInterval> queries;

    StagedRecords() = default;
    StagedRecords(const StagedRecords&) = delete;
    ~StagedRecords() {
        if (raw_all.p || offs_all.p || batch_table.p || idx_keys.p || idx_scal.p) {
            cudaSetDevice(dev);
            cudaDeviceSynchronize();
            raw_all.release(); offs_all.release(); batch_table.release();
            idx_keys.release(); idx_long_key.release(); idx_long_row.release(); idx_scal.release();
        }
    }
};

// ---------------------------------------------------------------------------------------------------------------
// Session: one BAM + one region set on one device.
// ---------------------------------------------------------------------------------------------------------------
class Session {
public:
    // dev >= 0 overrides the device opts names (device-output calls run where the caller's buffer is)
    Session(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
            const int32_t* loc, const int32_t* width, const int8_t* strand, const bsg_opts* opts, int dev = -1)
        : bamp_(open_bam(bampath)), bam_(*bamp_), opts_(effective_opts(opts)) {
        resolve_regions(bam_, R, seq_levels, n_levels, seq_idx, loc, width, strand, &rg_);
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
            fail(BSG_ECUDA, "no CUDA device available (libbamsignals_cuda has no CPU fallback)");
        if (dev < 0) dev = opts_.n_devices > 0 ? opts_.devices[0] : 0;
        if (dev < 0 || dev >= ndev || dev >= 16) fail(BSG_EARG, "invalid CUDA device index");
        ctx_ = &g_ctx[dev];
        ctx_->ensure_init(dev);
        ctx_->ev_next = 0;
        pool_ = &get_pool(opts_.inflate_threads);
        res_->dev = dev;
        memset(&tm_, 0, sizeof tm_);
        tm_.n_devices = 1;
    }

    // One shard of a multi-device call: regions already resolved, device chosen by the caller.
    Session(std::shared_ptr<BamFile> bam, Regions rg, const bsg_opts& o, int dev)
        : bamp_(std::move(bam)), bam_(*bamp_), opts_(o), rg_(std::move(rg)) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
            fail(BSG_ECUDA, "no CUDA device available (libbamsignals_cuda has no CPU fallback)");
        if (dev < 0 || dev >= ndev || dev >= 16) fail(BSG_EARG, "invalid CUDA device index");
        ctx_ = &g_ctx[dev];
        ctx_->ensure_init(dev);
        ctx_->ev_next = 0;
        pool_ = &get_pool(opts_.inflate_threads);
        res_->dev = dev;
        memset(&tm_, 0, sizeof tm_);
        tm_.n_devices = 1;
    }

    // A view of a staged session (bsg_stage_view): the resident records, options and device of `st`, the region set `rg`.
    // view_halo is how far around every region of rg the records are known to be resident (view_halo()).
    Session(const Session& st, Regions rg, int64_t view_halo)
        : bamp_(st.bamp_), bam_(*bamp_), opts_(st.opts_), rg_(std::move(rg)), ctx_(st.ctx_), res_(st.res_),
          is_view_(true), view_halo_(view_halo) {
        pool_ = &get_pool(opts_.inflate_threads);
        memset(&tm_, 0, sizeof tm_);
        tm_.n_devices = 1;
        tm_.bytes_compressed = st.tm_.bytes_compressed;
        tm_.bytes_inflated = st.tm_.bytes_inflated;
        tm_.n_batches = st.tm_.n_batches;
    }

    // The largest halo `a` around the regions of `rg` for which this staged session holds every record: each region
    // [loc, loc + width) with width > 0, widened by a on both sides and clamped at 0 as the planner clamps, must lie inside
    // one of the index queries the open sent (after their merge; the index returns every record that overlaps a query).
    // INT64_MAX when rg has no non-empty region.  BSG_EARG, naming the 1-based region, when some region has no such a >= 0.
    int64_t view_halo(const Regions& rg) const {
        const std::vector<QueryInterval>& q = res_->queries;
        int64_t halo = INT64_MAX;
        for (int64_t i = 0; i < rg.R; ++i) {
            if (rg.width[i] == 0) continue;
            const int64_t loc = rg.loc[i], end = loc + rg.width[i], p = std::max<int64_t>(0, loc);
            // the last query on this contig that begins at or before p (the merged queries are disjoint)
            auto it = std::upper_bound(q.begin(), q.end(), std::make_pair(rg.rid[i], p), [](const std::pair<int32_t, int64_t>& k, const QueryInterval& x) {
                return k.first != x.rid ? k.first < x.rid : k.second < x.beg;
            });
            int64_t a = -1;
            if (it != q.begin() && (it - 1)->rid == rg.rid[i]) {
                const QueryInterval& x = *(it - 1);
                a = x.end - end;
                if (x.beg > 0) a = std::min(a, loc - x.beg);
            }
            if (a < 0)
                fail(BSG_EARG, "region " + std::to_string(i + 1) + " of the view lies outside what the staged session fetched; "
                               "stage a session over it (or a wider ext_hint) to count it");
            halo = std::min(halo, a);
        }
        return halo;
    }

    // The fetch plan (index queries + BGZF header scan) depends only on the regions and `ext`: it can run on its own
    // thread while the caller builds and uploads the tiles (both take 10-15 ms for 100 k regions).
    void start_plan(int64_t ext) {
        if (ext < 0) fail(BSG_EARG, "negative 'ext' values don't make sense");           // src/bamsignals.cpp:243
        rg_.sorted_order();                              // lazily cached: compute it before two threads ask for it
        segs_.clear();
        plan_err_ = Error{0, ""};
        plan_ext_ = ext;
        plan_thread_ = std::thread([this, ext] {
            const double t0 = now_ms();
            Nvtx r("bsg:plan_fetch");
            try { plan_fetch(bam_, rg_, ext, kSegCBytes, *pool_, &segs_); }
            catch (Error& e) { plan_err_ = e; }
            catch (std::exception& e) { plan_err_ = Error{BSG_EARG, std::string("internal error: ") + e.what()}; }
            plan_ms_ = now_ms() - t0;
        });
    }

    // Work of a streaming call that needs neither the plan nor the device pipeline - building and uploading the tiles,
    // starting the result streamer - runs on a thread of its own next to the planner thread; stage() joins it before the
    // first batch is decoded (C2: 8-11 ms that used to sit in front of the first upload).
    void defer_setup(std::function<void()> f) {
        setup_err_ = Error{0, ""};
        setup_thread_ = std::thread([this, f] {
            Nvtx r("bsg:setup (tiles + streamer)");
            try {
                BSG_CUDA(cudaSetDevice(ctx_->dev));
                f();
            } catch (Error& e) { setup_err_ = e; }
            catch (std::exception& e) { setup_err_ = Error{BSG_EARG, std::string("internal error: ") + e.what()}; }
        });
    }
    void run_deferred() {
        if (!setup_thread_.joinable()) return;
        setup_thread_.join();
        if (setup_err_.code) throw setup_err_;
    }
    cudaStream_t setup_stream() const { return ctx_->s_d2h; }      // idle until the result streamer starts

    // Fetch + upload (+ decode unless keep_raw) everything the regions need with halo `ext`.
    void stage(int64_t ext, bool keep_raw) {
        if (ext < 0) fail(BSG_EARG, "negative 'ext' values don't make sense");           // src/bamsignals.cpp:243
        double t0 = now_ms();
        res_->keep_raw = keep_raw;
        res_->staged_ext = ext;
        if (plan_thread_.joinable()) {
            plan_thread_.join();
            if (plan_err_.code) throw plan_err_;
            if (plan_ext_ != ext) fail(BSG_EARG, "internal error: plan started with another halo");
            t0 = now_ms() - plan_ms_;                    // ms_plan reports the plan's own duration, ms_fetch what follows it
        } else {
            segs_.clear();
            res_->queries.clear();
            plan_fetch(bam_, rg_, ext, kSegCBytes, *pool_, &segs_, keep_raw ? &res_->queries : nullptr);
        }
        if (prefault_out_) { prefault_output(prefault_out_, prefault_total_); prefault_out_ = nullptr; }
        // 1 = device inflate, -1 = host zlib pool, 0 = default: device inflate unless the job is tiny.  A device-inflate
        // launch lasts as long as ONE BGZF block takes a single lane (a few ms) however few blocks there are, and a file
        // with a handful of index entry points leaves the device record walk a few long serial chains (the reference's
        // 4.5 MB fixture: 3 entry points, 19 ms per call); the worker pool inflates and walks such a job in well under a
        // millisecond.
        uint64_t plan_usize = 0;
        for (const Segment& sg : segs_) plan_usize += sg.usize;
        const bool gpu = opts_.gpu_inflate > 0 || (opts_.gpu_inflate == 0 && plan_usize > kSmallJobBytes);
        const int64_t batch_bytes = opts_.batch_bytes > 0 ? opts_.batch_bytes : (gpu ? kDefaultGpuBatch : kDefaultBatch);
        // group segments into batches
        batches_.clear();
        uint64_t max_batch = 0, total_bytes = 0, total_c = 0;
        int64_t rows_cap = 0;
        // Device inflate: a launch keeps n_sm x 64 BGZF blocks in flight and its time is that of ONE block, however many
        // streams are busy - so a batch is one such "wave" of blocks (~0.6 GB inflated on a B200), the first one half a
        // wave (nothing overlaps its upload).  opts.batch_bytes > 0 overrides with a byte limit.
        const uint64_t wave_blocks = (gpu && opts_.batch_bytes <= 0) ? uint64_t(inflate_wave_blocks(ctx_->n_sm)) : ~0ull;
        for (size_t i = 0; i < segs_.size();) {
            auto b = std::make_unique<Batch>();
            b->seg_first = i;
            const bool first_short = gpu && !keep_raw && opts_.batch_bytes <= 0 && i == 0;
            const uint64_t limit = uint64_t(batch_bytes);
            const uint64_t limit_blocks = first_short ? wave_blocks / 2 : wave_blocks;
            uint64_t acc = 0, nblk = 0;
            while (i < segs_.size() && (acc == 0 || (acc + segs_[i].usize <= limit && nblk + segs_[i].blocks.size() <= limit_blocks))) {
                acc += (segs_[i].usize + 15) & ~15ull;
                nblk += segs_[i].blocks.size();
                ++i;
            }
            b->seg_last = i;
            b->bytes = acc;
            if (acc >= (1ull << 32) - 64) fail(BSG_ENOMEM, "a single fetch segment exceeds 4 GiB");
            max_batch = std::max(max_batch, acc);
            for (size_t k = b->seg_first; k < b->seg_last; ++k) {
                rows_cap += int64_t((segs_[k].uend - segs_[k].ubeg) / kMinRecord) + 1;
                total_bytes += segs_[k].usize; total_c += segs_[k].csize;
            }
            batches_.push_back(std::move(b));
        }
        res_->rows_cap = (rows_cap + 3) & ~int64_t(3);
        tm_.bytes_compressed = int64_t(total_c);
        tm_.bytes_inflated = int64_t(total_bytes);
        tm_.n_batches = int64_t(batches_.size());
        tm_.ms_plan = now_ms() - t0;
        if (getenv("BSG_DEBUG"))
            fprintf(stderr, "[bsg] plan %.1f ms: %zu segments, %zu batches, %.1f MB compressed, %.1f MB inflated, rows_cap %lld\n",
                    tm_.ms_plan, segs_.size(), batches_.size(), total_c / 1e6, total_bytes / 1e6, (long long)res_->rows_cap);

        // device + pinned buffers
        DeviceCtx& c = *ctx_;
        const size_t max_offs = size_t(max_batch / kMinRecord) + 1;
        size_t max_segs = 0;
        for (auto& b : batches_) max_segs = std::max(max_segs, b->seg_last - b->seg_first);
        if (keep_raw) {
            size_t tot = 0;
            for (auto& b : batches_) tot += (b->bytes + 64 + 255) & ~255ull;
            res_->raw_all.ensure(tot + 64);
            size_t offs_tot = size_t(res_->rows_cap) + batches_.size() + 8;
            if (gpu) { offs_tot = 8; for (auto& b : batches_) offs_tot += size_t(b->bytes / kMinRecord) + 2; }
            res_->offs_all.ensure(offs_tot * sizeof(uint32_t));
        }
        ensure_table(res_->rows_cap);
        c.scalars.ensure(sizeof(DeviceScalars));
        BSG_CUDA(cudaMemsetAsync(c.scalars.p, 0, sizeof(DeviceScalars), c.s_comp));
        if (gpu) {
            run_pipeline_gpu(max_batch, max_offs);
            run_deferred();                              // (a job without batches)
            tm_.ms_fetch = now_ms() - t0 - tm_.ms_plan;
            return;
        }
        run_deferred();
        for (int s = 0; s < kSlots && s < int(batches_.size()); ++s) {
            c.h_raw[s].ensure(max_batch + 64);
            c.h_offs[s].ensure((max_offs + max_segs + 8) * sizeof(uint32_t));
            if (!keep_raw) {
                c.d_raw[s].ensure(max_batch + 64);
                c.d_offs[s].ensure((max_offs + 8) * sizeof(uint32_t));
            }
        }
        run_pipeline();
        tm_.ms_fetch = now_ms() - t0 - tm_.ms_plan;
    }

    // A staged call may only look as far around its regions as the session fetched: the reference widens every index
    // query by `ext` (src/bamsignals.cpp:255-256,457,487); with a smaller halo, reads near the region borders would
    // silently be missing.
    // A view may look as far as its regions' resident halo (view_halo()).
    void require_ext(int64_t ext) const {
        if (is_view_) {
            if (ext > view_halo_)
                fail(BSG_EARG, "this call needs a halo of " + std::to_string(ext) + " bp around the regions, the staged records reach " +
                               std::to_string(view_halo_) + " bp around every region of this view");
            return;
        }
        if (ext > res_->staged_ext)
            fail(BSG_EARG, "this call needs a halo of " + std::to_string(ext) + " bp around the regions, the session was staged with ext_hint = " +
                           std::to_string(res_->staged_ext));
    }

    // Staged sessions: decode + filter every resident raw batch again (K1) in ONE launch, timed.
    void decode_resident(Mode mode, const FilterParams& fp, int ss = 0) {
        DeviceCtx& c = *ctx_;
        fused_ = false;
        BSG_CUDA(cudaMemsetAsync(c.scalars.p, 0, sizeof(DeviceScalars), c.s_comp));
        if (res_->batches.empty()) return;
        ensure_table(res_->rows_cap);            // (a view's first table-path call on this device)
        Span sp{c.timing_event(), c.timing_event()};
        BSG_CUDA(cudaEventRecord(sp.a, c.s_comp));
        launch_decode_table(res_->batch_table.as<DecodeBatch>(), int(res_->batches.size()), res_->chunks, table(),
                            mode == MODE_COVERAGE, ss != 0, fp, c.scalars.as<DeviceScalars>(), c.s_comp);
        BSG_CUDA(cudaEventRecord(sp.b, c.s_comp));
        kt_.decode.push_back(sp); kt_.launches += 1;
    }

    // The caller's flat output buffer is usually freshly allocated (np.empty / R allocVector): its pages fault in on
    // first touch, which would otherwise happen inside the final D2H scatter.  Touch them on the worker pool now,
    // while the GPU is busy inflating (the workers are mostly idle in that phase).
    // Started before planning (measured: starting it after the plan makes it compete with the first batch's upload,
    // which is on the critical path; C2 272 -> 289 ms).
    // (the pre-faulting starts when the plan is done: page faults and the planner's allocations fight over the process's
    // mmap lock - plan 7 -> 15-23 ms when both ran together)
    void request_prefault(int32_t* out, int64_t total) { prefault_out_ = out; prefault_total_ = total; }
    void prefault_output(int32_t* out, int64_t total) {
        if (!out || total < (int64_t(1) << 22)) return;
        // One atomic `or 0` per page: a write fault that leaves the contents alone, so it may run concurrently with
        // the scatter of early tiles.  (MADV_POPULATE_WRITE was measured too: it holds the process's mmap lock for
        // whole ranges and starved the planner's allocations, plan 13 -> 39 ms.)
        const size_t bytes = size_t(total) * 4, piece = size_t(2) << 20;
        const int n = int((bytes + piece - 1) / piece);
        {
            std::lock_guard<std::mutex> g(pf_m_);
            pf_left_ += n;
        }
        uint8_t* base = reinterpret_cast<uint8_t*>(out);
        for (int k = 0; k < n; ++k)
            pool_->submit_low([this, base, bytes, piece, k](int) {
                const size_t lo = size_t(k) * piece, hi = std::min(bytes, lo + piece);
                for (size_t o = lo; o < hi; o += 4096) __atomic_fetch_or(base + o, uint8_t(0), __ATOMIC_RELAXED);
                std::lock_guard<std::mutex> g(pf_m_);
                if (--pf_left_ == 0) pf_cv_.notify_all();
            });
    }
    void wait_prefault() {
        std::unique_lock<std::mutex> lk(pf_m_);
        pf_cv_.wait(lk, [&] { return pf_left_ == 0; });
    }
    ~Session() {
        if (plan_thread_.joinable()) plan_thread_.join();
        if (setup_thread_.joinable()) setup_thread_.join();
        stop_streamer(true);
        wait_prefault();
        if (fused_rng_.p) {
            cudaSetDevice(ctx_->dev);
            cudaDeviceSynchronize();
            fused_rng_.release();
        }
    }                                            // res_: the resident records go with the last handle that shares them

    // Tiles depend only on the regions and on (mode, binsize, ss, layout): build + upload them before any device
    // work of the call is queued, and keep them for the next call of a staged session.
    // the layout must be the one allocateList gives (src/bamsignals.cpp:139-192): the host scatter trusts it
    void validate_layout(Mode mode, int32_t binsize, int ss, const int64_t* out_offsets) const {
        const int64_t R = rg_.R;
        if (!out_offsets) fail(BSG_EARG, "out_offsets is required");
        {
            const int64_t mult = ss ? 2 : 1;
            if (R > 0 && out_offsets[0] < 0) fail(BSG_EARG, "out_offsets must not be negative");
            for (int64_t i = 0; i < R; ++i) {
                const int64_t want = mode == MODE_COUNT ? mult
                                   : (mode == MODE_COVERAGE ? mult * int64_t(rg_.width[i])
                                                            : mult * ((int64_t(rg_.width[i]) + binsize - 1) / binsize));
                if (out_offsets[i + 1] - out_offsets[i] != want)
                    fail(BSG_EARG, "out_offsets[" + std::to_string(i + 1) + "] - out_offsets[" + std::to_string(i) + "] is " +
                                   std::to_string(out_offsets[i + 1] - out_offsets[i]) + ", the layout of this call needs " + std::to_string(want) +
                                   " (see bsg_output_layout)");
                // the stranded read table tells the strands apart by the sign of a read's end (kernels.cuh), so a read that
                // ends before position 0 is not counted: no region may reach there
                if (mode == MODE_COVERAGE && ss && rg_.loc[i] < 0)
                    fail(BSG_EARG, "strand-specific coverage needs regions that start at position 1 or later (region " +
                                   std::to_string(i + 1) + ")");
            }
        }
    }
    // up: the stream the tile table is uploaded on (and waited for); not the compute stream once inflates are queued on it
    // The tiles' out_off depends on where the kernels write: DeviceCtx::out in tile order, or the caller's device buffer
    // in the caller's layout (use_device_output) - the cached table is only reused for the same kind.
    void prepare_tiles(Mode mode, int32_t binsize, int ss, const int64_t* out_offsets, cudaStream_t up = nullptr) {
        Nvtx r("bsg:tiles");
        DeviceCtx& c = *ctx_;
        const int64_t R = rg_.R;
        if (!up) up = c.s_comp;
        if (!out_offsets) fail(BSG_EARG, "out_offsets is required");
        if (tiles_valid_ && my_tiles_gen_ == c.tiles_gen && tiles_mode_ == mode && tiles_binsize_ == binsize && tiles_ss_ == ss &&
            tiles_caller_ == dev_out_.on && tiles_offsets_.size() == size_t(R + 1) &&
            memcmp(tiles_offsets_.data(), out_offsets, size_t(R + 1) * 8) == 0)
            return;
        validate_layout(mode, binsize, ss, out_offsets);
        HostTiles& ht = ht_;
        ht = HostTiles();
        // Tile size: as large as shared memory allows (fewer halo re-reads), but small enough that the launch has
        // >= ~16 CTAs per SM: a few huge regions (C4: 24 whole chromosomes) must still fill 148 SMs.
        const int64_t total_ints = out_offsets[R];
        int tile_ints = kTileInts;
        while (tile_ints > 512 && total_ints / tile_ints < 148 * 16) tile_ints >>= 1;
        make_tiles(rg_, mode, binsize, ss, out_offsets, tile_ints, &ht);
        const int64_t nt = ht.size();
        // The device result buffer is laid out in TILE order (tile t at dev_off[t]): a run of consecutive tiles is one
        // contiguous D2H copy, whatever order the caller's regions came in; the host scatters tiles to the caller.
        tile_dev_off_.assign(size_t(nt) + 1, 0);
        for (int64_t t = 0; t < nt; ++t) tile_dev_off_[t + 1] = tile_dev_off_[t] + ht.ints[t];
        c.tiles_i32.ensure(size_t(nt) * 4 * sizeof(int32_t) + 64);
        c.tiles_i64.ensure(size_t(nt) * 3 * sizeof(int64_t) + 64);
        int32_t* ti = c.tiles_i32.as<int32_t>();
        int64_t* tl = c.tiles_i64.as<int64_t>();
        if (nt) {
            c.h_tiles.ensure(size_t(nt) * 24);
            uint8_t* h = c.h_tiles.as<uint8_t>();
            memcpy(h, ht.rid.data(), nt * 4); memcpy(h + nt * 4, ht.loc.data(), nt * 4);
            memcpy(h + nt * 8, ht.len.data(), nt * 4); memcpy(h + nt * 12, ht.strand.data(), nt * 4);
            memcpy(h + nt * 16, dev_out_.on ? ht.out_off.data() : tile_dev_off_.data(), nt * 8);
            BSG_CUDA(cudaMemcpyAsync(ti, h, nt * 16, cudaMemcpyHostToDevice, up));
            BSG_CUDA(cudaMemcpyAsync(tl, h + nt * 16, nt * 8, cudaMemcpyHostToDevice, up));
            BSG_CUDA(cudaStreamSynchronize(up));         // h_tiles is reused by the next call; the kernels that read the tiles are launched after this
        }
        my_tiles_gen_ = ++c.tiles_gen;
        n_tiles_ = nt;
        max_tile_ints_ = ht.max_tile_ints;
        tiles_mode_ = mode; tiles_binsize_ = binsize; tiles_ss_ = ss; tiles_caller_ = dev_out_.on;
        tiles_offsets_.assign(out_offsets, out_offsets + R + 1);
        tiles_valid_ = true;
    }

    // ---- counting: begin_count() / advance() / finish_count() ---------------------------------------------------------
    // The reference finishes a region as soon as the sorted read stream has passed its end + ext
    // (src/bamsignals.cpp:278); the same observation lets the result leave the device while later batches are still
    // being inflated: a tile is final once the last decoded record's (tid, pos) is >= (rid, end + ext).
    void begin_count(Mode mode, const FilterParams& fp, int32_t binsize, int ss, int64_t ext, int32_t* out,
                     const int64_t* out_offsets, int32_t* const* out_ptrs, bool want_output, cudaStream_t tiles_stream = nullptr) {
        DeviceCtx& c = *ctx_;
        const int64_t R = rg_.R;
        stop_streamer(true);                         // left over from a call that failed half-way (staged sessions persist)
        prepare_tiles(mode, binsize, ss, out_offsets, tiles_stream);
        cnt_ = CountState();
        cnt_.active = true; cnt_.mode = mode; cnt_.fp = fp; cnt_.binsize = binsize; cnt_.ss = ss;
        cnt_.out = out; cnt_.out_offsets = out_offsets; cnt_.out_ptrs = out_ptrs;
        const int64_t total = out_offsets[R];
        cnt_.want_output = want_output && total > 0 && !dev_out_.on;
        if (cnt_.want_output && !out && !out_ptrs) fail(BSG_EARG, "either out or out_ptrs must be given");
        tm_.n_tiles = n_tiles_;
        tm_.out_elems = total;
        if (dev_out_.on) {
            cnt_.dst = dev_out_.ptr;
        } else if (!runs_.res) {
            c.out.ensure(size_t(total) * sizeof(int32_t) + 64);
            cnt_.dst = c.out.as<int32_t>();
        }
        // (rid, end + ext) as one key, prefix-maxed over the tile order: tiles [0, t) are final iff final_key[t-1] <= frontier
        tile_final_key_.resize(size_t(n_tiles_));
        uint64_t run = 0;
        for (int64_t t = 0; t < n_tiles_; ++t) {
            const int64_t e = std::min<int64_t>(int64_t(ht_.loc[t]) + ht_.len[t] + ext, INT32_MAX);
            run = std::max(run, uint64_t(uint32_t(ht_.rid[t])) << 32 | uint64_t(uint32_t(std::max<int64_t>(e, 0))));
            tile_final_key_[t] = run;
        }
        os_bytes_ = 0;
        if (cnt_.want_output) start_streamer();
    }

    // Rows [0, rows) of the read table are decoded + filtered and `frontier` = (tid, pos) of the last of them:
    // count + ship every tile that can no longer change.
    void advance(int64_t rows, uint32_t f_tid, int32_t f_pos) {
        if (!cnt_.active) return;
        cnt_.rows_ready = rows;
        const uint64_t key = uint64_t(f_tid) << 32 | uint64_t(uint32_t(std::max(f_pos, 0)));
        const int64_t t_new = std::upper_bound(tile_final_key_.begin(), tile_final_key_.end(), key) - tile_final_key_.begin();
        // worth a launch + copy only in decent portions; runs are counted at the end of the call
        if (opts_.stream_min_ints < 0 || runs_.res) return;
        const int64_t min_ints = opts_.stream_min_ints > 0 ? opts_.stream_min_ints : (int64_t(4) << 20);
        if (t_new > cnt_.t_done && tile_dev_off_[t_new] - tile_dev_off_[cnt_.t_done] >= min_ints) count_tiles(cnt_.t_done, t_new);
    }

    void finish_count() {
        Nvtx r("bsg:finish_count+d2h");
        DeviceCtx& c = *ctx_;
        cnt_.rows_ready = res_->n_rows;
        if (n_tiles_ > cnt_.t_done || runs_.res) count_tiles(cnt_.t_done, n_tiles_);      // runs: also without tiles
        DeviceScalars* sc = c.scalars.as<DeviceScalars>();
        BSG_CUDA(cudaGetLastError());
        double scalar_bytes = double(sizeof(DeviceScalars));
        if (dev_out_.on || runs_.res) {
            // nothing of the result comes back: only the header (status, candidates) and the used kept[] slots
            DeviceScalars* hs = c.h_scalars.as<DeviceScalars>();
            const size_t head = offsetof(DeviceScalars, pad2), pitch = kKeptStride * sizeof(unsigned long long);
            BSG_CUDA(cudaMemcpyAsync(hs, sc, head, cudaMemcpyDeviceToHost, cnt_stream()));
            BSG_CUDA(cudaMemcpy2DAsync(hs->kept, pitch, sc->kept, pitch, sizeof(unsigned long long), kKeptSlots,
                                       cudaMemcpyDeviceToHost, cnt_stream()));
            scalar_bytes = double(head + kKeptSlots * sizeof(unsigned long long));
        } else {
            BSG_CUDA(cudaMemcpyAsync(c.h_scalars.p, sc, sizeof(DeviceScalars), cudaMemcpyDeviceToHost, cnt_stream()));
        }
        const double t_d2h = now_ms();
        stop_streamer(false);
        BSG_CUDA(cudaStreamSynchronize(cnt_stream()));
        BSG_CUDA(cudaStreamSynchronize(c.s_comp));
        hi_prio_ = false;
        tm_.ms_d2h = now_ms() - t_d2h;
        tm_.bytes_d2h = os_bytes_ + scalar_bytes;
        cnt_.active = false;
        const DeviceScalars* hs = c.h_scalars.as<DeviceScalars>();
        check_status(hs->status | (res_->keep_raw ? res_->idx.status : 0u));     // staged: the resident records' bits, every call
        tm_.records = res_->n_rows;
        tm_.records_kept = 0;
        for (int k = 0; k < kKeptSlots; ++k) tm_.records_kept += int64_t(hs->kept[k * kKeptStride]);
        if (fused_) tm_.records_kept = -1;                              // only the examined rows were filtered
        tm_.candidates = int64_t(hs->candidates);
    }

    void count(Mode mode, const FilterParams& fp, int32_t binsize, int ss, int32_t* out, const int64_t* out_offsets,
               int32_t* const* out_ptrs, bool want_output) {
        begin_count(mode, fp, binsize, ss, 0, out, out_offsets, out_ptrs, want_output);
        finish_count();
    }

    // Where the counting kernels of the next call write.  use_device_output: straight into the caller's device buffer
    // d_out at the caller's offsets (no DeviceCtx::out, no result streamer, nothing of the result crosses PCIe); every
    // library stream that writes d_out first waits for what `caller` had queued at this point (e.g. work on memory the
    // caller's allocator just handed out again).  use_host_output: the default, DeviceCtx::out in tile order + streamer.
    void use_device_output(int32_t* d_out, cudaStream_t caller) {
        BSG_CUDA(cudaEventRecord(ctx_->ev_caller, caller));
        dev_out_ = DeviceOutput{true, d_out};
        runs_ = RunsOutput{};
    }
    void use_host_output() { dev_out_ = DeviceOutput{}; runs_ = RunsOutput{}; }
    // The next call counts coverage or a profile as runs (count_runs) into `res`, and fills the caller's run_offsets
    // (R + 1 entries, or 2R + 1 when strand-specific).
    void use_runs_output(bsg_runs* res, int64_t* run_offsets) {
        dev_out_ = DeviceOutput{};
        runs_ = RunsOutput{res, run_offsets};
    }
    // bsg_output_layout() of bamCoverage (strand-specific with ss) for this session's regions: the tiles are cut from it
    std::vector<int64_t> coverage_layout(int ss) const {
        const int64_t mult = ss ? 2 : 1;
        std::vector<int64_t> off(size_t(rg_.R) + 1, 0);
        for (int64_t i = 0; i < rg_.R; ++i) off[i + 1] = off[i] + mult * rg_.width[i];
        return off;
    }
    // bsg_output_layout() of bamProfile (binsize >= 1) for this session's regions
    std::vector<int64_t> profile_layout(int32_t binsize, int ss) const {
        const int64_t mult = ss ? 2 : 1;
        std::vector<int64_t> off(size_t(rg_.R) + 1, 0);
        for (int64_t i = 0; i < rg_.R; ++i) off[i + 1] = off[i] + mult * ((int64_t(rg_.width[i]) + binsize - 1) / binsize);
        return off;
    }
    int device() const { return ctx_->dev; }
    const BamFile& bam() const { return bam_; }
    int64_t regions() const { return rg_.R; }

private:
    struct CountState {
        bool active = false, want_output = false;
        Mode mode = MODE_COUNT;
        FilterParams fp{};
        int32_t binsize = 1;
        int ss = 0;
        int32_t* out = nullptr;
        const int64_t* out_offsets = nullptr;
        int32_t* const* out_ptrs = nullptr;
        int32_t* dst = nullptr;                  // what the counting kernels write: DeviceCtx::out or the caller's d_out
        int64_t rows_ready = 0, t_done = 0;
    };
    struct DeviceOutput { bool on = false; int32_t* ptr = nullptr; };
    struct RunsOutput { bsg_runs* res = nullptr; int64_t* run_offsets = nullptr; };
    struct OutJob { int slot; int64_t t0, t1; cudaEvent_t computed; };

    cudaStream_t cnt_stream() const { return hi_prio_ ? ctx_->s_hi : ctx_->s_comp; }

    // K3 + K4/K5 for tiles [t0, t1) over the rows decoded so far, then hand them to the output streamer
    void count_tiles(int64_t t0, int64_t t1) {
        Nvtx r("bsg:join+count");
        DeviceCtx& c = *ctx_;
        cudaStream_t st = cnt_stream();
        const int64_t n = t1 - t0;
        const TileTable tt = tile_table(t0);
        DeviceScalars* sc = c.scalars.as<DeviceScalars>();
        int32_t* c0 = c.c0.as<int32_t>();
        int32_t* c1 = c.c1.as<int32_t>();
        if (fused_) { count_tiles_fused(tt, t0, t1, st); return; }
        {
            Span sp{c.timing_event(), c.timing_event()};
            BSG_CUDA(cudaEventRecord(sp.a, st));
            launch_join(table(), cnt_.rows_ready, tt, n, sc, st);
            BSG_CUDA(cudaEventRecord(sp.b, st));
            kt_.join.push_back(sp); kt_.launches += 1;
        }
        if (runs_.res) { count_runs(tt, n, st); cnt_.t_done = t1; return; }
        if (dev_out_.on) BSG_CUDA(cudaStreamWaitEvent(st, c.ev_caller, 0));
        {
            Span sp{c.timing_event(), c.timing_event()};
            BSG_CUDA(cudaEventRecord(sp.a, st));
            if (cnt_.mode == MODE_COUNT) launch_count(tt, n, c0, c1, cnt_.ss, cnt_.dst, sc, st);
            else if (cnt_.mode == MODE_PROFILE) launch_profile(tt, n, c0, c1, cnt_.ss, cnt_.binsize, max_tile_ints_, cnt_.dst, sc, st);
            else launch_coverage(tt, n, c0, c1, cnt_.ss, max_tile_ints_, cnt_.dst, sc, st);
            BSG_CUDA(cudaEventRecord(sp.b, st));
            kt_.count.push_back(sp); kt_.launches += 1;
            if (cnt_.want_output) ship_tiles(t0, t1, sp.b);
        }
        cnt_.t_done = t1;
    }

    // the device tile table from tile t0 on
    TileTable tile_table(int64_t t0) const {
        const int64_t nt = n_tiles_;
        int32_t* ti = ctx_->tiles_i32.as<int32_t>();
        int64_t* tl = ctx_->tiles_i64.as<int64_t>();
        return TileTable{ti + t0, ti + nt + t0, ti + 2 * nt + t0, ti + 3 * nt + t0, tl + t0, tl + nt + t0, tl + 2 * nt + t0};
    }

    // K3f + K4f (staged pileup calls, DESIGN.md §13): the tiles' row ranges from the resident index, then the counts
    // straight from the raw records.
    void count_tiles_fused(const TileTable& tt, int64_t t0, int64_t t1, cudaStream_t st) {
        DeviceCtx& c = *ctx_;
        const int64_t n = t1 - t0;
        fused_rng_.ensure(size_t(2 * n_tiles_) * sizeof(int64_t) + 64);
        int64_t* llo = fused_rng_.as<int64_t>() + t0;
        int64_t* lhi = fused_rng_.as<int64_t>() + n_tiles_ + t0;
        const ResidentView v = resident_view();
        {
            Span sp{c.timing_event(), c.timing_event()};
            BSG_CUDA(cudaEventRecord(sp.a, st));
            launch_join_fused(v, tt, llo, lhi, n, fused_h_, c.scalars.as<DeviceScalars>(), st);
            BSG_CUDA(cudaEventRecord(sp.b, st));
            kt_.join.push_back(sp); kt_.launches += 1;
        }
        if (dev_out_.on) BSG_CUDA(cudaStreamWaitEvent(st, c.ev_caller, 0));
        Span sp{c.timing_event(), c.timing_event()};
        BSG_CUDA(cudaEventRecord(sp.a, st));
        launch_pileup_fused(v, tt, llo, lhi, n, cnt_.ss, cnt_.mode == MODE_COUNT ? 0 : cnt_.binsize, max_tile_ints_, cnt_.fp, cnt_.dst, st);
        BSG_CUDA(cudaEventRecord(sp.b, st));
        kt_.count.push_back(sp); kt_.launches += 1;
        if (cnt_.want_output) ship_tiles(t0, t1, sp.b);
        cnt_.t_done = t1;
    }

    // Coverage (DESIGN.md §10, §12) or a profile (§11) as runs over ALL tiles (t0 == 0, advance() never counts early):
    // count pass + scans, the list spans come back (the only D2H besides the control scalars), the result is allocated at
    // its exact size, then the write pass.  A list is a region, or with ss one strand row of a region (list mult * i + a);
    // every tile holds one virtual tile per row: row a of the j-th of region i's n_i tiles, T_i its first, is
    // v = mult * T_i + a * n_i + j, so that a list's pieces are consecutive (identity when mult is 1).
    // Device memory: 28 bytes per virtual tile (+4 with ss), 24 per list, 8 per run.
    void count_runs(const TileTable& tt, int64_t nt, cudaStream_t st) {
        DeviceCtx& c = *ctx_;
        if (nt != n_tiles_) fail(BSG_EARG, "internal error: runs are counted over all tiles at once");
        const bool profile = cnt_.mode == MODE_PROFILE;
        const int64_t mult = cnt_.ss ? 2 : 1;
        const int64_t R = rg_.R, L = mult * R, nv = mult * nt;
        const int64_t up = mult == 2 ? 3 : 2;                  // uploaded per virtual tile: list, rel (and vt with ss)
        runs_tiles_.resize(size_t(nv * up));
        for (int64_t t0 = 0; t0 < nt;) {
            const int64_t i = ht_.region[t0];
            int64_t t1 = t0 + 1;
            while (t1 < nt && ht_.region[t1] == i) ++t1;
            for (int64_t t = t0; t < t1; ++t)
                for (int64_t a = 0; a < mult; ++a) {
                    const int64_t v = mult * t0 + a * (t1 - t0) + (t - t0);
                    runs_tiles_[v] = int32_t(mult * i + a);
                    runs_tiles_[nv + v] = int32_t((ht_.out_off[t] - tiles_offsets_[i]) / mult);
                    if (mult == 2) runs_tiles_[2 * nv + a * nt + t] = int32_t(v);
                }
            t0 = t1;
        }
        c.runs_i32.ensure(size_t(nv) * (up + 3) * sizeof(int32_t) + 64);
        c.runs_i64.ensure((size_t(nv) + 3 * size_t(L) + 1) * sizeof(int64_t) + 64);
        c.h_runs.ensure((size_t(L) + 1) * sizeof(int64_t));
        int32_t* ri = c.runs_i32.as<int32_t>();
        int64_t* rl = c.runs_i64.as<int64_t>();
        int32_t* rw = ri + up * nv;
        const RunTiles rt{ri, ri + nv, rw, rw + nv, rw + 2 * nv, rl, rl + nv, rl + nv + L};
        const int32_t* vt = mult == 2 ? ri + 2 * nv : nullptr;
        int64_t* run_off = rl + nv + 2 * L;
        int32_t* c0 = c.c0.as<int32_t>();
        int32_t* c1 = c.c1.as<int32_t>();
        Span sp{c.timing_event(), c.timing_event()};
        BSG_CUDA(cudaEventRecord(sp.a, st));
        if (nv) BSG_CUDA(cudaMemcpyAsync(ri, runs_tiles_.data(), size_t(nv * up) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        if (L) BSG_CUDA(cudaMemsetAsync(rt.rfirst, 0, size_t(L) * 2 * sizeof(int64_t), st));
        if (profile) launch_profile_runs(tt, nt, c0, c1, cnt_.ss, cnt_.binsize, max_tile_ints_, rt, vt, L, run_off, st);
        else launch_coverage_runs(tt, nt, c0, c1, cnt_.ss, max_tile_ints_, rt, vt, L, run_off, st);
        BSG_CUDA(cudaMemcpyAsync(c.h_runs.p, run_off, (size_t(L) + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        BSG_CUDA(cudaStreamSynchronize(st));
        BSG_CUDA(cudaGetLastError());
        memcpy(runs_.run_offsets, c.h_runs.p, (size_t(L) + 1) * sizeof(int64_t));
        bsg_runs& res = *runs_.res;
        res.dev = c.dev;
        res.n = runs_.run_offsets[L];
        const size_t bytes = size_t(std::max<int64_t>(res.n, 1)) * sizeof(int32_t);
        BSG_CUDA(cudaMalloc(&res.lengths, bytes));
        BSG_CUDA(cudaMalloc(&res.values, bytes));
        BSG_CUDA(cudaMemsetAsync(res.lengths, 0, bytes, st));
        if (profile) launch_profile_runs_write(tt, nt, c0, c1, cnt_.ss, cnt_.binsize, max_tile_ints_, rt, vt, run_off, res.lengths, res.values, st);
        else launch_coverage_runs_write(tt, nt, c0, c1, cnt_.ss, max_tile_ints_, rt, vt, run_off, res.lengths, res.values, st);
        BSG_CUDA(cudaEventRecord(sp.b, st));
        kt_.count.push_back(sp); kt_.launches += nt ? 3 : 1;
        tm_.out_elems = 2 * res.n;
        os_bytes_ += double((L + 1) * int64_t(sizeof(int64_t)));
    }

    // ---- output streamer: D2H on its own stream into a pinned ring, a host thread scatters tiles to the caller ------------
    void start_streamer() {
        DeviceCtx& c = *ctx_;
        for (int k = 0; k < kOutSlots; ++k) c.h_out[k].ensure(size_t(kD2HChunk));
        if (opts_.result_pack >= 0) {
            for (int k = 0; k < kOutSlots; ++k) c.g_pack[k].ensure(size_t(kD2HChunk / 4));
            c.h_pack_cnt.ensure(64);
            if (!c.g_pack_cnt.p) { c.g_pack_cnt.ensure(64); BSG_CUDA(cudaMemset(c.g_pack_cnt.p, 0, 64)); }
        }
        os_stop_ = false; os_abort_ = false;
        os_wait_ms_ = os_scatter_ms_ = 0; os_bytes_ = 0;
        os_jobs_.clear();
        os_err_ = Error{0, ""};
        os_thread_ = std::thread([this] { streamer_main(); });
    }
    // main thread: never blocks here, the streamer thread does the copies
    void ship_tiles(int64_t t0, int64_t t1, cudaEvent_t computed) {
        {
            std::lock_guard<std::mutex> g(os_m_);
            os_jobs_.push_back(OutJob{0, t0, t1, computed});
        }
        os_cv_.notify_all();
    }
    void streamer_main() {
        DeviceCtx& c = *ctx_;
        cudaSetDevice(c.dev);
        const int64_t cap = kD2HChunk / 4;
        nvtxNameOsThreadA(uint32_t(syscall(SYS_gettid)), "bsg result streamer");
        for (;;) {
            OutJob job;
            {
                std::unique_lock<std::mutex> lk(os_m_);
                os_cv_.wait(lk, [&] { return os_stop_ || !os_jobs_.empty(); });
                if (os_jobs_.empty()) return;
                job = os_jobs_.front();
                os_jobs_.pop_front();
            }
            if (os_abort_ || os_err_.code) continue;
            // pieces of <= 32 MiB at tile boundaries; the copy of piece k+1 is in flight while piece k is scattered
            std::vector<int64_t> cut{job.t0};
            for (int64_t p0 = job.t0; p0 < job.t1;) {
                int64_t p1 = p0 + 1;
                while (p1 < job.t1 && tile_dev_off_[p1 + 1] - tile_dev_off_[p0] <= cap) ++p1;
                cut.push_back(p1);
                p0 = p1;
            }
            const int np = int(cut.size()) - 1;
            cudaError_t e = cudaStreamWaitEvent(c.s_d2h, job.computed, 0);
            // A large portion crosses PCIe as ONE BYTE per element (+ the few elements above 254 as (index, value) pairs
            // written straight into pinned host memory): C2's 1.6 GB of int32 counts - more than its 1.2 GB of compressed
            // input - took 68 ms at the 23 GB/s the device-to-host path reaches next to the upload, longer than the whole
            // fetch pipeline.  The scatter below widens the bytes while it moves them.
            const int pack_div = opts_.result_pack < 0 ? 0 : (opts_.result_pack == 0 ? 64 : std::max(2, opts_.result_pack));
            std::vector<uint32_t> ovf_cap(size_t(np), 0u);          // 0 = this piece travels as int32
            auto issue = [&](int k) {
                const int slot = k % kOutSlots;
                const int64_t ints = tile_dev_off_[cut[k + 1]] - tile_dev_off_[cut[k]];
                const int32_t* src = c.out.as<int32_t>() + tile_dev_off_[cut[k]];
                cudaError_t r = cudaSuccess;
                if (pack_div > 0 && ints >= kPackMinInts && ints <= kD2HChunk / 4) {
                    const uint32_t cap = uint32_t(std::max<int64_t>(1024, ints / pack_div));
                    try { c.h_ovf[slot].ensure(size_t(cap) * sizeof(uint2)); } catch (const Error&) { return cudaErrorMemoryAllocation; }
                    ovf_cap[size_t(k)] = cap;
                    launch_pack_u8(src, ints, c.g_pack[slot].as<uint8_t>(), c.h_ovf[slot].as<uint2>(), cap, c.g_pack_cnt.as<uint32_t>() + slot, c.s_d2h);
                    launch_publish_reset(c.g_pack_cnt.as<uint32_t>() + slot, c.h_pack_cnt.as<uint32_t>() + slot, c.s_d2h);
                    r = cudaMemcpyAsync(c.h_out[slot].p, c.g_pack[slot].p, size_t(ints), cudaMemcpyDeviceToHost, c.s_d2h);
                    os_bytes_ += double(ints) + 4;
                } else {
                    r = cudaMemcpyAsync(c.h_out[slot].p, src, size_t(ints) * 4, cudaMemcpyDeviceToHost, c.s_d2h);
                    os_bytes_ += double(ints) * 4;
                }
                if (r == cudaSuccess) r = cudaEventRecord(c.ev_d2h[slot], c.s_d2h);
                return r;
            };
            for (int k = 0; k < np && k < kOutSlots - 1 && e == cudaSuccess; ++k) e = issue(k);
            for (int k = 0; k < np && e == cudaSuccess; ++k) {
                if (k + kOutSlots - 1 < np) e = issue(k + kOutSlots - 1);      // its slot was scattered in iteration k-1
                if (e != cudaSuccess) break;
                const int slot = k % kOutSlots;
                const double tw0 = now_ms();
                e = cudaEventSynchronize(c.ev_d2h[slot]);
                if (e != cudaSuccess) break;
                const double tw1 = now_ms();
                os_wait_ms_ += tw1 - tw0;
                const int64_t t_lo = cut[k], base = tile_dev_off_[t_lo], n = cut[k + 1] - t_lo;
                uint32_t n_ovf = 0;
                bool packed = ovf_cap[size_t(k)] != 0;
                if (packed) {
                    n_ovf = c.h_pack_cnt.as<uint32_t>()[slot];
                    os_bytes_ += 8.0 * std::min(n_ovf, ovf_cap[size_t(k)]);
                    if (n_ovf > ovf_cap[size_t(k)]) {
                        os_bytes_ += double(tile_dev_off_[cut[k + 1]] - base) * 4;
                        // too many large elements for the list: this piece travels again, as int32 (the copies already queued
                        // for the next pieces go first; it is the rare case)
                        e = cudaMemcpyAsync(c.h_out[slot].p, c.out.as<int32_t>() + base, size_t(tile_dev_off_[cut[k + 1]] - base) * 4,
                                            cudaMemcpyDeviceToHost, c.s_d2h);
                        if (e == cudaSuccess) e = cudaStreamSynchronize(c.s_d2h);
                        if (e != cudaSuccess) break;
                        packed = false;
                    }
                }
                auto dst_of = [&](int64_t t) -> int32_t* {
                    return cnt_.out ? cnt_.out + ht_.out_off[t]
                                    : (cnt_.out_ptrs[ht_.region[t]] ? cnt_.out_ptrs[ht_.region[t]] + (ht_.out_off[t] - cnt_.out_offsets[ht_.region[t]]) : nullptr);
                };
                const int64_t grain = std::max<int64_t>(1, n / (int64_t(pool_->size()) * 4));
                if (packed) {
                    const uint8_t* src = c.h_out[slot].as<uint8_t>();
                    pool_->parallel_for(n, grain, [&](int64_t a, int64_t b, int) {
                        for (int64_t t = t_lo + a; t < t_lo + b; ++t) {
                            int32_t* dst = dst_of(t);
                            if (!dst) continue;
                            widen_u8_to_i32(dst, src + (tile_dev_off_[t] - base), ht_.ints[t]);
                        }
                    });
                    const uint2* ov = c.h_ovf[slot].as<uint2>();
                    for (uint32_t j = 0; j < n_ovf; ++j) {          // the elements above 254, exactly
                        const int64_t pos = base + int64_t(ov[j].x);
                        const int64_t t = (std::upper_bound(tile_dev_off_.begin() + t_lo, tile_dev_off_.begin() + t_lo + n + 1, pos) - tile_dev_off_.begin()) - 1;
                        int32_t* dst = dst_of(t);
                        if (dst) dst[pos - tile_dev_off_[t]] = int32_t(ov[j].y);
                    }
                } else {
                    const int32_t* src = c.h_out[slot].as<int32_t>();
                    pool_->parallel_for(n, grain, [&](int64_t a, int64_t b, int) {
                        for (int64_t t = t_lo + a; t < t_lo + b; ++t) {
                            int32_t* dst = dst_of(t);
                            if (dst) copy_i32_stream(dst, src + (tile_dev_off_[t] - base), ht_.ints[t]);
                        }
                    });
                }
                os_scatter_ms_ += now_ms() - tw1;
            }
            if (e != cudaSuccess) {
                std::lock_guard<std::mutex> g(os_m_);
                if (!os_err_.code) os_err_ = Error{BSG_ECUDA, std::string("CUDA error in result copy: ") + cudaGetErrorString(e)};
            }
        }
    }
    void stop_streamer(bool abort) {
        if (!os_thread_.joinable()) return;
        {
            std::lock_guard<std::mutex> g(os_m_);
            os_stop_ = true;
            if (abort) os_abort_ = true;
        }
        os_cv_.notify_all();
        os_thread_.join();
        if (getenv("BSG_DEBUG")) fprintf(stderr, "[bsg] result streamer: %.1f ms waiting for copies, %.1f ms scattering\n", os_wait_ms_, os_scatter_ms_);
        if (!abort && os_err_.code) throw os_err_;
    }

public:
    void check_status(uint32_t status) {
        if (status & STATUS_BAD_CRC) fail(BSG_EFORMAT, "BGZF CRC32 mismatch in " + bam_.path());
        if (status & STATUS_BAD_DEFLATE) fail(BSG_EFORMAT, "BGZF inflate failed (corrupt DEFLATE stream or ISIZE mismatch) in " + bam_.path());
        if (status & STATUS_CORRUPT) fail(BSG_EFORMAT, "corrupt BAM record chain in " + bam_.path());
        if (status & STATUS_UNSORTED) fail(BSG_EUNSORTED, "BAM file is not coordinate-sorted: " + bam_.path());
    }

    void finish_timings(double t_start) {
        tm_.ms_decode = sum_ms(kt_.decode);
        tm_.ms_filter = sum_ms(kt_.filter);
        tm_.ms_join = sum_ms(kt_.join);
        tm_.ms_count = sum_ms(kt_.count);
        tm_.ms_kernels = tm_.ms_decode + tm_.ms_filter + tm_.ms_join + tm_.ms_count;
        if (!kt_.count.empty()) {
            const cudaEvent_t first = !kt_.decode.empty() ? kt_.decode.front().a
                                    : (!kt_.filter.empty() ? kt_.filter.front().a : kt_.join.front().a);
            float ms = 0;
            cudaEventElapsedTime(&ms, first, kt_.count.back().b);
            tm_.ms_device = ms;
        }
        tm_.n_launches = kt_.launches;
        tm_.ms_total = now_ms() - t_start;
        g_tm = tm_;
        kt_ = KernelTimes();
        ctx_->ev_next = 0;
    }
    const bsg_timings& timings() const { return tm_; }
    void kick_page_locking() { kick_pinning(bamp_, ctx_->dev); }
    void reset_counters() { int nd = tm_.n_devices; int64_t bc = tm_.bytes_compressed, bi = tm_.bytes_inflated, nb = tm_.n_batches;
        memset(&tm_, 0, sizeof tm_); tm_.n_devices = nd; tm_.bytes_compressed = bc; tm_.bytes_inflated = bi; tm_.n_batches = nb; }

private:
    ReadTable table() {
        DeviceCtx& c = *ctx_;
        return ReadTable{c.tab[0].as<int32_t>(), c.tab[1].as<int32_t>(), c.c0.as<int32_t>(), c.c1.as<int32_t>()};
    }
    void ensure_table(int64_t rows) {
        DeviceCtx& c = *ctx_;
        const size_t bytes = size_t(rows + 4) * 4;
        for (auto& b : c.tab) b.ensure(bytes);   // tid, pos
        c.c0.ensure(bytes); c.c1.ensure(bytes);
    }

    // Inflate + walk one batch on the pool; the last worker to finish marks it ready.
    void submit_batch(Batch* b, int slot) {
        DeviceCtx& c = *ctx_;
        uint8_t* stage = c.h_raw[slot].as<uint8_t>();
        uint32_t* offs = c.h_offs[slot].as<uint32_t>();
        const size_t ns = b->seg_last - b->seg_first;
        b->seg_base.resize(ns); b->seg_off_base.resize(ns); b->seg_count.assign(ns, 0);
        b->seg_blocks_left.reset(new std::atomic<int>[ns]);
        uint64_t base = 0, obase = 0;
        for (size_t k = 0; k < ns; ++k) {
            const Segment& s = segs_[b->seg_first + k];
            b->seg_base[k] = base; b->seg_off_base[k] = obase;
            base += (s.usize + 15) & ~15ull;
            obase += (s.uend - s.ubeg) / kMinRecord + 1;
            b->seg_blocks_left[k].store(int(s.blocks.size()));
        }
        b->segs_left.store(int(ns));
        b->ready = false;
        const bool crc = opts_.verify_crc != 0;
        auto seg_done = [this, b, stage, offs](size_t k) {
            // walk the block_size chain of segment k
            const Segment& s = segs_[b->seg_first + k];
            try {
                const uint64_t sb = b->seg_base[k];
                uint64_t p = sb + s.ubeg;
                const uint64_t e = sb + s.uend;
                uint32_t* o = offs + b->seg_off_base[k];
                int64_t n = 0;
                while (p < e) {
                    if (p + 4 > e) fail(BSG_EFORMAT, "truncated BAM record in " + bam_.path());
                    const int32_t bs = rd_i32(stage + p);
                    if (bs < 32 || p + 4 + uint64_t(bs) > e) fail(BSG_EFORMAT, "corrupt BAM record chain in " + bam_.path());
                    o[n++] = uint32_t(p);
                    p += 4 + uint64_t(bs);
                }
                b->seg_count[k] = n;
            } catch (Error& er) {
                std::lock_guard<std::mutex> g(b->m);
                if (!b->err.code) b->err = er;
            }
            if (b->segs_left.fetch_sub(1) == 1) {
                // finalize: compact the per-segment offset runs, append the end sentinel
                const size_t ns2 = b->seg_last - b->seg_first;
                int64_t n = 0;
                for (size_t q = 0; q < ns2; ++q) {
                    if (b->seg_off_base[q] != uint64_t(n) && b->seg_count[q])
                        memmove(offs + n, offs + b->seg_off_base[q], size_t(b->seg_count[q]) * 4);
                    n += b->seg_count[q];
                }
                const Segment& last = segs_[b->seg_last - 1];
                offs[n] = uint32_t(b->seg_base[ns2 - 1] + last.uend);
                b->n_records = n;
                std::lock_guard<std::mutex> g(b->m);
                b->ready = true;
                b->cv.notify_all();
            }
        };
        for (size_t k = 0; k < ns; ++k) {
            const Segment& s = segs_[b->seg_first + k];
            if (s.blocks.empty()) { pool_->submit([seg_done, k](int) { seg_done(k); }); continue; }
            const size_t group = 8;
            uint64_t ub = 0;
            for (size_t g0 = 0; g0 < s.blocks.size(); g0 += group) {
                const size_t g1 = std::min(s.blocks.size(), g0 + group);
                const uint64_t ub0 = ub;
                for (size_t q = g0; q < g1; ++q) ub += s.blocks[q].isize;
                pool_->submit([this, b, &s, k, g0, g1, ub0, stage, crc, seg_done](int) {
                    try {
                        thread_local Inflater inf;
                        uint64_t u = b->seg_base[k] + ub0;
                        for (size_t q = g0; q < g1; ++q) {
                            inf.inflate_block(bam_.data(), s.blocks[q], stage + u, crc);
                            u += s.blocks[q].isize;
                        }
                    } catch (Error& er) {
                        std::lock_guard<std::mutex> g(b->m);
                        if (!b->err.code) b->err = er;
                    }
                    if (b->seg_blocks_left[k].fetch_sub(int(g1 - g0)) == int(g1 - g0)) seg_done(k);
                });
            }
        }
    }

    void run_pipeline() {
        DeviceCtx& c = *ctx_;
        const size_t nb = batches_.size();
        res_->batches.clear();
        res_->n_rows = 0;
        size_t next_submit = 0;
        uint64_t raw_base = 0; int64_t offs_base = 0;
        double h2d_ms = 0;
        try {
        for (size_t commit = 0; commit < nb; ++commit) {
            while (next_submit < nb && next_submit < commit + kSlots) {
                const int slot = int(next_submit % kSlots);
                if (next_submit >= size_t(kSlots)) BSG_CUDA(cudaEventSynchronize(c.ev_free[slot]));
                submit_batch(batches_[next_submit].get(), slot);
                ++next_submit;
            }
            Batch* b = batches_[commit].get();
            {
                std::unique_lock<std::mutex> lk(b->m);
                b->cv.wait(lk, [&] { return b->ready; });
            }
            if (b->err.code) throw b->err;
            const int slot = int(commit % kSlots);
            const int64_t n = b->n_records;
            if (res_->n_rows + n > res_->rows_cap) fail(BSG_EFORMAT, "record count exceeds the planned table capacity");
            const double t0 = now_ms();
            uint8_t* d_raw; uint32_t* d_offs;
            if (res_->keep_raw) {
                d_raw = res_->raw_all.as<uint8_t>() + raw_base;
                d_offs = res_->offs_all.as<uint32_t>() + offs_base;
                res_->batches.push_back(ResidentBatch{raw_base, offs_base, n});
                raw_base += (b->bytes + 64 + 255) & ~255ull;
                offs_base += n + 1;
            } else {
                d_raw = c.d_raw[slot].as<uint8_t>();
                d_offs = c.d_offs[slot].as<uint32_t>();
            }
            BSG_CUDA(cudaMemcpyAsync(d_raw, c.h_raw[slot].p, b->bytes + 16, cudaMemcpyHostToDevice, c.s_copy));
            BSG_CUDA(cudaMemcpyAsync(d_offs, c.h_offs[slot].p, size_t(n + 1) * 4, cudaMemcpyHostToDevice, c.s_copy));
            BSG_CUDA(cudaEventRecord(c.ev_h2d[slot], c.s_copy));
            if (res_->keep_raw) {
                BSG_CUDA(cudaEventRecord(c.ev_free[slot], c.s_copy));
            } else {
                BSG_CUDA(cudaStreamWaitEvent(c.s_comp, c.ev_h2d[slot], 0));
                Span sp{c.timing_event(), c.timing_event()};
                BSG_CUDA(cudaEventRecord(sp.a, c.s_comp));
                if (!cnt_.active) fail(BSG_EARG, "internal error: streaming decode without a counting call");
                launch_decode(DecodeBatch{d_raw, d_offs, res_->n_rows, int32_t(n), 0}, table(), cnt_.mode == MODE_COVERAGE, cnt_.ss != 0, cnt_.fp,
                              c.scalars.as<DeviceScalars>(), c.s_comp);
                BSG_CUDA(cudaEventRecord(sp.b, c.s_comp));
                BSG_CUDA(cudaEventRecord(c.ev_free[slot], c.s_comp));
                kt_.decode.push_back(sp); kt_.launches += n > 0;
            }
            h2d_ms += now_ms() - t0;
            res_->n_rows += n;
        }
        } catch (...) {
            // workers still reference this Session and the staging slots: wait for every submitted batch
            for (size_t k = 0; k < next_submit; ++k) {
                std::unique_lock<std::mutex> lk(batches_[k]->m);
                batches_[k]->cv.wait(lk, [&] { return batches_[k]->ready; });
            }
            cudaStreamSynchronize(c.s_copy); cudaStreamSynchronize(c.s_comp);
            throw;
        }
        BSG_CUDA(cudaStreamSynchronize(c.s_copy));
        if (res_->keep_raw) build_resident_table();
        tm_.ms_h2d = h2d_ms;
        tm_.records = res_->n_rows;
    }

    // GPU-inflate pipeline: host ships compressed bytes; inflate, record walk and decode run on the device.
    //   upload(b):  descriptors + H2D of the compressed bytes into upload slot b % kUp              (copy stream)
    //   compute(b): inflate -> CRC (side stream) -> walk (count / scan / write) -> record count back (compute stream)
    //   finish(b):  K1 decode on the high-priority stream, frontier read-back, count + ship the tiles it finalises
    // The inflate kernel is persistent and takes every SM (227 KB of shared memory per CTA): K1 of batch b, launched when
    // the host has seen the walk of b end, runs only when inflate(b + 1) has drained, and finish(b) blocks the host
    // until then.  Everything that must not wait for that is therefore queued BEFORE finish(b): compute(b + 1) and
    // upload(b + 2).  (Round 1 queued upload(b + 1) after finish(b - 1): each H2D started when an inflate ended, copy
    // engine and SMs took turns - 88 ms for C2 whose kernels need 51 ms and whose H2D needs 37.)
    void run_pipeline_gpu(uint64_t max_batch, size_t max_offs) {
        DeviceCtx& c = *ctx_;
        const size_t nb = batches_.size();
        res_->batches.clear();
        res_->n_rows = 0;
        const std::vector<uint64_t>& ent = bam_.entry_points();
        uint64_t raw_base = 0; int64_t offs_base = 0;
        struct Up {             // what compute() and finish() need to know about an uploaded batch
            int n_blocks = 0, n_walkers = 0; uint32_t end_pos = 0, raw_end = 0; int scheme = 2;
            uint8_t* d_raw = nullptr; uint32_t* d_offs = nullptr; uint64_t raw_base = 0; int64_t offs_base = 0;
        };
        std::vector<Up> ups(nb);
        // the high-priority stream starts behind everything already queued on the compute stream (scalars reset, tiles)
        hi_prio_ = !res_->keep_raw;
        BSG_CUDA(cudaEventRecord(c.ev_order, c.s_comp));
        BSG_CUDA(cudaStreamWaitEvent(c.s_hi, c.ev_order, 0));
        std::vector<Span> inflate_spans, walk_spans, h2d_spans, crc_spans;
        const size_t dec_first = kt_.decode.size(), cnt_first = kt_.count.size();
        const bool dbg_tl = getenv("BSG_DEBUG") != nullptr;
        double t_desc = 0, t_copy = 0, t_wait = 0, t_finish = 0;
        std::vector<InflateBlock> blocks;
        std::vector<uint32_t> crcs;
        std::vector<uint2> walkers;
        struct CopyPiece { uint64_t file_off, dst_off, len; };
        std::vector<CopyPiece> pieces;
        int pin_slot = 0;

        auto upload = [&](size_t bi) {
            Batch* b = batches_[bi].get();
            const int slot = int(bi % kUp), rslot = int(bi & 1);
            Up& up = ups[bi];
            // ---- descriptors -----------------------------------------------------------------------------------------
            double tt = now_ms();
            nvtxRangePushA("bsg:batch descriptors");
            blocks.clear(); crcs.clear(); walkers.clear(); pieces.clear();
            // Compressed layout of the batch on the device: SPANS of the file, each one contiguous byte range copied as it
            // lies.  Consecutive segments whose gap in the file is small are one span (the gap's bytes ride along unused):
            // one DMA descriptor costs about as much as 160 KB of transfer, and a job like C2 (100 k scattered windows)
            // has 27 k segments of 45 KB with gaps of one to three BGZF blocks between them.
            uint64_t ubase = 0, cbase = 0;
            for (size_t k = b->seg_first; k < b->seg_last; ++k) {
                const Segment& sg = segs_[k];
                if (sg.blocks.empty()) continue;
                const uint64_t fbeg = sg.blocks.front().coff, fend = sg.blocks.back().coff + sg.blocks.back().csize;
                uint64_t span_file, span_dst;
                if (!pieces.empty() && fbeg >= pieces.back().file_off + pieces.back().len &&
                    fbeg - (pieces.back().file_off + pieces.back().len) <= kSpanGap) {
                    pieces.back().len = fend - pieces.back().file_off;
                } else {
                    cbase = (cbase + 15) & ~15ull;
                    pieces.push_back(CopyPiece{fbeg & ~3ull, cbase, fend - (fbeg & ~3ull)});      // word-aligned source and destination
                }
                span_file = pieces.back().file_off; span_dst = pieces.back().dst_off;
                cbase = span_dst + pieces.back().len;
                uint64_t u = ubase;
                // walkers: the segment start plus every index entry point strictly inside the segment
                auto it = std::upper_bound(ent.begin(), ent.end(), sg.vbeg);
                uint32_t prev = uint32_t(ubase + sg.ubeg);
                const uint32_t seg_end = uint32_t(ubase + sg.uend);
                for (const BlockInfo& blk : sg.blocks) {
                    while (it != ent.end() && (*it >> 16) < blk.coff) ++it;      // stale entries cost parallelism, not correctness
                    blocks.push_back(InflateBlock{uint32_t(span_dst + (blk.coff - span_file) + blk.hdr), blk.csize - blk.hdr - 8, uint32_t(u), blk.isize});
                    crcs.push_back(blk.crc);
                    for (; it != ent.end() && *it < sg.vend && (*it >> 16) == blk.coff; ++it) {
                        const uint64_t uo = *it & 0xffff;
                        if (uo > blk.isize) fail(BSG_EFORMAT, "index offset beyond its BGZF block in " + bam_.path());
                        const uint32_t pos = uint32_t(u + uo);
                        if (pos > prev && pos < seg_end) { walkers.push_back(make_uint2(prev, pos)); prev = pos; }
                    }
                    u += blk.isize;
                }
                if (seg_end > prev) walkers.push_back(make_uint2(prev, seg_end));
                ubase += (sg.usize + 15) & ~15ull;
            }
            if (cbase >= (1ull << 32) - 8192) fail(BSG_ENOMEM, "a batch's compressed bytes exceed 4 GiB");
            const uint32_t end_pos = walkers.empty() ? 0u : walkers.back().y;
            nvtxRangePop();
            t_desc += now_ms() - tt; tt = now_ms();
            // ---- buffers ------------------------------------------------------------------------------------------------
            // The upload overwrites the compressed bytes, descriptor arrays and walk scratch of its slot; their readers
            // were the inflate, walk and CRC kernels of batch bi - kUp, finished long ago (no wait in practice).
            BSG_CUDA(cudaEventSynchronize(c.ev_total[slot]));
            BSG_CUDA(cudaEventSynchronize(c.ev_crc[slot]));
            t_wait += now_ms() - tt; tt = now_ms();
            nvtxRangePushA("bsg:upload compressed (memcpy + H2D)");
            c.g_comp[slot].ensure(cbase + 4096);   // slack: the bit reader looks ahead, and a corrupt stream may run on for one round
            c.g_blocks[slot].ensure(blocks.size() * sizeof(InflateBlock) + 64);
            c.g_crc[slot].ensure(crcs.size() * 4 + 64);
            c.g_walkers[slot].ensure(walkers.size() * sizeof(uint2) + 64);
            c.g_counts[slot].ensure(walkers.size() * 4 + 64);
            c.g_base[slot].ensure(walkers.size() * 4 + 64);
            c.g_wscr[slot].ensure(walk_scratch_words(int(blocks.size()), int(walkers.size())) * 4);
            c.g_spec[slot].ensure(inflate_spec_words(int(blocks.size())) * 4);
            if (res_->keep_raw) {
                up.d_raw = res_->raw_all.as<uint8_t>() + raw_base;
                up.d_offs = res_->offs_all.as<uint32_t>() + offs_base;
            } else {
                // the raw buffer of the slot may still be read by the decode kernel of batch bi - 2; this batch's inflate
                // writes it next: a device-side dependency (ev_gfree in compute()), not a reason to hold the upload back
                c.g_raw[rslot].ensure(max_batch + 64);
                c.g_offs[rslot].ensure((max_offs + 8) * sizeof(uint32_t));
                up.d_raw = c.g_raw[rslot].as<uint8_t>();
                up.d_offs = c.g_offs[rslot].as<uint32_t>();
            }
            up.raw_base = raw_base; up.offs_base = offs_base;
            up.n_blocks = int(blocks.size()); up.n_walkers = int(walkers.size()); up.end_pos = end_pos; up.raw_end = uint32_t(ubase);
            {   // spans of less than a block and a half are cheapest followed one by one (C2: 16 kb index windows, ~500 records)
                uint32_t max_span = 0;
                for (const uint2& wk : walkers) max_span = std::max(max_span, wk.y - wk.x);
                up.scheme = opts_.walk_scheme == 1 ? 1 : (opts_.walk_scheme == 2 ? 2 : (max_span <= (96u << 10) ? 1 : 2));
            }
            // ---- compressed bytes -> device ------------------------------------------------------------------------------------
            Span sph{c.timing_event(), c.timing_event()};
            BSG_CUDA(cudaEventRecord(sph.a, c.s_copy));
            bool direct = true;
            for (const CopyPiece& pc : pieces) direct = direct && ensure_pinned(bam_, pc.file_off, pc.len);
            if (direct) {
                // the copy engine reads the page cache itself: one asynchronous copy per span and page-locked window (a
                // copy must stay inside ONE registered range: across two the driver answers "invalid argument")
                for (const CopyPiece& pc : pieces)
                    for (uint64_t o = 0; o < pc.len;) {
                        const uint64_t f = pc.file_off + o;
                        const uint64_t n = std::min<uint64_t>((f / kPinWindow + 1) * kPinWindow - f, pc.len - o);
                        BSG_CUDA(cudaMemcpyAsync(c.g_comp[slot].as<uint8_t>() + pc.dst_off + o, bam_.data() + f, n, cudaMemcpyHostToDevice, c.s_copy));
                        o += n;
                    }
                tm_.upload_mode = 1;
            } else {
                // Staging: file (page cache) -> pinned chunk -> device, chunk by chunk.  The pinned chunk mirrors a window
                // [c_lo, c_lo + kCompChunk) of the device buffer byte for byte, so every chunk is ONE H2D copy no matter how
                // many spans it holds.
                struct Part { const uint8_t* src; uint64_t pin_off, len; };
                size_t pi = 0; uint64_t done_in_piece = 0;
                while (pi < pieces.size()) {
                    const int ps = pin_slot; pin_slot = (pin_slot + 1) % kSlots;
                    c.h_raw[ps].ensure(kCompChunk + 64);
                    BSG_CUDA(cudaEventSynchronize(c.ev_pin[ps]));
                    uint8_t* pin = c.h_raw[ps].as<uint8_t>();
                    const uint64_t c_lo = pieces[pi].dst_off + done_in_piece;
                    uint64_t c_hi = c_lo;
                    std::vector<std::vector<Part>> tasks(1);
                    uint64_t task_bytes = 0;
                    while (pi < pieces.size()) {
                        const CopyPiece& pc = pieces[pi];
                        const uint64_t d0 = pc.dst_off + done_in_piece;
                        if (d0 - c_lo >= kCompChunk) break;
                        const uint64_t take = std::min<uint64_t>(pc.len - done_in_piece, kCompChunk - (d0 - c_lo));
                        // split long pieces into <= 1 MiB parts; group short ones into ~1 MiB tasks
                        for (uint64_t o = 0; o < take; o += (1u << 20)) {
                            const uint64_t n = std::min<uint64_t>(1u << 20, take - o);
                            if (task_bytes + n > (1u << 20) && !tasks.back().empty()) { tasks.emplace_back(); task_bytes = 0; }
                            tasks.back().push_back(Part{bam_.data() + pc.file_off + done_in_piece + o, d0 + o - c_lo, n});
                            task_bytes += n;
                        }
                        c_hi = d0 + take;
                        done_in_piece += take;
                        if (done_in_piece == pc.len) { ++pi; done_in_piece = 0; } else break;
                    }
                    pool_->parallel_for(int64_t(tasks.size()), 1, [&](int64_t a, int64_t e, int) {
                        for (int64_t t = a; t < e; ++t)
                            for (const Part& pt : tasks[t]) memcpy(pin + pt.pin_off, pt.src, pt.len);
                    });
                    BSG_CUDA(cudaMemcpyAsync(c.g_comp[slot].as<uint8_t>() + c_lo, pin, c_hi - c_lo, cudaMemcpyHostToDevice, c.s_copy));
                    BSG_CUDA(cudaEventRecord(c.ev_pin[ps], c.s_copy));
                }
            }
            // descriptors go through a pinned buffer of the slot (its previous use ended with the batch before last, whose
            // kernels the wait above covers), so nothing here blocks the host
            {
                const size_t nb_b = blocks.size() * sizeof(InflateBlock), nb_c = crcs.size() * 4, nb_w = walkers.size() * sizeof(uint2);
                const size_t o_c = (nb_b + 63) & ~size_t(63), o_w = o_c + ((nb_c + 63) & ~size_t(63));
                c.h_desc[slot].ensure(o_w + nb_w + 64);
                uint8_t* hd = c.h_desc[slot].as<uint8_t>();
                if (nb_b) memcpy(hd, blocks.data(), nb_b);
                if (nb_c) memcpy(hd + o_c, crcs.data(), nb_c);
                if (nb_w) memcpy(hd + o_w, walkers.data(), nb_w);
                if (nb_b) BSG_CUDA(cudaMemcpyAsync(c.g_blocks[slot].p, hd, nb_b, cudaMemcpyHostToDevice, c.s_copy));
                if (nb_c && opts_.verify_crc) BSG_CUDA(cudaMemcpyAsync(c.g_crc[slot].p, hd + o_c, nb_c, cudaMemcpyHostToDevice, c.s_copy));
                if (nb_w) BSG_CUDA(cudaMemcpyAsync(c.g_walkers[slot].p, hd + o_w, nb_w, cudaMemcpyHostToDevice, c.s_copy));
            }
            BSG_CUDA(cudaEventRecord(c.ev_up[slot], c.s_copy));
            BSG_CUDA(cudaEventRecord(sph.b, c.s_copy));
            h2d_spans.push_back(sph);
            nvtxRangePop();
            t_copy += now_ms() - tt;
            if (res_->keep_raw) {
                raw_base += (b->bytes + 64 + 255) & ~255ull;
                offs_base += int64_t((b->bytes) / kMinRecord) + 2;
            }
        };

        auto compute = [&](size_t bi) {
            const int slot = int(bi % kUp), rslot = int(bi & 1);
            const Up& up = ups[bi];
            nvtxRangePushA("bsg:launch inflate + crc + walk");
            BSG_CUDA(cudaStreamWaitEvent(c.s_comp, c.ev_up[slot], 0));
            if (!res_->keep_raw) BSG_CUDA(cudaStreamWaitEvent(c.s_comp, c.ev_gfree[rslot], 0));      // decode (+ CRC) of batch bi - 2
            Span sp{c.timing_event(), c.timing_event()};
            BSG_CUDA(cudaEventRecord(sp.a, c.s_comp));
            launch_inflate(c.g_blocks[slot].as<InflateBlock>(), up.n_blocks, c.g_comp[slot].as<uint8_t>(), up.d_raw,
                           up.scheme == 1 ? nullptr : c.g_spec[slot].as<uint32_t>(), c.scalars.as<DeviceScalars>(), c.s_comp);
            BSG_CUDA(cudaEventRecord(c.ev_inflated[slot], c.s_comp));
            BSG_CUDA(cudaEventRecord(sp.b, c.s_comp));
            inflate_spans.push_back(sp);
            if (opts_.verify_crc) {
                // integrity check on a side stream: it only reads the inflated bytes; the raw buffer is not recycled before
                // it has finished (finish()).
                BSG_CUDA(cudaStreamWaitEvent(c.s_aux, c.ev_inflated[slot], 0));
                Span spc{nullptr, nullptr};
                if (dbg_tl) { spc = Span{c.timing_event(), c.timing_event()}; BSG_CUDA(cudaEventRecord(spc.a, c.s_aux)); }
                launch_crc32(c.g_blocks[slot].as<InflateBlock>(), c.g_crc[slot].as<uint32_t>(), up.n_blocks, up.d_raw,
                             c.scalars.as<DeviceScalars>(), c.s_aux);
                if (dbg_tl) { BSG_CUDA(cudaEventRecord(spc.b, c.s_aux)); crc_spans.push_back(spc); }
                BSG_CUDA(cudaEventRecord(c.ev_crc[slot], c.s_aux));
                kt_.launches += up.n_blocks ? 1 : 0;
            }
            // The record walk has its own stream too.  Neither it nor the CRC kernel uses shared memory, and the inflate
            // kernel leaves 2 KB of every SM free: their CTAs run NEXT TO the persistent inflate CTAs of the following batch,
            // which is queued right behind this batch's inflate.  (Round 1: walk between two inflates on the compute stream,
            // 1.3 ms of every 5.7 ms batch period with the SMs nearly idle; on another stream it could not start at all while
            // an inflate launch held every SM.)
            cudaStream_t ws = (bi & 1) ? c.s_walk2 : c.s_walk;       // two streams: on deep data a walk outlasts an inflate launch, and the
                                                                     // walks of consecutive batches are independent chains of dependent loads
            BSG_CUDA(cudaStreamWaitEvent(ws, c.ev_inflated[slot], 0));
            Span spw{c.timing_event(), c.timing_event()};
            BSG_CUDA(cudaEventRecord(spw.a, ws));
            launch_walk(up.d_raw, c.g_walkers[slot].as<uint2>(), up.n_walkers, up.scheme, c.g_blocks[slot].as<InflateBlock>(), up.n_blocks,
                        up.scheme == 1 ? nullptr : c.g_spec[slot].as<uint32_t>(), c.g_wscr[slot].as<uint32_t>(),
                        c.g_counts[slot].as<uint32_t>(), c.g_base[slot].as<uint32_t>(), c.h_total.as<uint32_t>() + slot, up.d_offs, up.end_pos,
                        c.scalars.as<DeviceScalars>(), ws);
            BSG_CUDA(cudaEventRecord(spw.b, ws));
            walk_spans.push_back(spw);
            kt_.launches += (up.n_blocks ? 1 : 0) + ((up.n_walkers && up.n_blocks) ? (up.scheme == 1 ? 3 : 4) : 1);
            // (the record count lands in pinned host memory straight from the scan kernel: a 4-byte cudaMemcpy would queue
            // behind the 32 MiB result copies on the device-to-host engine - measured: up to 6 ms per batch)
            BSG_CUDA(cudaEventRecord(c.ev_total[slot], ws));
            nvtxRangePop();
        };

        auto finish = [&](size_t bi) {
            const int slot = int(bi % kUp), rslot = int(bi & 1);
            const Up& up = ups[bi];
            nvtxRangePushA("bsg:decode batch + stream out");
            BSG_CUDA(cudaEventSynchronize(c.ev_total[slot]));
            const int64_t n = int64_t(c.h_total.as<uint32_t>()[slot]);
            if (res_->n_rows + n > res_->rows_cap) fail(BSG_EFORMAT, "record count exceeds the planned table capacity");
            if (res_->keep_raw) {
                res_->batches.push_back(ResidentBatch{up.raw_base, up.offs_base, n});
            } else {
                // decode on the high-priority stream as soon as the walk of this batch is done (ev_total): it goes ahead of
                // whatever of the next batches has not started yet
                BSG_CUDA(cudaStreamWaitEvent(c.s_hi, c.ev_total[slot], 0));
                Span sp{c.timing_event(), c.timing_event()};
                BSG_CUDA(cudaEventRecord(sp.a, c.s_hi));
                if (!cnt_.active) fail(BSG_EARG, "internal error: streaming decode without a counting call");
                launch_decode(DecodeBatch{up.d_raw, up.d_offs, res_->n_rows, int32_t(n), 0}, table(), cnt_.mode == MODE_COVERAGE, cnt_.ss != 0, cnt_.fp,
                              c.scalars.as<DeviceScalars>(), c.s_hi);
                BSG_CUDA(cudaEventRecord(sp.b, c.s_hi));
                kt_.decode.push_back(sp); kt_.launches += n > 0;
                // K1 (and the CRC kernel) were the last readers of the raw buffer: inflate(bi + 2) may have it, without
                // waiting for the counting kernels queued below
                if (opts_.verify_crc) BSG_CUDA(cudaStreamWaitEvent(c.s_hi, c.ev_crc[slot], 0));
                BSG_CUDA(cudaEventRecord(c.ev_gfree[rslot], c.s_hi));
                if (n > 0 && cnt_.active) {
                    // (tid, pos) of the last decoded record = how far the sorted read stream has come: count + ship
                    // every tile it finalises while the next batches inflate
                    // (Polling for the frontier between upload chunks instead of blocking here was measured: no gain.)
                    ReadTable t = table();
                    int32_t* f = c.h_front.as<int32_t>();
                    launch_publish_pair(t.tid + (res_->n_rows + n - 1), t.pos + (res_->n_rows + n - 1), f, c.s_hi);      // not a memcpy: see compute()
                    BSG_CUDA(cudaEventRecord(c.ev_front[0], c.s_hi));
                    BSG_CUDA(cudaEventSynchronize(c.ev_front[0]));
                    advance(res_->n_rows + n, uint32_t(f[0]), f[1]);
                }
            }
            res_->n_rows += n;
            nvtxRangePop();
        };

        const double t_pipe0 = now_ms();
        size_t n_up = 0, n_comp = 0;
        auto upload_to = [&](size_t k) { for (; n_up < std::min(k + 1, nb); ++n_up) upload(n_up); };
        auto compute_to = [&](size_t k) { for (; n_comp < std::min(k + 1, nb); ++n_comp) compute(n_comp); };
        try {
            // two batches queued on the device, a third on its way: then the setup the call deferred (tiles, streamer),
            // on this thread, while the first batch uploads and inflates
            upload_to(1); compute_to(0); compute_to(1); upload_to(2);
            run_deferred();
            for (size_t bi = 0; bi < nb; ++bi) {
                compute_to(bi + 1);
                upload_to(bi + 2);
                const double tt = now_ms();
                finish(bi);
                t_finish += now_ms() - tt;
                if (dbg_tl) fprintf(stderr, "[bsg]   host: finish(%zu) entered %.2f, returned %.2f ms after the pipeline started\n", bi, tt - t_pipe0, now_ms() - t_pipe0);
            }
        } catch (...) {
            // queued copies and kernels still reference this call's buffers
            cudaStreamSynchronize(c.s_copy); cudaStreamSynchronize(c.s_comp); cudaStreamSynchronize(c.s_walk); cudaStreamSynchronize(c.s_walk2);
            cudaStreamSynchronize(c.s_aux); cudaStreamSynchronize(c.s_hi);
            throw;
        }
        BSG_CUDA(cudaStreamSynchronize(c.s_comp));
        BSG_CUDA(cudaStreamSynchronize(c.s_walk));
        BSG_CUDA(cudaStreamSynchronize(c.s_walk2));
        BSG_CUDA(cudaStreamSynchronize(c.s_hi));
        if (opts_.verify_crc) BSG_CUDA(cudaStreamSynchronize(c.s_aux));
        tm_.ms_inflate_gpu = sum_ms(inflate_spans);
        tm_.ms_h2d = sum_ms(h2d_spans);         // on the copy stream: the time the copy engine (and, when staging, the pool) needed
        if (getenv("BSG_DEBUG")) {
            fprintf(stderr, "[bsg] gpu pipeline host ms: descriptors %.1f, slot wait %.1f, memcpy+h2d %.1f, finish(wait total) %.1f; device inflate %.1f, walk %.1f\n",
                    t_desc, t_wait, t_copy, t_finish, tm_.ms_inflate_gpu, sum_ms(walk_spans));
            // device timeline of the batches relative to the first upload (ms): h2d, inflate, walk, decode
            auto rel = [&](cudaEvent_t e) { float ms = 0; cudaEventElapsedTime(&ms, h2d_spans[0].a, e); return ms; };
            for (size_t k = 0; k < nb && !h2d_spans.empty(); ++k) {
                fprintf(stderr, "[bsg]   batch %zu: h2d %.2f-%.2f inflate %.2f-%.2f walk %.2f-%.2f", k, rel(h2d_spans[k].a), rel(h2d_spans[k].b),
                        rel(inflate_spans[k].a), rel(inflate_spans[k].b), rel(walk_spans[k].a), rel(walk_spans[k].b));
                if (!res_->keep_raw && k < dec_first + nb && dec_first + k < kt_.decode.size())
                    fprintf(stderr, " decode %.2f-%.2f", rel(kt_.decode[dec_first + k].a), rel(kt_.decode[dec_first + k].b));
                if (k < crc_spans.size()) fprintf(stderr, " crc %.2f-%.2f", rel(crc_spans[k].a), rel(crc_spans[k].b));
                fprintf(stderr, "\n");
            }
            for (size_t k = cnt_first; k < kt_.count.size(); ++k)
                fprintf(stderr, "[bsg]   count launch %zu: join %.2f-%.2f count %.2f-%.2f\n", k - cnt_first, rel(kt_.join[k].a), rel(kt_.join[k].b),
                        rel(kt_.count[k].a), rel(kt_.count[k].b));
        }
        BSG_CUDA(cudaMemcpyAsync(c.h_scalars.p, c.scalars.p, sizeof(DeviceScalars), cudaMemcpyDeviceToHost, c.s_comp));
        BSG_CUDA(cudaStreamSynchronize(c.s_comp));
        check_status(c.h_scalars.as<DeviceScalars>()->status);
        if (res_->keep_raw) build_resident_table();
        tm_.records = res_->n_rows;
    }

    void build_resident_table() {
        DeviceCtx& c = *ctx_;
        std::vector<DecodeBatch> tab;
        int chunks = 0;
        int64_t row0 = 0;
        for (auto& rb : res_->batches) {
            if (rb.n > 0) {
                tab.push_back(DecodeBatch{res_->raw_all.as<uint8_t>() + rb.raw_base, res_->offs_all.as<uint32_t>() + rb.offs_base, row0, int32_t(rb.n), chunks});
                chunks += int((rb.n + kDecodeChunk - 1) / kDecodeChunk);
            }
            row0 += rb.n;
        }
        res_->batches.resize(tab.size());
        res_->chunks = chunks;
        res_->batch_table.ensure(tab.size() * sizeof(DecodeBatch) + 64);
        if (!tab.empty()) BSG_CUDA(cudaMemcpy(res_->batch_table.p, tab.data(), tab.size() * sizeof(DecodeBatch), cudaMemcpyHostToDevice));
        BSG_CUDA(cudaStreamSynchronize(c.s_comp));
        build_resident_index(row0);
    }

    // The record index of the fused pileup step (DESIGN.md §13), built once per staged session by two passes of K0i
    // over every resident record (the open call's ms_decode):
    //   pass 0: a key per 32 rows, the unsorted / corrupt status bits, reach = max(pos + span) and
    //           the span buckets;
    //   host:   the long-span threshold T = 2^k - 1 for the smallest k >= 6 that leaves at most 1/64 of the rows with
    //           span > T (C2: reads ~100 bp, 1 % spliced with a 100-10,000 bp N => T = 127, the spliced reads are long);
    //   pass 1: the long list (rows with span > T), sorted by key on the host.
    // The status bits do not fail the open: every staged call raises them, as K1 does on the table path.
    void build_resident_index(int64_t n_rows) {
        DeviceCtx& c = *ctx_;
        res_->idx = ResidentIndexHost();
        const int nb = int(res_->batches.size());
        if (n_rows <= 0 || nb == 0) return;
        res_->idx.n = n_rows;
        const int64_t n_keys = (n_rows + kIndexStride - 1) / kIndexStride;
        res_->idx_keys.ensure(size_t(n_keys) * sizeof(uint64_t));
        res_->idx_scal.ensure(sizeof(IndexScalars));
        IndexScalars* isc = res_->idx_scal.as<IndexScalars>();
        cudaStream_t st = c.s_comp;
        Span sp0{c.timing_event(), c.timing_event()};
        BSG_CUDA(cudaMemsetAsync(isc, 0, sizeof(IndexScalars), st));
        BSG_CUDA(cudaEventRecord(sp0.a, st));
        launch_resident_index(res_->batch_table.as<DecodeBatch>(), nb, res_->chunks, 0, 0, res_->idx_keys.as<unsigned long long>(), nullptr,
                              nullptr, isc, st);
        BSG_CUDA(cudaEventRecord(sp0.b, st));
        kt_.decode.push_back(sp0); kt_.launches += 1;
        IndexScalars hs;
        BSG_CUDA(cudaMemcpyAsync(&hs, isc, sizeof hs, cudaMemcpyDeviceToHost, st));
        BSG_CUDA(cudaStreamSynchronize(st));
        res_->idx.n_keys = n_keys;
        res_->idx.status = hs.status;
        res_->idx.reach = int64_t(hs.reach);
        int k = 6;
        for (; k < kSpanBuckets; ++k) {
            uint64_t above = 0;
            for (int b = k; b < kSpanBuckets; ++b) above += hs.bucket_n[b];
            if (above * 64 <= uint64_t(n_rows)) break;
        }
        res_->idx.long_span = k < kSpanBuckets ? (1u << k) - 1u : ~0u;
        uint64_t n_long = 0;
        for (int b = 0; b < kSpanBuckets; ++b) {
            if (b < k) res_->idx.short_max = std::max(res_->idx.short_max, int64_t(hs.bucket_max[b]));
            else { res_->idx.long_max = std::max(res_->idx.long_max, int64_t(hs.bucket_max[b])); n_long += hs.bucket_n[b]; }
        }
        if (n_long) {
            res_->idx_long_key.ensure(size_t(n_long) * sizeof(uint64_t));
            res_->idx_long_row.ensure(size_t(n_long) * sizeof(int2));
            Span sp1{c.timing_event(), c.timing_event()};
            BSG_CUDA(cudaMemsetAsync(&isc->n_long, 0, sizeof(uint32_t), st));
            BSG_CUDA(cudaEventRecord(sp1.a, st));
            launch_resident_index(res_->batch_table.as<DecodeBatch>(), nb, res_->chunks, 1, res_->idx.long_span, nullptr,
                                  res_->idx_long_key.as<unsigned long long>(), res_->idx_long_row.as<int2>(), isc, st);
            BSG_CUDA(cudaEventRecord(sp1.b, st));
            kt_.decode.push_back(sp1); kt_.launches += 1;
            std::vector<uint64_t> lk(n_long);
            std::vector<int2> lr(n_long);
            BSG_CUDA(cudaMemcpyAsync(lk.data(), res_->idx_long_key.p, n_long * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            BSG_CUDA(cudaMemcpyAsync(lr.data(), res_->idx_long_row.p, n_long * sizeof(int2), cudaMemcpyDeviceToHost, st));
            BSG_CUDA(cudaStreamSynchronize(st));
            // pass 1 appends in CTA completion order: sort into row order (key, then batch and record for equal keys)
            std::vector<uint32_t> ord(n_long);
            for (uint32_t j = 0; j < uint32_t(n_long); ++j) ord[j] = j;
            std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) {
                if (lk[a] != lk[b]) return lk[a] < lk[b];
                return lr[a].x != lr[b].x ? lr[a].x < lr[b].x : lr[a].y < lr[b].y;
            });
            std::vector<uint64_t> keys(n_long);
            std::vector<int2> rows(n_long);
            for (size_t j = 0; j < n_long; ++j) { keys[j] = lk[ord[j]]; rows[j] = lr[ord[j]]; }
            res_->idx.n_long = int64_t(n_long);
            BSG_CUDA(cudaMemcpy(res_->idx_long_key.p, keys.data(), n_long * sizeof(uint64_t), cudaMemcpyHostToDevice));
            BSG_CUDA(cudaMemcpy(res_->idx_long_row.p, rows.data(), n_long * sizeof(int2), cudaMemcpyHostToDevice));
        }
    }

    ResidentView resident_view() const {
        return ResidentView{res_->batch_table.as<DecodeBatch>(), int(res_->batches.size()), res_->idx.n, res_->idx_keys.as<unsigned long long>(),
                            res_->idx.n_keys, res_->idx_long_key.as<unsigned long long>(), res_->idx_long_row.as<int2>(), res_->idx.n_long, res_->idx.long_span};
    }

    // Key ranges around a tile that hold every read the call can count there, in int64 from the session's spans and the
    // call's shift / midpoint / tlen bound.  A read's pileup coordinate is pos + D, D = offset (forward) or
    // span - 1 - offset (reverse), offset = shift or |tlen| / 2 + shift; a kept read has tmin <= |tlen| <= tmax, where
    // |tlen| is >= 0 or INT_MIN (abs() leaves INT_MIN negative).  If a coordinate could wrap around int32 (K1 computes it
    // in int32), the ranges are the whole contig.  The kernels' exact per-read test decides what counts.
    FusedHalos fused_halos(const FilterParams& p) const {
        int64_t omin = p.shift, omax = p.shift;
        if (p.midpoint) {
            int64_t amin = INT32_MIN, amax = INT32_MAX;
            if (p.have_tlen) { amax = p.tmax; if (p.tmin > INT32_MIN) amin = std::max<int64_t>(p.tmin, 0); }
            omin = amin / 2 + p.shift;       // truncating division, as the kernels' int32 a / 2
            omax = amax / 2 + p.shift;
        }
        const int64_t big = int64_t(1) << 40;
        if (std::max(std::abs(omin), std::abs(omax)) + res_->idx.reach + 2 > INT32_MAX) return FusedHalos{big, big, big, big};
        auto halo = [&](int64_t smax, int64_t* lo, int64_t* hi) {
            *lo = std::max(omax, std::max<int64_t>(smax, 1) - 1 - omin);
            *hi = std::max(-omin, omax);
        };
        FusedHalos h;
        halo(res_->idx.short_max, &h.s_lo, &h.s_hi);
        halo(res_->idx.long_max, &h.l_lo, &h.l_hi);
        return h;
    }

    // Rows the fused join examines with halos h: K3f itself, run over all tiles on the device (its candidate count comes
    // back; ~0.1 ms, against 27-49 ms for four host binary searches per tile over the sampled keys on C2).  Cached for
    // the last kEstCache (tile table, halos) pairs, so a session that alternates a few parameter sets pays it once per set.
    int64_t fused_rows_estimate(const FusedHalos& h) {
        for (const EstEntry& e : est_cache_)
            if (e.gen == my_tiles_gen_ && memcmp(&e.h, &h, sizeof h) == 0) return e.rows;
        DeviceCtx& c = *ctx_;
        DeviceScalars* sc = c.scalars.as<DeviceScalars>();
        fused_rng_.ensure(size_t(2 * n_tiles_) * sizeof(int64_t) + 64);
        BSG_CUDA(cudaMemsetAsync(&sc->candidates, 0, sizeof(sc->candidates), c.s_comp));
        launch_join_fused(resident_view(), tile_table(0), fused_rng_.as<int64_t>(), fused_rng_.as<int64_t>() + n_tiles_, n_tiles_, h, sc,
                          c.s_comp);
        DeviceScalars* hs = c.h_scalars.as<DeviceScalars>();
        BSG_CUDA(cudaMemcpyAsync(&hs->candidates, &sc->candidates, sizeof(sc->candidates), cudaMemcpyDeviceToHost, c.s_comp));
        BSG_CUDA(cudaStreamSynchronize(c.s_comp));
        const int64_t rows = int64_t(hs->candidates);
        if (est_cache_.size() >= size_t(kEstCache)) est_cache_.erase(est_cache_.begin());
        est_cache_.push_back(EstEntry{my_tiles_gen_, h, rows});
        return rows;
    }

public:
    // Staged pileup calls (after prepare_tiles): the fused step when opts.resident_scheme is 2, or when it is 0 and the
    // rows the fused join would examine are at most kFusedShare of the resident rows; else K1 over every resident record.
    void prepare_resident_pileup(Mode mode, const FilterParams& fp) {
        const int scheme = opts_.resident_scheme;
        bool fused = scheme == 2;
        FusedHalos h{};
        if (scheme != 1) {
            h = fused_halos(fp);
            if (scheme != 2) fused = double(fused_rows_estimate(h)) <= kFusedShare * double(res_->idx.n);
        }
        if (!fused) { decode_resident(mode, fp); return; }
        BSG_CUDA(cudaMemsetAsync(ctx_->scalars.p, 0, sizeof(DeviceScalars), ctx_->s_comp));
        fused_ = true;
        fused_h_ = h;
    }

private:
    std::thread setup_thread_;
    Error setup_err_{0, ""};
    int32_t* prefault_out_ = nullptr;
    int64_t prefault_total_ = 0;
    std::shared_ptr<BamFile> bamp_;
    const BamFile& bam_;
    bsg_opts opts_;
    Regions rg_;
    DeviceCtx* ctx_ = nullptr;
    Pool* pool_ = nullptr;
    std::vector<Segment> segs_;
    std::vector<std::unique_ptr<Batch>> batches_;
    std::shared_ptr<StagedRecords> res_ = std::make_shared<StagedRecords>();
    bool is_view_ = false;
    int64_t view_halo_ = 0;
    uint64_t my_tiles_gen_ = 0;
    std::thread plan_thread_;
    Error plan_err_{0, ""};
    int64_t plan_ext_ = 0;
    double plan_ms_ = 0;
    // the fused pileup step of staged sessions (build_resident_index, prepare_resident_pileup)
    DevBuf fused_rng_;
    bool fused_ = false;                 // this call counts through K3f + K4f
    FusedHalos fused_h_{};
    struct EstEntry { uint64_t gen; FusedHalos h; int64_t rows; };
    static constexpr int kEstCache = 8;
    std::vector<EstEntry> est_cache_;    // fused_rows_estimate's cache, oldest first
    // background pre-faulting of the caller's output buffer
    std::mutex pf_m_;
    std::condition_variable pf_cv_;
    int pf_left_ = 0;
    // counting state + output streamer
    CountState cnt_;
    bool hi_prio_ = false;           // decode/count kernels of this call go to the high-priority stream
    HostTiles ht_;
    std::vector<int64_t> tile_dev_off_;
    std::vector<uint64_t> tile_final_key_;
    std::thread os_thread_;
    std::mutex os_m_;
    std::condition_variable os_cv_;
    std::deque<OutJob> os_jobs_;
    bool os_stop_ = false;
    std::atomic<bool> os_abort_{false};
    Error os_err_{0, ""};
    double os_wait_ms_ = 0, os_scatter_ms_ = 0, os_bytes_ = 0;
    // cached tiles
    bool tiles_valid_ = false, tiles_caller_ = false;
    DeviceOutput dev_out_;
    RunsOutput runs_;
    std::vector<int32_t> runs_tiles_;           // list, rel (and vt) of every virtual tile (uploaded by count_runs)
    Mode tiles_mode_ = MODE_COUNT;
    int32_t tiles_binsize_ = 0;
    int tiles_ss_ = 0;
    std::vector<int64_t> tiles_offsets_;
    int64_t n_tiles_ = 0;
    int max_tile_ints_ = 0;
    KernelTimes kt_;
    bsg_timings tm_;
};

FilterParams make_params(const int32_t* tlen_filter, int32_t mapqual, int32_t shift, int32_t requiredF, int32_t filteredF,
                         int32_t pe_mid, int32_t tspan) {
    FilterParams p;
    memset(&p, 0, sizeof p);
    p.mapqual = mapqual;
    p.required = uint32_t(requiredF);
    p.filtered = uint32_t(filteredF);
    p.have_tlen = tlen_filter != nullptr;
    if (tlen_filter) { p.tmin = tlen_filter[0]; p.tmax = tlen_filter[1]; }
    p.midpoint = pe_mid != 0;
    p.shift = shift;
    p.tspan = tspan != 0;
    return p;
}

int64_t ext_pileup(const int32_t* tlen_filter, int32_t shift, int32_t pe_mid) {
    if (pe_mid && !tlen_filter) fail(BSG_EARG, "pe_mid requires a tlen_filter");      // the reference would read tlen_filter[1]
    return std::abs(int64_t(shift)) + (pe_mid ? int64_t(tlen_filter[1]) : 0);         // src/bamsignals.cpp:457
}
int64_t ext_coverage(const int32_t* tlen_filter, int32_t tspan) {
    if (tspan && !tlen_filter) fail(BSG_EARG, "tspan requires a tlen_filter");
    return tspan ? int64_t(tlen_filter[1]) : 0;                                       // src/bamsignals.cpp:487
}

// A call on several devices: the regions are cut into contiguous shards in (chromosome, start) order, balanced by
// the compressed bytes between their index positions; every shard runs the whole pipeline on its own device in its
// own host thread and writes straight into the caller's per-region destinations.  No exchange step, no collective:
// every output element has exactly one owner (SURVEY 8e).
void run_multi_device(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                      const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                      const bsg_opts& o, Mode mode, const FilterParams& fp, int32_t binsize, int ss, int64_t ext,
                      int32_t* out, const int64_t* out_offsets, int32_t* const* out_ptrs, double t0) {
    if (!out_offsets) fail(BSG_EARG, "out_offsets is required");
    if (!out && !out_ptrs) fail(BSG_EARG, "either out or out_ptrs must be given");
    const int nd = o.n_devices;
    std::shared_ptr<BamFile> bam = open_bam(bampath);
    Regions rg;
    resolve_regions(*bam, R, seq_levels, n_levels, seq_idx, loc, width, strand, &rg);
    // Units of the shards are PIECES, not regions: a region with many output ints (C4: 24 whole chromosomes) is cut
    // into bin-aligned sub-intervals exactly like the counting tiles (make_tiles: each behaves like a region of its own,
    // DESIGN 3), so that a handful of huge regions still spreads over all devices and the shards balance by reads.
    HostTiles pc;
    {
        const int64_t total_ints = R > 0 ? out_offsets[R] : 0;
        int64_t piece_ints = std::max<int64_t>(kTileInts, total_ints / (int64_t(nd) * 64));
        piece_ints = std::min<int64_t>((piece_ints + 7) & ~int64_t(7), int64_t(1) << 30);
        make_tiles(rg, mode, binsize, ss, out_offsets, int(piece_ints), &pc);
    }
    const int64_t P = pc.size();
    std::vector<int64_t> order(P);
    for (int64_t i = 0; i < P; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
        return pc.rid[a] != pc.rid[b] ? pc.rid[a] < pc.rid[b] : (pc.loc[a] != pc.loc[b] ? pc.loc[a] < pc.loc[b] : a < b);
    });
    // cut points at equal compressed-byte quantiles of the pieces' index positions (compressed bytes ~ reads)
    std::vector<int64_t> cut(nd + 1, P);
    cut[0] = 0;
    if (P > 0) {
        std::vector<uint64_t> off(P);
        for (int64_t k = 0; k < P; ++k) off[k] = bam->approx_coffset(pc.rid[order[k]], pc.loc[order[k]]);
        for (int64_t k = 1; k < P; ++k) off[k] = std::max(off[k], off[k - 1]);
        const uint64_t lo = off.front(), hi = std::max(off.back(), lo + 1);
        for (int d = 1; d < nd; ++d) {
            const uint64_t target = lo + (hi - lo) * uint64_t(d) / uint64_t(nd);
            int64_t c = std::lower_bound(off.begin(), off.end(), target) - off.begin();
            c = std::max(c, P * d / (4 * nd));                    // never starve a device completely on odd indexes
            cut[d] = std::max(cut[d - 1], std::min<int64_t>(c, P));
        }
    }
    get_pool(o.inflate_threads);                                   // create the shared worker pool before the device threads race for it
    std::vector<bsg_timings> tms(nd);
    std::vector<Error> errs(nd, Error{0, ""});
    std::vector<std::thread> th;
    for (int d = 0; d < nd; ++d)
        th.emplace_back([&, d] {
            try {
                const int64_t n = cut[d + 1] - cut[d];
                Regions sub;
                sub.R = n;
                sub.rid.resize(n); sub.loc.resize(n); sub.width.resize(n); sub.strand.resize(n);
                std::vector<int64_t> loff(n + 1, 0);
                std::vector<int32_t*> lptr(n);
                for (int64_t k = 0; k < n; ++k) {
                    const int64_t t = order[cut[d] + k], i = pc.region[t];
                    sub.rid[k] = pc.rid[t]; sub.loc[k] = pc.loc[t]; sub.width[k] = pc.len[t]; sub.strand[k] = int8_t(pc.strand[t]);
                    loff[k + 1] = loff[k] + pc.ints[t];
                    lptr[k] = out ? out + pc.out_off[t] : (out_ptrs[i] ? out_ptrs[i] + (pc.out_off[t] - out_offsets[i]) : nullptr);
                }
                Session s(bam, std::move(sub), o, o.devices[d]);
                s.start_plan(ext);
                s.prepare_tiles(mode, binsize, ss, loff.data());
                s.begin_count(mode, fp, binsize, ss, ext, nullptr, loff.data(), lptr.data(), true);
                s.stage(ext, false);
                s.finish_count();
                s.finish_timings(t0);
                s.kick_page_locking();
                tms[d] = s.timings();
            } catch (Error& e) { errs[d] = e; }
            catch (std::exception& e) { errs[d] = Error{BSG_EARG, std::string("internal error: ") + e.what()}; }
        });
    for (auto& t : th) t.join();
    for (auto& e : errs) if (e.code) throw e;
    // aggregate: counters add up, times are the slowest device's
    bsg_timings a;
    memset(&a, 0, sizeof a);
    for (const bsg_timings& t : tms) {
        a.records += t.records; a.records_kept += t.records_kept; a.bytes_compressed += t.bytes_compressed;
        a.bytes_inflated += t.bytes_inflated; a.candidates += t.candidates; a.out_elems += t.out_elems;
        a.n_tiles += t.n_tiles; a.n_batches += t.n_batches; a.n_launches += t.n_launches;
        a.ms_plan = std::max(a.ms_plan, t.ms_plan); a.ms_fetch = std::max(a.ms_fetch, t.ms_fetch);
        a.ms_h2d = std::max(a.ms_h2d, t.ms_h2d); a.ms_d2h = std::max(a.ms_d2h, t.ms_d2h);
        a.ms_decode = std::max(a.ms_decode, t.ms_decode); a.ms_filter = std::max(a.ms_filter, t.ms_filter);
        a.ms_join = std::max(a.ms_join, t.ms_join); a.ms_count = std::max(a.ms_count, t.ms_count);
        a.ms_inflate_gpu = std::max(a.ms_inflate_gpu, t.ms_inflate_gpu); a.ms_kernels = std::max(a.ms_kernels, t.ms_kernels);
        a.ms_device = std::max(a.ms_device, t.ms_device); a.bytes_d2h += t.bytes_d2h;
    }
    a.n_devices = nd;
    a.ms_total = now_ms() - t0;
    g_tm = a;
}

void validate_devices(const bsg_opts& o) {
    if (o.n_devices < 0 || o.n_devices > 16) fail(BSG_EARG, "n_devices must be between 0 and 16");
    for (int a = 0; a < o.n_devices; ++a)
        for (int b = a + 1; b < o.n_devices; ++b)
            if (o.devices[a] == o.devices[b]) fail(BSG_EARG, "the same CUDA device is listed twice");
}

// Device-output calls (bsg_*_device): the device that owns d_out, or -1 when d_out is NULL and the layout is empty.
// Everything the caller could get wrong is refused before anything is written.
int output_device(const int32_t* d_out, int64_t R, const int64_t* out_offsets) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
        cudaGetLastError();
        fail(BSG_ECUDA, "no CUDA device available (libbamsignals_cuda has no CPU fallback)");
    }
    if (!out_offsets) fail(BSG_EARG, "out_offsets is required");
    if (R < 0) fail(BSG_EARG, "negative region count");
    if (!d_out) {
        if (out_offsets[R] == 0) return -1;
        fail(BSG_EARG, "d_out is NULL but the layout has " + std::to_string(out_offsets[R]) + " elements");
    }
    if (reinterpret_cast<uintptr_t>(d_out) & 3) fail(BSG_EARG, "d_out must be 4-byte aligned");
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, d_out) != cudaSuccess) {
        cudaGetLastError();
        fail(BSG_EARG, "d_out is not a pointer CUDA knows");
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)
        fail(BSG_EARG, std::string("d_out must be device or managed memory, not ") +
                       (a.type == cudaMemoryTypeHost ? "page-locked host memory" : "unregistered host memory"));
    return a.device;
}

// With ss, bsg_coverage_ss / bsg_coverage_ss_device refuse a layout that is not the stranded one before any device work,
// so that a caller who passes bamCoverage's unstranded offsets learns it even without a GPU (validate_layout checks the
// layout again once the regions are resolved).
void check_stranded_layout(int64_t R, const int32_t* width, const int64_t* out_offsets) {
    if (!out_offsets) fail(BSG_EARG, "out_offsets is required");
    if (R < 0 || (R > 0 && !width)) fail(BSG_EARG, "invalid region arrays");
    for (int64_t i = 0; i < R; ++i)
        if (out_offsets[i + 1] - out_offsets[i] != 2 * int64_t(width[i]))
            fail(BSG_EARG, "out_offsets[" + std::to_string(i + 1) + "] - out_offsets[" + std::to_string(i) + "] is " +
                           std::to_string(out_offsets[i + 1] - out_offsets[i]) + ", strand-specific coverage needs 2 x width = " +
                           std::to_string(2 * int64_t(width[i])) + " (see bsg_output_layout with binsize 1 and ss)");
}

// The device a bsg_*_device call runs on: the one that owns d_out; opts may name it, but only that one.
int device_for_output(const int32_t* d_out, int64_t R, const int64_t* out_offsets, const bsg_opts* opts) {
    const int dev = output_device(d_out, R, out_offsets);
    const bsg_opts o = effective_opts(opts);
    validate_devices(o);
    if (o.n_devices > 1) fail(BSG_EARG, "device output runs on one device: n_devices must be 0 or 1");
    if (o.n_devices == 1 && dev >= 0 && o.devices[0] != dev)
        fail(BSG_EARG, "d_out is on CUDA device " + std::to_string(dev) + ", opts.devices[0] names device " + std::to_string(o.devices[0]));
    return dev >= 0 ? dev : (o.n_devices == 1 ? o.devices[0] : 0);
}

// Device-output calls run with the buffer's device current - `stream` 0 is that device's legacy stream - and give the
// calling thread its current device back when they return (a torch caller's current device must not change under it).
struct KeepCurrentDevice {
    int prev = -1;
    KeepCurrentDevice() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
    ~KeepCurrentDevice() { if (prev >= 0) cudaSetDevice(prev); }
    KeepCurrentDevice(const KeepCurrentDevice&) = delete;
};

template <class F>
int guarded(F&& f) {
    try {
        std::lock_guard<std::mutex> g(g_mu);
        f();
        return BSG_OK;
    } catch (Error& e) {
        g_err = e.msg;
        cudaGetLastError();
        return e.code;
    } catch (std::bad_alloc&) {
        g_err = "out of host memory";
        return BSG_ENOMEM;
    } catch (std::exception& e) {
        g_err = std::string("internal error: ") + e.what();
        return BSG_EARG;
    }
}

}  // namespace
}  // namespace bsg

using namespace bsg;

struct bsg_stage {
    std::unique_ptr<Session> s;
};

namespace {
// open staged sessions: bsg_shutdown() ends them (their device memory and streams are about to go away); the handles stay
// valid to pass to bsg_stage_close(), every other use is refused
std::vector<bsg_stage*> g_stages;

// live run-length results: bsg_shutdown() frees their device memory, the handles stay valid for bsg_runs_free()
std::vector<bsg_runs*> g_runs;

// A bsg_runs_read destination: true for device (or managed) memory on the result's device, false for host memory.
bool runs_destination(const int32_t* p, const bsg_runs* r, const char* what) {
    if (!p) fail(BSG_EARG, std::string(what) + " is NULL");
    if (reinterpret_cast<uintptr_t>(p) & 3) fail(BSG_EARG, std::string(what) + " must be 4-byte aligned");
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        fail(BSG_EARG, std::string(what) + " is not a pointer CUDA knows");
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) return false;
    if (a.device != r->dev)
        fail(BSG_EARG, std::string(what) + " is on CUDA device " + std::to_string(a.device) + ", the result on device " + std::to_string(r->dev));
    return true;
}

// the device that owns d_out must be the session's (-1: empty layout, nothing is written)
void check_staged_output(const bsg_stage* st, const int32_t* d_out, const int64_t* out_offsets) {
    const int dev = output_device(d_out, st->s->regions(), out_offsets);
    if (dev >= 0 && dev != st->s->device())
        fail(BSG_EARG, "d_out is on CUDA device " + std::to_string(dev) + ", the staged session on device " + std::to_string(st->s->device()));
}
}

extern "C" {

int bsg_pileup(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
               const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
               int32_t mapqual, int32_t binsize, int32_t shift, int32_t ss, int32_t requiredF, int32_t filteredF,
               int32_t pe_mid, int32_t /*maxgap*/, int32_t* out, const int64_t* out_offsets, int32_t* const* out_ptrs,
               const bsg_opts* opts) {
    return guarded([&] {
        const double t0 = now_ms();
        const bsg_opts o = effective_opts(opts);
        validate_devices(o);
        if (o.n_devices > 1) {
            run_multi_device(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, o,
                             binsize <= 0 ? MODE_COUNT : MODE_PROFILE, make_params(tlen_filter, mapqual, shift, requiredF, filteredF, pe_mid, 0),
                             binsize, ss != 0, ext_pileup(tlen_filter, shift, pe_mid), out, out_offsets, out_ptrs, t0);
            return;
        }
        const bool dbg = getenv("BSG_DEBUG") != nullptr;
        Session s(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, opts);
        const double t1 = now_ms();
        const int64_t ext = ext_pileup(tlen_filter, shift, pe_mid);
        const Mode mode = binsize <= 0 ? MODE_COUNT : MODE_PROFILE;
        s.start_plan(ext);
        s.validate_layout(mode, binsize, ss != 0, out_offsets);
        const double t2 = now_ms();
        const FilterParams fp = make_params(tlen_filter, mapqual, shift, requiredF, filteredF, pe_mid, 0);
        if (out && out_offsets) s.request_prefault(out, out_offsets[R]);
        s.defer_setup([&] { s.begin_count(mode, fp, binsize, ss != 0, ext, out, out_offsets, out_ptrs, true, s.setup_stream()); });
        const double t3 = now_ms();
        s.stage(ext, false);
        const double t4 = now_ms();
        s.finish_count();
        const double t5 = now_ms();
        s.finish_timings(t0);
        s.kick_page_locking();
        if (dbg) fprintf(stderr, "[bsg] call host ms: open+regions %.1f, tiles %.1f, begin_count %.1f, stage %.1f, finish_count %.1f\n",
                         t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4);
    });
}

int bsg_coverage(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                 const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                 int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan, int32_t maxgap, int32_t* out,
                 const int64_t* out_offsets, int32_t* const* out_ptrs, const bsg_opts* opts) {
    return bsg_coverage_ss(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, tlen_filter, mapqual, requiredF,
                           filteredF, tspan, 0, maxgap, out, out_offsets, out_ptrs, opts);
}

int bsg_coverage_ss(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                    const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                    int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan, int32_t ss, int32_t /*maxgap*/,
                    int32_t* out, const int64_t* out_offsets, int32_t* const* out_ptrs, const bsg_opts* opts) {
    return guarded([&] {
        const double t0 = now_ms();
        if (ss) check_stranded_layout(R, width, out_offsets);
        const bsg_opts o = effective_opts(opts);
        validate_devices(o);
        if (o.n_devices > 1) {
            run_multi_device(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, o, MODE_COVERAGE,
                             make_params(tlen_filter, mapqual, 0, requiredF, filteredF, 0, tspan), 1, ss != 0,
                             ext_coverage(tlen_filter, tspan), out, out_offsets, out_ptrs, t0);
            return;
        }
        Session s(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, opts);
        const int64_t ext = ext_coverage(tlen_filter, tspan);
        s.start_plan(ext);
        s.validate_layout(MODE_COVERAGE, 1, ss != 0, out_offsets);
        const FilterParams fp = make_params(tlen_filter, mapqual, 0, requiredF, filteredF, 0, tspan);
        if (out && out_offsets) s.request_prefault(out, out_offsets[R]);
        s.defer_setup([&] { s.begin_count(MODE_COVERAGE, fp, 1, ss != 0, ext, out, out_offsets, out_ptrs, true, s.setup_stream()); });
        s.stage(ext, false);
        s.finish_count();
        s.finish_timings(t0);
        s.kick_page_locking();
    });
}

int bsg_pileup_device(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                      const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                      int32_t mapqual, int32_t binsize, int32_t shift, int32_t ss, int32_t requiredF, int32_t filteredF,
                      int32_t pe_mid, int32_t /*maxgap*/, int32_t* d_out, const int64_t* out_offsets, void* stream,
                      const bsg_opts* opts) {
    return guarded([&] {
        const double t0 = now_ms();
        KeepCurrentDevice keep;
        const int dev = device_for_output(d_out, R, out_offsets, opts);
        Session s(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, opts, dev);
        const int64_t ext = ext_pileup(tlen_filter, shift, pe_mid);
        const Mode mode = binsize <= 0 ? MODE_COUNT : MODE_PROFILE;
        s.start_plan(ext);
        s.validate_layout(mode, binsize, ss != 0, out_offsets);
        s.use_device_output(d_out, static_cast<cudaStream_t>(stream));
        const FilterParams fp = make_params(tlen_filter, mapqual, shift, requiredF, filteredF, pe_mid, 0);
        s.defer_setup([&] { s.begin_count(mode, fp, binsize, ss != 0, ext, nullptr, out_offsets, nullptr, false, s.setup_stream()); });
        s.stage(ext, false);
        s.finish_count();
        s.finish_timings(t0);
        s.kick_page_locking();
    });
}

int bsg_coverage_device(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                        const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                        int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan, int32_t maxgap,
                        int32_t* d_out, const int64_t* out_offsets, void* stream, const bsg_opts* opts) {
    return bsg_coverage_ss_device(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, tlen_filter, mapqual, requiredF,
                                  filteredF, tspan, 0, maxgap, d_out, out_offsets, stream, opts);
}

int bsg_coverage_ss_device(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                           const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                           int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan, int32_t ss, int32_t /*maxgap*/,
                           int32_t* d_out, const int64_t* out_offsets, void* stream, const bsg_opts* opts) {
    return guarded([&] {
        const double t0 = now_ms();
        if (ss) check_stranded_layout(R, width, out_offsets);
        KeepCurrentDevice keep;
        const int dev = device_for_output(d_out, R, out_offsets, opts);
        Session s(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, opts, dev);
        const int64_t ext = ext_coverage(tlen_filter, tspan);
        s.start_plan(ext);
        s.validate_layout(MODE_COVERAGE, 1, ss != 0, out_offsets);
        s.use_device_output(d_out, static_cast<cudaStream_t>(stream));
        const FilterParams fp = make_params(tlen_filter, mapqual, 0, requiredF, filteredF, 0, tspan);
        s.defer_setup([&] { s.begin_count(MODE_COVERAGE, fp, 1, ss != 0, ext, nullptr, out_offsets, nullptr, false, s.setup_stream()); });
        s.stage(ext, false);
        s.finish_count();
        s.finish_timings(t0);
        s.kick_page_locking();
    });
}

int64_t bsg_output_layout(int64_t R, const int32_t* width, int32_t binsize, int32_t ss, int64_t* offsets) {
    const int64_t mult = ss ? 2 : 1;
    int64_t acc = 0;
    for (int64_t i = 0; i < R; ++i) {
        offsets[i] = acc;
        acc += binsize <= 0 ? mult : mult * ((int64_t(width[i]) + binsize - 1) / binsize);
    }
    offsets[R] = acc;
    return acc;
}

int bsg_stage_open(bsg_stage** st, const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                   const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                   int32_t ext_hint, const bsg_opts* opts) {
    if (!st) { g_err = "null stage pointer"; return BSG_EARG; }
    *st = nullptr;
    return guarded([&] {
        const double t0 = now_ms();
        auto h = std::make_unique<bsg_stage>();
        h->s.reset(new Session(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, opts));
        h->s->stage(ext_hint, true);
        h->s->finish_timings(t0);
        h->s->kick_page_locking();
        g_stages.push_back(h.get());
        *st = h.release();
    });
}

int bsg_stage_view(bsg_stage** view, const bsg_stage* st, int64_t R, const char* const* seq_levels, int32_t n_levels,
                   const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand) {
    if (!view) { g_err = "null view pointer"; return BSG_EARG; }
    *view = nullptr;
    if (!st) { g_err = "null stage"; return BSG_EARG; }
    return guarded([&] {
        if (!st->s) fail(BSG_EARG, "this staged session was ended by bsg_shutdown()");
        const double t0 = now_ms();
        const Session& s = *st->s;
        Regions rg;
        resolve_regions(s.bam(), R, seq_levels, n_levels, seq_idx, loc, width, strand, &rg);
        const int64_t halo = s.view_halo(rg);
        auto h = std::make_unique<bsg_stage>();
        h->s.reset(new Session(s, std::move(rg), halo));
        memset(&g_tm, 0, sizeof g_tm);
        g_tm.ms_total = now_ms() - t0;
        g_stages.push_back(h.get());
        *view = h.release();
    });
}

int bsg_pileup_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift,
                      int32_t ss, int32_t requiredF, int32_t filteredF, int32_t pe_mid, int32_t* out,
                      const int64_t* out_offsets) {
    if (!st) { g_err = "null stage"; return BSG_EARG; }
    return guarded([&] {
        if (!st->s) fail(BSG_EARG, "this staged session was ended by bsg_shutdown()");
        const double t0 = now_ms();
        st->s->reset_counters();
        st->s->require_ext(ext_pileup(tlen_filter, shift, pe_mid));
        st->s->use_host_output();
        st->s->prepare_tiles(binsize <= 0 ? MODE_COUNT : MODE_PROFILE, binsize, ss != 0, out_offsets);
        const FilterParams fp = make_params(tlen_filter, mapqual, shift, requiredF, filteredF, pe_mid, 0);
        st->s->prepare_resident_pileup(binsize <= 0 ? MODE_COUNT : MODE_PROFILE, fp);
        st->s->count(binsize <= 0 ? MODE_COUNT : MODE_PROFILE, fp, binsize, ss != 0, out, out_offsets, nullptr, out != nullptr);
        st->s->finish_timings(t0);
    });
}

int bsg_coverage_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                        int32_t filteredF, int32_t tspan, int32_t* out, const int64_t* out_offsets) {
    return bsg_coverage_ss_staged(st, tlen_filter, mapqual, requiredF, filteredF, tspan, 0, out, out_offsets);
}

int bsg_coverage_ss_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                           int32_t filteredF, int32_t tspan, int32_t ss, int32_t* out, const int64_t* out_offsets) {
    if (!st) { g_err = "null stage"; return BSG_EARG; }
    return guarded([&] {
        if (!st->s) fail(BSG_EARG, "this staged session was ended by bsg_shutdown()");
        const double t0 = now_ms();
        st->s->reset_counters();
        st->s->require_ext(ext_coverage(tlen_filter, tspan));
        st->s->use_host_output();
        st->s->prepare_tiles(MODE_COVERAGE, 1, ss != 0, out_offsets);
        const FilterParams fp = make_params(tlen_filter, mapqual, 0, requiredF, filteredF, 0, tspan);
        st->s->decode_resident(MODE_COVERAGE, fp, ss != 0);
        st->s->count(MODE_COVERAGE, fp, 1, ss != 0, out, out_offsets, nullptr, out != nullptr);
        st->s->finish_timings(t0);
    });
}

int bsg_pileup_staged_device(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift,
                             int32_t ss, int32_t requiredF, int32_t filteredF, int32_t pe_mid, int32_t* d_out,
                             const int64_t* out_offsets, void* stream) {
    if (!st) { g_err = "null stage"; return BSG_EARG; }
    return guarded([&] {
        if (!st->s) fail(BSG_EARG, "this staged session was ended by bsg_shutdown()");
        const double t0 = now_ms();
        KeepCurrentDevice keep;
        check_staged_output(st, d_out, out_offsets);
        BSG_CUDA(cudaSetDevice(st->s->device()));
        const Mode mode = binsize <= 0 ? MODE_COUNT : MODE_PROFILE;
        st->s->reset_counters();
        st->s->require_ext(ext_pileup(tlen_filter, shift, pe_mid));
        st->s->use_device_output(d_out, static_cast<cudaStream_t>(stream));
        st->s->prepare_tiles(mode, binsize, ss != 0, out_offsets);
        const FilterParams fp = make_params(tlen_filter, mapqual, shift, requiredF, filteredF, pe_mid, 0);
        st->s->prepare_resident_pileup(mode, fp);
        st->s->count(mode, fp, binsize, ss != 0, nullptr, out_offsets, nullptr, false);
        st->s->finish_timings(t0);
    });
}

int bsg_coverage_staged_device(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                               int32_t filteredF, int32_t tspan, int32_t* d_out, const int64_t* out_offsets, void* stream) {
    return bsg_coverage_ss_staged_device(st, tlen_filter, mapqual, requiredF, filteredF, tspan, 0, d_out, out_offsets, stream);
}

int bsg_coverage_ss_staged_device(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                                  int32_t filteredF, int32_t tspan, int32_t ss, int32_t* d_out, const int64_t* out_offsets,
                                  void* stream) {
    if (!st) { g_err = "null stage"; return BSG_EARG; }
    return guarded([&] {
        if (!st->s) fail(BSG_EARG, "this staged session was ended by bsg_shutdown()");
        const double t0 = now_ms();
        KeepCurrentDevice keep;
        check_staged_output(st, d_out, out_offsets);
        BSG_CUDA(cudaSetDevice(st->s->device()));
        st->s->reset_counters();
        st->s->require_ext(ext_coverage(tlen_filter, tspan));
        st->s->use_device_output(d_out, static_cast<cudaStream_t>(stream));
        st->s->prepare_tiles(MODE_COVERAGE, 1, ss != 0, out_offsets);
        const FilterParams fp = make_params(tlen_filter, mapqual, 0, requiredF, filteredF, 0, tspan);
        st->s->decode_resident(MODE_COVERAGE, fp, ss != 0);
        st->s->count(MODE_COVERAGE, fp, 1, ss != 0, nullptr, out_offsets, nullptr, false);
        st->s->finish_timings(t0);
    });
}

int bsg_coverage_runs(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                      const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                      int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan, int32_t maxgap,
                      int64_t* run_offsets, bsg_runs** runs, const bsg_opts* opts) {
    return bsg_coverage_runs_ss(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, tlen_filter, mapqual, requiredF,
                                filteredF, tspan, 0, maxgap, run_offsets, runs, opts);
}

int bsg_coverage_runs_ss(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                         const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                         int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan, int32_t ss, int32_t /*maxgap*/,
                         int64_t* run_offsets, bsg_runs** runs, const bsg_opts* opts) {
    if (!runs) { g_err = "runs must not be NULL"; return BSG_EARG; }
    *runs = nullptr;
    return guarded([&] {
        const double t0 = now_ms();
        const bsg_opts o = effective_opts(opts);
        validate_devices(o);
        if (o.n_devices > 1) fail(BSG_EARG, "run-length coverage runs on one device: n_devices must be 0 or 1");
        if (!run_offsets) fail(BSG_EARG, "run_offsets is required");
        KeepCurrentDevice keep;
        Session s(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, opts);
        const int64_t ext = ext_coverage(tlen_filter, tspan);
        const std::vector<int64_t> dense = s.coverage_layout(ss != 0);
        s.start_plan(ext);
        auto res = std::make_unique<bsg_runs>();
        s.use_runs_output(res.get(), run_offsets);
        const FilterParams fp = make_params(tlen_filter, mapqual, 0, requiredF, filteredF, 0, tspan);
        s.defer_setup([&] { s.begin_count(MODE_COVERAGE, fp, 1, ss != 0, ext, nullptr, dense.data(), nullptr, false, s.setup_stream()); });
        s.stage(ext, false);
        s.finish_count();
        s.finish_timings(t0);
        s.kick_page_locking();
        res->live = true;
        g_runs.push_back(res.get());
        *runs = res.release();
    });
}

int bsg_coverage_runs_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF,
                             int32_t tspan, int64_t* run_offsets, bsg_runs** runs) {
    return bsg_coverage_runs_ss_staged(st, tlen_filter, mapqual, requiredF, filteredF, tspan, 0, run_offsets, runs);
}

int bsg_coverage_runs_ss_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF,
                                int32_t tspan, int32_t ss, int64_t* run_offsets, bsg_runs** runs) {
    if (!runs) { g_err = "runs must not be NULL"; return BSG_EARG; }
    *runs = nullptr;
    if (!st) { g_err = "null stage"; return BSG_EARG; }
    return guarded([&] {
        if (!st->s) fail(BSG_EARG, "this staged session was ended by bsg_shutdown()");
        if (!run_offsets) fail(BSG_EARG, "run_offsets is required");
        const double t0 = now_ms();
        KeepCurrentDevice keep;
        BSG_CUDA(cudaSetDevice(st->s->device()));
        st->s->reset_counters();
        st->s->require_ext(ext_coverage(tlen_filter, tspan));
        auto res = std::make_unique<bsg_runs>();
        st->s->use_runs_output(res.get(), run_offsets);
        const std::vector<int64_t> dense = st->s->coverage_layout(ss != 0);
        st->s->prepare_tiles(MODE_COVERAGE, 1, ss != 0, dense.data());
        const FilterParams fp = make_params(tlen_filter, mapqual, 0, requiredF, filteredF, 0, tspan);
        st->s->decode_resident(MODE_COVERAGE, fp, ss != 0);
        st->s->count(MODE_COVERAGE, fp, 1, ss != 0, nullptr, dense.data(), nullptr, false);
        st->s->finish_timings(t0);
        st->s->use_host_output();
        res->live = true;
        g_runs.push_back(res.get());
        *runs = res.release();
    });
}

int bsg_profile_runs(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                     const int32_t* loc, const int32_t* width, const int8_t* strand, const int32_t* tlen_filter,
                     int32_t mapqual, int32_t binsize, int32_t shift, int32_t ss, int32_t requiredF, int32_t filteredF,
                     int32_t pe_mid, int32_t /*maxgap*/, int64_t* run_offsets, bsg_runs** runs, const bsg_opts* opts) {
    if (!runs) { g_err = "runs must not be NULL"; return BSG_EARG; }
    *runs = nullptr;
    return guarded([&] {
        const double t0 = now_ms();
        const bsg_opts o = effective_opts(opts);
        validate_devices(o);
        if (o.n_devices > 1) fail(BSG_EARG, "run-length profiles run on one device: n_devices must be 0 or 1");
        if (!run_offsets) fail(BSG_EARG, "run_offsets is required");
        if (binsize < 1) fail(BSG_EARG, "run-length profiles need binsize >= 1 (bamCount has no runs form)");
        const int64_t ext = ext_pileup(tlen_filter, shift, pe_mid);
        KeepCurrentDevice keep;
        Session s(bampath, R, seq_levels, n_levels, seq_idx, loc, width, strand, opts);
        const std::vector<int64_t> dense = s.profile_layout(binsize, ss != 0);
        s.start_plan(ext);
        auto res = std::make_unique<bsg_runs>();
        s.use_runs_output(res.get(), run_offsets);
        const FilterParams fp = make_params(tlen_filter, mapqual, shift, requiredF, filteredF, pe_mid, 0);
        s.defer_setup([&] { s.begin_count(MODE_PROFILE, fp, binsize, ss != 0, ext, nullptr, dense.data(), nullptr, false, s.setup_stream()); });
        s.stage(ext, false);
        s.finish_count();
        s.finish_timings(t0);
        s.kick_page_locking();
        res->live = true;
        g_runs.push_back(res.get());
        *runs = res.release();
    });
}

int bsg_profile_runs_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift,
                            int32_t ss, int32_t requiredF, int32_t filteredF, int32_t pe_mid, int64_t* run_offsets,
                            bsg_runs** runs) {
    if (!runs) { g_err = "runs must not be NULL"; return BSG_EARG; }
    *runs = nullptr;
    if (!st) { g_err = "null stage"; return BSG_EARG; }
    return guarded([&] {
        if (!st->s) fail(BSG_EARG, "this staged session was ended by bsg_shutdown()");
        if (!run_offsets) fail(BSG_EARG, "run_offsets is required");
        if (binsize < 1) fail(BSG_EARG, "run-length profiles need binsize >= 1 (bamCount has no runs form)");
        const double t0 = now_ms();
        KeepCurrentDevice keep;
        BSG_CUDA(cudaSetDevice(st->s->device()));
        st->s->reset_counters();
        st->s->require_ext(ext_pileup(tlen_filter, shift, pe_mid));
        auto res = std::make_unique<bsg_runs>();
        st->s->use_runs_output(res.get(), run_offsets);
        const std::vector<int64_t> dense = st->s->profile_layout(binsize, ss != 0);
        st->s->prepare_tiles(MODE_PROFILE, binsize, ss != 0, dense.data());
        const FilterParams fp = make_params(tlen_filter, mapqual, shift, requiredF, filteredF, pe_mid, 0);
        st->s->decode_resident(MODE_PROFILE, fp);
        st->s->count(MODE_PROFILE, fp, binsize, ss != 0, nullptr, dense.data(), nullptr, false);
        st->s->finish_timings(t0);
        st->s->use_host_output();
        res->live = true;
        g_runs.push_back(res.get());
        *runs = res.release();
    });
}

int bsg_runs_read(const bsg_runs* runs, int32_t* lengths, int32_t* values, void* stream) {
    if (!runs) { g_err = "runs must not be NULL"; return BSG_EARG; }
    return guarded([&] {
        if (!runs->live) fail(BSG_EARG, "this result was freed by bsg_shutdown()");
        if (runs->n == 0) return;
        KeepCurrentDevice keep;
        const bool dev_l = runs_destination(lengths, runs, "lengths"), dev_v = runs_destination(values, runs, "values");
        BSG_CUDA(cudaSetDevice(runs->dev));
        // on the caller's stream: ordered after what it has queued; synchronous like every call
        cudaStream_t s = static_cast<cudaStream_t>(stream);
        const size_t bytes = size_t(runs->n) * sizeof(int32_t);
        BSG_CUDA(cudaMemcpyAsync(lengths, runs->lengths, bytes, dev_l ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
        BSG_CUDA(cudaMemcpyAsync(values, runs->values, bytes, dev_v ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
        BSG_CUDA(cudaStreamSynchronize(s));
    });
}

void bsg_runs_free(bsg_runs* runs) {
    if (!runs) return;
    std::lock_guard<std::mutex> g(g_mu);
    g_runs.erase(std::remove(g_runs.begin(), g_runs.end(), runs), g_runs.end());
    KeepCurrentDevice keep;
    delete runs;
}

void bsg_stage_close(bsg_stage* st) {
    if (!st) return;
    std::lock_guard<std::mutex> g(g_mu);
    g_stages.erase(std::remove(g_stages.begin(), g_stages.end(), st), g_stages.end());
    delete st;                                   // returns the session's resident device memory
}

const char* bsg_last_error(void) { return g_err.c_str(); }

int bsg_get_timings(bsg_timings* t) {
    if (!t) return BSG_EARG;
    *t = g_tm;
    return BSG_OK;
}

int bsg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void bsg_shutdown(void) {
    std::lock_guard<std::mutex> g(g_mu);
    stop_pin_thread();
    for (bsg_stage* st : g_stages) st->s.reset();
    {
        KeepCurrentDevice keep;
        for (bsg_runs* r : g_runs) r->release();
    }
    for (auto& c : g_ctx) c.release();
    g_pool.reset();
    g_bams.clear();
}

int64_t bsg_debug_plan(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels, const int32_t* seq_idx,
                       const int32_t* loc, const int32_t* width, const int8_t* strand, int64_t ext, int64_t* n_segments,
                       int64_t* bytes_compressed, int64_t* bytes_inflated, int32_t* tid_out, int32_t* pos_out, int64_t cap) {
    int64_t n_rec = 0;
    const int rc = guarded([&] {
        if (ext < 0) fail(BSG_EARG, "negative 'ext' values don't make sense");
        std::shared_ptr<BamFile> bam = open_bam(bampath);
        Regions rg;
        resolve_regions(*bam, R, seq_levels, n_levels, seq_idx, loc, width, strand, &rg);
        std::vector<Segment> segs;
        plan_fetch(*bam, rg, ext, kSegCBytes, get_pool(0), &segs);
        int64_t cb = 0, ub = 0;
        Inflater inf;
        std::vector<uint8_t> buf;
        for (const Segment& sg : segs) {
            cb += int64_t(sg.csize); ub += int64_t(sg.usize);
            buf.resize(sg.usize + 8);
            uint64_t u = 0;
            for (const BlockInfo& b : sg.blocks) { inf.inflate_block(bam->data(), b, buf.data() + u, true); u += b.isize; }
            for (uint64_t p = sg.ubeg; p < sg.uend;) {          // the block_size chain, as the walk kernels follow it
                if (p + 4 > sg.uend) fail(BSG_EFORMAT, "truncated BAM record in " + bam->path());
                const int32_t bs = rd_i32(buf.data() + p);
                if (bs < 32 || p + 4 + uint64_t(bs) > sg.uend) fail(BSG_EFORMAT, "corrupt BAM record chain in " + bam->path());
                if (n_rec < cap && tid_out && pos_out) { tid_out[n_rec] = rd_i32(buf.data() + p + 4); pos_out[n_rec] = rd_i32(buf.data() + p + 8); }
                ++n_rec;
                p += 4 + uint64_t(bs);
            }
        }
        if (n_segments) *n_segments = int64_t(segs.size());
        if (bytes_compressed) *bytes_compressed = cb;
        if (bytes_inflated) *bytes_inflated = ub;
    });
    return rc == BSG_OK ? n_rec : int64_t(rc);
}

int bsg_write_sam_as_bam_and_index(const char* sampath, const char* bampath) {
    return guarded([&] {
        // a cached handle of a file this call replaces must not survive it
        const std::string p = bampath ? bampath : "";
        for (auto it = g_bams.begin(); it != g_bams.end();) it = (*it)->path() == p ? g_bams.erase(it) : it + 1;
        write_sam_as_bam_and_index(sampath, bampath);
    });
}

const char* bsg_version(void) { return "bamsignals_cuda 0.1.0 (sm_100a)"; }

}  // extern "C"
