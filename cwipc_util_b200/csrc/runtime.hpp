// runtime.hpp -- device plumbing shared by every translation unit of libcwipc_util_cuda:
// per-thread streams, stream-ordered device memory, refcounted point storage, launch accounting.
//
// Design notes (see DESIGN.md §3):
//  * one stream per (host thread, device); a cloud remembers the stream that produced it
//    ("home") and an event recorded when its contents became valid.  A consumer on another
//    stream waits on that event; the storage is returned to the pool on its home stream after
//    waiting for every foreign reader.  No global lock is held while work is queued.
//  * device memory comes from a private cudaMemPool per device (cudaMallocFromPoolAsync) with the release
//    threshold raised, so steady-state frames never reach cudaMalloc; the device's default pool is not touched.
//  * there is NO host fallback: every entry point that needs a device fails loudly without one.
#pragma once

#include <cuda_runtime.h>
#include <atomic>
#include <cstddef>
#include <cstdint>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "cwipc_util_cuda.h"

namespace cwcu {

// ---- logging (logging.cpp); mirrors src/logging.cpp + include/cwipc_util/internal/logging.hpp ----
void log(cwipc_log_level level, const std::string &module, const std::string &message);
void log_set_errorbuf(char **errorbuf);
cwipc_log_level log_get_level();

// ---- errors ----
struct CudaError {
    cudaError_t code;
    std::string what;
};
[[noreturn]] void throw_cuda(cudaError_t e, const char *expr, const char *file, int line);
#define CWCU_CHECK(expr)                                                      \
    do {                                                                      \
        cudaError_t _e = (expr);                                              \
        if (_e != cudaSuccess) ::cwcu::throw_cuda(_e, #expr, __FILE__, __LINE__); \
    } while (0)

// ---- devices and streams ----
int device_count();                 // 0 when no usable device
int current_device();               // thread-local selection (default $CWIPC_CUDA_DEVICE or 0)
bool set_current_device(int dev);
cudaStream_t thread_stream(int dev); // the calling thread's stream on `dev` (created on first use)
int sm_count(int dev);

// RAII: make `dev` the CUDA-current device of this thread for the scope.
struct DeviceGuard {
    int prev;
    explicit DeviceGuard(int dev);
    ~DeviceGuard();
};

// ---- memory ----
void *dmalloc(size_t bytes, cudaStream_t s);      // never returns nullptr for bytes>0 (throws)
void dfree(void *p, cudaStream_t s) noexcept;
// Small page-locked scratch owned by the calling thread (count readbacks etc.), >= bytes, 16B aligned.
void *thread_pinned(size_t bytes);
bool is_pinned_host(const void *p);
// Host <-> device copies of point buffers for callers that hand us ordinary (pageable) memory, as an unchanged
// python/cwipc/util.py caller does.  The driver stages such copies itself, one caller at a time; here every caller
// thread copies through its OWN page-locked ring (4 x 2 MB), chunk by chunk, so that the host-side memcpy of one chunk
// overlaps the DMA of the one before it and the copies of several threads overlap each other.  Page-locked
// memory and small buffers take the plain cudaMemcpyAsync.  $CWIPC_CUDA_STAGING=0 switches the ring off.
//   copy_from_host: returns once `src` has been read completely (the transfer itself may still be in flight on `s`);
//                   returns true when `src` was page-locked (the DMA engine reads it later: the caller decides whether to wait).
//   copy_to_host:   returns once `dst` holds the bytes.
bool copy_from_host(void *dst, const void *src, size_t bytes, cudaStream_t s);
void copy_to_host(void *dst, const void *src, size_t bytes, cudaStream_t s);
// Device workspace owned by the calling thread (one per device), at least `bytes` long, that is ALL
// ZERO when handed out and that the caller must leave all zero again (the kernel that consumes an
// entry clears it), so that steady-state calls need no memset.  Work on it must be queued on `s`,
// the thread's stream.  Call thread_zeroed_invalidate() when a failure may have left it dirty.
void *thread_zeroed(int dev, size_t bytes, cudaStream_t s);
// Head of that workspace, shared by the kernels that need a few zero-initialised words per launch and clear them
// again before they exit (so that no launch needs a memset):
//   words 0,1    voxel table: claimed-slot count, error flag                    (downsample.cu)
//   word  2      bbox_octree_kernel: last-block ticket
//   words 4,5    radix_fused_kernel: grid barrier
//   word  6      stats_threshold_kernel: last-block ticket
//   bytes 256..  compact_kernel: ticket, total, done, pad, then one 64-bit look-back word per 2048-point tile
constexpr size_t ZW_HEADER_BYTES = 65536;
constexpr size_t ZW_COMPACT_OFFSET = 256;
constexpr size_t ZW_COMPACT_TILES = (ZW_HEADER_BYTES - ZW_COMPACT_OFFSET - 16) / 8;
void thread_zeroed_invalidate(int dev);

// Scratch block, released at scope exit.  Scratch comes from a per-thread, per-device arena (one cudaMallocAsync'd
// block, bump allocation) when it is requested on the thread's own stream: kernels of successive calls of one thread
// are ordered on that stream, so the bytes can be reused without any driver call.  The arena rewinds when the last
// live Scratch of the thread is released (i.e. at the end of every filter call); a call that outgrows it chains a
// larger block, and the blocks are merged at the next rewind.  Other streams fall back to cudaMallocAsync.
void *scratch_alloc(size_t bytes, cudaStream_t s, bool *from_arena);
void scratch_free(void *p, cudaStream_t s, bool from_arena) noexcept;

struct Scratch {
    void *p = nullptr;
    cudaStream_t s = nullptr;
    bool arena = false;
    Scratch() = default;
    Scratch(size_t bytes, cudaStream_t stream) : s(stream) { p = bytes ? scratch_alloc(bytes, stream, &arena) : nullptr; }
    Scratch(const Scratch &) = delete;
    Scratch &operator=(const Scratch &) = delete;
    Scratch(Scratch &&o) noexcept : p(o.p), s(o.s), arena(o.arena) { o.p = nullptr; }
    Scratch &operator=(Scratch &&o) noexcept {
        if (this != &o) { release(); p = o.p; s = o.s; arena = o.arena; o.p = nullptr; }
        return *this;
    }
    ~Scratch() { release(); }
    void release() noexcept { if (p) { scratch_free(p, s, arena); p = nullptr; } }
    template <class T> T *as() const { return static_cast<T *>(p); }
};

// Wait until everything queued on `s` so far has completed.  Polls for $CWIPC_CUDA_SPIN_US (default 20) microseconds
// -- the usual wait is a count readback behind one or two short kernels -- then naps $CWIPC_CUDA_SLEEP_US (default 20)
// between polls, so that many caller threads can share few cores (measured: 15 threads on 4 cores lose nothing against
// 10 polling threads on 16).  CWIPC_CUDA_SLEEP_US=0 blocks in the driver instead (interrupt wake-up, slow in VMs).
void stream_sync(cudaStream_t s);

// ---- events ----
cudaEvent_t event_acquire(int dev);      // timing disabled; created on (and only ever reused on) `dev`
void event_release(int dev, cudaEvent_t e) noexcept;
void trim_device(int dev);               // release cached device memory (see cwipc_cuda_trim)

// ---- point storage ----
// `count` valid 16-byte points at d_pts (capacity >= count).  Immutable once `ready` has fired.
struct Storage {
    int dev = 0;
    cwipc_point *d_pts = nullptr;
    size_t capacity = 0;
    size_t count = 0;
    cudaStream_t home = nullptr;
    cudaEvent_t ready = nullptr;
    std::mutex mu;
    struct Reader {
        cudaStream_t stream;
        cudaEvent_t event;
        int dev; // device of `stream` (and of `event`)
    };
    std::vector<Reader> readers; // latest read per foreign stream
    // A box known to contain every point (not necessarily tight), when a producer had one for free.
    bool has_bounds = false;
    float bounds_min[3] = {0, 0, 0}, bounds_max[3] = {0, 0, 0};

    Storage(int dev, size_t capacity, cudaStream_t home);
    ~Storage();
    Storage(const Storage &) = delete;
    Storage &operator=(const Storage &) = delete;

    void mark_ready();                    // record `ready` on home (call after the producing work is queued)

private:
    friend class ReadLease;
    void acquire_for_read(cudaStream_t s); // make `s` wait until contents are valid
    void release_after_read(cudaStream_t s); // note that work queued so far on `s` reads this storage
};
using StoragePtr = std::shared_ptr<Storage>;

// `s` reads `st` for the scope: the constructor makes `s` wait until the contents are valid, the destructor notes that
// the work queued on `s` so far reads them, so that the storage's free on its home stream waits for that work on every
// way out of the scope.  Hold it inside the DeviceGuard of `s`'s device, and hold `st` longer than the lease.  The
// destructor does not throw: a failure to record the reader (a broken CUDA context) is logged as an ERROR.
class ReadLease {
public:
    ReadLease(Storage &st, cudaStream_t s) : m_st(st), m_s(s) { m_st.acquire_for_read(m_s); }
    ~ReadLease();
    ReadLease(const ReadLease &) = delete;
    ReadLease &operator=(const ReadLease &) = delete;

private:
    Storage &m_st;
    cudaStream_t m_s;
};

// ---- launch accounting / profiling ----
extern std::atomic<uint64_t> g_kernel_launches;
struct LaunchScope {
    const char *name;
    cudaStream_t s;
    size_t bytes;
    cudaEvent_t e0 = nullptr;
    LaunchScope(const char *name, cudaStream_t s, size_t algorithmic_bytes);
    ~LaunchScope();
};
void check_launch(const char *name);

// launch("kernel_name", stream, algorithmic_bytes, [&]{ kernel<<<grid, block, smem, stream>>>(args...); });
// algorithmic_bytes: the bytes this launch must move at minimum (DESIGN.md section 4); only used by the profile.
template <class F>
inline void launch(const char *name, cudaStream_t s, size_t algorithmic_bytes, F &&f) {
    LaunchScope scope(name, s, algorithmic_bytes);
    f();
    check_launch(name);
}
// Shared-memory carve-out preference of a kernel (a percentage of the SM's shared memory, cudaSharedmemCarveoutMaxShared
// = 100, or -1 = the driver's choice), applied once per kernel and device.  Kernels of several streams can only share an
// SM when its L1 / shared-memory split suits them all, so the kernels of the frame chain state a common preference;
// `dflt` < -1 leaves the kernel alone.  $CWIPC_CUDA_CARVEOUT overrides `dflt` for every kernel (tuning only).
constexpr int CHAIN_CARVEOUT = -2; // default preference of the frame chain's kernels (-2: none stated)
void tune_kernel(const void *func, int dflt, bool fixed = false); // fixed: $CWIPC_CUDA_CARVEOUT does not apply
template <class K>
inline void tune_kernel(K *kernel, int dflt, bool fixed = false) { tune_kernel(reinterpret_cast<const void *>(kernel), dflt, fixed); }

// bytes that are only known after a readback (e.g. survivors written by a compaction)
void profile_add_bytes(const char *name, size_t bytes);

void profile_enable(bool on);
void profile_reset();
std::string profile_report_json();

inline size_t div_up(size_t a, size_t b) { return (a + b - 1) / b; }

} // namespace cwcu
