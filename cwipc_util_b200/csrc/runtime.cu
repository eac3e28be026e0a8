// runtime.cu -- streams, memory pool, storage lifetime, launch accounting.  See runtime.hpp.
#include "runtime.hpp"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <map>
#include <sstream>

namespace cwcu {

void throw_cuda(cudaError_t e, const char *expr, const char *file, int line) {
    std::ostringstream os;
    os << "CUDA error " << (int)e << " (" << cudaGetErrorName(e) << ": " << cudaGetErrorString(e) << ") at " << file << ":" << line << " in " << expr;
    throw CudaError{e, os.str()};
}

// ------------------------------------------------------------------------------------------
// devices
// ------------------------------------------------------------------------------------------
namespace {

struct DeviceState {
    std::once_flag once;
    int sm_count = 0;
    std::mutex mu;
    std::vector<cudaStream_t> idle_streams; // streams returned by exited threads
    std::vector<std::pair<void *, size_t>> idle_zeroed; // workspaces returned by exited threads (contents unknown)
    std::vector<std::pair<char *, size_t>> idle_arena;  // scratch arena blocks returned by exited threads
    std::vector<cudaEvent_t> idle_events;               // timing-disabled events; an event belongs to the device it was created on
    cudaMemPool_t pool = nullptr;                       // the library's own stream-ordered pool on this device
};

int g_ndev = -1;
std::once_flag g_ndev_once;
DeviceState *g_devs = nullptr;

void init_devices() {
    // The library does not touch process-wide CUDA settings.  A host that drives one GPU from more than 8 threads (one
    // stream each) should export CUDA_DEVICE_MAX_CONNECTIONS=32 before the first CUDA call so that the streams do not
    // share hardware queues (bench.py does; measured +3.5 % frame throughput).
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        n = 0;
    }
    g_devs = new DeviceState[n > 0 ? n : 1];
    g_ndev = n;
}

void init_device(int dev) {
    DeviceState &st = g_devs[dev];
    std::call_once(st.once, [&] {
        DeviceGuard g(dev);
        cudaDeviceProp prop;
        CWCU_CHECK(cudaGetDeviceProperties(&prop, dev));
        st.sm_count = prop.multiProcessorCount;
        // A private pool (the device's default pool, which the host application and other libraries may use, is left
        // alone).  Freed blocks stay cached in it, so steady-state frames never reach cudaMalloc; cwipc_cuda_trim()
        // hands the cache back to the driver.
        cudaMemPoolProps props;
        memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        CWCU_CHECK(cudaMemPoolCreate(&st.pool, &props));
        uint64_t threshold = UINT64_MAX;
        CWCU_CHECK(cudaMemPoolSetAttribute(st.pool, cudaMemPoolAttrReleaseThreshold, &threshold));
    });
}

int default_device() {
    const char *env = getenv("CWIPC_CUDA_DEVICE");
    if (env && *env) return atoi(env);
    return 0;
}

struct ThreadState {
    int device = -1; // -1: not chosen yet
    std::vector<cudaStream_t> streams; // per device
    void *pinned = nullptr;
    size_t pinned_size = 0;
    cudaEvent_t sync_event[64] = {nullptr}; // per device, created with cudaEventBlockingSync
    struct Arena {
        std::vector<std::pair<char *, size_t>> blocks; // the last one is the current one
        size_t offset = 0;  // in the current block
        size_t used = 0;    // bytes handed out since the last rewind (all blocks)
        int live = 0;       // Scratch objects alive
    };
    std::vector<Arena> arenas; // per device
    struct Zeroed {
        void *p = nullptr;
        size_t size = 0;
        bool dirty = false;
    };
    std::vector<Zeroed> zeroed; // per device
    // page-locked staging ring for copies from / to pageable caller memory (copy_from_host / copy_to_host)
    static constexpr int STAGE_SLOTS = 4;
    static constexpr size_t STAGE_CHUNK = (size_t)2 << 20;
    struct Stage {
        char *ring = nullptr;
        cudaEvent_t done[STAGE_SLOTS] = {nullptr, nullptr, nullptr, nullptr}; // the last transfer that used the slot
        int dev[STAGE_SLOTS] = {-1, -1, -1, -1};                              // device that event was created on
        bool pending[STAGE_SLOTS] = {false, false, false, false};
        unsigned next = 0;
    } stage;
    static std::mutex &idle_stage_mu() { static std::mutex *m = new std::mutex; return *m; }           // (never destroyed: threads may
    static std::vector<Stage> &idle_stages() { static auto *v = new std::vector<Stage>; return *v; }  //  exit after main returns)
    ~ThreadState() {
        // the staging ring (8 MB of page-locked memory) goes back to a process-wide list, so that hosts which start a thread per
        // frame do not pin more and more memory; its transfers are waited for first (errors ignored: CUDA may be shutting down)
        if (stage.ring) {
            for (int i = 0; i < STAGE_SLOTS; i++) {
                if (stage.pending[i] && stage.done[i]) (void)cudaEventSynchronize(stage.done[i]);
                stage.pending[i] = false;
            }
            (void)cudaGetLastError();
            std::lock_guard<std::mutex> lk(idle_stage_mu());
            idle_stages().push_back(stage);
            stage.ring = nullptr;
        }
        // give streams back so that thread churn does not leak them
        if (g_devs) {
            for (size_t d = 0; d < streams.size(); d++) {
                if (streams[d]) {
                    std::lock_guard<std::mutex> lk(g_devs[d].mu);
                    g_devs[d].idle_streams.push_back(streams[d]);
                }
            }
        }
        if (g_devs) {
            for (size_t d = 0; d < zeroed.size(); d++) {
                if (zeroed[d].p) {
                    std::lock_guard<std::mutex> lk(g_devs[d].mu);
                    g_devs[d].idle_zeroed.emplace_back(zeroed[d].p, zeroed[d].size);
                }
            }
        }
        if (g_devs) {
            for (size_t d = 0; d < arenas.size(); d++) {
                std::lock_guard<std::mutex> lk(g_devs[d].mu);
                for (auto &b : arenas[d].blocks) g_devs[d].idle_arena.push_back(b);
            }
        }
        // the pinned scratch is deliberately not freed: the CUDA runtime may already be gone
    }
};
thread_local ThreadState t_state;

} // namespace

int device_count() {
    std::call_once(g_ndev_once, init_devices);
    return g_ndev;
}

int current_device() {
    if (t_state.device < 0) t_state.device = default_device();
    return t_state.device;
}

bool set_current_device(int dev) {
    if (dev < 0 || dev >= device_count()) return false;
    t_state.device = dev;
    return true;
}

int sm_count(int dev) {
    init_device(dev);
    return g_devs[dev].sm_count;
}

DeviceGuard::DeviceGuard(int dev) : prev(-1) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) CWCU_CHECK(cudaSetDevice(dev));
}
DeviceGuard::~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) (void)cudaSetDevice(prev);
}

cudaStream_t thread_stream(int dev) {
    if (dev < 0 || dev >= device_count()) throw CudaError{cudaErrorInvalidDevice, "no such CUDA device: " + std::to_string(dev)};
    init_device(dev);
    if ((int)t_state.streams.size() <= dev) t_state.streams.resize(dev + 1, nullptr);
    if (!t_state.streams[dev]) {
        DeviceState &st = g_devs[dev];
        {
            std::lock_guard<std::mutex> lk(st.mu);
            if (!st.idle_streams.empty()) {
                t_state.streams[dev] = st.idle_streams.back();
                st.idle_streams.pop_back();
            }
        }
        if (!t_state.streams[dev]) {
            DeviceGuard g(dev);
            cudaStream_t s;
            CWCU_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
            t_state.streams[dev] = s;
        }
    }
    return t_state.streams[dev];
}

// ------------------------------------------------------------------------------------------
// memory
// ------------------------------------------------------------------------------------------
void *dmalloc(size_t bytes, cudaStream_t s) {
    if (bytes == 0) bytes = 16;
    int dev = 0;
    CWCU_CHECK(cudaGetDevice(&dev));
    init_device(dev);
    void *p = nullptr;
    CWCU_CHECK(cudaMallocFromPoolAsync(&p, bytes, g_devs[dev].pool, s));
    return p;
}

void dfree(void *p, cudaStream_t s) noexcept {
    if (!p) return;
    cudaError_t e = cudaFreeAsync(p, s);
    if (e != cudaSuccess) (void)cudaGetLastError();
}

void *scratch_alloc(size_t bytes, cudaStream_t s, bool *from_arena) {
    int dev = 0;
    CWCU_CHECK(cudaGetDevice(&dev));
    *from_arena = false;
    if ((int)t_state.streams.size() <= dev || t_state.streams[dev] != s) return dmalloc(bytes, s); // not this thread's stream
    if ((int)t_state.arenas.size() <= dev) t_state.arenas.resize(dev + 1);
    auto &a = t_state.arenas[dev];
    const size_t need = (bytes + 255) & ~(size_t)255;
    if (a.blocks.empty()) { // adopt a block an exited thread left behind, if it is large enough
        DeviceState &st = g_devs[dev];
        bool adopted = false;
        {
            std::lock_guard<std::mutex> lk(st.mu);
            for (size_t i = 0; i < st.idle_arena.size(); i++) {
                if (st.idle_arena[i].second >= need) {
                    a.blocks.push_back(st.idle_arena[i]);
                    st.idle_arena.erase(st.idle_arena.begin() + (long)i);
                    adopted = true;
                    break;
                }
            }
        }
        if (adopted) CWCU_CHECK(cudaDeviceSynchronize()); // its previous owner's stream may still be draining (rare: thread start-up)
        a.offset = 0;
    }
    if (a.blocks.empty() || a.offset + need > a.blocks.back().second) {
        size_t cap = a.blocks.empty() ? ((size_t)8 << 20) : a.blocks.back().second * 2;
        while (cap < need) cap *= 2;
        a.blocks.emplace_back(static_cast<char *>(dmalloc(cap, s)), cap);
        a.offset = 0;
    }
    char *p = a.blocks.back().first + a.offset;
    a.offset += need;
    a.used += need;
    a.live++;
    *from_arena = true;
    return p;
}

void scratch_free(void *p, cudaStream_t s, bool from_arena) noexcept {
    if (!from_arena) {
        dfree(p, s);
        return;
    }
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    if ((int)t_state.arenas.size() <= dev) return;
    auto &a = t_state.arenas[dev];
    if (--a.live > 0) return;
    // rewind; if the call needed more than one block, replace them by one that holds everything
    if (a.blocks.size() > 1) {
        size_t cap = a.blocks.back().second;
        while (cap < a.used) cap *= 2;
        for (auto &b : a.blocks) dfree(b.first, s);
        a.blocks.clear();
        void *q = nullptr;
        if (cudaMallocFromPoolAsync(&q, cap, g_devs[dev].pool, s) == cudaSuccess) a.blocks.emplace_back(static_cast<char *>(q), cap);
        else (void)cudaGetLastError();
    }
    a.offset = 0;
    a.used = 0;
    a.live = 0;
}

void *thread_pinned(size_t bytes) {
    if (bytes < 4096) bytes = 4096;
    if (t_state.pinned_size < bytes) {
        if (t_state.pinned) (void)cudaFreeHost(t_state.pinned);
        t_state.pinned = nullptr;
        t_state.pinned_size = 0;
        void *p = nullptr;
        CWCU_CHECK(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
        t_state.pinned = p;
        t_state.pinned_size = bytes;
    }
    return t_state.pinned;
}

void *thread_zeroed(int dev, size_t bytes, cudaStream_t s) {
    if ((int)t_state.zeroed.size() <= dev) t_state.zeroed.resize(dev + 1);
    auto &z = t_state.zeroed[dev];
    if (!z.p) { // adopt a workspace an exited thread left behind
        DeviceState &st = g_devs[dev];
        bool adopted = false;
        {
            std::lock_guard<std::mutex> lk(st.mu);
            if (!st.idle_zeroed.empty()) {
                z.p = st.idle_zeroed.back().first;
                z.size = st.idle_zeroed.back().second;
                z.dirty = true;
                st.idle_zeroed.pop_back();
                adopted = true;
            }
        }
        // its previous owner's stream may still be draining: rare (thread start-up), so simply wait
        if (adopted) CWCU_CHECK(cudaDeviceSynchronize());
    }
    if (z.size < bytes) {
        if (z.p) dfree(z.p, s);
        z.p = nullptr;
        z.size = 0;
        size_t want = 1;
        while (want < bytes) want <<= 1;
        z.p = dmalloc(want, s);
        z.size = want;
        z.dirty = true;
    }
    if (z.dirty) {
        CWCU_CHECK(cudaMemsetAsync(z.p, 0, z.size, s));
        z.dirty = false;
    }
    return z.p;
}

void thread_zeroed_invalidate(int dev) {
    if ((int)t_state.zeroed.size() > dev) t_state.zeroed[dev].dirty = true;
}

void stream_sync(cudaStream_t s) {
    static const long spin_ns = [] {
        const char *e = getenv("CWIPC_CUDA_SPIN_US");
        return (e && *e) ? atol(e) * 1000L : 20000L;
    }();
    static const long sleep_ns = [] { // > 0: after the polling budget, poll every sleep_ns instead of blocking in the driver
        const char *e = getenv("CWIPC_CUDA_SLEEP_US");
        return (e && *e) ? atol(e) * 1000L : 20000L;
    }();
    static const bool spin_given = [] { const char *e = getenv("CWIPC_CUDA_SPIN_US"); return e && *e; }();
    static std::atomic<int> waiters{0};
    struct WaiterScope {
        std::atomic<int> &c;
        int mine;
        explicit WaiterScope(std::atomic<int> &c_) : c(c_), mine(c_.fetch_add(1) + 1) {}
        ~WaiterScope() { c.fetch_sub(1); }
    } scope(waiters);
    // one or two callers: polling costs nothing and saves the ~60 us a nap overshoots by (single-call latency);
    // many callers: short polling budget, then naps
    const long budget_ns = (!spin_given && scope.mine <= 2) ? 500000L : spin_ns;
    int dev = 0;
    CWCU_CHECK(cudaGetDevice(&dev));
    cudaEvent_t &ev = t_state.sync_event[dev & 63];
    if (!ev) CWCU_CHECK(cudaEventCreateWithFlags(&ev, cudaEventBlockingSync | cudaEventDisableTiming));
    CWCU_CHECK(cudaEventRecord(ev, s));
    timespec t0;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    while (true) {
        const cudaError_t q = cudaEventQuery(ev);
        if (q == cudaSuccess) return;
        if (q != cudaErrorNotReady) throw_cuda(q, "cudaEventQuery(sync)", __FILE__, __LINE__);
        timespec t1;
        clock_gettime(CLOCK_MONOTONIC, &t1);
        if ((t1.tv_sec - t0.tv_sec) * 1000000000L + (t1.tv_nsec - t0.tv_nsec) >= budget_ns) break;
    }
    if (sleep_ns > 0) {
        // few cores, many waiting threads: give the core away between polls (a blocking wait in the driver wakes up
        // through an interrupt, which is slow in virtual machines)
        const timespec nap = {0, sleep_ns};
        while (true) {
            nanosleep(&nap, nullptr);
            const cudaError_t q = cudaEventQuery(ev);
            if (q == cudaSuccess) return;
            if (q != cudaErrorNotReady) throw_cuda(q, "cudaEventQuery(sync)", __FILE__, __LINE__);
        }
    }
    CWCU_CHECK(cudaEventSynchronize(ev)); // blocks (cudaEventBlockingSync): the thread sleeps until the GPU interrupt
}

// ------------------------------------------------------------------------------------------
// staged copies from / to pageable host memory
// ------------------------------------------------------------------------------------------
namespace {
bool staging_enabled() {
    static const bool on = [] { const char *e = getenv("CWIPC_CUDA_STAGING"); return !(e && *e == '0'); }();
    return on;
}
constexpr size_t STAGE_MIN_BYTES = (size_t)1 << 20; // below this the driver's own path is as good

void host_wait_event(cudaEvent_t ev) {
    timespec t0;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    while (true) {
        const cudaError_t q = cudaEventQuery(ev);
        if (q == cudaSuccess) return;
        if (q != cudaErrorNotReady) throw_cuda(q, "cudaEventQuery(stage)", __FILE__, __LINE__);
        timespec t1;
        clock_gettime(CLOCK_MONOTONIC, &t1);
        if ((t1.tv_sec - t0.tv_sec) * 1000000000L + (t1.tv_nsec - t0.tv_nsec) >= 30000L) { // a chunk takes 40-200 us: nap between polls
            const timespec nap = {0, 10000L};
            nanosleep(&nap, nullptr);
        }
    }
}

struct StageRing {
    ThreadState::Stage &st;
    int dev;
    explicit StageRing(int dev_) : st(t_state.stage), dev(dev_) {
        if (!st.ring) { // adopt a ring an exited thread left behind, else pin a new one
            {
                std::lock_guard<std::mutex> lk(ThreadState::idle_stage_mu());
                auto &idle = ThreadState::idle_stages();
                if (!idle.empty()) {
                    st = idle.back();
                    idle.pop_back();
                }
            }
            if (!st.ring) {
                void *p = nullptr;
                CWCU_CHECK(cudaHostAlloc(&p, ThreadState::STAGE_SLOTS * ThreadState::STAGE_CHUNK, cudaHostAllocPortable));
                st.ring = static_cast<char *>(p);
            }
        }
    }
    char *slot(int i) const { return st.ring + (size_t)i * ThreadState::STAGE_CHUNK; }
    void wait(int i) { // until the last transfer that used slot i is done
        if (st.pending[i]) {
            host_wait_event(st.done[i]);
            st.pending[i] = false;
        }
    }
    void record(int i, cudaStream_t s) {
        if (st.done[i] && st.dev[i] != dev) { // an event belongs to the device it was created on
            (void)cudaEventDestroy(st.done[i]);
            st.done[i] = nullptr;
        }
        if (!st.done[i]) {
            CWCU_CHECK(cudaEventCreateWithFlags(&st.done[i], cudaEventDisableTiming));
            st.dev[i] = dev;
        }
        CWCU_CHECK(cudaEventRecord(st.done[i], s));
        st.pending[i] = true;
    }
};
} // namespace

// what the CUDA runtime knows about a caller's pointer: page-locked host memory, memory the driver addresses itself
// (device or managed), or ordinary host memory
enum class HostKind { Pageable, Pinned, DriverAddressable };
static HostKind host_kind(const void *p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return HostKind::Pageable;
    }
    if (attr.type == cudaMemoryTypeHost) return HostKind::Pinned;
    if (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) return HostKind::DriverAddressable;
    return HostKind::Pageable;
}

bool copy_from_host(void *dst, const void *src, size_t bytes, cudaStream_t s) {
    if (bytes == 0) return false;
    const HostKind kind = host_kind(src);
    const bool pinned = kind == HostKind::Pinned;
    if (kind != HostKind::Pageable || bytes < STAGE_MIN_BYTES || !staging_enabled()) {
        // (a device or managed pointer is the driver's business: never touched by the host-side memcpy below)
        CWCU_CHECK(cudaMemcpyAsync(dst, src, bytes, kind == HostKind::DriverAddressable ? cudaMemcpyDefault : cudaMemcpyHostToDevice, s));
        return pinned;
    }
    int dev = 0;
    CWCU_CHECK(cudaGetDevice(&dev));
    StageRing ring(dev);
    for (size_t off = 0; off < bytes; off += ThreadState::STAGE_CHUNK) {
        const size_t len = std::min(ThreadState::STAGE_CHUNK, bytes - off);
        const int i = (int)ring.st.next;
        ring.st.next = (ring.st.next + 1) % ThreadState::STAGE_SLOTS;
        ring.wait(i);
        memcpy(ring.slot(i), static_cast<const char *>(src) + off, len);
        CWCU_CHECK(cudaMemcpyAsync(static_cast<char *>(dst) + off, ring.slot(i), len, cudaMemcpyHostToDevice, s));
        ring.record(i, s);
    }
    return false;
}

void copy_to_host(void *dst, const void *src, size_t bytes, cudaStream_t s) {
    if (bytes == 0) return;
    const HostKind kind = (bytes < STAGE_MIN_BYTES || !staging_enabled()) ? HostKind::Pinned : host_kind(dst);
    if (kind != HostKind::Pageable) {
        CWCU_CHECK(cudaMemcpyAsync(dst, src, bytes, kind == HostKind::DriverAddressable ? cudaMemcpyDefault : cudaMemcpyDeviceToHost, s));
        stream_sync(s);
        return;
    }
    int dev = 0;
    CWCU_CHECK(cudaGetDevice(&dev));
    StageRing ring(dev);
    constexpr int SLOTS = ThreadState::STAGE_SLOTS;
    const size_t chunk = ThreadState::STAGE_CHUNK, nchunks = (bytes + chunk - 1) / chunk;
    // chunk c travels through slot (base + c) % SLOTS; up to SLOTS transfers are in flight while the oldest is copied out
    const unsigned base = ring.st.next;
    auto issue = [&](size_t c) {
        const int i = (int)((base + c) % SLOTS);
        ring.wait(i);
        const size_t off = c * chunk, len = std::min(chunk, bytes - off);
        CWCU_CHECK(cudaMemcpyAsync(ring.slot(i), static_cast<const char *>(src) + off, len, cudaMemcpyDeviceToHost, s));
        ring.record(i, s);
    };
    for (size_t c = 0; c < std::min<size_t>(nchunks, SLOTS); c++) issue(c);
    for (size_t c = 0; c < nchunks; c++) {
        const int i = (int)((base + c) % SLOTS);
        ring.wait(i);
        const size_t off = c * chunk, len = std::min(chunk, bytes - off);
        memcpy(static_cast<char *>(dst) + off, ring.slot(i), len);
        if (c + SLOTS < nchunks) issue(c + SLOTS);
    }
    ring.st.next = (unsigned)((base + nchunks) % SLOTS);
}

void tune_kernel(const void *func, int dflt, bool fixed) {
    static const int forced = [] {
        const char *e = getenv("CWIPC_CUDA_CARVEOUT");
        return (e && *e) ? atoi(e) : -2;
    }();
    const int want = (!fixed && forced >= -1) ? forced : dflt;
    if (want < -1) return;
    int dev = 0;
    CWCU_CHECK(cudaGetDevice(&dev));
    // applied once per (kernel, device); the per-thread list keeps the steady-state launch path free of locks
    thread_local std::vector<std::pair<const void *, int>> seen;
    for (const auto &e : seen)
        if (e.first == func && e.second == dev) return;
    seen.emplace_back(func, dev);
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, int> done;
    {
        std::lock_guard<std::mutex> lk(mu);
        auto it = done.find({func, dev});
        if (it != done.end() && it->second == want) return;
        done[{func, dev}] = want;
    }
    CWCU_CHECK(cudaFuncSetAttribute(func, cudaFuncAttributePreferredSharedMemoryCarveout, want));
}

bool is_pinned_host(const void *p) {
    if (!p) return false;
    cudaPointerAttributes attr;
    cudaError_t e = cudaPointerGetAttributes(&attr, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

// ------------------------------------------------------------------------------------------
// events
// ------------------------------------------------------------------------------------------
// One pool per device: cudaEventRecord wants the event and the stream on the same device, so an event freed by a cloud on
// device 0 must never be handed to a cloud on device 1 (one process, one thread per GPU: DESIGN.md section 7).
cudaEvent_t event_acquire(int dev) {
    init_device(dev);
    DeviceState &st = g_devs[dev];
    {
        std::lock_guard<std::mutex> lk(st.mu);
        if (!st.idle_events.empty()) {
            cudaEvent_t e = st.idle_events.back();
            st.idle_events.pop_back();
            return e;
        }
    }
    DeviceGuard g(dev);
    cudaEvent_t e;
    CWCU_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return e;
}

void event_release(int dev, cudaEvent_t e) noexcept {
    if (!e || !g_devs || dev < 0 || dev >= g_ndev) return;
    std::lock_guard<std::mutex> lk(g_devs[dev].mu);
    g_devs[dev].idle_events.push_back(e);
}

// Hand cached memory back to the driver: idle arenas / workspaces of exited threads, the calling thread's own arena and
// zeroed workspace on `dev`, and everything the pool holds beyond what is in use.
void trim_device(int dev) {
    if (dev < 0 || dev >= device_count()) return;
    init_device(dev);
    DeviceGuard g(dev);
    DeviceState &st = g_devs[dev];
    CWCU_CHECK(cudaDeviceSynchronize());
    std::vector<void *> drop;
    {
        std::lock_guard<std::mutex> lk(st.mu);
        for (auto &b : st.idle_arena) drop.push_back(b.first);
        for (auto &z : st.idle_zeroed) drop.push_back(z.first);
        st.idle_arena.clear();
        st.idle_zeroed.clear();
    }
    if ((int)t_state.arenas.size() > dev && t_state.arenas[dev].live == 0) {
        for (auto &b : t_state.arenas[dev].blocks) drop.push_back(b.first);
        t_state.arenas[dev].blocks.clear();
        t_state.arenas[dev].offset = t_state.arenas[dev].used = 0;
    }
    if ((int)t_state.zeroed.size() > dev && t_state.zeroed[dev].p) {
        drop.push_back(t_state.zeroed[dev].p);
        t_state.zeroed[dev] = ThreadState::Zeroed();
    }
    for (void *p : drop) CWCU_CHECK(cudaFree(p));
    CWCU_CHECK(cudaMemPoolTrimTo(st.pool, 0));
}

// ------------------------------------------------------------------------------------------
// storage
// ------------------------------------------------------------------------------------------
Storage::Storage(int dev_, size_t capacity_, cudaStream_t home_) : dev(dev_), capacity(capacity_), home(home_) {
    DeviceGuard g(dev);
    d_pts = capacity ? static_cast<cwipc_point *>(dmalloc(capacity * sizeof(cwipc_point), home)) : nullptr;
    ready = event_acquire(dev);
}

Storage::~Storage() {
    // Runs on whichever thread drops the last reference.  Order the free after every reader.
    try {
        DeviceGuard g(dev);
        for (auto &r : readers) {
            (void)cudaStreamWaitEvent(home, r.event, 0);
            event_release(r.dev, r.event);
        }
        dfree(d_pts, home);
        event_release(dev, ready);
    } catch (...) {
    }
}

void Storage::mark_ready() { CWCU_CHECK(cudaEventRecord(ready, home)); }

void Storage::acquire_for_read(cudaStream_t s) {
    if (s != home) CWCU_CHECK(cudaStreamWaitEvent(s, ready, 0));
}

void Storage::release_after_read(cudaStream_t s) {
    if (s == home) return;
    std::lock_guard<std::mutex> lk(mu);
    for (auto &r : readers) {
        if (r.stream == s) {
            CWCU_CHECK(cudaEventRecord(r.event, s));
            return;
        }
    }
    // `s` is a stream of the CUDA-current device (the caller holds a DeviceGuard for it), which need not be this->dev
    int sdev = 0;
    CWCU_CHECK(cudaGetDevice(&sdev));
    cudaEvent_t e = event_acquire(sdev);
    CWCU_CHECK(cudaEventRecord(e, s));
    readers.push_back(Reader{s, e, sdev});
}

ReadLease::~ReadLease() {
    try {
        m_st.release_after_read(m_s);
    } catch (const CudaError &e) {
        log(CWIPC_LOG_LEVEL_ERROR, "cwipc_util", "cannot record a reader of a pointcloud: " + e.what);
    } catch (const std::exception &e) {
        log(CWIPC_LOG_LEVEL_ERROR, "cwipc_util", std::string("cannot record a reader of a pointcloud: ") + e.what());
    }
}

// ------------------------------------------------------------------------------------------
// launch accounting / profiling
// ------------------------------------------------------------------------------------------
std::atomic<uint64_t> g_kernel_launches{0};

namespace {
std::atomic<bool> g_profile_on{false};
std::mutex g_profile_mu;
struct ProfRec {
    const char *name;
    cudaEvent_t e0, e1;
    size_t bytes;
};
struct ProfAcc {
    uint64_t launches = 0;
    double ms = 0.0;
    double bytes = 0.0;
};
std::vector<ProfRec> g_profile_recs;
std::map<std::string, ProfAcc> g_profile_acc;

void profile_drain_locked() {
    for (auto &r : g_profile_recs) {
        float ms = 0.f;
        if (cudaEventSynchronize(r.e1) == cudaSuccess && cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) {
            auto &acc = g_profile_acc[r.name];
            acc.launches += 1;
            acc.ms += ms;
            acc.bytes += (double)r.bytes;
        } else {
            (void)cudaGetLastError();
        }
        (void)cudaEventDestroy(r.e0);
        (void)cudaEventDestroy(r.e1);
    }
    g_profile_recs.clear();
}
} // namespace

LaunchScope::LaunchScope(const char *name_, cudaStream_t s_, size_t bytes_) : name(name_), s(s_), bytes(bytes_) {
    g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
    if (g_profile_on.load(std::memory_order_relaxed)) {
        if (cudaEventCreate(&e0) == cudaSuccess) (void)cudaEventRecord(e0, s);
        else e0 = nullptr;
    }
}

LaunchScope::~LaunchScope() {
    if (!e0) return;
    cudaEvent_t e1 = nullptr;
    if (cudaEventCreate(&e1) != cudaSuccess) {
        (void)cudaEventDestroy(e0);
        return;
    }
    (void)cudaEventRecord(e1, s);
    std::lock_guard<std::mutex> lk(g_profile_mu);
    g_profile_recs.push_back({name, e0, e1, bytes});
    if (g_profile_recs.size() > 8192) profile_drain_locked();
}

void check_launch(const char *name) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        std::ostringstream os;
        os << "kernel launch failed: " << name << ": " << cudaGetErrorName(e) << ": " << cudaGetErrorString(e);
        throw CudaError{e, os.str()};
    }
}

void profile_enable(bool on) { g_profile_on.store(on); }

void profile_add_bytes(const char *name, size_t bytes) {
    if (!g_profile_on.load(std::memory_order_relaxed)) return;
    std::lock_guard<std::mutex> lk(g_profile_mu);
    g_profile_acc[name].bytes += (double)bytes;
}

void profile_reset() {
    std::lock_guard<std::mutex> lk(g_profile_mu);
    profile_drain_locked();
    g_profile_acc.clear();
}

std::string profile_report_json() {
    std::lock_guard<std::mutex> lk(g_profile_mu);
    profile_drain_locked();
    std::ostringstream os;
    os << "{";
    bool first = true;
    for (auto &kv : g_profile_acc) {
        if (!first) os << ", ";
        first = false;
        os << "\"" << kv.first << "\": {\"launches\": " << kv.second.launches << ", \"total_ms\": " << kv.second.ms << ", \"bytes\": " << (uint64_t)kv.second.bytes << "}";
    }
    os << "}";
    return os.str();
}

} // namespace cwcu
