// pointcloud.cpp -- device-resident cwipc_pointcloud, leak counters, metadata collection.
// ref: src/cwipc_util.cpp:24-430
#include "pointcloud.hpp"

#include <cstdlib>
#include <cstring>

#include "kernels.hpp"

namespace cwcu {

// ---- metadata ------------------------------------------------------------------------------
MetadataCollection::~MetadataCollection() {
    for (auto &it : m_items)
        if (it.dealloc) it.dealloc(it.pointer);
}
int MetadataCollection::count() { return (int)m_items.size(); }
const std::string &MetadataCollection::name(int idx) { return m_items[idx].name; }
const std::string &MetadataCollection::description(int idx) { return m_items[idx].description; }
void *MetadataCollection::pointer(int idx) { return m_items[idx].pointer; }
size_t MetadataCollection::size(int idx) { return m_items[idx].size; }
void MetadataCollection::_add(const std::string &name, const std::string &description, void *pointer, size_t size, deallocfunc dealloc) {
    m_items.push_back(Item{name, description, pointer, size, dealloc});
}
void MetadataCollection::_move(cwipc_metadata *other) {
    // ownership of every item passes to `other`; like the reference this assumes `other` is ours
    auto *dst = static_cast<MetadataCollection *>(other);
    for (auto &it : m_items) dst->m_items.push_back(it);
    m_items.clear();
}

// ---- leak accounting (ref: src/cwipc_util.cpp:89-93, 420-430) --------------------------------
namespace {
std::mutex g_count_mu;
int g_alloc = 0, g_dealloc = 0;
} // namespace

void count_alloc() {
    std::lock_guard<std::mutex> lk(g_count_mu);
    g_alloc++;
}
void count_dealloc() {
    std::lock_guard<std::mutex> lk(g_count_mu);
    g_dealloc++;
}

// ---- the cloud -----------------------------------------------------------------------------
DevicePointcloud::DevicePointcloud(StoragePtr store, uint64_t timestamp, float cellsize) : m_store(std::move(store)), m_timestamp(timestamp), m_cellsize(cellsize) {
    if (m_store) count_alloc();
}

DevicePointcloud *DevicePointcloud::from_host(const cwipc_point *points, size_t npoint, uint64_t timestamp, bool sync) {
    const int dev = current_device();
    if (device_count() <= 0) throw CudaError{cudaErrorNoDevice, "libcwipc_util_cuda needs a CUDA device and found none (there is no CPU fallback)"};
    cudaStream_t s = thread_stream(dev);
    DeviceGuard g(dev);
    // Pageable source memory has been read completely when copy_from_host returns (it travels through the calling
    // thread's page-locked ring); page-locked memory is read by the DMA engine later, so wait unless the caller opted out.
    bool pinned = false;
    StoragePtr store = new_storage(dev, npoint, s, [&](Storage &out) {
        if (npoint) pinned = copy_from_host(out.d_pts, points, npoint * sizeof(cwipc_point), s);
        return npoint;
    });
    if (sync && npoint && pinned) stream_sync(s);
    return new DevicePointcloud(store, timestamp, 0.f);
}

void DevicePointcloud::free() {
    if (m_store) {
        m_store.reset();
        count_dealloc();
    }
    delete m_metadata;
    m_metadata = nullptr;
    // As in the reference (src/cwipc_util.cpp:149-163, 731-733) the C++ shell itself stays alive:
    // callers may still hold the pointer and free() twice must be harmless.
}

cwipc_pointcloud *DevicePointcloud::_shallowcopy() {
    auto *rv = new DevicePointcloud(m_store, m_timestamp, m_cellsize);
    rv->m_exact_size = m_exact_size;
    return rv;
}

void DevicePointcloud::_set_cellsize(float cellsize) {
    if (cellsize < 0 && m_store) {
        // ref: src/cwipc_util.cpp:173-204 -- prevPoint never advances, so the heuristic is the
        // minimum distance from any later point to the FIRST point.
        StoragePtr st = m_store;
        cellsize = guarded<float>("cwipc_util", 0.f, [&] {
            DeviceGuard g(st->dev);
            cudaStream_t s = thread_stream(st->dev);
            ReadLease lease(*st, s);
            return min_distance_to_first(st->d_pts, st->count, s);
        });
    }
    m_cellsize = cellsize;
}

int DevicePointcloud::count() {
    if (!m_store) {
        log(CWIPC_LOG_LEVEL_WARNING, "cwipc_util", "count: NULL pointcloud");
        return 0;
    }
    return (int)m_store->count;
}

size_t DevicePointcloud::get_uncompressed_size() {
    if (!m_store) {
        log(CWIPC_LOG_LEVEL_WARNING, "cwipc_util", "get_uncompressed_size: NULL pointcloud");
        return 0;
    }
    return m_store->count * sizeof(cwipc_point);
}

int DevicePointcloud::copy_uncompressed(struct cwipc_point *pointbuf, size_t size) {
    if (!m_store) {
        log(CWIPC_LOG_LEVEL_WARNING, "cwipc_util", "copy_uncompressed: NULL pointcloud");
        return 0;
    }
    const size_t need = m_store->count * sizeof(cwipc_point);
    if (m_exact_size ? size != need : size < need) {
        log(CWIPC_LOG_LEVEL_ERROR, "cwipc_util", "copy_uncompressed: buffer too small");
        return -1;
    }
    if (need == 0) return 0;
    StoragePtr st = m_store;
    return guarded<int>("cwipc_util", -1, [&] {
        DeviceGuard g(st->dev);
        cudaStream_t s = thread_stream(st->dev);
        ReadLease lease(*st, s);
        copy_to_host(pointbuf, st->d_pts, need, s); // returns when pointbuf is complete
        return (int)st->count;
    });
}

size_t DevicePointcloud::copy_packet(uint8_t *packet, size_t size) {
    if (!m_store) {
        log(CWIPC_LOG_LEVEL_WARNING, "cwipc_util", "copy_packet: NULL pointcloud");
        return 0;
    }
    const size_t dataSize = get_uncompressed_size();
    const size_t need = sizeof(cwipc_cwipcdump_header) + dataSize;
    if (packet == nullptr) return need;
    if (size != need) return 0;
    cwipc_cwipcdump_header hdr;
    memset(&hdr, 0, sizeof(hdr));
    memcpy(hdr.hdr, CWIPC_CWIPCDUMP_HEADER, 4);
    hdr.magic = CWIPC_CWIPCDUMP_VERSION;
    hdr.timestamp = m_timestamp;
    hdr.cellsize = m_cellsize;
    hdr.unused = 0;
    hdr.size = dataSize;
    memcpy(packet, &hdr, sizeof(hdr));
    if (copy_uncompressed(reinterpret_cast<cwipc_point *>(packet + sizeof(hdr)), dataSize) < 0) return 0;
    return need;
}

cwipc_metadata *DevicePointcloud::access_metadata() {
    if (!m_metadata) m_metadata = new MetadataCollection();
    return m_metadata;
}

StoragePtr storage_of(cwipc_pointcloud *pc, const char *who) {
    if (auto *mine = dynamic_cast<DevicePointcloud *>(pc)) {
        if (!mine->storage()) log(CWIPC_LOG_LEVEL_WARNING, who, "pointcloud has been freed");
        return mine->storage();
    }
    // foreign implementation: pull its points through the public interface and upload them
    const size_t bytes = pc->get_uncompressed_size();
    const size_t n = bytes / sizeof(cwipc_point);
    std::vector<cwipc_point> host(n);
    if (n && pc->copy_uncompressed(host.data(), bytes) < 0) {
        log(CWIPC_LOG_LEVEL_WARNING, who, "cannot obtain points of foreign pointcloud");
        return nullptr;
    }
    return guarded<StoragePtr>(who, nullptr, [&] {
        const int dev = current_device();
        cudaStream_t s = thread_stream(dev);
        DeviceGuard g(dev);
        StoragePtr store = new_storage(dev, n, s, [&](Storage &out) {
            if (n) (void)copy_from_host(out.d_pts, host.data(), bytes, s);
            return n;
        });
        stream_sync(s);
        return store;
    });
}

} // namespace cwcu

extern "C" int cwipc_dangling_allocations(bool log) {
    int alloc, dealloc;
    {
        std::lock_guard<std::mutex> lk(cwcu::g_count_mu);
        alloc = cwcu::g_alloc;
        dealloc = cwcu::g_dealloc;
    }
    const int dangling = alloc - dealloc;
    if (log && dangling != 0) {
        cwcu::log(CWIPC_LOG_LEVEL_WARNING, "cwipc_pointcloud",
                  std::to_string(dangling) + " free() mismatch. nAlloc=" + std::to_string(alloc) + ", nFree=" + std::to_string(dealloc));
    }
    return dangling < 0 ? -dangling : dangling;
}
