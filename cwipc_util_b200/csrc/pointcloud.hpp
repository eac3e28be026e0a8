// pointcloud.hpp -- the device-resident cwipc_pointcloud.
// ref: src/cwipc_util.cpp:24-87 (metadata), :94-410 (cwipc_impl / cwipc_uncompressed_impl)
#pragma once

#include "runtime.hpp"

namespace cwcu {

class MetadataCollection : public cwipc_metadata {
    struct Item {
        std::string name, description;
        void *pointer;
        size_t size;
        deallocfunc dealloc;
    };
    std::vector<Item> m_items;

public:
    ~MetadataCollection() override;
    int count() override;
    const std::string &name(int idx) override;
    const std::string &description(int idx) override;
    void *pointer(int idx) override;
    size_t size(int idx) override;
    void _add(const std::string &name, const std::string &description, void *pointer, size_t size, deallocfunc dealloc) override;
    void _move(cwipc_metadata *other) override;
};

// Points live in HBM as 16-byte cwipc_point records and reach the host only through
// copy_uncompressed / copy_packet (the lazy-copy model of the reference's readme.md:9-11).
class DevicePointcloud : public cwipc_pointcloud {
    StoragePtr m_store; // nullptr after free()
    uint64_t m_timestamp = 0;
    float m_cellsize = 0.f;
    MetadataCollection *m_metadata = nullptr;
    // Clouds made from a caller's point array (cwipc_from_points / cwipc_from_packet / read_debugdump) are the
    // reference's cwipc_uncompressed_impl, whose copy_uncompressed wants the EXACT size (src/cwipc_util.cpp:393-397);
    // filter results are its cwipc_impl, which accepts any buffer that is large enough (:226-231).
    bool m_exact_size = false;

public:
    DevicePointcloud(StoragePtr store, uint64_t timestamp, float cellsize);
    ~DevicePointcloud() override {}

    // host -> device.  sync=true returns after the copy has completed (caller may reuse the buffer).
    static DevicePointcloud *from_host(const cwipc_point *points, size_t npoint, uint64_t timestamp, bool sync);

    const StoragePtr &storage() const { return m_store; }
    void set_exact_size(bool on) { m_exact_size = on; }

    void free() override;
    cwipc_pointcloud *_shallowcopy() override;
    uint64_t timestamp() override { return m_timestamp; }
    float cellsize() override { return m_cellsize; }
    void _set_cellsize(float cellsize) override;
    void _set_timestamp(uint64_t timestamp) override { m_timestamp = timestamp; }
    int count() override;
    size_t get_uncompressed_size() override;
    int copy_uncompressed(struct cwipc_point *pointbuf, size_t size) override;
    size_t copy_packet(uint8_t *packet, size_t size) override;
    cwipc_pcl_pointcloud access_pcl_pointcloud() override { return nullptr; }
    cwipc_metadata *access_metadata() override;
};

// The filters accept any cwipc_pointcloud.  A cloud made by this library is used in place; a
// foreign implementation (another DLL's subclass) is imported through copy_uncompressed.
// Returns nullptr (after logging) if the points cannot be obtained.
StoragePtr storage_of(cwipc_pointcloud *pc, const char *who);

void count_alloc();
void count_dealloc();

// Run `body` translating any CudaError / std::exception into an ERROR log + `fallback`.
template <class R, class F>
R guarded(const char *module, R fallback, F &&body) {
    try {
        return body();
    } catch (const CudaError &e) {
        log(CWIPC_LOG_LEVEL_ERROR, module, e.what);
    } catch (const std::exception &e) {
        log(CWIPC_LOG_LEVEL_ERROR, module, std::string("std exception: ") + e.what());
    }
    return fallback;
}

// The shape of every entry point that reads a cloud: NULL -> `fallback` (silent, as the reference's filters); the cloud's
// storage (`fallback` when it cannot be had); its device, the calling thread's stream there and a ReadLease on the
// storage for the whole of `body(in, dev, stream)`; any exception -> an ERROR log naming `who` and `fallback`.
template <class R, class Body>
R read_entry(const char *who, cwipc_pointcloud *pc, R fallback, Body &&body) {
    if (pc == nullptr) return fallback;
    return guarded<R>(who, fallback, [&]() -> R {
        StoragePtr in = storage_of(pc, who);
        if (!in) return fallback;
        DeviceGuard g(in->dev);
        cudaStream_t s = thread_stream(in->dev);
        ReadLease lease(*in, s);
        return body(in, in->dev, s);
    });
}

// The shape of an entry point that reads no cloud: `body(dev, stream)` runs with `dev` current and the calling thread's
// stream there; any exception -> an ERROR log naming `who` and `fallback`.
template <class R, class Body>
R device_entry(const char *who, R fallback, int dev, Body &&body) {
    return guarded<R>(who, fallback, [&]() -> R {
        DeviceGuard g(dev);
        return body(dev, thread_stream(dev));
    });
}

// A new storage of `capacity` points on `dev` whose home is `s`: `fill(out)` queues the work that writes out.d_pts and
// returns the number of points.  `subset_of`, when not null, is a cloud that holds every result point: its box, if it has
// one, is the result's too, so that the kNN grid of a following filter need not measure one.  The storage is marked ready
// last, so that readers on other streams wait for the fill.
template <class Fill>
StoragePtr new_storage(int dev, size_t capacity, cudaStream_t s, Fill &&fill, const Storage *subset_of = nullptr) {
    auto out = std::make_shared<Storage>(dev, capacity, s);
    out->count = fill(*out);
    if (subset_of && subset_of->has_bounds) {
        out->has_bounds = true;
        std::copy(subset_of->bounds_min, subset_of->bounds_min + 3, out->bounds_min);
        std::copy(subset_of->bounds_max, subset_of->bounds_max + 3, out->bounds_max);
    }
    out->mark_ready();
    return out;
}

// A filter result: a new cloud holding `out`, with the given timestamp and cellsize (cellsize < 0: estimated from the
// points, as cwipc_pointcloud::_set_cellsize does).
inline cwipc_pointcloud *new_result(StoragePtr out, uint64_t timestamp, float cellsize) {
    auto *rv = new DevicePointcloud(std::move(out), timestamp, 0.f);
    rv->_set_cellsize(cellsize);
    return rv;
}

} // namespace cwcu
