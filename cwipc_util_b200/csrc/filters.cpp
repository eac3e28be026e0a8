// filters.cpp -- the C-ABI filter entry points: argument rules, cellsize/timestamp propagation,
// per-tile grouping and error behaviour of the reference, with the arithmetic done by the CUDA
// kernels in pointops.cu / downsample.cu / outliers.cu.
// ref: src/cwipc_filters.cpp:30-418
#include <algorithm>
#include <cmath>
#include <cstring>

#include "kernels.hpp"
#include "pointcloud.hpp"
#include "radix_sort.hpp"

using namespace cwcu;

namespace {

// A one-input filter whose result keeps the input's timestamp and cellsize: `body(in, dev, stream)` -> StoragePtr.
// NULL input: NULL, silently (ref: src/cwipc_filters.cpp:282-284).
template <class Body>
cwipc_pointcloud *unary_filter(const char *who, cwipc_pointcloud *pc, Body &&body) {
    return read_entry<cwipc_pointcloud *>(who, pc, nullptr, [&](const StoragePtr &in, int dev, cudaStream_t s) {
        return new_result(body(in, dev, s), pc->timestamp(), pc->cellsize());
    });
}

// cwipc_downsample's voxel size: voxelsize >= 0 selects the octree-split path, < 0 one global grid; the size is |voxelsize|,
// and the cloud's own cellsize wins when it is larger.  ref: src/cwipc_filters.cpp:42-46, :103-107
struct VoxelSize {
    bool octree_split;
    float cellsize;
};
VoxelSize voxel_size(cwipc_pointcloud *pc, float voxelsize) {
    const bool octree_split = !(voxelsize < 0);
    const float cellsize = octree_split ? voxelsize : -voxelsize, own = pc->cellsize();
    return {octree_split, own >= cellsize ? own : cellsize};
}

const float *bounds_of(const Storage &in, float box[6]) {
    if (!in.has_bounds) return nullptr;
    memcpy(box, in.bounds_min, 3 * sizeof(float));
    memcpy(box + 3, in.bounds_max, 3 * sizeof(float));
    return box;
}

// cwipc_cuda_transform's arguments checked, and the matrix slot of every tile value: slot[v] = i for tiles[i] == v, else the
// tile-0 entry's slot when there is one.  A bad argument throws (-> NULL and one ERROR log).
void transform_slots(const double *matrices, const uint8_t *tiles, int n, uint16_t slot[256]) {
    auto bad = [](const std::string &what) { throw CudaError{cudaErrorInvalidValue, what}; };
    if (n < 1) bad("n must be at least 1");
    if (matrices == nullptr || tiles == nullptr) bad("matrices and tiles must not be NULL");
    std::fill(slot, slot + 256, TRANSFORM_NONE);
    for (int i = 0; i < n; i++) { // a repeat is met by i == 256 at the latest
        if (slot[tiles[i]] != TRANSFORM_NONE) bad("tile value " + std::to_string(tiles[i]) + " is listed twice");
        slot[tiles[i]] = (uint16_t)i;
    }
    for (int i = 0; i < n; i++) {
        const double *m = matrices + 16 * i;
        for (int k = 0; k < 16; k++)
            if (!std::isfinite(m[k])) bad("matrix " + std::to_string(i) + " has a non-finite entry");
        if (!(m[12] == 0.0 && m[13] == 0.0 && m[14] == 0.0 && m[15] == 1.0)) bad("the last row of matrix " + std::to_string(i) + " is not (0, 0, 0, 1)");
    }
    if (slot[0] != TRANSFORM_NONE)
        for (int v = 1; v < 256; v++)
            if (slot[v] == TRANSFORM_NONE) slot[v] = slot[0];
}

} // namespace

extern "C" {

// keep iff tile == 0 || point.tile == tile; stable; empty in -> empty out.  ref: src/cwipc_filters.cpp:281-306
cwipc_pointcloud *cwipc_tilefilter(cwipc_pointcloud *pc, int tile) {
    return unary_filter("cwipc_tilefilter", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        if (tile == 0) return in; // keeps every point: storage is immutable, so share it
        if (tile < 0 || tile > 255) return new_storage(dev, 0, s, [](Storage &) -> size_t { return 0; }); // `tile == pt.a` with an 8-bit pt.a can never hold
        return new_storage(dev, in->count, s, [&](Storage &out) { return compact_points(in->d_pts, in->count, out.d_pts, tile_equals(tile), dev, s); }, in.get());
    });
}

// (tile & mask) != 0, the variant python/cwipc/registration/util.py:98-112 builds in numpy
cwipc_pointcloud *cwipc_cuda_tilefilter_masked(cwipc_pointcloud *pc, int mask) {
    return unary_filter("cwipc_tilefilter_masked", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        return new_storage(dev, in->count, s, [&](Storage &out) { return compact_points(in->d_pts, in->count, out.d_pts, tile_mask(mask & 0xff), dev, s); }, in.get());
    });
}

// ref: src/cwipc_filters.cpp:333-360
cwipc_pointcloud *cwipc_crop(cwipc_pointcloud *pc, float bbox[6]) {
    return unary_filter("cwipc_crop", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        return new_storage(dev, in->count, s, [&](Storage &out) { return compact_points(in->d_pts, in->count, out.d_pts, crop_box(bbox), dev, s); }, in.get());
    });
}

// ref: src/cwipc_filters.cpp:308-331
cwipc_pointcloud *cwipc_tilemap(cwipc_pointcloud *pc, uint8_t map[256]) {
    return unary_filter("cwipc_tilemap", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        return new_storage(dev, in->count, s, [&](Storage &out) {
            tilemap_points(in->d_pts, in->count, out.d_pts, map, s);
            return in->count;
        });
    });
}

// ref: src/cwipc_filters.cpp:362-386
cwipc_pointcloud *cwipc_colormap(cwipc_pointcloud *pc, uint32_t clearBits, uint32_t setBits) {
    return unary_filter("cwipc_colormap", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        return new_storage(dev, in->count, s, [&](Storage &out) {
            colormap_points(in->d_pts, in->count, out.d_pts, clearBits, setBits, s);
            return in->count;
        });
    });
}

// Every point moved by the 4x4 matrix of its tile value (see include/cwipc_util_cuda.h).  One kernel, no host wait.  The
// result has no known box: the input's does not bound the moved points, and a stale box would mislead the kNN grid of
// cwipc_remove_outliers.
cwipc_pointcloud *cwipc_cuda_transform(cwipc_pointcloud *pc, const double *matrices, const uint8_t *tiles, int n) {
    return unary_filter("cwipc_cuda_transform", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        uint16_t slot[256];
        transform_slots(matrices, tiles, n, slot);
        return new_storage(dev, in->count, s, [&](Storage &out) {
            transform_points(in->d_pts, in->count, out.d_pts, matrices, slot, n, dev, s);
            return in->count;
        });
    });
}

// concatenation; timestamp and cellsize are the minima.  ref: src/cwipc_filters.cpp:388-418
cwipc_pointcloud *cwipc_join(cwipc_pointcloud *pc1, cwipc_pointcloud *pc2) {
    if (pc2 == nullptr) return nullptr;
    return read_entry<cwipc_pointcloud *>("cwipc_join", pc1, nullptr, [&](const StoragePtr &a, int dev, cudaStream_t s) -> cwipc_pointcloud * {
        StoragePtr b = storage_of(pc2, "cwipc_join");
        if (!b) return nullptr;
        ReadLease lease_b(*b, s);
        StoragePtr out = new_storage(dev, a->count + b->count, s, [&](Storage &o) {
            if (a->count) CWCU_CHECK(cudaMemcpyAsync(o.d_pts, a->d_pts, a->count * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
            if (b->count) {
                // a cloud on another device: an explicit peer copy (memory of a private pool is not reachable through UVA alone)
                if (b->dev != dev) CWCU_CHECK(cudaMemcpyPeerAsync(o.d_pts + a->count, dev, b->d_pts, b->dev, b->count * sizeof(cwipc_point), s));
                else CWCU_CHECK(cudaMemcpyAsync(o.d_pts + a->count, b->d_pts, b->count * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
            }
            return a->count + b->count;
        });
        return new_result(out, std::min(pc1->timestamp(), pc2->timestamp()), std::min(pc1->cellsize(), pc2->cellsize()));
    });
}

// Voxel-grid downsample.  voxelsize > 0: the reference's octree-split path (a grid per 64-voxel
// octree leaf, so voxels cut by a leaf face come out once per leaf); voxelsize < 0: one global grid.
// The cloud's own cellsize wins when it is larger.  ref: src/cwipc_filters.cpp:30-172
cwipc_pointcloud *cwipc_downsample(cwipc_pointcloud *pc, float voxelsize) {
    return read_entry<cwipc_pointcloud *>("cwipc_downsample", pc, nullptr, [&](const StoragePtr &in, int dev, cudaStream_t s) -> cwipc_pointcloud * {
        const auto [octree_split, cellsize] = voxel_size(pc, voxelsize);
        return new_result(downsample_points(in, cellsize, octree_split, dev, s), pc->timestamp(), cellsize);
    });
}

// cwipc_downsample of every tile group on its own, the results one after another:
// join(downsample(tilefilter(pc, t1)), downsample(tilefilter(pc, t2)), ...) over the distinct tile values in first-appearance
// order, tile 0 meaning "every point" as cwipc_tilefilter(pc, 0) does.  Every group is downsampled exactly as cwipc_downsample
// downsamples the cloud tilefilter(pc, t) (its points in input order; the centroid scale from the group's own count).
// ref: python/cwipc/registration/util.py:170-182, src/cwipc_filters.cpp:239-256
cwipc_pointcloud *cwipc_cuda_downsample_pertile(cwipc_pointcloud *pc, float voxelsize) {
    return read_entry<cwipc_pointcloud *>("cwipc_cuda_downsample_pertile", pc, nullptr, [&](const StoragePtr &in, int dev, cudaStream_t s) -> cwipc_pointcloud * {
        const VoxelSize vs = voxel_size(pc, voxelsize);
        const size_t n = in->count;
        StoragePtr out;
        std::vector<size_t> counts;
        const std::vector<int> tiles = tiles_in_first_appearance_order(in->d_pts, n, s, &counts);
        // a group's failure names its tile
        auto in_group = [](int tile, auto &&body) {
            try {
                return body();
            } catch (const CudaError &e) {
                throw CudaError{e.code, "tile " + std::to_string(tile) + ": " + e.what};
            }
        };
        if (tiles.size() <= 1) { // the whole cloud is the only group (or there is none: an empty cloud, no tile to name)
            auto whole = [&] { return downsample_points(in, vs.cellsize, vs.octree_split, dev, s); };
            out = tiles.empty() ? whole() : in_group(tiles[0], whole);
        } else {
            // the non-zero groups side by side in one buffer; the tile-0 group is the input itself
            std::vector<int> split;
            size_t nsplit = 0;
            for (size_t i = 0; i < tiles.size(); i++) {
                if (tiles[i] == 0) continue;
                split.push_back(tiles[i]);
                nsplit += counts[i];
            }
            Scratch grouped(nsplit * sizeof(cwipc_point), s);
            split_by_tile(in->d_pts, n, split, nsplit, grouped.as<cwipc_point>(), dev, s);
            // a group keeps at most all of its points: room for the sum of the group sizes
            const bool has_zero = split.size() < tiles.size();
            out = new_storage(dev, has_zero ? n + nsplit : n, s, [&](Storage &o) {
                size_t total = 0, offset = 0;
                bool first = true;
                for (size_t i = 0; i < tiles.size(); i++) {
                    const cwipc_point *src = in->d_pts;
                    size_t cnt = n;
                    if (tiles[i] != 0) {
                        src = grouped.as<cwipc_point>() + offset;
                        cnt = counts[i];
                        offset += cnt;
                    }
                    const DownsampleRange r = in_group(tiles[i], [&] { return downsample_range(src, cnt, vs.cellsize, vs.octree_split, o.d_pts + total, dev, s); });
                    total += r.count;
                    // a box that holds every group's centroids
                    for (int a = 0; a < 3; a++) {
                        o.bounds_min[a] = first ? r.bounds_min[a] : std::min(o.bounds_min[a], r.bounds_min[a]);
                        o.bounds_max[a] = first ? r.bounds_max[a] : std::max(o.bounds_max[a], r.bounds_max[a]);
                    }
                    first = false;
                }
                o.has_bounds = true;
                return total;
            });
        }
        return new_result(out, pc->timestamp(), vs.cellsize);
    });
}

// Statistical outlier removal, whole cloud or once per distinct tile value (first-appearance order,
// tile 0 meaning "every point" exactly as cwipc_tilefilter(pc, 0) does).  ref: src/cwipc_filters.cpp:181-278
cwipc_pointcloud *cwipc_remove_outliers(cwipc_pointcloud *pc, int kNeighbors, float stddevMulThresh, bool perTile) {
    return unary_filter("cwipc_remove_outliers", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        const float spacing = pc->cellsize();
        const size_t n = in->count;
        float box[6];
        const float *bounds = bounds_of(*in, box);
        if (!perTile)
            return new_storage(dev, n, s, [&](Storage &out) { return remove_outliers_points(in->d_pts, n, out.d_pts, kNeighbors, stddevMulThresh, spacing, bounds, dev, s); }, in.get());
        std::vector<int> tiles = tiles_in_first_appearance_order(in->d_pts, n, s);
        const bool has_zero = std::find(tiles.begin(), tiles.end(), 0) != tiles.end();
        static const bool sequential = getenv("CWIPC_CUDA_SOR_PER_TILE") && !strcmp(getenv("CWIPC_CUDA_SOR_PER_TILE"), "sequential"); // tests only
        return new_storage(dev, has_zero ? 2 * n : n, s, [&](Storage &out) -> size_t {
            if (!has_zero && kNeighbors >= 1 && n > (size_t)kNeighbors && !sequential) {
                // every group at once: one search index with the tile rank as a band of cells (outliers.cu)
                return remove_outliers_per_tile(in->d_pts, n, out.d_pts, tiles, kNeighbors, stddevMulThresh, spacing, bounds, dev, s);
            }
            // tile 0 among the values (the whole cloud is a group of its own, src/cwipc_filters.cpp:281-306) or fewer points
            // than neighbours: group after group
            size_t total = 0;
            for_each_tile_group(in->d_pts, n, tiles, dev, s, [&](const cwipc_point *src, size_t cnt) {
                total += remove_outliers_points(src, cnt, out.d_pts + total, kNeighbors, stddevMulThresh, spacing, bounds, dev, s);
            });
            return total;
        }, in.get());
    });
}

// ---- diagnostic hooks used by the parity tests ---------------------------------------------------
int cwipc_cuda_knn_mean_distances(cwipc_pointcloud *pc, int kNeighbors, float *dist, size_t ndist) {
    if (dist == nullptr) return -1;
    return read_entry<int>("cwipc_cuda_knn_mean_distances", pc, -1, [&](const StoragePtr &in, int dev, cudaStream_t s) -> int {
        if (ndist < in->count) return -1;
        if (in->count == 0) return 0;
        Scratch d(in->count * sizeof(float), s);
        float box[6];
        knn_mean_distances(in->d_pts, in->count, kNeighbors, pc->cellsize(), bounds_of(*in, box), d.as<float>(), dev, s);
        CWCU_CHECK(cudaMemcpyAsync(dist, d.p, in->count * sizeof(float), cudaMemcpyDeviceToHost, s));
        stream_sync(s);
        return (int)in->count;
    });
}

// ---- partitioned clouds: building blocks for a cloud spread over several GPUs as x-slabs ---------------
// The library runs the whole protocol itself in slab.cpp (cwipc_cuda_slab_*).  These are its steps one call at a time, for
// callers that move the data between the parts by their own means (cwipc_util_b200/slab.py) and for the tests.

int cwipc_cuda_octree_replay(cwipc_pointcloud *pc, float cellsize, struct cwipc_cuda_octree_state *state, float bounds[6]) {
    if (state == nullptr || bounds == nullptr) return -1;
    return read_entry<int>("cwipc_cuda_octree_replay", pc, -1, [&](const StoragePtr &in, int dev, cudaStream_t s) -> int {
        if (!(cellsize > 0.f)) return -1;
        octree_replay(in->d_pts, in->count, cellsize, *state, bounds, dev, s);
        return 0;
    });
}

cwipc_pointcloud *cwipc_cuda_downsample_planned(cwipc_pointcloud *pc, float voxelsize, const struct cwipc_cuda_octree_state *state, const float bounds[6]) {
    if (state == nullptr || bounds == nullptr) return nullptr;
    return read_entry<cwipc_pointcloud *>("cwipc_cuda_downsample_planned", pc, nullptr, [&](const StoragePtr &in, int dev, cudaStream_t s) -> cwipc_pointcloud * {
        const auto [octree_split, cellsize] = voxel_size(pc, voxelsize);
        return new_result(downsample_points_planned(in, cellsize, octree_split, *state, bounds, dev, s), pc->timestamp(), cellsize);
    });
}

cwipc_pointcloud *cwipc_cuda_from_device_points(const void *dev_points, int npoint, uint64_t timestamp) {
    if (npoint < 0 || (npoint > 0 && dev_points == nullptr)) return nullptr;
    return device_entry<cwipc_pointcloud *>("cwipc_cuda_from_device_points", nullptr, current_device(), [&](int dev, cudaStream_t s) -> cwipc_pointcloud * {
        StoragePtr out = new_storage(dev, (size_t)npoint, s, [&](Storage &o) {
            if (npoint) CWCU_CHECK(cudaMemcpyAsync(o.d_pts, dev_points, (size_t)npoint * sizeof(cwipc_point), cudaMemcpyDefault, s));
            return (size_t)npoint;
        });
        stream_sync(s); // the caller may reuse its buffer on return
        return new DevicePointcloud(out, timestamp, 0.f);
    });
}

int cwipc_cuda_knn_query(cwipc_pointcloud *pc, int kNeighbors, int nquery, float *mean, float *kth2) {
    if (mean == nullptr || nquery < 0) return -1;
    return read_entry<int>("cwipc_cuda_knn_query", pc, -1, [&](const StoragePtr &in, int dev, cudaStream_t s) -> int {
        if ((size_t)nquery > in->count) return -1;
        if (nquery == 0) return 0;
        Scratch d(in->count * sizeof(float), s), kth(in->count * sizeof(float), s);
        float box[6];
        knn_mean_distances(in->d_pts, in->count, kNeighbors, pc->cellsize(), bounds_of(*in, box), d.as<float>(), dev, s, kth.as<float>(), (size_t)nquery);
        CWCU_CHECK(cudaMemcpyAsync(mean, d.p, (size_t)nquery * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (kth2) CWCU_CHECK(cudaMemcpyAsync(kth2, kth.p, (size_t)nquery * sizeof(float), cudaMemcpyDeviceToHost, s));
        stream_sync(s);
        return nquery;
    });
}

// ---- device-resident per-point distances of a slab (so that only the few open queries ever reach the host) ----
// The buffers are plain device blocks, not the per-call arena: they outlive the call that made them.
struct cwipc_cuda_distances {
    int dev = 0;
    size_t n = 0;     // queries
    Scratch mean;     // float[n]
    Scratch open_idx; // uint32[nopen]
    Scratch kth;      // float[n]: (k+1)-th smallest squared distance found so far (+inf where fewer points were seen)
    size_t nopen = 0;
};

namespace {
Scratch persistent_scratch(size_t bytes, cudaStream_t s) {
    Scratch sc;
    sc.p = dmalloc(bytes, s);
    sc.s = s;
    return sc;
}
} // namespace

cwipc_cuda_distances *cwipc_cuda_knn_query_open(cwipc_pointcloud *pc, int kNeighbors, int nquery, float x_lo, float x_hi, int *nopen) {
    if (nquery < 0 || nopen == nullptr) return nullptr;
    return read_entry<cwipc_cuda_distances *>("cwipc_cuda_knn_query_open", pc, nullptr, [&](const StoragePtr &in, int dev, cudaStream_t s) -> cwipc_cuda_distances * {
        if ((size_t)nquery > in->count) return nullptr;
        auto h = std::make_unique<cwipc_cuda_distances>();
        h->dev = dev;
        h->n = (size_t)nquery;
        *nopen = 0;
        if (nquery == 0) return h.release();
        h->mean = persistent_scratch((size_t)nquery * sizeof(float), s);
        h->open_idx = persistent_scratch((size_t)nquery * sizeof(uint32_t), s);
        h->kth = persistent_scratch((size_t)nquery * sizeof(float), s);
        float box[6];
        h->nopen = knn_open_queries(in->d_pts, in->count, (size_t)nquery, kNeighbors, pc->cellsize(), bounds_of(*in, box), x_lo, x_hi, h->mean.as<float>(), h->kth.as<float>(),
                                    h->open_idx.as<uint32_t>(), dev, s);
        *nopen = (int)h->nopen;
        return h.release();
    });
}

// indices (into the first nquery points), coordinates and current (k+1)-th squared distances of the open queries, to host
int cwipc_cuda_distances_open(cwipc_cuda_distances *h, cwipc_pointcloud *pc, uint32_t *idx, struct cwipc_point *points, float *kth2) {
    if (h == nullptr || pc == nullptr) return -1;
    if (h->nopen == 0) return 0;
    return read_entry<int>("cwipc_cuda_distances_open", pc, -1, [&](const StoragePtr &in, int, cudaStream_t s) -> int {
        Scratch q(h->nopen * sizeof(cwipc_point), s);
        gather_points(in->d_pts, h->open_idx.as<uint32_t>(), h->nopen, q.as<cwipc_point>(), s);
        if (idx) CWCU_CHECK(cudaMemcpyAsync(idx, h->open_idx.p, h->nopen * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        if (points) CWCU_CHECK(cudaMemcpyAsync(points, q.p, h->nopen * sizeof(cwipc_point), cudaMemcpyDeviceToHost, s));
        Scratch kq(h->nopen * sizeof(float), s);
        if (kth2) {
            gather_floats(h->kth.as<float>(), h->open_idx.as<uint32_t>(), h->nopen, kq.as<float>(), s);
            CWCU_CHECK(cudaMemcpyAsync(kth2, kq.p, h->nopen * sizeof(float), cudaMemcpyDeviceToHost, s));
        }
        stream_sync(s);
        return (int)h->nopen;
    });
}

// mean[idx[i]] = values[i] for the open queries (values in the order cwipc_cuda_distances_open returned them)
int cwipc_cuda_distances_patch(cwipc_cuda_distances *h, const float *values, int n) {
    if (h == nullptr || n < 0 || (size_t)n != h->nopen || (n > 0 && values == nullptr)) return -1;
    if (n == 0) return 0;
    return device_entry<int>("cwipc_cuda_distances_patch", -1, h->dev, [&](int, cudaStream_t s) -> int {
        Scratch v((size_t)n * sizeof(float), s);
        CWCU_CHECK(cudaMemcpyAsync(v.p, values, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, s));
        scatter_floats(v.as<float>(), h->open_idx.as<uint32_t>(), (size_t)n, h->mean.as<float>(), s);
        stream_sync(s);
        return n;
    });
}

int cwipc_cuda_distances_stats(cwipc_cuda_distances *h, double sums[2]) {
    if (h == nullptr || sums == nullptr) return -1;
    return device_entry<int>("cwipc_cuda_distances_stats", -1, h->dev, [&](int, cudaStream_t s) -> int {
        distance_stats(h->mean.as<float>(), h->n, sums, s);
        return 0;
    });
}

cwipc_pointcloud *cwipc_cuda_distances_filter(cwipc_pointcloud *pc, cwipc_cuda_distances *h, double threshold) {
    if (h == nullptr) return nullptr;
    return unary_filter("cwipc_cuda_distances_filter", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        if (h->n != in->count) throw CudaError{cudaErrorInvalidValue, "one distance per point is required"};
        return new_storage(dev, in->count, s, [&](Storage &out) { return compact_points(in->d_pts, in->count, out.d_pts, distance_at_most(h->mean.as<float>(), threshold), dev, s); },
                           in.get());
    });
}

void cwipc_cuda_distances_free(cwipc_cuda_distances *h) {
    if (h == nullptr) return;
    try {
        DeviceGuard g(h->dev);
        delete h;
    } catch (...) {
    }
}

int cwipc_cuda_knn_lists(cwipc_pointcloud *pc, const struct cwipc_point *queries, const float *limits, int nq, int kNeighbors, float *lists) {
    if (nq < 0 || (nq > 0 && (queries == nullptr || lists == nullptr))) return -1;
    return read_entry<int>("cwipc_cuda_knn_lists", pc, -1, [&](const StoragePtr &in, int dev, cudaStream_t s) -> int {
        if (nq == 0) return 0;
        const size_t kk = (size_t)kNeighbors + 1;
        Scratch q((size_t)nq * sizeof(cwipc_point), s), l((size_t)nq * kk * sizeof(float), s), lim(limits ? (size_t)nq * sizeof(float) : 0, s);
        CWCU_CHECK(cudaMemcpyAsync(q.p, queries, (size_t)nq * sizeof(cwipc_point), cudaMemcpyHostToDevice, s));
        if (limits) CWCU_CHECK(cudaMemcpyAsync(lim.p, limits, (size_t)nq * sizeof(float), cudaMemcpyHostToDevice, s));
        float box[6];
        knn_lists(in->d_pts, in->count, q.as<cwipc_point>(), limits ? lim.as<float>() : nullptr, (size_t)nq, kNeighbors, pc->cellsize(), bounds_of(*in, box), l.as<float>(), dev, s);
        CWCU_CHECK(cudaMemcpyAsync(lists, l.p, (size_t)nq * kk * sizeof(float), cudaMemcpyDeviceToHost, s));
        stream_sync(s);
        return nq;
    });
}

int cwipc_cuda_knn_merge_lists(const float *lists, int nlists, int nq, int kNeighbors, float *mean, float *kth2) {
    if (nq < 0 || nlists < 1 || (nq > 0 && (lists == nullptr || mean == nullptr))) return -1;
    if (nq == 0) return 0;
    return device_entry<int>("cwipc_cuda_knn_merge_lists", -1, current_device(), [&](int, cudaStream_t s) -> int {
        const size_t kk = (size_t)kNeighbors + 1, total = (size_t)nlists * nq * kk;
        Scratch l(total * sizeof(float), s), m((size_t)nq * sizeof(float), s), kt((size_t)nq * sizeof(float), s);
        CWCU_CHECK(cudaMemcpyAsync(l.p, lists, total * sizeof(float), cudaMemcpyHostToDevice, s));
        knn_merge_lists(l.as<float>(), (size_t)nlists, (size_t)nq, kNeighbors, m.as<float>(), kt.as<float>(), s);
        CWCU_CHECK(cudaMemcpyAsync(mean, m.p, (size_t)nq * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (kth2) CWCU_CHECK(cudaMemcpyAsync(kth2, kt.p, (size_t)nq * sizeof(float), cudaMemcpyDeviceToHost, s));
        stream_sync(s);
        return nq;
    });
}

int cwipc_cuda_distance_stats(const float *dist, size_t ndist, double sums[2]) {
    if (sums == nullptr || (ndist > 0 && dist == nullptr)) return -1;
    return device_entry<int>("cwipc_cuda_distance_stats", -1, current_device(), [&](int, cudaStream_t s) -> int {
        Scratch d(ndist * sizeof(float), s);
        if (ndist) CWCU_CHECK(cudaMemcpyAsync(d.p, dist, ndist * sizeof(float), cudaMemcpyHostToDevice, s));
        distance_stats(d.as<float>(), ndist, sums, s);
        return 0;
    });
}

double cwipc_cuda_outlier_threshold(double sum, double sq, double n, float stddevMulThresh) { return outlier_threshold(sum, sq, n, stddevMulThresh); }

cwipc_pointcloud *cwipc_cuda_filter_by_distance(cwipc_pointcloud *pc, const float *dist, size_t ndist, double threshold) {
    return unary_filter("cwipc_cuda_filter_by_distance", pc, [&](const StoragePtr &in, int dev, cudaStream_t s) -> StoragePtr {
        if (ndist != in->count || (ndist > 0 && dist == nullptr)) throw CudaError{cudaErrorInvalidValue, "one distance per point is required"};
        Scratch d(ndist * sizeof(float), s);
        if (ndist) CWCU_CHECK(cudaMemcpyAsync(d.p, dist, ndist * sizeof(float), cudaMemcpyHostToDevice, s));
        return new_storage(dev, in->count, s, [&](Storage &out) { return compact_points(in->d_pts, in->count, out.d_pts, distance_at_most(d.as<float>(), threshold), dev, s); },
                           in.get());
    });
}

// Diagnostic: the library's stable LSD radix sort on bits [begin_bit, end_bit) of host words, in place.
int cwipc_cuda_sort_u64(uint64_t *words, size_t n, int begin_bit, int end_bit) {
    if (n > 0 && words == nullptr) return -1;
    if (n == 0) return 0;
    return device_entry<int>("cwipc_cuda_sort_u64", -1, current_device(), [&](int dev, cudaStream_t s) -> int {
        Scratch a(n * sizeof(uint64_t), s), b(n * sizeof(uint64_t), s);
        CWCU_CHECK(cudaMemcpyAsync(a.p, words, n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        const uint64_t *sorted = radix_sort_u64(a.as<uint64_t>(), b.as<uint64_t>(), n, begin_bit, end_bit, dev, s);
        CWCU_CHECK(cudaMemcpyAsync(words, sorted, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        stream_sync(s);
        return 0;
    });
}

int cwipc_cuda_downsample_keys(cwipc_pointcloud *pc, float voxelsize, uint64_t *keys, size_t nkeys) {
    if (keys == nullptr) return -1;
    return read_entry<int>("cwipc_cuda_downsample_keys", pc, -1, [&](const StoragePtr &in, int dev, cudaStream_t s) -> int {
        if (nkeys < in->count) return -1;
        if (in->count == 0) return 0;
        const auto [octree_split, cellsize] = voxel_size(pc, voxelsize);
        downsample_keys_to_host(in, cellsize, octree_split, keys, dev, s);
        return (int)in->count;
    });
}

} // extern "C"
