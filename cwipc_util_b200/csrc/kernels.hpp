// kernels.hpp -- host-callable launchers of the filter kernels.  All work is queued on the given
// stream; functions that return a count synchronise that stream once to read it back.
#pragma once

#include "runtime.hpp"

namespace cwcu {

// ---- pointops.cu: stable compaction and per-point maps -------------------------------------
enum class PredKind : int { TileEquals = 0, TileMask = 1, CropBox = 2, DistanceAtMost = 3 };

struct Predicate {
    PredKind kind = PredKind::TileEquals;
    int tile = 0;                 // TileEquals (0 keeps everything) / TileMask
    float box[6] = {0, 0, 0, 0, 0, 0}; // CropBox: minx,maxx,miny,maxy,minz,maxz
    const float *dist = nullptr;  // DistanceAtMost: keep iff !(dist[i] > threshold)
    double threshold = 0.0;
    const double *threshold_dev = nullptr; // when not null the threshold is read from device memory instead
};

// Stable compaction of in[0..n) by `pred` into out (capacity >= n).  Returns the number kept.
size_t compact_points(const cwipc_point *in, size_t n, cwipc_point *out, const Predicate &pred, int dev, cudaStream_t s);

// One link of a chain of compactions into the same `out`: keeps the points of `tile` with !(dist[i] > *threshold_dev),
// writing from position *d_base (device word; 0 when null) and leaving base + kept in *d_total.  No read-back; n > 0.
void compact_tile_group_chained(const cwipc_point *in, size_t n, cwipc_point *out, int tile, const float *dist, const double *threshold_dev, const uint32_t *d_base,
                                uint32_t *d_total, cudaStream_t s);

void tilemap_points(const cwipc_point *in, size_t n, cwipc_point *out, const uint8_t map[256], cudaStream_t s);
// cwipc_cuda_transform: out[i] = in[i] with x, y, z moved by matrices[slot[tile]] (nmat row-major 4x4 doubles, affine),
// or copied when slot[tile] == TRANSFORM_NONE.  1 <= nmat <= 256.  One kernel, no host wait.
constexpr uint16_t TRANSFORM_NONE = 0xffff; // 16-bit slots: 256 matrices and "none"
void transform_points(const cwipc_point *in, size_t n, cwipc_point *out, const double *matrices, const uint16_t slot[256], int nmat, int dev, cudaStream_t s);
void colormap_points(const cwipc_point *in, size_t n, cwipc_point *out, uint32_t clearBits, uint32_t setBits, cudaStream_t s);
// min over i>=1 of |p_i - p_0| (float), 0 when n < 2.  ref: src/cwipc_util.cpp:173-204
float min_distance_to_first(const cwipc_point *in, size_t n, cudaStream_t s);
// distinct tile values in first-appearance order. ref: src/cwipc_filters.cpp:239-249
// counts (nullable) receives the number of points of each, in the same order (same pass, same read-back).
std::vector<int> tiles_in_first_appearance_order(const cwipc_point *in, size_t n, cudaStream_t s, std::vector<size_t> *counts = nullptr);
// Stable split by tile value: the points of tiles[0], then those of tiles[1], ..., each group in input order, into out.
// `tiles` are distinct and non-zero; points of other values are left out.  nkept = the number of points written.
void split_by_tile(const cwipc_point *in, size_t n, const std::vector<int> &tiles, size_t nkept, cwipc_point *out, int dev, cudaStream_t s);

// The reference's synthetic cloud (src/cwipc_synthetic.cpp:182-222) generated in HBM: side x side points, row hi at height
// hi * dh, column ai at angle ai * da.  d_radius[hi] (float), d_sin[ai] / d_cos[ai] (double) are the host's own libm values
// (3 * side numbers), so the geometry is bit-identical to the host generator; colours use the device's double sin.
void synthetic_points(cwipc_point *out, int side, float dh, float da, const float *d_radius, const double *d_sin, const double *d_cos, float angle, bool eyes_lit, cudaStream_t s);

// ---- downsample.cu -------------------------------------------------------------------------
struct DownsampleResult {
    StoragePtr out;    // nullptr on failure
    bool failed = false;
    std::string error; // reference-compatible error text when failed
};
// cellsize > 0 already resolved against the cloud's own cellsize.  octree_split selects the
// reference's positive-size path (per-octree-leaf grids) vs the single global grid.
DownsampleResult downsample_points(const StoragePtr &in, float cellsize, bool octree_split, int dev, cudaStream_t s);
// The same downsample of pts[0..n), written to dst (room for n points) instead of a new cloud: the voxels come out exactly as
// downsample_points gives them for a cloud of these n points.  Returns their number and the input's bounding box.
struct DownsampleRange {
    bool failed = false;
    std::string error;
    size_t count = 0;
    bool has_bounds = false; // false when n == 0
    float bounds_min[3] = {0, 0, 0}, bounds_max[3] = {0, 0, 0};
};
DownsampleRange downsample_range(const cwipc_point *pts, size_t n, float cellsize, bool octree_split, cwipc_point *dst, int dev, cudaStream_t s);
// Octree bounding box of pcl::octree::OctreePointCloud after inserting points in order (a cloud partitioned
// over several GPUs is replayed part by part, the state travelling from rank to rank).  A state that starts a replay is
// all zero.
void octree_replay(const cwipc_point *in, size_t n, float cellsize, cwipc_cuda_octree_state &state, float bounds[6], int dev, cudaStream_t s);
DownsampleResult downsample_points_planned(const StoragePtr &in, float cellsize, bool octree_split, const cwipc_cuda_octree_state &state, const float bounds[6], int dev,
                                           cudaStream_t s);
// global bounding box of in[0..n), n > 0 (synchronises the stream)
void global_bbox(const cwipc_point *in, size_t n, float gmin[3], float gmax[3], int dev, cudaStream_t s);
// diagnostic: sort keys (without the index bits) per input point, to host
void downsample_keys_to_host(const StoragePtr &in, float cellsize, bool octree_split, uint64_t *host_keys, int dev, cudaStream_t s);

// ---- outliers.cu ---------------------------------------------------------------------------
// Statistical outlier removal on in[0..n) (one group).  Appends survivors to out (capacity >= n),
// returns the number kept.  `hint_spacing` is the cloud's cellsize (0 if unknown).
// `bounds` (min xyz, max xyz), when not null, is a box known to contain every point; it saves the bounding-box pass.
size_t remove_outliers_points(const cwipc_point *in, size_t n, cwipc_point *out, int k, float stddev_mul, float hint_spacing, const float *bounds, int dev, cudaStream_t s);
// cwipc_remove_outliers(perTile=true) in one pass (ref: src/cwipc_filters.cpp:238-261): `tiles` = the distinct, NON-ZERO tile
// values in first-appearance order; one search index over the whole cloud with the tile rank as a band of cells, one kNN
// launch, per-group statistics and thresholds on the device, the groups' survivors chained into `out` in `tiles` order.
// Needs n > k.  group_kept (nullable) receives the survivors per group.
size_t remove_outliers_per_tile(const cwipc_point *in, size_t n, cwipc_point *out, const std::vector<int> &tiles, int k, float stddev_mul, float hint_spacing, const float *bounds,
                                int dev, cudaStream_t s);
// First pass only: mean distance to the k nearest neighbours per point, original order, device array.
// Only the first `nquery` points are queries (the rest are candidates only); d_kth, when not null, receives the
// (k+1)-th smallest squared distance of every query.
void knn_mean_distances(const cwipc_point *in, size_t n, int k, float hint_spacing, const float *bounds, float *d_dist, int dev, cudaStream_t s, float *d_kth = nullptr,
                        size_t nquery = (size_t)-1);
// The k+1 smallest squared distances (ascending, +inf padded) from each of nq device-resident query points to the cloud.
// d_limits (nullable): per query, only distances <= limit are reported (a bound on its (k+1)-th distance found elsewhere)
void knn_lists(const cwipc_point *in, size_t n, const cwipc_point *d_queries, const float *d_limits, size_t nq, int k, float hint_spacing, const float *bounds, float *d_lists, int dev,
               cudaStream_t s);
void gather_floats(const float *values, const uint32_t *idx, size_t n, float *out, cudaStream_t s);
// lists laid out [nlists][nq][k+1]; mean distance to the k nearest (and k-th squared distance) of the merged lists
void knn_merge_lists(const float *d_lists, size_t nlists, size_t nq, int k, float *d_mean, float *d_kth, cudaStream_t s);
// sum d, sum (float)(d*d), both in double (synchronises the stream)
void distance_stats(const float *d_dist, size_t n, double out[2], cudaStream_t s);
double outlier_threshold(double sum, double sq, double n, float stddev_mul);
// Slab protocol: indices i < nquery whose (k+1)-th neighbour sphere (kth2[i], squared) is not strictly inside the covered
// interval (x_lo, x_hi); kth2 == nullptr marks every query.  Returns their number (synchronises the stream).
size_t mark_open_queries(const cwipc_point *pts, const float *kth2, size_t nquery, float x_lo, float x_hi, uint32_t *open_idx, int dev, cudaStream_t s);
void gather_points(const cwipc_point *pts, const uint32_t *idx, size_t n, cwipc_point *out, cudaStream_t s);
// the same with the indices in the low 32 bits of 64-bit words
void gather_points(const cwipc_point *pts, const uint64_t *words, size_t n, cwipc_point *out, cudaStream_t s);
void scatter_floats(const float *values, const uint32_t *idx, size_t n, float *out, cudaStream_t s);

// ---- runtime.cu ----------------------------------------------------------------------------
void flush_l2(int dev, cudaStream_t s);

} // namespace cwcu
