// downsample.cu -- voxel-grid downsample as hand-written sm_100a kernels.
//
// Reference semantics (src/cwipc_filters.cpp:30-172 over pcl::VoxelGrid, pcl::CentroidPoint and
// pcl::octree::OctreePointCloud, restated in SURVEY.md App. A.3/A.4 and in oracle/cwipc_oracle.c):
//   * voxel of a point:  (int)floorf(x * inv) per axis with inv = 1.0f / cellsize (float arithmetic);
//   * positive voxelsize: the cloud is first split by an octree of resolution 64*cellsize whose origin
//     is anchored on the FIRST point (leaf faces at p0 + m*res, double arithmetic); every leaf gets its
//     own voxel grid, so a voxel cut by a leaf face is emitted once per leaf.  Output order = leaves in
//     depth-first (Morton, x most significant) order, voxels inside a leaf by (z, y, x);
//   * negative voxelsize: one grid over the whole cloud, output ordered by (z, y, x);
//   * per voxel: xyz = mean, rgb = (uint)(float sum / n) (truncation), tile = OR of the tiles.  Here the colour is the exact
//     floor(sum / n): the reference's result wherever its float sum is exact (every channel sum below 2^24).
//
// Pipeline (one stream; N points in, V voxels out):
//   voxel_stream_kernel   16 B/pt read   ONE pass over the points.  Warps stream 256-point tiles into shared memory
//                                        (cp.async, double buffered, 128-byte-row swizzle); every lane walks 8
//                                        CONSECUTIVE points and merges runs of equal (leaf, voxel) in registers, the
//                                        lanes' partial runs are joined by a segmented shuffle scan, and only whole
//                                        runs reach the voxel hash table in L2 (one probe + 5 RED per run, 7 for clouds
//                                        over 16.8 M points).  In
//                                        octree mode the same pass computes the 256-point chunk boxes, the block that
//                                        finishes last replays PCL's sequential octree-box growth from them, and keys
//                                        are taken relative to the first point (the leaf PARTITION depends on p0 and
//                                        the resolution only), so nothing has to be known before the pass.
//   voxel_words_kernel    12 B/voxel     list of claimed voxels -> sort words [final key | claim index]
//   radix_sort_u64        16 B/voxel/pass
//   voxel_emit_kernel     64 B/voxel     slot -> centroid / colour / tile, 16 B/voxel written; clears the slot
// One host round trip (voxel count + octree box + flags).  Algorithmic bytes: 16*N in + 16*V out.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>

#include "device_utils.cuh"
#include "kernels.hpp"
#include "pointcloud.hpp"
#include "radix_sort.hpp"

namespace cwcu {

namespace {

constexpr int WL_RADIX = 72;     // voxel-in-leaf coordinate range per axis (64 + misalignment + guard)
constexpr int WL_BITS = 19;      // 72^3 = 373248 < 2^19
constexpr int MAX_OCTREE_DEPTH = 14;
constexpr int REL_BIAS = 16384;  // leaf index relative to the first point's box, biased into 15 bits

struct OctreeBox {
    double min[3];
    double max[3];
    float gmin[3];
    float gmax[3];
    int depth;
    int error; // 1: runaway growth (non-finite input)
    // fused pass only: leaf index of the final octree = leaf index relative to the first point's box + shift
    int shift[3];
    int fallback; // 1: the relative keys cannot be trusted (rounding at a leaf face): redo with the two-pass path
    double m0[3]; // min corner of the first point's box: what the relative leaf indices count from
};

// ---- per-chunk bounding boxes --------------------------------------------------------------------------
constexpr int BB_THREADS = 1024;
constexpr int BB_ITEMS = 4;
constexpr int BB_CHUNK = BB_THREADS * BB_ITEMS; // points per bounding-box chunk of the stand-alone bbox kernel
__device__ __forceinline__ void chunk_bbox_block(const cwipc_point *__restrict__ pts, uint32_t n, float *chunk_bbox) {
    __shared__ float s_cb[6][BB_THREADS / 32];
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int j = 0; j < BB_ITEMS; j++) {
        const uint32_t i = blockIdx.x * BB_CHUNK + j * BB_THREADS + threadIdx.x;
        if (i < n) {
            const Point16 p = ld_point_stream(pts, i);
            lo[0] = fminf(lo[0], p.x); hi[0] = fmaxf(hi[0], p.x);
            lo[1] = fminf(lo[1], p.y); hi[1] = fmaxf(hi[1], p.y);
            lo[2] = fminf(lo[2], p.z); hi[2] = fmaxf(hi[2], p.z);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; a++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(FULL_MASK, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(FULL_MASK, hi[a], o));
        }
    }
    const unsigned warp = threadIdx.x >> 5;
    if (lane_id() == 0) {
#pragma unroll
        for (int a = 0; a < 3; a++) {
            s_cb[a][warp] = lo[a];
            s_cb[3 + a][warp] = hi[a];
        }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float v = s_cb[threadIdx.x][0];
        for (int w = 1; w < BB_THREADS / 32; w++) v = threadIdx.x < 3 ? fminf(v, s_cb[threadIdx.x][w]) : fmaxf(v, s_cb[threadIdx.x][w]);
        __stcg(chunk_bbox + (size_t)blockIdx.x * 6 + threadIdx.x, v);
    }
}

// ---- global bbox + octree bounding box replay ------------------------------------------------
// PCL grows the octree box sequentially while inserting points (OctreePointCloud::adoptBoundingBoxToPoint):
// a point outside [min, max) doubles the box, moving `min` down by the old side on every axis the point
// does not exceed upward.  The final `min` (hence leaf keys and leaf visiting order) depends on the
// input order, so the replay below finds, in order, each point that violates the current box.
__device__ __forceinline__ bool violates(const double *mn, const double *mx, float lx, float ly, float lz, float hx, float hy, float hz) {
    return (double)lx < mn[0] || (double)ly < mn[1] || (double)lz < mn[2] || (double)hx >= mx[0] || (double)hy >= mx[1] || (double)hz >= mx[2];
}

// box of the octree after its first point (getKeyBitSize() on the empty tree: depth 1, box padded symmetrically to
// side 2*res): min = c - res up to double rounding, restated operation by operation
__host__ __device__ __forceinline__ void octree_first_box(const float c[3], double res, double mn[3], double mx[3]) {
    const double eps = (double)1.1920929e-07f; // std::numeric_limits<float>::epsilon(), promoted as in PCL
    for (int a = 0; a < 3; a++) {
        mn[a] = (double)c[a] - res / 2;
        mx[a] = (double)c[a] + res / 2;
    }
    const double side = (double)(1 << 1) * res;
    for (int a = 0; a < 3; a++) {
        const double oversize = (side - (mx[a] - mn[a])) / 2.0;
        if (oversize > eps) {
            mn[a] -= oversize;
            mx[a] += oversize;
        }
    }
}

// Boxes of SUPER consecutive chunks, kept by atomic max on an order-preserving encoding in which 0 means "nothing yet"
// (the words live in the all-zero workspace and are cleared again by the block that reads them):
//   word a     = ~enc(min over the points of coordinate a)       word 3 + a = enc(max ...)
__device__ __forceinline__ uint32_t enc_float(float x) {
    const uint32_t b = __float_as_uint(x);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float dec_float(uint32_t e) { return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e); }

// Called by a whole block of THREADS threads.  chunk_bbox holds one box per CHUNK consecutive points; super_bbox (or
// nullptr) one encoded box per SUPER chunks, searched first (with 256-point chunks an 8 M-point cloud has 31 K of them).
// The replay continues from `seed` (a cloud partitioned over several GPUs is replayed part by part); seed.valid == 0: it
// starts from this cloud's first point.
template <int THREADS, int CHUNK, int SUPER>
__device__ __forceinline__ void octree_box_block(const cwipc_point *__restrict__ pts, uint32_t n, const float *chunk_bbox, uint32_t nchunks, uint32_t *super_bbox, double res,
                                                  int do_octree, const cwipc_cuda_octree_state &seed, OctreeBox *__restrict__ out) {
    __shared__ float s_red[6][32];
    __shared__ double s_min[3], s_max[3];
    __shared__ int s_depth, s_error;
    __shared__ uint32_t s_cursor, s_first;
    const unsigned tid = threadIdx.x, warp = tid >> 5, lane = lane_id();

    // global bounding box
    const uint32_t nsuper = (nchunks + SUPER - 1) / SUPER;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (super_bbox) {
        for (uint32_t c = tid; c < nsuper; c += THREADS) {
#pragma unroll
            for (int a = 0; a < 3; a++) {
                lo[a] = fminf(lo[a], dec_float(~__ldcg(super_bbox + (size_t)c * 8 + a)));
                hi[a] = fmaxf(hi[a], dec_float(__ldcg(super_bbox + (size_t)c * 8 + 3 + a)));
            }
        }
    } else {
        for (uint32_t c = tid; c < nchunks; c += THREADS) {
#pragma unroll
            for (int a = 0; a < 3; a++) {
                lo[a] = fminf(lo[a], __ldcg(chunk_bbox + (size_t)c * 6 + a));
                hi[a] = fmaxf(hi[a], __ldcg(chunk_bbox + (size_t)c * 6 + 3 + a));
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 3; a++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(FULL_MASK, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(FULL_MASK, hi[a], o));
        }
        if (lane == 0) {
            s_red[a][warp] = lo[a];
            s_red[3 + a][warp] = hi[a];
        }
    }
    __syncthreads();
    if (tid < 6) {
        float v = s_red[tid][0];
        for (int w = 1; w < THREADS / 32; w++) v = tid < 3 ? fminf(v, s_red[tid][w]) : fmaxf(v, s_red[tid][w]);
        if (tid < 3) out->gmin[tid] = v;
        else out->gmax[tid - 3] = v;
    }
    if (!do_octree) {
        if (tid == 0) { out->depth = 0; out->error = 0; }
        return;
    }

    const double eps = (double)1.1920929e-07f;
    if (tid == 0 && seed.valid) {
        for (int a = 0; a < 3; a++) {
            s_min[a] = seed.min[a];
            s_max[a] = seed.max[a];
        }
        s_depth = seed.depth;
        s_error = 0;
        s_cursor = 0;
    } else if (tid == 0) {
        const Point16 p0 = ld_point(pts, 0);
        const float c[3] = {p0.x, p0.y, p0.z};
        double mn[3], mx[3];
        octree_first_box(c, res, mn, mx);
        for (int a = 0; a < 3; a++) {
            s_min[a] = mn[a];
            s_max[a] = mx[a];
        }
        s_depth = 1;
        s_error = 0;
        s_cursor = 1;
    }
    while (true) {
        __syncthreads();
        if (tid == 0) s_first = 0xffffffffu;
        __syncthreads();
        const uint32_t cursor = s_cursor;
        uint32_t c_begin = cursor / CHUNK, c_end = nchunks;
        if (super_bbox) {
            // first super chunk at or after the cursor whose box sticks out; then only its chunks are looked at
            for (uint32_t sc = cursor / (CHUNK * SUPER) + tid; sc < nsuper; sc += THREADS) {
                const uint32_t *b = super_bbox + (size_t)sc * 8;
                if (violates(s_min, s_max, dec_float(~__ldcg(b)), dec_float(~__ldcg(b + 1)), dec_float(~__ldcg(b + 2)), dec_float(__ldcg(b + 3)), dec_float(__ldcg(b + 4)),
                             dec_float(__ldcg(b + 5)))) {
                    atomicMin(&s_first, sc);
                    break;
                }
            }
            __syncthreads();
            const uint32_t scstar = s_first;
            if (scstar == 0xffffffffu) break;
            __syncthreads();
            if (tid == 0) s_first = 0xffffffffu;
            __syncthreads();
            c_begin = max(c_begin, scstar * SUPER);
            c_end = min(nchunks, (scstar + 1) * SUPER);
        }
        // first chunk at or after the cursor whose box sticks out
        for (uint32_t c = c_begin + tid; c < c_end; c += THREADS) {
            const float *b = chunk_bbox + (size_t)c * 6;
            if (violates(s_min, s_max, __ldcg(b), __ldcg(b + 1), __ldcg(b + 2), __ldcg(b + 3), __ldcg(b + 4), __ldcg(b + 5))) {
                atomicMin(&s_first, c);
                break;
            }
        }
        __syncthreads();
        const uint32_t cstar = s_first;
        if (cstar == 0xffffffffu) {
            if (!super_bbox) break;
            __syncthreads();
            if (tid == 0) s_cursor = c_end * CHUNK; // (cannot happen: a box sticks out through one of its points, and those before the cursor do not)
            continue;
        }
        __syncthreads();
        if (tid == 0) s_first = 0xffffffffu;
        __syncthreads();
        // first violating point of that chunk, not before the cursor
        for (uint32_t i = cstar * CHUNK + tid; i < (cstar + 1) * CHUNK && i < n; i += THREADS) {
            if (i >= cursor) {
                const Point16 p = ld_point(pts, i);
                if (violates(s_min, s_max, p.x, p.y, p.z, p.x, p.y, p.z)) atomicMin(&s_first, i);
            }
        }
        __syncthreads();
        const uint32_t istar = s_first;
        if (tid == 0) {
            if (istar == 0xffffffffu) {
                s_cursor = (cstar + 1) * CHUNK; // only already-replayed points of this chunk stick out
            } else {
                const Point16 p = ld_point(pts, istar);
                const double q[3] = {(double)p.x, (double)p.y, (double)p.z};
                while (true) {
                    bool upper[3], any = false;
                    for (int a = 0; a < 3; a++) {
                        upper[a] = q[a] >= s_max[a];
                        any = any || upper[a] || q[a] < s_min[a];
                    }
                    if (!any) break;
                    if (s_depth >= 30) {
                        s_error = 1;
                        break;
                    }
                    double side = (double)(1 << s_depth) * res;
                    for (int a = 0; a < 3; a++)
                        if (!upper[a]) s_min[a] -= side;
                    s_depth++;
                    side = (double)(1 << s_depth) * res - eps;
                    for (int a = 0; a < 3; a++) s_max[a] = s_min[a] + side;
                }
                s_cursor = istar + 1;
            }
        }
        __syncthreads();
        if (s_error) break;
    }
    __syncthreads();
    if (tid == 0) {
        for (int a = 0; a < 3; a++) {
            out->min[a] = s_min[a];
            out->max[a] = s_max[a];
            out->shift[a] = 0;
        }
        out->depth = s_depth;
        out->error = s_error;
        out->fallback = 0;
    }
    if (super_bbox) // leave the workspace all zero
        for (uint32_t i = tid; i < nsuper * 8; i += THREADS) super_bbox[i] = 0u;
}

// One launch: every block boxes its 4096-point chunk; the block that finishes last reduces the chunk boxes
// and replays the octree growth (the classic "last block" pattern: fence, ticket, fence).
__global__ void __launch_bounds__(BB_THREADS) bbox_octree_kernel(const cwipc_point *__restrict__ pts, uint32_t n, float *chunk_bbox, uint32_t nchunks, double res, int do_octree,
                                                                cwipc_cuda_octree_state seed, uint32_t *__restrict__ done_counter, OctreeBox *__restrict__ out) {
    __shared__ bool s_last;
    chunk_bbox_block(pts, n, chunk_bbox);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t ticket = atomicAdd(done_counter, 1u);
        s_last = ticket == nchunks - 1;
        if (s_last) *done_counter = 0; // leave the counter clean for the next call
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    octree_box_block<BB_THREADS, BB_CHUNK, 1>(pts, n, chunk_bbox, nchunks, nullptr, res, do_octree, seed, out);
}

// ---- key generation --------------------------------------------------------------------------
struct KeyParams {
    int octree;       // 1: [morton | voxel-in-leaf], 0: PCL's linear voxel index
    float inv;        // 1.0f / cellsize
    int idxbits;
    // octree mode
    double omin[3];
    double res;
    double inv_res;   // 1.0 / res (filter only; ties are decided by the exact division)
    double inv_cs;    // 1.0 / (double)cellsize
    int depth;
    // single-grid mode
    int minb[3];
    int div[3];
};

__host__ __device__ __forceinline__ uint64_t spread3(uint32_t v) { // bit i -> bit 3i, v < 2^21
    uint64_t x = v & 0x1fffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__host__ __device__ __forceinline__ uint32_t compact3(uint64_t x) { // inverse of spread3
    x &= 0x1249249249249249ull;
    x = (x | x >> 2) & 0x10c30c30c30c30c3ull;
    x = (x | x >> 4) & 0x100f00f00f00f00full;
    x = (x | x >> 8) & 0x1f0000ff0000ffull;
    x = (x | x >> 16) & 0x1f00000000ffffull;
    x = (x | x >> 32) & 0x1fffffull;
    return (uint32_t)x;
}

// Leaf lookup tables (octree mode): the leaf index of a coordinate is a step function of the float32 value, so the
// smallest float at which every step happens is found once, with the very double arithmetic of the generic path, and a
// point then costs two or three float compares per axis instead of double-precision subtract / divide / floor.
// Leaf slot m of axis a covers the floats in [thr[a][m], thr[a][m + 1]).
constexpr int KT_LEAVES = 32;
struct KeyTables {
    float thr[3][KT_LEAVES + 1];
    int origin[3][KT_LEAVES];       // voxel-coordinate origin of the leaf (a per-leaf constant <= every voxel coordinate in it)
    uint64_t bits[3][KT_LEAVES];    // the leaf's contribution to the key, already in the axis' position
    float inv_res_f;                // 1 / res in float: first guess of the slot
    int relative;                   // 1: leaf indices relative to the first point's box (fused pass), 0: final Morton bits
    // Fused pass: which side of a leaf face a coordinate lies on is decided by floor(((double)x - min) / res), against the box
    // of the first point here and against the final box (a whole number of leaf pitches lower) by the reference.  Both
    // agree whenever x - min is computed exactly, i.e. for every float that is not tiny next to res; for a face F at (nearly)
    // zero, floats with |x - F| < 2^-36 res (several double ulps of the widest possible box, 2^14 res) can fall on
    // different sides.  risk[a] = 2^-36 res when axis a has such a face (else 0), fz[a] = the face (0 when it is exactly
    // zero, where the two boxes are checked against each other by the last block), zero_ok[a] = the face is exactly zero.
    float risk[3];
    float fz[3];
    int zero_ok[3];
};

// leaf index of a coordinate against an octree origin: (unsigned)(((double)x - min) / res), PCL genOctreeKeyforPoint
__host__ __device__ __forceinline__ long long leaf_floor(float x, double mn, double res) {
    const double q = floor(((double)x - mn) / res);
    return q >= 4.0e18 ? (long long)4000000000000000000ll : (q <= -4.0e18 ? (long long)-4000000000000000000ll : (long long)q); // the cast is undefined beyond 2^63
}
__host__ __device__ __forceinline__ int leaf_origin(double mn, long long leaf, double res, double inv_cs) { return (int)floor((mn + (double)leaf * res) * inv_cs) - 2; }

__host__ __device__ __forceinline__ float next_up(float x) {
#ifdef __CUDA_ARCH__
    return nextafterf(x, INFINITY);
#else
    return std::nextafter(x, INFINITY);
#endif
}
__host__ __device__ __forceinline__ float next_down(float x) {
#ifdef __CUDA_ARCH__
    return nextafterf(x, -INFINITY);
#else
    return std::nextafter(x, -INFINITY);
#endif
}

// floats in their numeric order as signed integers (and back): bisection over "the smallest float such that ..."
__host__ __device__ __forceinline__ int32_t float_order(float x) {
    int32_t b;
    memcpy(&b, &x, 4);
    return b >= 0 ? b : (int32_t)(0x80000000u - (uint32_t)b);
}
__host__ __device__ __forceinline__ float order_float(int32_t k) {
    const int32_t b = k >= 0 ? k : (int32_t)(0x80000000u - (uint32_t)k);
    float x;
    memcpy(&x, &b, 4);
    return x;
}

// smallest float whose leaf index (against mn) is >= leaf.  The leaf index is monotone in the coordinate, so this is a
// bisection over the float ordering: first in a window of +-32 floats around the face, else over all finite floats
// (e.g. a face at 0, where the neighbouring floats are denormals that vanish in (double)x - mn).
__host__ __device__ __forceinline__ bool leaf_threshold(double mn, double res, long long leaf, float *out) {
    const float face = (float)(mn + (double)leaf * res);
    if (!(face == face) || fabsf(face) > 3.0e38f) return false;
    long long lo = (long long)float_order(face) - 32, hi = (long long)float_order(face) + 32; // invariant: leaf(lo) < leaf <= leaf(hi)
    const long long kmin = float_order(-3.4028234e38f), kmax = float_order(3.4028234e38f);
    if (lo < kmin || hi > kmax || !(leaf_floor(order_float((int32_t)lo), mn, res) < leaf) || !(leaf_floor(order_float((int32_t)hi), mn, res) >= leaf)) {
        lo = kmin;
        hi = kmax;
        if (!(leaf_floor(order_float((int32_t)lo), mn, res) < leaf) || !(leaf_floor(order_float((int32_t)hi), mn, res) >= leaf)) return false;
    }
    while (hi - lo > 1) {
        const long long mid = lo + (hi - lo) / 2;
        if (leaf_floor(order_float((int32_t)mid), mn, res) >= leaf) hi = mid;
        else lo = mid;
    }
    *out = order_float((int32_t)hi);
    return true;
}

// Generic key of a point (any cloud extent): returns the sort key WITHOUT index bits; *bad is set when a coordinate
// is out of the supported range.
__device__ __forceinline__ uint64_t voxel_key(const Point16 &p, const KeyParams &kp, bool *bad) {
    const float f[3] = {floorf(__fmul_rn(p.x, kp.inv)), floorf(__fmul_rn(p.y, kp.inv)), floorf(__fmul_rn(p.z, kp.inv))};
    if (!(fabsf(f[0]) < 4194304.f && fabsf(f[1]) < 4194304.f && fabsf(f[2]) < 4194304.f)) {
        *bad = true; // |voxel coordinate| >= 2^22 (or NaN): float voxel arithmetic is no longer exact
        return 0;
    }
    if (!kp.octree) {
        // ijk = (int)(floor(x*inv) - (float)min_b); idx = i + j*dx + k*dx*dy   (pcl voxel_grid.hpp)
        const int64_t i = (int)(f[0] - (float)kp.minb[0]), j = (int)(f[1] - (float)kp.minb[1]), k = (int)(f[2] - (float)kp.minb[2]);
        return (uint64_t)(i + j * (int64_t)kp.div[0] + k * (int64_t)kp.div[0] * (int64_t)kp.div[1]);
    }
    const float c[3] = {p.x, p.y, p.z};
    uint32_t leaf[3], w[3];
#pragma unroll
    for (int a = 0; a < 3; a++) {
        // OctreePointCloud::genOctreeKeyforPoint: (unsigned)((double)x - min) / res), double arithmetic
        // The quotient is only needed truncated: multiply by the reciprocal, and redo it with the exact
        // division whenever the product lands within 1e-9 of a leaf face (the two differ by < 1e-11).
        const double num = (double)c[a] - kp.omin[a];
        double rel = num * kp.inv_res;
        const double fr = rel - floor(rel);
        if (!(fr > 1e-9 && fr < 1.0 - 1e-9)) rel = num / kp.res;
        leaf[a] = (uint32_t)rel;
        // Any per-leaf constant keeps the (z,y,x) order inside a leaf; this one is <= every voxel
        // coordinate that can occur in the leaf, and the leaf spans < 70 voxels.
        const int origin = leaf_origin(kp.omin[a], (long long)leaf[a], kp.res, kp.inv_cs);
        const int wi = (int)f[a] - origin;
        if (wi < 0 || wi >= WL_RADIX || rel < 0.0 || leaf[a] >= (1u << kp.depth)) *bad = true;
        w[a] = (uint32_t)min(max(wi, 0), WL_RADIX - 1);
    }
    const uint64_t morton = (spread3(leaf[0]) << 2) | (spread3(leaf[1]) << 1) | spread3(leaf[2]);
    const uint64_t wlin = ((uint64_t)w[2] * WL_RADIX + w[1]) * WL_RADIX + w[0];
    return (morton << WL_BITS) | wlin;
}

__global__ void __launch_bounds__(256) voxel_keygen_kernel(const cwipc_point *__restrict__ pts, uint32_t n, KeyParams kp, uint64_t *__restrict__ keys, int with_index,
                                                            uint32_t *__restrict__ error_flag) {
    bool bad = false;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const Point16 p = ld_point_stream(pts, i);
        const uint64_t k = voxel_key(p, kp, &bad);
        keys[i] = with_index ? ((k << kp.idxbits) | i) : k;
    }
    if (bad) atomicOr(error_flag, 1u);
}

// ---- the voxel hash table ---------------------------------------------------------------------------------
// Every voxel owns one 64-byte slot (two L2 sectors): key, tile OR, point count, fixed-point coordinate sums RELATIVE to
// the voxel's own origin and colour sums.  Sums are integers, so the result does not depend on the order in which runs
// arrive (deterministic), and the origin-relative offsets of float coordinates are exact in double, so the centroid is
// the correctly rounded mean whatever the cloud's extent.  A voxel of n points sums up to 255 n per colour channel,
// which passes 2^32 from n = 16 843 010 on: calls with more points than that use the WIDE layout, in which every colour
// sum has 64 bits of its own (two more RED per run, measurably slower, hence not the default).
struct __align__(64) VoxelSlot {
    unsigned long long keyp1;      // key + 1; 0 = empty                       } one 16-byte probe
    uint32_t tile;                 // OR of the tile bytes                      }
    uint32_t count;                // wide layout: points                       }
    unsigned long long sx, sy, sz; // two's-complement fixed-point sums of (x - voxel origin) * 2^shift
    unsigned long long c[3];       // colour sums.  Narrow: sum r | sum g << 32, sum b | count << 32.  Wide: sum r, sum g, sum b
};
constexpr uint32_t VS_NARROW_MAX_POINTS = 16843009; // 255 * 16843009 = 2^32 - 1: the largest call whose 32-bit colour sums cannot overflow
static_assert(sizeof(VoxelSlot) == 64, "one slot per 64 bytes");

struct TableHeader { // first 64 bytes of the zeroed workspace (layout of the whole head: runtime.hpp, ZW_HEADER_BYTES)
    uint32_t count; // claimed slots
    uint32_t error; // out-of-range coordinate seen
    uint32_t pad[14]; // pad[0]: last-block ticket of the bbox / stream kernels; pad[2..3]: barrier words of radix_fused_kernel; pad[4]: stats ticket;
                      // pad[5]: stream kernel flags (1: table overflow, 2: a point too close to a leaf face for the relative keys)
};
constexpr uint32_t VS_FLAG_OVERFLOW = 1u, VS_FLAG_AMBIGUOUS = 2u;

__device__ __forceinline__ uint32_t hash_key(uint64_t k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return (uint32_t)k;
}

// ---- the streaming pass -------------------------------------------------------------------------------------
constexpr int VS_L = 8;                       // consecutive points per lane per tile
constexpr int VS_TILE = 32 * VS_L;            // points per warp tile (= points per chunk box)
constexpr int VS_WARPS = 8;
constexpr int VS_THREADS = VS_WARPS * 32;
constexpr int VS_QCAP = 80;                   // queued runs per warp (>= 64: a tile end can add two per lane)
constexpr int VS_REC = 3;                     // 16-byte words per queued run: key | sx, sy | sz, rb gn tl
constexpr int VS_MAX_PROBES = 1 << 14;
constexpr int VS_SUPER = 64;                  // tiles per super chunk of the octree replay's search (16384 points)

enum { VS_LINEAR = 0, VS_TABLES = 1, VS_FUSED = 2 };

// a run of consecutive points of one (leaf, voxel), in registers
struct Run {
    uint64_t key;
    long long sx, sy, sz;      // sums of (coordinate - voxel origin) * 2^shift
    uint32_t rb, gn, tl;       // sum r | sum b << 16 ; sum g | count << 16 (<= 256 points) ; OR of the rgbt words
};

struct __align__(16) WarpStage {
    uint4 pts[2][VS_TILE];        // 8 KB: two stages of 256 points, 16-byte chunks XOR-swizzled inside every 128-byte row
    uint4 queue[VS_QCAP * VS_REC]; // 3.75 KB: closed runs waiting for their trip to the table
    uint4 heads[32 * VS_REC];      // 1.5 KB: every lane's first run of the tile (it may continue the previous lane's last run)
};

struct StreamArgs {
    const cwipc_point *pts;
    uint32_t n, ntiles;
    KeyParams kp;
    float cs;                     // cellsize
    double scale;                 // 2^shift
    VoxelSlot *table;
    uint32_t slot_mask, claim_limit;
    uint64_t *list_keys;          // key of claim c
    uint32_t *list_slots;         // slot of claim c
    TableHeader *header;
    // fused pass: chunk boxes, octree replay, table check
    float *chunk_bbox;
    uint32_t *super_bbox;         // in the zeroed workspace, behind the table
    double res;
    OctreeBox *box_out;
};

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ uint4 ld_volatile_v4(const void *p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void run_add(Run &a, long long sx, long long sy, long long sz, uint32_t rb, uint32_t gn, uint32_t tl) {
    a.sx += sx;
    a.sy += sy;
    a.sz += sz;
    a.rb += rb;
    a.gn += gn;
    a.tl |= tl;
}

__device__ __forceinline__ void queue_store(uint4 *q, uint32_t pos, const Run &r) {
    q[pos * VS_REC + 0] = make_uint4((uint32_t)r.key, (uint32_t)(r.key >> 32), (uint32_t)r.sx, (uint32_t)((unsigned long long)r.sx >> 32));
    q[pos * VS_REC + 1] = make_uint4((uint32_t)r.sy, (uint32_t)((unsigned long long)r.sy >> 32), (uint32_t)r.sz, (uint32_t)((unsigned long long)r.sz >> 32));
    q[pos * VS_REC + 2] = make_uint4(r.rb, r.gn, r.tl, 0u);
}
__device__ __forceinline__ Run queue_load(const uint4 *q, uint32_t pos) {
    const uint4 a = q[pos * VS_REC + 0], b = q[pos * VS_REC + 1], c = q[pos * VS_REC + 2];
    Run r;
    r.key = ((uint64_t)a.y << 32) | a.x;
    r.sx = (long long)(((unsigned long long)a.w << 32) | a.z);
    r.sy = (long long)(((unsigned long long)b.y << 32) | b.x);
    r.sz = (long long)(((unsigned long long)b.w << 32) | b.z);
    r.rb = c.x;
    r.gn = c.y;
    r.tl = c.z;
    return r;
}

// ---- explicit state spaces: the table is global memory and the queue is shared memory, whatever the compiler can prove
// (through a pointer in a struct it falls back to generic ATOM / LD, which wait for their result) ----
__device__ __forceinline__ void red_add_u64(void *gaddr, unsigned long long v) { asm volatile("red.global.add.u64 [%0], %1;" ::"l"(gaddr), "l"(v) : "memory"); }
__device__ __forceinline__ void red_add_u32(void *gaddr, uint32_t v) { asm volatile("red.global.add.u32 [%0], %1;" ::"l"(gaddr), "r"(v) : "memory"); }
__device__ __forceinline__ void red_or_u32(void *gaddr, uint32_t v) { asm volatile("red.global.or.b32 [%0], %1;" ::"l"(gaddr), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned long long atom_cas_u64(void *gaddr, unsigned long long cmp, unsigned long long val) {
    unsigned long long old;
    asm volatile("atom.global.cas.b64 %0, [%1], %2, %3;" : "=l"(old) : "l"(gaddr), "l"(cmp), "l"(val) : "memory");
    return old;
}
__device__ __forceinline__ uint32_t atom_add_u32(void *gaddr, uint32_t v) {
    uint32_t old;
    asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(gaddr), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr) : "memory");
    return v;
}

struct DrainCtx { // by value: a reference to the kernel's parameter block would be read through generic loads
    VoxelSlot *table;
    uint64_t *list_keys;
    uint32_t *list_slots;
    TableHeader *header;
    uint32_t slot_mask, claim_limit;
};

// one queued run: find or claim its slot (the first probe `h` is already in flight), add the sums (WIDE: slot layout)
template <bool WIDE>
__device__ __forceinline__ void flush_run(const DrainCtx &c, bool active, uint64_t key, uint32_t slot, uint4 h, const uint4 &q0, const uint4 &q1, const uint4 &q2, bool &claimed,
                                          bool &lost, uint32_t &slot_out) {
    claimed = false;
    lost = false;
    slot_out = slot;
    if (!active) return;
    const unsigned long long want = key + 1ull;
    uint32_t seen_tile = 0;
    int probes = 0;
    while (true) {
        unsigned long long cur = ((unsigned long long)h.y << 32) | h.x;
        if (cur == 0ull) {
            cur = atom_cas_u64(&c.table[slot].keyp1, 0ull, want);
            if (cur == 0ull) { // claimed: one list entry per voxel
                claimed = true;
                break;
            }
        }
        if (cur == want) {
            seen_tile = h.z; // possibly stale, always a subset of the bits already there
            break;
        }
        slot = (slot + 1u) & c.slot_mask;
        if (++probes > VS_MAX_PROBES) { // table (nearly) full: give up, the host repeats the call with a larger one
            lost = true;
            return;
        }
        h = ld_volatile_v4(&c.table[slot]);
    }
    slot_out = slot;
    VoxelSlot *sl = c.table + slot;
    red_add_u64(&sl->sx, ((unsigned long long)q0.w << 32) | q0.z);
    red_add_u64(&sl->sy, ((unsigned long long)q1.y << 32) | q1.x);
    red_add_u64(&sl->sz, ((unsigned long long)q1.w << 32) | q1.z);
    if constexpr (WIDE) {
        red_add_u64(&sl->c[0], q2.x & 0xffffu);
        red_add_u64(&sl->c[1], q2.y & 0xffffu);
        red_add_u64(&sl->c[2], q2.x >> 16);
        red_add_u32(&sl->count, q2.y >> 16);
    } else {
        red_add_u64(&sl->c[0], (unsigned long long)(q2.x & 0xffffu) | ((unsigned long long)(q2.y & 0xffffu) << 32));
        red_add_u64(&sl->c[1], (unsigned long long)(q2.x >> 16) | ((unsigned long long)(q2.y >> 16) << 32));
    }
    const uint32_t tl = q2.z >> 24;
    if ((seen_tile & tl) != tl) red_or_u32(&sl->tile, tl);
}

// All 32 lanes: the queued runs go to the table, two runs per lane and pass with both 16-byte probes in flight together
// (claim with a 64-bit CAS when the slot is empty, linear probing), then fire-and-forget L2 reductions (RED).  Claims are
// appended to the voxel list with one counter update per warp and pass.
// `seen` is the largest claim count this warp has seen so far (returned by its own counter updates): no extra load.
template <bool WIDE>
__device__ __noinline__ uint32_t drain_queue(uint32_t qaddr, uint32_t qn, DrainCtx c, unsigned lane, uint32_t seen) {
    __syncwarp();
    // more voxels than the table was sized for: stop claiming (the host repeats the call with a full-size table)
    if (seen >= c.claim_limit) {
        if (lane == 0) red_or_u32(&c.header->pad[5], VS_FLAG_OVERFLOW);
        __syncwarp();
        return seen;
    }
    for (uint32_t base = 0; base < qn; base += 64) {
        const uint32_t r0 = base + lane, r1 = base + 32 + lane;
        const bool act0 = r0 < qn, act1 = r1 < qn;
        uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0, a2 = a0, b0 = a0, b1 = a0, b2 = a0, ha = a0, hb = a0;
        uint64_t keya = 0, keyb = 0;
        uint32_t slota = 0, slotb = 0;
        if (act0) {
            a0 = lds_v4(qaddr + r0 * (16 * VS_REC));
            keya = ((uint64_t)a0.y << 32) | a0.x;
            slota = hash_key(keya) & c.slot_mask;
            ha = ld_volatile_v4(&c.table[slota]);
        }
        if (act1) {
            b0 = lds_v4(qaddr + r1 * (16 * VS_REC));
            keyb = ((uint64_t)b0.y << 32) | b0.x;
            slotb = hash_key(keyb) & c.slot_mask;
            hb = ld_volatile_v4(&c.table[slotb]);
        }
        if (act0) {
            a1 = lds_v4(qaddr + r0 * (16 * VS_REC) + 16);
            a2 = lds_v4(qaddr + r0 * (16 * VS_REC) + 32);
        }
        if (act1) {
            b1 = lds_v4(qaddr + r1 * (16 * VS_REC) + 16);
            b2 = lds_v4(qaddr + r1 * (16 * VS_REC) + 32);
        }
        bool cla, clb, losta, lostb;
        flush_run<WIDE>(c, act0, keya, slota, ha, a0, a1, a2, cla, losta, slota);
        flush_run<WIDE>(c, act1, keyb, slotb, hb, b0, b1, b2, clb, lostb, slotb);
        if (__any_sync(FULL_MASK, losta || lostb)) {
            if (losta || lostb) red_or_u32(&c.header->pad[5], VS_FLAG_OVERFLOW);
        }
        const unsigned cma = __ballot_sync(FULL_MASK, cla), cmb = __ballot_sync(FULL_MASK, clb);
        if (cma | cmb) {
            uint32_t first = 0;
            if (lane == 0) first = atom_add_u32(&c.header->count, (uint32_t)(__popc(cma) + __popc(cmb)));
            first = __shfl_sync(FULL_MASK, first, 0);
            seen = first + (uint32_t)(__popc(cma) + __popc(cmb));
            const unsigned lt = lanemask_lt();
            if (cla) {
                const uint32_t i = first + __popc(cma & lt);
                if (i < c.claim_limit) {
                    c.list_keys[i] = keya;
                    c.list_slots[i] = slota;
                } else {
                    red_or_u32(&c.header->pad[5], VS_FLAG_OVERFLOW);
                }
            }
            if (clb) {
                const uint32_t i = first + __popc(cma) + __popc(cmb & lt);
                if (i < c.claim_limit) {
                    c.list_keys[i] = keyb;
                    c.list_slots[i] = slotb;
                } else {
                    red_or_u32(&c.header->pad[5], VS_FLAG_OVERFLOW);
                }
            }
        }
    }
    __syncwarp();
    return seen;
}

// Build the leaf tables of the fused pass inside the block: leaf indices relative to the box of the first point
// (slot m = relative leaf m - 15, i.e. +-16 leaves = +-1024 voxels around p0; points further out take the generic path).
__device__ __forceinline__ void build_relative_tables(KeyTables &tab, const double m0[3], double res, double inv_cs, uint32_t *flags) {
    const unsigned tid = threadIdx.x;
    if (tid < 3 * (KT_LEAVES + 1)) {
        const int a = tid / (KT_LEAVES + 1), m = tid % (KT_LEAVES + 1);
        const long long leaf = (long long)m - 15;
        float x = INFINITY;
        if (!leaf_threshold(m0[a], res, leaf, &x)) {
            atomicOr(flags, VS_FLAG_AMBIGUOUS);
            x = INFINITY;
        }
        tab.thr[a][m] = x;
        if (m < KT_LEAVES) {
            tab.origin[a][m] = leaf_origin(m0[a], leaf, res, inv_cs);
            tab.bits[a][m] = (uint64_t)(leaf + REL_BIAS) << (WL_BITS + 15 * (2 - a));
        }
    }
    if (tid == 0) {
        tab.inv_res_f = (float)(1.0 / res);
        tab.relative = 1;
    }
    __syncthreads();
    if (tid < 3) {
        const float near0 = (float)(res * 2.9802322387695312e-08); // 2^-25 res: floats are denser than double ulps of res below this
        float risk = 0.f, fz = 0.f;
        int zero_ok = 0;
        for (int m = 0; m <= KT_LEAVES; m++) {
            if (fabsf(tab.thr[tid][m]) < near0) {
                risk = (float)(res * 1.4551915228366852e-11); // 2^-36 res
                const double face = m0[tid] + (double)((long long)m - 15) * res;
                zero_ok = face == 0.0;
                fz = zero_ok ? 0.f : tab.thr[tid][m];
            }
        }
        tab.risk[tid] = risk;
        tab.fz[tid] = fz;
        tab.zero_ok[tid] = zero_ok;
    }
}

// The leaf of a point that is not in the open run's leaf: float bounds of the leaf per axis, the leaf's voxel origin and key
// bits.  A leaf spans 64 voxels, so this runs once per tile and lane plus once per leaf crossing.
struct LeafState {
    float lo[3], hi[3];
    int org[3];
    uint64_t bits;
    uint32_t flags; // 1: out of range, 2: on a leaf face of the first point's box (fused pass)
};

template <int MODE>
__device__ __forceinline__ void lookup_leaf(const KeyTables *tab, float cx, float cy, float cz, const double *m0, double res, double inv_res, double inv_cs, int depth,
                                         LeafState *out) {
    const float c[3] = {cx, cy, cz};
    LeafState ls;
    ls.bits = 0;
    ls.flags = 0;
    bool in_table = true;
#pragma unroll
    for (int ax = 0; ax < 3; ax++) {
        int g = (int)floorf(__fmul_rn(__fsub_rn(c[ax], tab->thr[ax][1]), tab->inv_res_f)) + 1;
        g = min(max(g, 0), KT_LEAVES - 1);
        if (c[ax] < tab->thr[ax][g]) g = max(g - 1, 0);
        else if (c[ax] >= tab->thr[ax][g + 1]) g = min(g + 1, KT_LEAVES - 1);
        ls.lo[ax] = tab->thr[ax][g];
        ls.hi[ax] = tab->thr[ax][g + 1];
        ls.org[ax] = tab->origin[ax][g];
        ls.bits |= tab->bits[ax][g];
        in_table = in_table && c[ax] >= ls.lo[ax] && c[ax] < ls.hi[ax];
    }
    if (!in_table) {
        // outside the tables (more than 16 leaves from the first point / more than 32 leaves across): double arithmetic
        // per point, and no leaf bounds, so the next point starts a run of its own
        ls.bits = 0;
#pragma unroll
        for (int ax = 0; ax < 3; ax++) {
            ls.lo[ax] = INFINITY;
            ls.hi[ax] = -INFINITY;
            const double num = (double)c[ax] - m0[ax];
            double rel = num * inv_res;
            const double fr = rel - floor(rel);
            if (!(fr > 1e-9 && fr < 1.0 - 1e-9)) {
                rel = num / res;
                if (MODE == VS_FUSED) ls.flags |= 2u; // on a leaf face: the final box may round the other way
            }
            const long long leaf = (long long)floor(rel);
            ls.org[ax] = leaf_origin(m0[ax], leaf, res, inv_cs);
            if (MODE == VS_FUSED) {
                if (leaf < -REL_BIAS || leaf >= REL_BIAS) ls.flags |= 1u;
                ls.bits |= (uint64_t)((leaf + REL_BIAS) & 0x7fff) << (WL_BITS + 15 * (2 - ax));
            } else {
                if (leaf < 0 || leaf >= (1ll << depth)) ls.flags |= 1u;
                ls.bits |= (spread3((uint32_t)leaf) << (2 - ax)) << WL_BITS;
            }
        }
    }
    *out = ls;
}

// WIDE: slot layout (VoxelSlot)
template <int MODE, bool WIDE>
__global__ void __launch_bounds__(VS_THREADS, 2) voxel_stream_kernel(const __grid_constant__ StreamArgs a, const __grid_constant__ KeyTables g_tab) {
    extern __shared__ __align__(128) unsigned char vs_smem_raw[];
    WarpStage *stages = reinterpret_cast<WarpStage *>(vs_smem_raw);
    KeyTables &tab = *reinterpret_cast<KeyTables *>(vs_smem_raw + sizeof(WarpStage) * VS_WARPS);
    __shared__ double s_m0[3];
    __shared__ bool s_last;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const unsigned lt = lanemask_lt(), le = lt | (1u << lane);
    WarpStage &ws = stages[warp];

    if (MODE == VS_TABLES) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(&g_tab); // kernel parameter (constant bank) -> shared
        uint32_t *dst = reinterpret_cast<uint32_t *>(&tab);
        for (uint32_t i = threadIdx.x; i < sizeof(KeyTables) / 4; i += VS_THREADS) dst[i] = src[i];
    }
    if (MODE == VS_FUSED) {
        if (threadIdx.x == 0) {
            const Point16 p0 = ld_point(a.pts, 0);
            const float c[3] = {p0.x, p0.y, p0.z};
            double mn[3], mx[3];
            octree_first_box(c, a.res, mn, mx);
            s_m0[0] = mn[0];
            s_m0[1] = mn[1];
            s_m0[2] = mn[2];
        }
        __syncthreads();
        build_relative_tables(tab, s_m0, a.res, a.kp.inv_cs, &a.header->pad[5]);
    }
    __syncthreads();

    const float inv = a.kp.inv;
    const uint32_t gw = blockIdx.x * VS_WARPS + warp, nw = gridDim.x * VS_WARPS;
    const Point16 *gpts = reinterpret_cast<const Point16 *>(a.pts);
    bool bad = false, amb = false;
    uint32_t qn = 0;
    const uint32_t qaddr = (uint32_t)__cvta_generic_to_shared(ws.queue);
    uint32_t seen_claims = 0;
    auto drain = [&](uint32_t count) { // the context is read from the parameter bank at the call, not kept in registers
        DrainCtx dctx;
        dctx.table = a.table;
        dctx.list_keys = a.list_keys;
        dctx.list_slots = a.list_slots;
        dctx.header = a.header;
        dctx.slot_mask = a.slot_mask;
        dctx.claim_limit = a.claim_limit;
        seen_claims = drain_queue<WIDE>(qaddr, count, dctx, lane, seen_claims);
    };

    // lane `lane` copies points c*32 + lane (c = 0..7) of a tile: 512 contiguous bytes per instruction.  Point i of the tile
    // lands in 16-byte chunk (i & ~7) | ((i & 7) ^ ((i >> 3) & 7)): the chunks of a 128-byte row are XOR-swizzled with the
    // row number, so that the lanes, each reading its OWN row front to back, hit eight different banks groups per phase.
    auto issue = [&](uint32_t tile, int st) {
        const uint32_t base = tile * VS_TILE;
#pragma unroll
        for (int c = 0; c < VS_L; c++) {
            const uint32_t i = (uint32_t)c * 32u + lane;
            const uint32_t gi = base + i;
            const bool in = gi < a.n;
            cp_async16(&ws.pts[st][(i & ~7u) | ((i & 7u) ^ ((i >> 3) & 7u))], gpts + (in ? gi : 0u), in ? 16u : 0u);
        }
    };

    uint32_t tile = gw;
    int st = 0;
    if (tile < a.ntiles) issue(tile, 0);
    cp_async_commit();
    for (; tile < a.ntiles; tile += nw, st ^= 1) {
        if (tile + nw < a.ntiles) issue(tile + nw, st ^ 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncwarp();

        const uint32_t base = tile * VS_TILE;
        const uint32_t cnt = min((uint32_t)VS_TILE, a.n - base);
        Run cur;
        cur.key = 0; cur.sx = cur.sy = cur.sz = 0; cur.rb = cur.gn = cur.tl = 0;
        float cf0 = 0.f, cf1 = 0.f, cf2 = 0.f; // the open run's voxel coordinates
        uint64_t head_key = 0;                 // key of the lane's first run once it is closed (its sums wait in ws.heads)
        bool have = false;
        int nclosed = 0;
        // state of the open run's leaf (octree modes): float bounds per axis, voxel origin, key bits
        float lo0 = INFINITY, hi0 = -INFINITY, lo1 = INFINITY, hi1 = -INFINITY, lo2 = INFINITY, hi2 = -INFINITY;
        int org0 = 0, org1 = 0, org2 = 0;
        uint64_t leafbits = 0;
        double od0 = 0.0, od1 = 0.0, od2 = 0.0; // the open run's voxel origin (float product, promoted)
        if (MODE == VS_FUSED) {
            // chunk box of the tile (for the octree replay): a sweep of its own, so that the six extrema do not stay in
            // registers across the run loop
            float bmin0 = INFINITY, bmin1 = INFINITY, bmin2 = INFINITY, bmax0 = -INFINITY, bmax1 = -INFINITY, bmax2 = -INFINITY;
            // a leaf face at (nearly) zero on some axis (the first point sits on a coordinate plane): floats within `risk` of
            // it, other than an exact zero, are left to the two-pass path.  0 < |d| < risk  <=>  (bits(|d|) - 1) < (bits(risk) - 1)
            // as unsigned integers; an axis without such a face has risk = 0 and never matches.
            const float fz0 = tab.fz[0], fz1 = tab.fz[1], fz2 = tab.fz[2];
            const uint32_t rk0 = __float_as_uint(tab.risk[0]) - 1u, rk1 = __float_as_uint(tab.risk[1]) - 1u, rk2 = __float_as_uint(tab.risk[2]) - 1u;
            const bool any_risk = (tab.risk[0] > 0.f) | (tab.risk[1] > 0.f) | (tab.risk[2] > 0.f);
#pragma unroll
            for (int j = 0; j < VS_L; j++) {
                const uint4 raw = ws.pts[st][lane * VS_L + ((unsigned)j ^ (lane & 7u))];
                if (lane * VS_L + j < cnt) {
                    const float x = __uint_as_float(raw.x), y = __uint_as_float(raw.y), z = __uint_as_float(raw.z);
                    bmin0 = fminf(bmin0, x); bmax0 = fmaxf(bmax0, x);
                    bmin1 = fminf(bmin1, y); bmax1 = fmaxf(bmax1, y);
                    bmin2 = fminf(bmin2, z); bmax2 = fmaxf(bmax2, z);
                    if (any_risk) {
                        const uint32_t ux = (__float_as_uint(x - fz0) & 0x7fffffffu) - 1u, uy = (__float_as_uint(y - fz1) & 0x7fffffffu) - 1u,
                                       uz = (__float_as_uint(z - fz2) & 0x7fffffffu) - 1u;
                        if ((tab.risk[0] > 0.f && ux < rk0) | (tab.risk[1] > 0.f && uy < rk1) | (tab.risk[2] > 0.f && uz < rk2)) amb = true;
                    }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                bmin0 = fminf(bmin0, __shfl_xor_sync(FULL_MASK, bmin0, o)); bmax0 = fmaxf(bmax0, __shfl_xor_sync(FULL_MASK, bmax0, o));
                bmin1 = fminf(bmin1, __shfl_xor_sync(FULL_MASK, bmin1, o)); bmax1 = fmaxf(bmax1, __shfl_xor_sync(FULL_MASK, bmax1, o));
                bmin2 = fminf(bmin2, __shfl_xor_sync(FULL_MASK, bmin2, o)); bmax2 = fmaxf(bmax2, __shfl_xor_sync(FULL_MASK, bmax2, o));
            }
            if (lane < 6) {
                const float v = lane == 0 ? bmin0 : lane == 1 ? bmin1 : lane == 2 ? bmin2 : lane == 3 ? bmax0 : lane == 4 ? bmax1 : bmax2;
                __stcg(a.chunk_bbox + (size_t)tile * 6 + lane, v);
                atomicMax(a.super_bbox + (size_t)(tile / VS_SUPER) * 8 + lane, lane < 3 ? ~enc_float(v) : enc_float(v));
            }
        }

#pragma unroll 2
        for (int j = 0; j < VS_L; j++) {
            if (qn > (uint32_t)(VS_QCAP - 32)) {
                drain(qn);
                qn = 0;
            }
            const uint32_t li = lane * VS_L + j;
            const bool valid = li < cnt;
            const uint4 raw = ws.pts[st][lane * VS_L + ((unsigned)j ^ (lane & 7u))];
            Point16 p;
            p.x = __uint_as_float(raw.x);
            p.y = __uint_as_float(raw.y);
            p.z = __uint_as_float(raw.z);
            p.rgbt = raw.w;
            const float f0 = floorf(__fmul_rn(p.x, inv)), f1 = floorf(__fmul_rn(p.y, inv)), f2 = floorf(__fmul_rn(p.z, inv));
            bool same_leaf = true;
            if (MODE != VS_LINEAR) same_leaf = p.x >= lo0 && p.x < hi0 && p.y >= lo1 && p.y < hi1 && p.z >= lo2 && p.z < hi2;
            const bool same = have && same_leaf && f0 == cf0 && f1 == cf1 && f2 == cf2;
            const bool closing = valid && have && !same;
            const unsigned qm = __ballot_sync(FULL_MASK, closing && nclosed > 0);
            if (closing) {
                if (nclosed == 0) {
                    queue_store(ws.heads, lane, cur);
                    head_key = cur.key;
                } else {
                    queue_store(ws.queue, qn + __popc(qm & lt), cur);
                }
                nclosed++;
            }
            qn += __popc(qm);
            if (valid && !same) {
                // ---- a new run starts here ----
                if (!(fabsf(f0) < 4194304.f && fabsf(f1) < 4194304.f && fabsf(f2) < 4194304.f)) bad = true; // |voxel coordinate| >= 2^22 or NaN
                if (MODE == VS_LINEAR) {
                    const int64_t i0 = (int)(f0 - (float)a.kp.minb[0]), i1 = (int)(f1 - (float)a.kp.minb[1]), i2 = (int)(f2 - (float)a.kp.minb[2]);
                    cur.key = (uint64_t)(i0 + i1 * (int64_t)a.kp.div[0] + i2 * (int64_t)a.kp.div[0] * (int64_t)a.kp.div[1]);
                } else {
                    if (!(have && same_leaf)) {
                        // ---- ... in another leaf (rare: a leaf spans 64 voxels) ----
                        LeafState ls;
                        lookup_leaf<MODE>(&tab, p.x, p.y, p.z, MODE == VS_FUSED ? s_m0 : a.kp.omin, a.kp.res, a.kp.inv_res, a.kp.inv_cs, a.kp.depth, &ls);
                        lo0 = ls.lo[0]; hi0 = ls.hi[0]; lo1 = ls.lo[1]; hi1 = ls.hi[1]; lo2 = ls.lo[2]; hi2 = ls.hi[2];
                        org0 = ls.org[0]; org1 = ls.org[1]; org2 = ls.org[2];
                        leafbits = ls.bits;
                        if (ls.flags & 1u) bad = true;
                        if (ls.flags & 2u) amb = true;
                    }
                    const int w0 = (int)f0 - org0, w1 = (int)f1 - org1, w2 = (int)f2 - org2;
                    if ((unsigned)w0 >= (unsigned)WL_RADIX || (unsigned)w1 >= (unsigned)WL_RADIX || (unsigned)w2 >= (unsigned)WL_RADIX) bad = true;
                    cur.key = leafbits | (uint64_t)(uint32_t)((w2 * WL_RADIX + w1) * WL_RADIX + w0); // (out of range: flagged above, the result is discarded)
                }
                cur.sx = cur.sy = cur.sz = 0;
                cur.rb = cur.gn = cur.tl = 0;
                cf0 = f0;
                cf1 = f1;
                cf2 = f2;
                od0 = (double)__fmul_rn(f0, a.cs);
                od1 = (double)__fmul_rn(f1, a.cs);
                od2 = (double)__fmul_rn(f2, a.cs);
                have = true;
            }
            if (valid) {
                // (coordinate - voxel origin) is exact in double; the scale is a power of two
                cur.sx += __double2ll_rn(((double)p.x - od0) * a.scale);
                cur.sy += __double2ll_rn(((double)p.y - od1) * a.scale);
                cur.sz += __double2ll_rn(((double)p.z - od2) * a.scale);
                cur.rb += p.rgbt & 0x00ff00ffu;
                cur.gn += ((p.rgbt >> 8) & 0xffu) + 0x10000u;
                cur.tl |= p.rgbt;
            }
        }

        // ---- join the lanes' partial runs: a run that crosses lane boundaries is summed by a segmented scan ----
        const bool has_t = have;
        const bool single = has_t && nclosed == 0;          // the whole segment is one run
        const uint64_t EMPTY_T = ~0ull, EMPTY_F = ~0ull - 1ull; // never valid keys (the low 19 bits of a key are < 72^3)
        const uint64_t tkey = has_t ? cur.key : EMPTY_T;
        const uint64_t firstkey = !has_t ? EMPTY_F : (single ? cur.key : head_key);
        const uint64_t prev_tkey = __shfl_up_sync(FULL_MASK, tkey, 1);
        const uint64_t next_first = __shfl_down_sync(FULL_MASK, firstkey, 1);
        const bool cont = lane > 0 && single && prev_tkey == cur.key;   // my (only) run continues the previous lane's tail run
        const bool absorbed = lane < 31 && has_t && next_first == cur.key; // my tail run continues in the next lane
        const unsigned seg_heads = __ballot_sync(FULL_MASK, !cont);
        const int seg_start = 31 - __clz(seg_heads & le);
        Run tail = cur;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long tx = __shfl_up_sync(FULL_MASK, tail.sx, o), ty = __shfl_up_sync(FULL_MASK, tail.sy, o), tz = __shfl_up_sync(FULL_MASK, tail.sz, o);
            const uint32_t trb = __shfl_up_sync(FULL_MASK, tail.rb, o), tgn = __shfl_up_sync(FULL_MASK, tail.gn, o), ttl = __shfl_up_sync(FULL_MASK, tail.tl, o);
            if ((int)lane - o >= seg_start) run_add(tail, tx, ty, tz, trb, tgn, ttl);
        }
        // the run that ends where my segment starts is joined to my first run when that one is not my only run
        const long long px = __shfl_up_sync(FULL_MASK, tail.sx, 1), py = __shfl_up_sync(FULL_MASK, tail.sy, 1), pz = __shfl_up_sync(FULL_MASK, tail.sz, 1);
        const uint32_t prb = __shfl_up_sync(FULL_MASK, tail.rb, 1), pgn = __shfl_up_sync(FULL_MASK, tail.gn, 1), ptl = __shfl_up_sync(FULL_MASK, tail.tl, 1);
        const bool push_tail = has_t && !absorbed, push_head = has_t && !single;
        const unsigned mt = __ballot_sync(FULL_MASK, push_tail), mh = __ballot_sync(FULL_MASK, push_head);
        if (qn + __popc(mt) + __popc(mh) > (uint32_t)VS_QCAP) { // the queue is drained when it is (nearly) full: dense passes
            drain(qn);
            qn = 0;
        }
        if (push_tail) queue_store(ws.queue, qn + __popc(mt & lt), tail);
        qn += __popc(mt);
        if (push_head) {
            Run head = queue_load(ws.heads, lane);
            if (lane > 0 && prev_tkey == head_key) run_add(head, px, py, pz, prb, pgn, ptl);
            queue_store(ws.queue, qn + __popc(mh & lt), head);
        }
        qn += __popc(mh);
        __syncwarp();
    }
    cp_async_wait<0>();
    if (qn > 0) drain(qn);
    if (bad) atomicOr(&a.header->error, 1u);
    if (amb) atomicOr(&a.header->pad[5], VS_FLAG_AMBIGUOUS);

    if (MODE != VS_FUSED) return;
    // ---- the block that finishes last: global box, octree replay, and the check that relative keys are final keys ----
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t ticket = atomicAdd(&a.header->pad[0], 1u);
        s_last = ticket == gridDim.x - 1;
        if (s_last) a.header->pad[0] = 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    octree_box_block<VS_THREADS, VS_TILE, VS_SUPER>(a.pts, a.n, a.chunk_bbox, a.ntiles, a.super_bbox, a.res, 1, cwipc_cuda_octree_state{}, a.box_out);
    __syncthreads();
    // shift of the leaf indices: (m0 - final min) / res must be a whole number (the box only ever moves by multiples of res),
    // and every table threshold inside the cloud's extent must be a threshold of the FINAL box too
    __shared__ int s_fallback;
    if (threadIdx.x == 0) s_fallback = 0;
    __syncthreads();
    if (threadIdx.x < 3) {
        const int ax = threadIdx.x;
        const double q = (s_m0[ax] - a.box_out->min[ax]) / a.res;
        const double r = rint(q);
        if (!(fabs(q - r) <= 1e-12 * fmax(1.0, fabs(q))) || r < 0.0 || r > 1.0e9) atomicOr(&s_fallback, 1);
        a.box_out->shift[ax] = (int)r;
    }
    __syncthreads();
    if (threadIdx.x < 3 * (KT_LEAVES + 1)) {
        const int ax = threadIdx.x / (KT_LEAVES + 1), m = threadIdx.x % (KT_LEAVES + 1);
        const float x = tab.thr[ax][m];
        const float gmin = a.box_out->gmin[ax], gmax = a.box_out->gmax[ax];
        (void)gmin;
        (void)gmax;
        if (x == x && fabsf(x) < 3.0e38f) { // every face of the table (the relation is affine: faces outside the cloud agree too)
            const long long sh = (long long)a.box_out->shift[ax];
            const long long want = (long long)m - 15 + sh;
            const double mn = a.box_out->min[ax];
            const float risk = tab.risk[ax];
            if (risk > 0.f && fabsf(x - tab.fz[ax]) < 4.f * risk) {
                // a face at (nearly) zero: floats closer to it than `risk` were excluded point by point (VS_FLAG_AMBIGUOUS); the
                // face itself when it is exactly zero, and everything from `risk` on, must fall on the same side for both boxes
                const float fz = tab.fz[ax];
                const float probe[4] = {fz + risk, fz - risk, tab.zero_ok[ax] ? 0.f : fz + risk, tab.zero_ok[ax] ? -0.f : fz - risk};
                for (int i = 0; i < 4; i++)
                    if (leaf_floor(probe[i], mn, a.res) != leaf_floor(probe[i], s_m0[ax], a.res) + sh) atomicOr(&s_fallback, 1);
            } else if (leaf_floor(x, mn, a.res) != want || leaf_floor(next_down(x), mn, a.res) != want - 1) {
                atomicOr(&s_fallback, 1);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        a.box_out->fallback = s_fallback;
        a.box_out->m0[0] = s_m0[0];
        a.box_out->m0[1] = s_m0[1];
        a.box_out->m0[2] = s_m0[2];
    }
}

// claimed voxels -> sort words [final key | claim index].  Fused pass: relative leaf indices become the final octree's
// Morton code here, on V entries instead of N points.
__global__ void __launch_bounds__(256) voxel_words_kernel(const uint64_t *__restrict__ list_keys, uint32_t v, int cbits, int relative, int sx, int sy, int sz, int depth,
                                                           uint64_t *__restrict__ words, TableHeader *__restrict__ header) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= v) return;
    uint64_t key = list_keys[c];
    if (relative) {
        const long long lx = (long long)((key >> (WL_BITS + 30)) & 0x7fff) - REL_BIAS + sx;
        const long long ly = (long long)((key >> (WL_BITS + 15)) & 0x7fff) - REL_BIAS + sy;
        const long long lz = (long long)((key >> WL_BITS) & 0x7fff) - REL_BIAS + sz;
        (void)depth; // the final box contains every point: 0 <= leaf < 2^depth
        const uint64_t morton = (spread3((uint32_t)lx) << 2) | (spread3((uint32_t)ly) << 1) | spread3((uint32_t)lz);
        key = (morton << WL_BITS) | (key & ((1ull << WL_BITS) - 1ull));
    }
    words[c] = (key << cbits) | c;
}

// how to get a voxel's integer coordinates back from its key (they fix the origin its sums are relative to)
struct EmitGeom {
    int mode;        // VS_LINEAR: key = PCL's linear index; VS_TABLES: [Morton(leaf) | voxel-in-leaf]; VS_FUSED: [relative leaf x, y, z | voxel-in-leaf]
    double mn[3];    // octree min corner the leaf indices count from (final box, or the first point's box)
    double res, inv_cs;
    int minb[3], div[3];
};

__device__ __forceinline__ void voxel_of_key(uint64_t key, const EmitGeom &g, float v[3]) {
    if (g.mode == VS_LINEAR) {
        const uint64_t dx = (uint64_t)g.div[0], dy = (uint64_t)g.div[1];
        v[0] = (float)(g.minb[0] + (int)(key % dx));
        v[1] = (float)(g.minb[1] + (int)((key / dx) % dy));
        v[2] = (float)(g.minb[2] + (int)(key / (dx * dy)));
        return;
    }
    const uint32_t wlin = (uint32_t)(key & ((1ull << WL_BITS) - 1ull));
    const int w[3] = {(int)(wlin % WL_RADIX), (int)((wlin / WL_RADIX) % WL_RADIX), (int)(wlin / (WL_RADIX * WL_RADIX))};
#pragma unroll
    for (int a = 0; a < 3; a++) {
        long long leaf;
        if (g.mode == VS_FUSED) leaf = (long long)((key >> (WL_BITS + 15 * (2 - a))) & 0x7fff) - REL_BIAS;
        else leaf = (long long)compact3((key >> WL_BITS) >> (2 - a));
        v[a] = (float)(leaf_origin(g.mn[a], leaf, g.res, g.inv_cs) + w[a]); // the very expression the keys were made with
    }
}

// mean xyz (exact sum, one rounding), colour floor(sum / n) (pcl::CentroidPoint's truncated float average wherever its
// float sum is exact), OR of tiles
template <bool WIDE>
__device__ __forceinline__ Point16 finalize_voxel(const VoxelSlot &s, const float v[3], float cs, double inv_scale) {
    Point16 o;
    const uint32_t cnt = WIDE ? s.count : (uint32_t)(s.c[1] >> 32);
    const double dn = (double)cnt;
    o.x = (float)((double)__fmul_rn(v[0], cs) + ((double)(long long)s.sx * inv_scale) / dn);
    o.y = (float)((double)__fmul_rn(v[1], cs) + ((double)(long long)s.sy * inv_scale) / dn);
    o.z = (float)((double)__fmul_rn(v[2], cs) + ((double)(long long)s.sz * inv_scale) / dn);
    uint32_t r, g, b; // floor(sum / n) <= 255
    if constexpr (WIDE) {
        r = (uint32_t)(s.c[0] / cnt);
        g = (uint32_t)(s.c[1] / cnt);
        b = (uint32_t)(s.c[2] / cnt);
    } else {
        r = (uint32_t)s.c[0] / cnt;
        g = (uint32_t)(s.c[0] >> 32) / cnt;
        b = (uint32_t)s.c[1] / cnt;
    }
    o.rgbt = r | (g << 8) | (b << 16) | ((s.tile & 0xffu) << 24);
    return o;
}

// One output point per sorted list entry; the slot is read once and cleared, so the table is all zero
// again when the kernel ends (no memset between calls).
template <bool WIDE>
__global__ void __launch_bounds__(256) voxel_emit_kernel(const uint64_t *__restrict__ sorted, uint32_t v, uint32_t cmask, const uint64_t *__restrict__ list_keys,
                                                          const uint32_t *__restrict__ list_slots, VoxelSlot *__restrict__ table, EmitGeom geom, float cs, double inv_scale,
                                                          cwipc_point *__restrict__ out, TableHeader *__restrict__ header) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j == 0) header->count = 0;
    if (j >= v) return;
    const uint32_t c = (uint32_t)sorted[j] & cmask;
    VoxelSlot *sl = table + list_slots[c];
    uint4 *raw = reinterpret_cast<uint4 *>(sl);
    union {
        uint4 q[4];
        VoxelSlot s;
    } u;
    u.q[0] = raw[0];
    u.q[1] = raw[1];
    u.q[2] = raw[2];
    u.q[3] = raw[3];
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    raw[0] = zero;
    raw[1] = zero;
    raw[2] = zero;
    raw[3] = zero;
    float vox[3];
    voxel_of_key(list_keys[c], geom, vox);
    st_point(out, j, finalize_voxel<WIDE>(u.s, vox, cs, inv_scale));
}

// a pass that failed half way: clear the claimed slots (the list knows them) and the header words
__global__ void __launch_bounds__(256) voxel_clear_kernel(uint32_t v, const uint32_t *__restrict__ list_slots, VoxelSlot *__restrict__ table, TableHeader *__restrict__ header) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j == 0) {
        header->count = 0;
        header->error = 0;
        header->pad[5] = 0;
    }
    if (j >= v) return;
    uint4 *raw = reinterpret_cast<uint4 *>(table + list_slots[j]);
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    raw[0] = zero;
    raw[1] = zero;
    raw[2] = zero;
    raw[3] = zero;
}

// the "last block" ticket of bbox_octree_kernel / voxel_stream_kernel: a word of the thread's zeroed workspace header (pad[0])
uint32_t *bbox_counter(int dev, cudaStream_t s) {
    TableHeader *h = static_cast<TableHeader *>(thread_zeroed(dev, ZW_HEADER_BYTES, s));
    return &h->pad[0];
}

struct Plan {
    Plan() {
        memset(&kp, 0, sizeof(kp));
        memset(&tables, 0, sizeof(tables));
    }
    KeyParams kp;
    int keybits = 0;
    float gmin[3] = {0, 0, 0}, gmax[3] = {0, 0, 0};
    bool use_tables = false;
    KeyTables tables;
};

// One launch + one readback: bounding box of the points and the octree box after inserting them in order
// (continuing from `seed` when it is valid).
OctreeBox measure_box(const cwipc_point *pts, size_t n, float cellsize, bool octree_split, int dev, cudaStream_t s, const cwipc_cuda_octree_state &seed = {}) {
    const uint32_t nchunks = (uint32_t)div_up(n, BB_CHUNK);
    Scratch chunk_bbox((size_t)nchunks * 6 * sizeof(float), s);
    Scratch box(sizeof(OctreeBox), s);
    const float octree_cellsize = 64 * cellsize;           // ref: src/cwipc_filters.cpp:113-114 (float)
    const double res = (double)octree_cellsize;
    launch("bbox_octree_kernel", s, 16 * (size_t)n, [&] {
        bbox_octree_kernel<<<nchunks, BB_THREADS, 0, s>>>(pts, (uint32_t)n, chunk_bbox.as<float>(), nchunks, res, octree_split ? 1 : 0, seed, bbox_counter(dev, s), box.as<OctreeBox>());
    });
    OctreeBox *h = static_cast<OctreeBox *>(thread_pinned(sizeof(OctreeBox)));
    CWCU_CHECK(cudaMemcpyAsync(h, box.p, sizeof(OctreeBox), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
    return *h;
}

// Leaf lookup tables against the FINAL octree box (two-pass path); false when an axis spans more than KT_LEAVES leaves.
bool build_key_tables(const KeyParams &kp, const OctreeBox &ob, KeyTables &tab) {
    memset(&tab, 0, sizeof(tab));
    tab.inv_res_f = (float)(1.0 / kp.res);
    tab.relative = 0;
    for (int a = 0; a < 3; a++) {
        if (!(ob.gmin[a] <= ob.gmax[a]) || (double)ob.gmin[a] < kp.omin[a]) return false;
        const long long first = leaf_floor(ob.gmin[a], kp.omin[a], kp.res), last = leaf_floor(ob.gmax[a], kp.omin[a], kp.res);
        if (first < 0 || last < first || last - first + 1 > (long long)KT_LEAVES || last >= (1ll << kp.depth)) return false;
        // slot 0 must start one leaf pitch below slot 1's threshold for the kernel's first guess: thr[a][0] is the first
        // leaf's own lower threshold (no point lies below it)
        for (int m = 0; m <= KT_LEAVES; m++) {
            const long long leaf = first + m;
            tab.thr[a][m] = INFINITY;
            if (m < KT_LEAVES) {
                tab.origin[a][m] = 0;
                tab.bits[a][m] = 0;
            }
            if (leaf > last + 1) continue;
            if (m == 0) {
                tab.thr[a][0] = -INFINITY;
            } else {
                float x;
                if (!leaf_threshold(kp.omin[a], kp.res, leaf, &x)) return false; // did not converge: generic path
                tab.thr[a][m] = x;
            }
            if (m < KT_LEAVES && leaf <= last) {
                tab.origin[a][m] = leaf_origin(kp.omin[a], leaf, kp.res, kp.inv_cs);
                tab.bits[a][m] = (spread3((uint32_t)leaf) << (2 - a)) << WL_BITS;
            }
        }
        // the kernel's first guess is floor((x - thr[1]) / res) + 1: thr[1] must be finite
        if (!std::isfinite(tab.thr[a][1])) {
            float x;
            if (!leaf_threshold(kp.omin[a], kp.res, first + 1, &x)) return false;
            tab.thr[a][1] = x;
        }
    }
    return true;
}

// The key parameters that depend on the voxel size alone: all the fused pass needs (its idxbits stays 0).
void fill_key_params(KeyParams &kp, float cellsize, bool octree_split) {
    memset(&kp, 0, sizeof(kp));
    kp.octree = octree_split ? 1 : 0;
    kp.inv = 1.0f / cellsize;
    kp.res = (double)(64 * cellsize);
    kp.inv_res = 1.0 / kp.res;
    kp.inv_cs = 1.0 / (double)cellsize;
}

// Key layout and limits from the measured (or supplied) boxes.  An input that cannot be downsampled throws.
Plan derive_plan(const OctreeBox &ob, size_t n, float cellsize, bool octree_split) {
    Plan plan;
    KeyParams &kp = plan.kp;
    fill_key_params(kp, cellsize, octree_split);
    kp.idxbits = std::max(1, bit_length((uint64_t)n - 1));
    float maxabs = 0.f;
    for (int a = 0; a < 3; a++) {
        maxabs = std::max(maxabs, std::max(std::fabs(ob.gmin[a]), std::fabs(ob.gmax[a])));
        plan.gmin[a] = ob.gmin[a];
        plan.gmax[a] = ob.gmax[a];
    }
    if (!std::isfinite(maxabs)) throw CudaError{cudaErrorInvalidValue, "pointcloud contains non-finite coordinates"};
    if (octree_split) {
        if (ob.error || ob.depth > MAX_OCTREE_DEPTH)
            throw CudaError{cudaErrorInvalidValue,
                            "pointcloud extent too large for voxel size (octree depth " + std::to_string(ob.depth) + " > " + std::to_string(MAX_OCTREE_DEPTH) + ")"};
        for (int a = 0; a < 3; a++) kp.omin[a] = ob.min[a];
        kp.depth = ob.depth;
        plan.keybits = WL_BITS + 3 * ob.depth;
        plan.use_tables = build_key_tables(kp, ob, plan.tables);
    } else {
        // ref: pcl VoxelGrid::applyFilter -- index-overflow guard, then min_b / div_b from the float bbox
        const float inv = kp.inv;
        const int64_t dx = (int64_t)((ob.gmax[0] - ob.gmin[0]) * inv) + 1;
        const int64_t dy = (int64_t)((ob.gmax[1] - ob.gmin[1]) * inv) + 1;
        const int64_t dz = (int64_t)((ob.gmax[2] - ob.gmin[2]) * inv) + 1;
        if (dx * dy * dz > (int64_t)INT32_MAX) // PCL copies the input and leaves its leaf layout empty; cwipc's tile pass then throws out_of_range
            throw CudaError{cudaErrorInvalidValue, "VoxelGrid std exception: leaf size is too small for the input dataset (integer indices would overflow)"};
        uint64_t cells = 1;
        for (int a = 0; a < 3; a++) {
            kp.minb[a] = (int)std::floor(ob.gmin[a] * inv);
            const int maxb = (int)std::floor(ob.gmax[a] * inv);
            kp.div[a] = maxb - kp.minb[a] + 1;
            cells *= (uint64_t)kp.div[a];
        }
        plan.keybits = std::max(1, bit_length(cells - 1));
    }
    return plan;
}

constexpr size_t VS_SMEM_BYTES = sizeof(WarpStage) * VS_WARPS + sizeof(KeyTables);

template <int MODE, bool WIDE>
void launch_stream(const StreamArgs &args, const KeyTables &tab, int dev, cudaStream_t s) {
    static std::once_flag once[64];
    std::call_once(once[dev & 63], [&] {
        CWCU_CHECK(cudaFuncSetAttribute(voxel_stream_kernel<MODE, WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VS_SMEM_BYTES));
        // two blocks of 106 KB per SM need the largest carve-out
        CWCU_CHECK(cudaFuncSetAttribute(voxel_stream_kernel<MODE, WIDE>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    });
    // persistent warps: two blocks of eight warps per SM, every warp takes tiles gw, gw + nw, ...
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min(div_up((size_t)args.ntiles, (size_t)VS_WARPS), (size_t)sm_count(dev) * 2));
    launch("voxel_stream_kernel", s, 16 * (size_t)args.n, [&] { voxel_stream_kernel<MODE, WIDE><<<grid, VS_THREADS, VS_SMEM_BYTES, s>>>(args, tab); });
}

// hash table size: room for n / 4 voxels (at most half full) when the cloud is large -- a downsample that keeps more than a
// quarter of its points is rare, and is repeated with room for n voxels when it happens
void table_size(size_t n, bool full, size_t &claim_limit, size_t &capacity) {
    claim_limit = (full || n <= ((size_t)1 << 18)) ? n : std::max(n / 4, (size_t)1 << 18);
    capacity = 1024;
    while (capacity < 2 * claim_limit) capacity <<= 1;
}

} // namespace

namespace {
// pts[0..n) -> voxels.  `dest(v)` is called once, when the voxel count v is known, and returns room for them.  `planned`
// and `bounds` (both or neither): the octree box and the bounding box of the whole cloud pts belongs to.  An input that
// cannot be downsampled throws.
DownsampleRange downsample_impl(const cwipc_point *pts, size_t n, float cellsize, bool octree_split, const cwipc_cuda_octree_state *planned, const float *bounds,
                                const std::function<cwipc_point *(size_t)> &dest, int dev, cudaStream_t s) {
    DownsampleRange result;
    if (n == 0) {
        if (!octree_split) throw CudaError{cudaErrorInvalidValue, "VoxelGrid filter produced empty pointcloud"}; // ref: src/cwipc_filters.cpp:58-62
        // no octree leaves: an empty, non-NULL cloud (python/test_cwipc_util.py:589-594)
        (void)dest(0);
        return result;
    }
    if (!(cellsize > 0.f) || !std::isfinite(cellsize)) throw CudaError{cudaErrorInvalidValue, "invalid voxel size " + std::to_string(cellsize)};
    // fixed-point scale of the voxel-relative offsets: |offset| <= cellsize (1 + eps), n of them must fit 2^62 (a part of a
    // partitioned cloud uses the count of the whole cloud: same scale, same rounding as the one-GPU call)
    int shift = 61 - bit_length(std::max((uint64_t)n, planned ? planned->points : 0));
    {
        int e;
        (void)std::frexp(cellsize, &e); // cellsize < 2^e
        shift -= e;
    }
    shift = std::max(-60, std::min(shift, 100));
    const double scale = std::ldexp(1.0, shift), inv_scale = std::ldexp(1.0, -shift);

    const uint32_t ntiles = (uint32_t)div_up(n, (size_t)VS_TILE);
    // CWIPC_CUDA_DS_PATH (tests only; results never depend on it): "twopass" = bounding box / octree replay first, then the
    // streaming pass with leaf tables of the final box; "generic" = same without tables (double arithmetic per run);
    // "smalltable" = start with a table that overflows early.  Default: the fused single pass.
    const char *force = getenv("CWIPC_CUDA_DS_PATH");
    const bool force_twopass = force && (!strcmp(force, "twopass") || !strcmp(force, "generic"));
    const bool force_generic = force && !strcmp(force, "generic");
    const bool force_small = force && !strcmp(force, "smalltable");
    bool fused = octree_split && !planned && !force_twopass;
    bool full_table = false;
    const bool wide = n > VS_NARROW_MAX_POINTS; // slot layout (VoxelSlot)
    OctreeBox ob;
    memset(&ob, 0, sizeof(ob));
    if (planned) {
        for (int a = 0; a < 3; a++) {
            ob.min[a] = planned->min[a];
            ob.max[a] = planned->max[a];
            ob.gmin[a] = bounds[a];
            ob.gmax[a] = bounds[3 + a];
        }
        ob.depth = planned->depth;
    }
    Plan plan;
    bool have_plan = false;
    // an input error the stream pass finds; the table is cleared before it is thrown, so the workspace stays valid
    std::string input_error;

    for (int attempt = 0; attempt < 4; attempt++) {
        if (!fused && !have_plan) {
            if (!planned) ob = measure_box(pts, n, cellsize, octree_split, dev, s);
            plan = derive_plan(ob, n, cellsize, octree_split);
            have_plan = true;
        }
        size_t claim_limit, capacity;
        table_size(n, full_table, claim_limit, capacity);
        if (force_small && !full_table) claim_limit = std::min<size_t>(claim_limit, 1000);
        const size_t nsuper = div_up((size_t)ntiles, (size_t)VS_SUPER);
        uint8_t *wsp = static_cast<uint8_t *>(thread_zeroed(dev, ZW_HEADER_BYTES + capacity * sizeof(VoxelSlot) + nsuper * 32, s));
        TableHeader *header = reinterpret_cast<TableHeader *>(wsp);
        VoxelSlot *table = reinterpret_cast<VoxelSlot *>(wsp + ZW_HEADER_BYTES);
        try {
            Scratch list_keys(claim_limit * sizeof(uint64_t), s), list_slots(claim_limit * sizeof(uint32_t), s);
            Scratch chunk_bbox(fused ? (size_t)ntiles * 6 * sizeof(float) : 0, s), box(sizeof(OctreeBox), s);
            StreamArgs args;
            memset(&args, 0, sizeof(args));
            args.pts = pts;
            args.n = (uint32_t)n;
            args.ntiles = ntiles;
            args.cs = cellsize;
            args.scale = scale;
            args.table = table;
            args.slot_mask = (uint32_t)(capacity - 1);
            args.claim_limit = (uint32_t)claim_limit;
            args.list_keys = list_keys.as<uint64_t>();
            args.list_slots = list_slots.as<uint32_t>();
            args.header = header;
            args.res = (double)(64 * cellsize);
            if (fused) {
                fill_key_params(args.kp, cellsize, true);
                args.chunk_bbox = chunk_bbox.as<float>();
                args.super_bbox = reinterpret_cast<uint32_t *>(wsp + ZW_HEADER_BYTES + capacity * sizeof(VoxelSlot));
                args.box_out = box.as<OctreeBox>();
                wide ? launch_stream<VS_FUSED, true>(args, plan.tables, dev, s) : launch_stream<VS_FUSED, false>(args, plan.tables, dev, s);
            } else {
                args.kp = plan.kp;
                if (!octree_split) wide ? launch_stream<VS_LINEAR, true>(args, plan.tables, dev, s) : launch_stream<VS_LINEAR, false>(args, plan.tables, dev, s);
                else {
                    if (!plan.use_tables || force_generic) { // no usable tables: empty ones send every run through the generic path
                        memset(&plan.tables, 0, sizeof(plan.tables));
                        for (int a = 0; a < 3; a++)
                            for (int m = 0; m <= KT_LEAVES; m++) plan.tables.thr[a][m] = m == 0 ? INFINITY : -INFINITY;
                        plan.tables.inv_res_f = 0.f;
                    }
                    wide ? launch_stream<VS_TABLES, true>(args, plan.tables, dev, s) : launch_stream<VS_TABLES, false>(args, plan.tables, dev, s);
                }
            }
            // one round trip: voxel count, flags, and (fused pass) the boxes
            struct Readback {
                uint32_t head[8];
                OctreeBox box;
            };
            Readback *h = static_cast<Readback *>(thread_pinned(sizeof(Readback)));
            CWCU_CHECK(cudaMemcpyAsync(h->head, header, sizeof(h->head), cudaMemcpyDeviceToHost, s));
            if (fused) CWCU_CHECK(cudaMemcpyAsync(&h->box, box.p, sizeof(OctreeBox), cudaMemcpyDeviceToHost, s));
            stream_sync(s);
            const size_t claimed = h->head[0];
            const uint32_t err = h->head[1], flags = h->head[7];
            auto clear_table = [&] {
                const size_t listed = std::min(claimed, claim_limit);
                if ((flags & VS_FLAG_OVERFLOW) && claimed > claim_limit) {
                    thread_zeroed_invalidate(dev); // claims beyond the list cannot be found again: wipe the workspace
                } else {
                    launch("voxel_clear_kernel", s, 64 * listed, [&] {
                        voxel_clear_kernel<<<(unsigned)std::max<size_t>(1, div_up(listed, 256)), 256, 0, s>>>((uint32_t)listed, list_slots.as<uint32_t>(), table, header);
                    });
                }
            };
            if (fused) {
                ob = h->box;
                const bool redo = (flags & VS_FLAG_AMBIGUOUS) != 0 || ob.fallback != 0 || ob.error != 0 || ob.depth > MAX_OCTREE_DEPTH;
                if (redo) { // a point on a leaf face, or an extent the relative keys do not cover: the two-pass path decides
                    clear_table();
                    fused = false;
                    continue;
                }
            }
            if (err != 0) {
                clear_table();
                input_error = "point coordinates out of range for voxel size " + std::to_string(cellsize) + " (|x/voxelsize| must stay below 2^22)";
                break;
            }
            if (flags & VS_FLAG_OVERFLOW) {
                clear_table();
                if (full_table) throw CudaError{cudaErrorUnknown, "downsample: voxel table overflow with a full-size table"};
                full_table = true;
                continue;
            }
            const size_t v = claimed;
            int keybits, depth = 0;
            if (fused) {
                depth = ob.depth;
                keybits = WL_BITS + 3 * depth;
                for (int a = 0; a < 3; a++) {
                    plan.gmin[a] = ob.gmin[a];
                    plan.gmax[a] = ob.gmax[a];
                }
            } else {
                keybits = plan.keybits;
            }
            const int cbits = std::max(1, bit_length((uint64_t)v - 1));
            if (keybits + cbits > 64) {
                clear_table();
                input_error = "pointcloud too large for 64-bit voxel sort words (" + std::to_string(keybits) + " key bits + " + std::to_string(cbits) + " index bits)";
                break;
            }
            Scratch words(v * sizeof(uint64_t), s), other(v * sizeof(uint64_t), s);
            launch("voxel_words_kernel", s, 16 * v, [&] {
                voxel_words_kernel<<<(unsigned)std::max<size_t>(1, div_up(v, 256)), 256, 0, s>>>(list_keys.as<uint64_t>(), (uint32_t)v, cbits, fused ? 1 : 0, ob.shift[0], ob.shift[1], ob.shift[2],
                                                                                                 depth, words.as<uint64_t>(), header);
            });
            const uint64_t *sorted = radix_sort_u64(words.as<uint64_t>(), other.as<uint64_t>(), v, cbits, cbits + keybits, dev, s);
            cwipc_point *dst = dest(v);
            EmitGeom geom;
            memset(&geom, 0, sizeof(geom));
            geom.mode = fused ? VS_FUSED : (octree_split ? VS_TABLES : VS_LINEAR);
            geom.res = args.res;
            geom.inv_cs = 1.0 / (double)cellsize;
            for (int a = 0; a < 3; a++) {
                geom.mn[a] = fused ? ob.m0[a] : plan.kp.omin[a];
                geom.minb[a] = plan.kp.minb[a];
                geom.div[a] = std::max(1, plan.kp.div[a]);
            }
            launch("voxel_emit_kernel", s, 16 * v, [&] {
                (wide ? voxel_emit_kernel<true> : voxel_emit_kernel<false>)<<<(unsigned)std::max<size_t>(1, div_up(v, 256)), 256, 0, s>>>(
                    sorted, (uint32_t)v, (uint32_t)((1ull << cbits) - 1ull), list_keys.as<uint64_t>(), list_slots.as<uint32_t>(), table, geom, cellsize, inv_scale, dst, header);
            });
            result.count = v;
            // centroids lie inside the input's bounding box: hand it on so that a following filter need not recompute it
            result.has_bounds = true;
            for (int a = 0; a < 3; a++) {
                result.bounds_min[a] = plan.gmin[a];
                result.bounds_max[a] = plan.gmax[a];
            }
            return result;
        } catch (...) {
            thread_zeroed_invalidate(dev);
            throw;
        }
    }
    if (!input_error.empty()) throw CudaError{cudaErrorInvalidValue, input_error};
    throw CudaError{cudaErrorUnknown, "downsample: no attempt succeeded"};
}

// a new cloud of exactly the voxels
StoragePtr downsample_to_cloud(const StoragePtr &in, float cellsize, bool octree_split, const cwipc_cuda_octree_state *planned, const float *bounds, int dev, cudaStream_t s) {
    StoragePtr out;
    const DownsampleRange r = downsample_impl(in->d_pts, in->count, cellsize, octree_split, planned, bounds, [&](size_t v) {
        out = std::make_shared<Storage>(dev, v, s);
        return out->d_pts;
    }, dev, s);
    out->count = r.count;
    out->has_bounds = r.has_bounds;
    memcpy(out->bounds_min, r.bounds_min, sizeof(out->bounds_min));
    memcpy(out->bounds_max, r.bounds_max, sizeof(out->bounds_max));
    out->mark_ready();
    return out;
}
} // namespace

StoragePtr downsample_points(const StoragePtr &in, float cellsize, bool octree_split, int dev, cudaStream_t s) {
    return downsample_to_cloud(in, cellsize, octree_split, nullptr, nullptr, dev, s);
}

// the scale of the centroid sums comes from n, as for a cloud of these n points
DownsampleRange downsample_range(const cwipc_point *pts, size_t n, float cellsize, bool octree_split, cwipc_point *dst, int dev, cudaStream_t s) {
    return downsample_impl(pts, n, cellsize, octree_split, nullptr, nullptr, [dst](size_t) { return dst; }, dev, s);
}

// Partitioned clouds: the octree box and the bounding box of the WHOLE cloud are supplied by the caller.  An empty part
// contributes nothing, in either mode.
StoragePtr downsample_points_planned(const StoragePtr &in, float cellsize, bool octree_split, const cwipc_cuda_octree_state &state, const float bounds[6], int dev, cudaStream_t s) {
    if (in->count == 0) return new_storage(dev, 0, s, [](Storage &) -> size_t { return 0; });
    if (octree_split && !state.valid) throw CudaError{cudaErrorInvalidValue, "planned downsample needs the octree state of the whole cloud"};
    return downsample_to_cloud(in, cellsize, octree_split, &state, bounds, dev, s);
}

// Continue the octree bounding-box replay over this cloud's points; also returns its bounding box.
void octree_replay(const cwipc_point *in, size_t n, float cellsize, cwipc_cuda_octree_state &state, float bounds[6], int dev, cudaStream_t s) {
    for (int a = 0; a < 3; a++) {
        bounds[a] = INFINITY;
        bounds[3 + a] = -INFINITY;
    }
    if (n == 0) return;
    const OctreeBox ob = measure_box(in, n, cellsize, true, dev, s, state);
    if (ob.error) throw CudaError{cudaErrorInvalidValue, "octree replay: runaway growth (non-finite coordinates?)"};
    for (int a = 0; a < 3; a++) {
        state.min[a] = ob.min[a];
        state.max[a] = ob.max[a];
        bounds[a] = ob.gmin[a];
        bounds[3 + a] = ob.gmax[a];
    }
    state.depth = ob.depth;
    state.valid = 1;
    state.points += n;
}

void global_bbox(const cwipc_point *in, size_t n, float gmin[3], float gmax[3], int dev, cudaStream_t s) {
    const OctreeBox ob = measure_box(in, n, 0.f, false, dev, s); // no octree: the cell size is not used
    memcpy(gmin, ob.gmin, sizeof(ob.gmin));
    memcpy(gmax, ob.gmax, sizeof(ob.gmax));
}

void downsample_keys_to_host(const StoragePtr &in, float cellsize, bool octree_split, uint64_t *host_keys, int dev, cudaStream_t s) {
    const size_t n = in->count;
    if (n == 0) return;
    const Plan plan = derive_plan(measure_box(in->d_pts, n, cellsize, octree_split, dev, s), n, cellsize, octree_split);
    Scratch keys(n * sizeof(uint64_t), s);
    Scratch flag(sizeof(uint32_t), s);
    CWCU_CHECK(cudaMemsetAsync(flag.p, 0, sizeof(uint32_t), s));
    launch("voxel_keygen_kernel", s, 24 * (size_t)n, [&] { voxel_keygen_kernel<<<stream_grid(n, dev), 256, 0, s>>>(in->d_pts, (uint32_t)n, plan.kp, keys.as<uint64_t>(), 0, flag.as<uint32_t>()); });
    CWCU_CHECK(cudaMemcpyAsync(host_keys, keys.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
}

} // namespace cwcu
