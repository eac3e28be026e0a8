// outliers.cu -- statistical outlier removal (exact k-nearest-neighbour statistics) on sm_100a.
//
// Reference semantics (src/cwipc_filters.cpp:181-211 over pcl::StatisticalOutlierRemoval ->
// pcl::search::KdTree -> FLANN KDTreeSingleIndex with L2_Simple<float>; SURVEY.md App. A.5):
//   for every point: the k+1 smallest float distances^2  ((dx*dx + dy*dy) + dz*dz, no FMA) to ALL
//   points (itself included); d_i = (float)( sum_{j=1..k} sqrt((double)d2_j) / k );
//   mean/variance of d in double (squares taken in float); keep iff !(d_i > mean + mul*stddev).
//
// The kd-tree is replaced by a uniform grid in Morton order with a dense table pyramid:
//   knn_keygen_kernel   16 B read + 8 B   key = [Morton(cell) | point index]
//   radix_sort_u64      P x (8+8) B       (shared with downsample)
//   knn_layout_kernel   8+16 B read, 16 B points re-laid out in cell order (every cell, and every aligned
//                                         2^l-cube of cells, is one contiguous range of the array) and the
//                                         dense (begin,end) table of every level, scattered from the
//                                         positions where the Morton prefix changes
//   knn_tile_kernel     one warp per 32 consecutive queries, one lane per query.  Candidates = the cells
//                       within Rc cell pitches of the queries' bounding box, streamed into shared memory
//                       by TMA bulk copies (one per cell range, double buffered); per lane an adaptive
//                       threshold + bitonic merge keeps the k+1 smallest distances in sorted registers.
//                       A query is final when its (k+1)-th distance is within Rc pitches; the rest is queued.
//   knn_second_kernel   (clouds of 256 K points and more) the queued queries of a group that lie side by side are
//                       scanned once more over the cells within their own bound, lanes = queries as above.
//   knn_far_kernel      one warp per queued query: depth-first search of the table pyramid (an implicit
//                       octree), four nearest open nodes per step, pruned by the running (k+1)-th best.  The
//                       search starts at the <= 2x2x2 nodes around the query that cover the ball of a first
//                       bound (farthest corner of the smallest node around its cell that holds k+1 points).
//                       kNeighbors 64..511: no main pass, this kernel alone, lists of 4/8/16 registers per lane.
//   stats_kernel        sum d, sum (float)(d*d) in double, fixed two-level order (deterministic)
//   compact_kernel      keep mask + stable compaction (pointops.cu)
// Exactness never depends on the grid pitch; the pitch only moves work between the two passes.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "device_utils.cuh"
#include "kernels.hpp"
#include "radix_sort.hpp"

namespace cwcu {

namespace {

constexpr int KG_MAX_LEVELS = 14; // levels 0..13 (at most 13 bits per axis)

struct GridParams {
    float gmin[3];
    float inv_h;   // 1 / cell pitch
    float h;       // cell pitch
    float rc;      // cover radius of the main pass, in cell pitches (<= 1)
    float rc_far;  // open queries whose (k+1)-th distance so far is within this many pitches get a second scan (knn_second_kernel)
    int second_min; // ... when at least this many of them share a query group
    int second_max; // ... and the scan lists at most this many candidates per open query
    int gdim[3];   // cells per axis at level 0
    int idxbits;
    int top_level; // level at which the whole grid is one cell
    // per-tile mode: the points of tile rank b live in the cells [b << band_bits, (b << band_bits) + xdim) along x, i.e. band
    // b is exactly the level-`band_bits` node (b, 0, 0): one index, one launch, and no neighbour from another tile.
    // bands == 1 otherwise (band_bits == top_level, xdim == gdim[0]).
    int bands;
    int band_bits;
    int xdim;      // cells along x of ONE band (gdim[0] spans all bands)
    uint32_t table_off[KG_MAX_LEVELS]; // first entry of each level's table (entries are uint2)
};
struct BandLut {
    uint8_t rank[256]; // tile value -> band
};

__host__ __device__ __forceinline__ int level_dim(int gdim, int level) { return ((gdim - 1) >> level) + 1; }

__device__ __forceinline__ uint32_t table_index(const GridParams &gp, int level, uint32_t x, uint32_t y, uint32_t z) {
    const uint32_t dx = (uint32_t)level_dim(gp.gdim[0], level), dy = (uint32_t)level_dim(gp.gdim[1], level);
    return gp.table_off[level] + (z * dy + y) * dx + x;
}

__device__ __forceinline__ uint64_t spread3(uint32_t v) { // bit i -> bit 3i, v < 2^21
    uint64_t x = v & 0x1fffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}
__device__ __forceinline__ uint32_t compact3(uint64_t x) { // inverse of spread3
    x &= 0x1249249249249249ull;
    x = (x | x >> 2) & 0x10c30c30c30c30c3ull;
    x = (x | x >> 4) & 0x100f00f00f00f00full;
    x = (x | x >> 8) & 0x1f0000ff0000ffull;
    x = (x | x >> 16) & 0x1f00000000ffffull;
    x = (x | x >> 32) & 0x1fffffull;
    return (uint32_t)x;
}
__device__ __forceinline__ uint64_t morton3(uint32_t x, uint32_t y, uint32_t z) { return (spread3(x) << 2) | (spread3(y) << 1) | spread3(z); }

// cell coordinate in cell units (float), monotone in the coordinate
__device__ __forceinline__ float cell_u(float x, float gmin, float inv_h) { return __fmul_rn(__fsub_rn(x, gmin), inv_h); }
__device__ __forceinline__ int cell_of(float u, int gdim) { return min(max((int)floorf(u), 0), gdim - 1); }

// FLANN L2_Simple<float>: ((dx*dx) + (dy*dy)) + (dz*dz), every operation rounded to float
__device__ __forceinline__ float dist2(const Point16 &a, const Point16 &b) {
    const float dx = __fsub_rn(a.x, b.x), dy = __fsub_rn(a.y, b.y), dz = __fsub_rn(a.z, b.z);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

__global__ void __launch_bounds__(256) knn_keygen_kernel(const cwipc_point *__restrict__ pts, uint32_t n, const __grid_constant__ GridParams gp, const __grid_constant__ BandLut lut,
                                                          uint64_t *__restrict__ keys, uint2 *__restrict__ table, uint32_t table_words2) {
    // the table pyramid (and the far-query counter behind it) must start empty: cleared here, two launches before
    // knn_layout_kernel fills it, instead of by a separate memset
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < table_words2; i += gridDim.x * blockDim.x) table[i] = make_uint2(0u, 0u);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const Point16 p = ld_point_stream(pts, i);
        uint32_t cx = cell_of(cell_u(p.x, gp.gmin[0], gp.inv_h), gp.xdim);
        const uint32_t cy = cell_of(cell_u(p.y, gp.gmin[1], gp.inv_h), gp.gdim[1]);
        const uint32_t cz = cell_of(cell_u(p.z, gp.gmin[2], gp.inv_h), gp.gdim[2]);
        if (gp.bands > 1) cx += (uint32_t)lut.rank[pt_tile(p)] << gp.band_bits;
        keys[i] = (morton3(cx, cy, cz) << gp.idxbits) | i;
    }
}

// ---- cell-ordered layout + table pyramid in one pass over the sorted keys ------------------------------
// (a) points are re-laid out in cell order; (b) (begin, end) of every node of every level: position i
// starts a new level-l node iff the Morton codes of i-1 and i differ above bit 3l.  The thread at such
// a position writes `begin` of the node it opens and `end` of the node it closes, for every level at
// which it is a boundary; empty nodes keep the (0,0) of the memset.
__global__ void __launch_bounds__(256) knn_layout_kernel(const uint64_t *__restrict__ sorted, uint32_t n, GridParams gp, const cwipc_point *__restrict__ pts,
                                                          cwipc_point *__restrict__ spts, uint2 *__restrict__ table) {
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint64_t word = sorted[i];
        st_point(spts, i, ld_point(pts, (size_t)(word & idxmask)));
        const uint64_t code = word >> gp.idxbits;
        int top; // highest level at which position i opens a node
        uint64_t prev = 0;
        if (i == 0) {
            top = gp.top_level;
        } else {
            prev = sorted[i - 1] >> gp.idxbits;
            const uint64_t diff = code ^ prev;
            top = diff ? min((63 - __clzll((long long)diff)) / 3, gp.top_level) : -1;
        }
        if (top >= 0) {
            const uint32_t cx = compact3(code >> 2), cy = compact3(code >> 1), cz = compact3(code);
            const uint32_t px = compact3(prev >> 2), py = compact3(prev >> 1), pz = compact3(prev);
            for (int l = 0; l <= top; l++) {
                table[table_index(gp, l, cx >> l, cy >> l, cz >> l)].x = i;
                if (i > 0) table[table_index(gp, l, px >> l, py >> l, pz >> l)].y = i;
            }
        }
        if (i == n - 1) {
            const uint32_t cx = compact3(code >> 2), cy = compact3(code >> 1), cz = compact3(code);
            for (int l = 0; l <= gp.top_level; l++) table[table_index(gp, l, cx >> l, cy >> l, cz >> l)].y = n;
        }
    }
}

// ---- TMA 1-D bulk copy + mbarrier (sm_90+/sm_100a PTX; SASS: UBLKCP / SYNCS) -----------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    long long t0 = 0;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
        if (!done) {
            // a bulk copy completes in microseconds; fail loudly (sticky launch error) rather than hang the device
            if (t0 == 0) t0 = clock64();
            else if (clock64() - t0 > 4000000000ll) __trap();
        }
    } while (!done);
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}

// ---- register sorting networks (fully unrolled, static indices only) ---------------------------------
template <int N>
__device__ __forceinline__ void bitonic_sort_asc(float (&a)[N]) {
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int i = 0; i < N; i++) {
                const int l = i ^ j;
                if (l > i) {
                    const float lo = fminf(a[i], a[l]), hi = fmaxf(a[i], a[l]);
                    const bool up = (i & k) == 0;
                    a[i] = up ? lo : hi;
                    a[l] = up ? hi : lo;
                }
            }
        }
    }
}
template <int N>
__device__ __forceinline__ void bitonic_merge_asc(float (&a)[N]) { // bitonic in, ascending out
#pragma unroll
    for (int j = N >> 1; j > 0; j >>= 1) {
#pragma unroll
        for (int i = 0; i < N; i++) {
            const int l = i ^ j;
            if (l > i) {
                const float lo = fminf(a[i], a[l]), hi = fmaxf(a[i], a[l]);
                a[i] = lo;
                a[l] = hi;
            }
        }
    }
}

struct FarEntry {
    uint32_t q;  // index in cell (sorted) order
    float bound; // valid upper bound on the (k+1)-th squared distance, +inf if unknown
};

// ---- main pass: one warp per 32 consecutive (cell-ordered) queries, one lane per query ---------------
// Queries that share a level-1 node (a 2x2x2 block of cells) are processed together: their candidate
// set is every cell within rc pitches of their common bounding box (at most 4x4x4 cells).  Lane 0
// streams the candidates' 16-byte records into a double-buffered shared-memory ring with TMA bulk
// copies (one per contiguous cell range); every lane then scans the same records as broadcast 128-bit
// shared loads.  Per lane, distances below the running (k+1)-th best are parked in a shared-memory
// column and merged into a sorted register array 16 at a time by bitonic networks, so the
// per-candidate cost is a distance, a compare and a predicated store.
constexpr int KT_WARPS = 2;  // small blocks: a block's registers and shared memory stay allocated until its slowest warp is done
constexpr int KT_THREADS = KT_WARPS * 32;
constexpr int KT_CH = 128;     // candidates per stage
constexpr int KT_STAGES = 2;
constexpr int KT_GROUP_LEVEL = 2; // queries are grouped by level-1 node (2x2x2 cells): ~one warp of queries per group on surface data, and a
                                  // candidate box of 4x4x4 cells instead of the 6x6x6 a level-2 group needs (3.4x fewer candidates per query)
constexpr int KT_GROUP_SPAN = 1 << KT_GROUP_LEVEL;
constexpr int KT_MAXR = (KT_GROUP_SPAN + 2) * (KT_GROUP_SPAN + 2) * (KT_GROUP_SPAN + 2); // cells of the largest candidate box (rc <= 1 on both sides)
constexpr int KT_BUF = 16;     // parked distances per lane
constexpr int KT_BLOCKS_PER_SM = 12; // register budget 85/thread (24 warps per SM): more resident warps hide the scan's latency

struct __align__(128) KnnWarpSmem {
    Point16 cand[KT_STAGES][KT_CH]; // 4096 B
    float buf[KT_BUF][32];          // 2048 B
    uint2 ranges[KT_MAXR];          // 512 B
    uint64_t mbar[KT_STAGES];
    float pbox[7];                  // knn_second_kernel: box and radius (cell units) of the group being listed
    uint32_t xoff;                  //   first cell (x) of the group's band (per-tile mode)
    uint32_t cursor;                //   next cell of the box to be listed
};

__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(FULL_MASK, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL_MASK, v, o));
    return v;
}

template <int KCAP>
__global__ void __launch_bounds__(KT_THREADS, KT_BLOCKS_PER_SM) knn_tile_kernel(const cwipc_point *__restrict__ spts, const uint64_t *__restrict__ sorted, uint32_t n, GridParams gp, int kk, int k,
                                                               const uint2 *__restrict__ table, float *__restrict__ dist_out, float *__restrict__ kth_out, uint32_t nquery,
                                                               FarEntry *__restrict__ far_list, uint32_t *__restrict__ far_count) {
    extern __shared__ __align__(128) unsigned char knn_smem_raw[];
    constexpr int B = KCAP < KT_BUF ? KCAP : KT_BUF;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    KnnWarpSmem &ws = reinterpret_cast<KnnWarpSmem *>(knn_smem_raw)[warp];
    const unsigned lt = lanemask_lt();
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < KT_STAGES; st++) mbar_init(&ws.mbar[st], 1);
        mbar_fence_init();
    }
    __syncwarp();
    uint32_t phase_bits = 0; // bit st: parity the next wait on stage st must see

    const uint32_t warps_total = (gridDim.x * blockDim.x) >> 5;
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    const int extra = KCAP - kk; // leading slots pinned at -inf so that best[KCAP-1] is the kk-th smallest
    const uint32_t nitems = (n + 31u) >> 5;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);
    const float rc = gp.rc;
    // every point within `reach` of a query is inside the scanned cells (0.01 pitch covers the rounding of cell_u)
    const float reach = (rc - 0.01f) * gp.h;
    const float reach2 = reach * reach * 0.999999f;

    for (uint32_t item = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; item < nitems; item += warps_total) {
        const uint32_t qi = item * 32u + lane;
        const uint32_t qs = qi < n ? qi : n - 1u;
        const uint64_t word = sorted[qs];
        // only the first `nquery` points (original order) are queries; the rest are candidates only (halo points)
        const bool active = qi < n && (uint32_t)(word & idxmask) < nquery;
        const uint64_t code = word >> gp.idxbits;
        const Point16 q = spts16[qs];
        const float ux = cell_u(q.x, gp.gmin[0], gp.inv_h), uy = cell_u(q.y, gp.gmin[1], gp.inv_h), uz = cell_u(q.z, gp.gmin[2], gp.inv_h);
        const uint32_t band = gp.bands > 1 ? (compact3(code >> 2) >> gp.band_bits) : 0u; // per-tile mode: the query's tile rank

        // groups: runs of lanes inside one level-KT_GROUP_LEVEL node (codes are non-decreasing along the lanes)
        const uint64_t node2 = code >> (3 * KT_GROUP_LEVEL);
        const uint64_t prev_node2 = __shfl_up_sync(FULL_MASK, node2, 1);
        const unsigned heads = __ballot_sync(FULL_MASK, (lane == 0) || (node2 != prev_node2));
        const int m = __popc(heads);
        const int ord = __popc(heads & (lt | (1u << lane))) - 1;

        for (int g = 0; g < m; g++) {
            const bool live = active && ord == g;

            // ---- bounding box of the group's queries (cell units) and the cells within rc of it ----
            const float lox = warp_min(live ? ux : INFINITY), loy = warp_min(live ? uy : INFINITY), loz = warp_min(live ? uz : INFINITY);
            const float hix = warp_max(live ? ux : -INFINITY), hiy = warp_max(live ? uy : -INFINITY), hiz = warp_max(live ? uz : -INFINITY);
            uint32_t nr = 0, total = 0;
            // a group never spans two bands (band_bits >= KT_GROUP_LEVEL): its candidates are the cells of its own band only
            const uint32_t xoff = gp.bands > 1 ? (__reduce_max_sync(FULL_MASK, live ? band : 0u) << gp.band_bits) : 0u;
            if (lox <= hix) { // the group has at least one live query (always, except for padding lanes)
                const int cx0 = max((int)floorf(lox - rc), 0), cx1 = min((int)floorf(hix + rc), gp.xdim - 1);
                const int cy0 = max((int)floorf(loy - rc), 0), cy1 = min((int)floorf(hiy + rc), gp.gdim[1] - 1);
                const int cz0 = max((int)floorf(loz - rc), 0), cz1 = min((int)floorf(hiz + rc), gp.gdim[2] - 1);
                const int nbx = cx1 - cx0 + 1, nby = cy1 - cy0 + 1, nbz = cz1 - cz0 + 1;
                const int nb = nbx * nby * nbz; // <= KT_MAXR: the queries span at most KT_GROUP_SPAN cells per axis and rc <= 1
                const float rc2 = rc * rc;
                // cells that overlap the queries' box first: their points tighten the running bound early,
                // so most candidates of the surrounding shell fail the threshold test without being parked
                for (int shell = 0; shell < 2; shell++) {
                    for (int t0 = 0; t0 < nb; t0 += 32) {
                        const int t = t0 + (int)lane;
                        uint2 r = make_uint2(0u, 0u);
                        if (t < nb) {
                            const int ix = cx0 + t % nbx, iy = cy0 + (t / nbx) % nby, iz = cz0 + t / (nbx * nby);
                            const float dx = fmaxf(fmaxf((float)ix - hix, lox - (float)(ix + 1)), 0.f);
                            const float dy = fmaxf(fmaxf((float)iy - hiy, loy - (float)(iy + 1)), 0.f);
                            const float dz = fmaxf(fmaxf((float)iz - hiz, loz - (float)(iz + 1)), 0.f);
                            const float dd = dx * dx + dy * dy + dz * dz;
                            if (shell == 0 ? dd == 0.f : (dd > 0.f && dd <= rc2)) r = table[table_index(gp, 0, (uint32_t)ix + xoff, (uint32_t)iy, (uint32_t)iz)];
                        }
                        const unsigned has = __ballot_sync(FULL_MASK, r.y > r.x);
                        if (r.y > r.x) ws.ranges[nr + __popc(has & lt)] = r;
                        nr += __popc(has);
                        total += warp_sum(r.y - r.x);
                    }
                }
            }
            __syncwarp();

            // ---- stream the candidates through the ring, keep the kk smallest distances per lane ----
            float best[KCAP];
#pragma unroll
            for (int j = 0; j < KCAP; j++) best[j] = (j < extra) ? -INFINITY : INFINITY;
            float tau = live ? INFINITY : -INFINITY;
            uint32_t bcnt = 0;

            const uint32_t nchunks = (total + KT_CH - 1) / KT_CH;
            uint32_t ri = 0, roff = 0; // producer cursor (lane 0)
            auto fill = [&](int st, uint32_t chunk) {
                const uint32_t cnt = min((uint32_t)KT_CH, total - chunk * KT_CH);
                mbar_arrive_expect_tx(&ws.mbar[st], cnt * 16u);
                uint32_t filled = 0;
                while (filled < cnt) {
                    const uint2 r = ws.ranges[ri];
                    const uint32_t len = r.y - r.x;
                    const uint32_t take = min(len - roff, cnt - filled);
                    bulk_g2s(&ws.cand[st][filled], spts16 + r.x + roff, take * 16u, &ws.mbar[st]);
                    filled += take;
                    roff += take;
                    if (roff == len) {
                        ri++;
                        roff = 0;
                    }
                }
            };
            if (lane == 0 && nchunks > 0) {
                fill(0, 0);
                if (nchunks > 1) fill(1, 1);
            }
            for (uint32_t chunk = 0; chunk < nchunks; chunk++) {
                const int st = (int)(chunk & 1u);
                mbar_wait(&ws.mbar[st], (phase_bits >> st) & 1u);
                phase_bits ^= 1u << st;
                const uint32_t cnt = min((uint32_t)KT_CH, total - chunk * KT_CH);
                const bool last_chunk = chunk + 1 == nchunks;
                for (uint32_t c = 0; c < cnt; c += 4) {
                    if (c + 4 <= cnt) { // (all but the last step of the last chunk: no per-candidate bound check)
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            const Point16 cand = ws.cand[st][c + u]; // same address in every lane: one broadcast load
                            const float d2 = dist2(q, cand);
                            if (d2 < tau) {
                                ws.buf[bcnt][lane] = d2;
                                bcnt++;
                            }
                        }
                    } else {
                        for (uint32_t u = c; u < cnt; u++) {
                            const float d2 = dist2(q, ws.cand[st][u]);
                            if (d2 < tau) {
                                ws.buf[bcnt][lane] = d2;
                                bcnt++;
                            }
                        }
                    }
                    const bool finish = last_chunk && c + 4 >= cnt;
                    if (finish || __any_sync(FULL_MASK, bcnt > (uint32_t)(B - 4))) {
                        // merge the parked distances: sort them, keep the KCAP smallest of (best U parked), re-sort
                        float s[B];
#pragma unroll
                        for (int j = 0; j < B; j++) s[j] = ((uint32_t)j < bcnt) ? ws.buf[j][lane] : INFINITY;
                        bitonic_sort_asc<B>(s);
#pragma unroll
                        for (int j = 0; j < B; j++) best[KCAP - 1 - j] = fminf(best[KCAP - 1 - j], s[j]);
                        bitonic_merge_asc<KCAP>(best);
                        bcnt = 0;
                        if (live) tau = best[KCAP - 1];
                    }
                }
                __syncwarp();
                if (lane == 0 && chunk + 2 < nchunks) fill(st, chunk + 2);
            }

            const float worst = best[KCAP - 1];
            const bool done = live && (gp.top_level == 0 || worst <= reach2);
            // the group's open queries are queued side by side (one atomic per group): knn_second_kernel finds them together again
            const unsigned fm = __ballot_sync(FULL_MASK, live && !done);
            if (fm) {
                uint32_t slot = 0;
                if (lane == (unsigned)(__ffs(fm) - 1)) slot = atomicAdd(far_count, (uint32_t)__popc(fm));
                slot = __shfl_sync(FULL_MASK, slot, __ffs(fm) - 1);
                if (live && !done) {
                    FarEntry e;
                    e.q = qi;
                    e.bound = worst;
                    far_list[slot + __popc(fm & lt)] = e;
                }
            }
            if (!done) continue;
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < KCAP; j++)
                if (j > extra) sum += sqrt((double)best[j]); // j == extra is the query itself (distance 0)
            dist_out[(size_t)(word & idxmask)] = (float)(sum / (double)k);
            if (kth_out) kth_out[(size_t)(word & idxmask)] = worst;
        }
        __syncwarp();
    }
}


// ---- second scan: the open queries whose neighbours are known to lie within rc_far pitches --------------
// An open query leaves the main pass with a valid bound on its (k+1)-th distance.  Where many queries are open (raw,
// noisy clouds: a thick shell rather than a surface) they sit side by side in the queue, group by group, and scanning
// the cells within the bound of their common box once more -- 32 queries per candidate load, as in the main pass --
// costs a fraction of one tree search per query.  Same lanes-are-queries scheme as knn_tile_kernel; the box can be
// larger than the range list, which is then filled and scanned piece by piece.  Queries whose bound exceeds rc_far
// pitches (isolated points) move on to far_list2 for knn_far_kernel.
template <int KCAP>
__global__ void __launch_bounds__(KT_THREADS, KT_BLOCKS_PER_SM) knn_second_kernel(const cwipc_point *__restrict__ spts, const uint64_t *__restrict__ sorted, GridParams gp, int kk, int k,
                                                                 const uint2 *__restrict__ table, float *__restrict__ dist_out, float *__restrict__ kth_out,
                                                                 const FarEntry *__restrict__ far_list, const uint32_t *__restrict__ far_count, uint32_t second_from,
                                                                 FarEntry *__restrict__ far_list2, uint32_t *__restrict__ far_count2) {
    extern __shared__ __align__(128) unsigned char knn_smem_raw[];
    constexpr int B = KCAP < KT_BUF ? KCAP : KT_BUF;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    KnnWarpSmem &ws = reinterpret_cast<KnnWarpSmem *>(knn_smem_raw)[warp];
    const unsigned lt = lanemask_lt();
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < KT_STAGES; st++) mbar_init(&ws.mbar[st], 1);
        mbar_fence_init();
    }
    __syncwarp();
    uint32_t phase_bits = 0;

    const uint32_t warps_total = (gridDim.x * blockDim.x) >> 5;
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    const int extra = KCAP - kk;
    const uint32_t nent = *far_count;
    // Few open queries are isolated points, which the tree search serves best; many (one query in eight or more: a dense,
    // noisy shell rather than a surface) are each other's neighbours, and that is what this scan is for.
    if (nent < second_from) return;
    const uint32_t nitems = (nent + 31u) >> 5;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);

    for (uint32_t item = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; item < nitems; item += warps_total) {
        const uint32_t ei = item * 32u + lane;
        const bool valid = ei < nent;
        const FarEntry ent = far_list[valid ? ei : nent - 1u];
        const uint64_t word = sorted[ent.q];
        const uint64_t code = word >> gp.idxbits;
        const Point16 q = spts16[ent.q];
        // radius in cell units that holds every neighbour of the query (0.02 pitch covers the rounding of cell_u)
        const float need = sqrtf(ent.bound) * gp.inv_h * 1.000001f + 0.02f;
        // groups: runs of lanes inside one level-KT_GROUP_LEVEL node (what the main pass queued together)
        const uint64_t node2 = code >> (3 * KT_GROUP_LEVEL);
        bool active = valid && need <= gp.rc_far; // (a bound of +inf or NaN is not)
        {
            // a scan serves every open query of the group at once; for a few lonely ones the tree search is cheaper
            const unsigned peers = __match_any_sync(FULL_MASK, node2) & __ballot_sync(FULL_MASK, active);
            active = active && __popc(peers) >= gp.second_min;
        }
        {
            const unsigned fm = __ballot_sync(FULL_MASK, valid && !active);
            if (fm) {
                uint32_t slot = 0;
                if (lane == (unsigned)(__ffs(fm) - 1)) slot = atomicAdd(far_count2, (uint32_t)__popc(fm));
                slot = __shfl_sync(FULL_MASK, slot, __ffs(fm) - 1);
                if (valid && !active) far_list2[slot + __popc(fm & lt)] = ent;
            }
        }
        if (!__any_sync(FULL_MASK, active)) continue;

        const uint64_t prev_node2 = __shfl_up_sync(FULL_MASK, node2, 1);
        const unsigned heads = __ballot_sync(FULL_MASK, (lane == 0) || (node2 != prev_node2));
        const int m = __popc(heads);
        const int ord = __popc(heads & (lt | (1u << lane))) - 1;

        for (int g = 0; g < m; g++) {
            const bool live = active && ord == g;
            if (!__any_sync(FULL_MASK, live)) continue;
            {
                const float ux = cell_u(q.x, gp.gmin[0], gp.inv_h), uy = cell_u(q.y, gp.gmin[1], gp.inv_h), uz = cell_u(q.z, gp.gmin[2], gp.inv_h);
                const float lx = warp_min(live ? ux : INFINITY), ly = warp_min(live ? uy : INFINITY), lz = warp_min(live ? uz : INFINITY);
                const float hx = warp_max(live ? ux : -INFINITY), hy = warp_max(live ? uy : -INFINITY), hz = warp_max(live ? uz : -INFINITY);
                const float pr = warp_max(live ? need : 0.f);
                const uint32_t band = gp.bands > 1 ? __reduce_max_sync(FULL_MASK, live ? (compact3(code >> 2) >> gp.band_bits) : 0u) : 0u;
                if (lane == 0) {
                    ws.pbox[0] = lx; ws.pbox[1] = ly; ws.pbox[2] = lz;
                    ws.pbox[3] = hx; ws.pbox[4] = hy; ws.pbox[5] = hz;
                    ws.pbox[6] = pr;
                    ws.xoff = band << gp.band_bits;
                    ws.cursor = 0u;
                }
            }
            __syncwarp();

            float best[KCAP];
#pragma unroll
            for (int j = 0; j < KCAP; j++) best[j] = (j < extra) ? -INFINITY : INFINITY;
            // everything up to the bound (inclusive) is collected: at least kk points are
            float tau = live ? __uint_as_float(__float_as_uint(ent.bound) + 1u) : -INFINITY;
            uint32_t bcnt = 0;
            bool first = true, rejected = false;

            while (true) {
                // ---- list cell ranges from the cursor on, until the list is full or the box is complete ----
                uint32_t total = 0;
                bool box_done;
                {
                    const float plox = ws.pbox[0], ploy = ws.pbox[1], ploz = ws.pbox[2], phix = ws.pbox[3], phiy = ws.pbox[4], phiz = ws.pbox[5], prad = ws.pbox[6];
                    const uint32_t xoff = ws.xoff;
                    uint32_t nr = 0, cursor = ws.cursor;
                    const int cx0 = max((int)floorf(plox - prad), 0), cx1 = min((int)floorf(phix + prad), gp.xdim - 1);
                    const int cy0 = max((int)floorf(ploy - prad), 0), cy1 = min((int)floorf(phiy + prad), gp.gdim[1] - 1);
                    const int cz0 = max((int)floorf(ploz - prad), 0), cz1 = min((int)floorf(phiz + prad), gp.gdim[2] - 1);
                    const int nbx = cx1 - cx0 + 1, nby = cy1 - cy0 + 1, nbz = cz1 - cz0 + 1;
                    const uint32_t nb = (uint32_t)max(nbx * nby * nbz, 0);
                    const float prad2 = prad * prad;
                    while (cursor < nb) {
                        const int t = (int)(cursor + lane);
                        uint2 r = make_uint2(0u, 0u);
                        if (t < (int)nb) {
                            const int ix = cx0 + t % nbx, iy = cy0 + (t / nbx) % nby, iz = cz0 + t / (nbx * nby);
                            const float dx = fmaxf(fmaxf((float)ix - phix, plox - (float)(ix + 1)), 0.f);
                            const float dy = fmaxf(fmaxf((float)iy - phiy, ploy - (float)(iy + 1)), 0.f);
                            const float dz = fmaxf(fmaxf((float)iz - phiz, ploz - (float)(iz + 1)), 0.f);
                            if (dx * dx + dy * dy + dz * dz <= prad2) r = table[table_index(gp, 0, (uint32_t)ix + xoff, (uint32_t)iy, (uint32_t)iz)];
                        }
                        const unsigned has = __ballot_sync(FULL_MASK, r.y > r.x);
                        if (r.y > r.x) ws.ranges[nr + __popc(has & lt)] = r;
                        nr += __popc(has);
                        total += warp_sum(r.y - r.x);
                        cursor += 32u;
                        if (nr > (uint32_t)(KT_MAXR - 32)) break; // the list is full: scan what it holds, then go on
                    }
                    box_done = cursor >= nb;
                    __syncwarp();
                    if (lane == 0) ws.cursor = cursor;
                }
                __syncwarp();
                if (first) {
                    // The scan costs `total` distance evaluations per lane whatever the number of open queries it serves; the
                    // tree search costs a few thousand instructions per query.  Scattered open queries (isolated points far
                    // from the surface: a large box, few of them) are left to the tree search.
                    first = false;
                    const uint32_t nlive = (uint32_t)__popc(__ballot_sync(FULL_MASK, live));
                    if (!box_done || total > nlive * (uint32_t)gp.second_max) {
                        rejected = true;
                        break;
                    }
                }

                // ---- stream the listed candidates through the ring (as knn_tile_kernel does) ----
                const uint32_t nchunks = (total + KT_CH - 1) / KT_CH;
                uint32_t ri = 0, roff = 0; // producer cursor (lane 0)
                auto fill = [&](int st, uint32_t chunk) {
                    const uint32_t cnt = min((uint32_t)KT_CH, total - chunk * KT_CH);
                    mbar_arrive_expect_tx(&ws.mbar[st], cnt * 16u);
                    uint32_t filled = 0;
                    while (filled < cnt) {
                        const uint2 r = ws.ranges[ri];
                        const uint32_t len = r.y - r.x;
                        const uint32_t take = min(len - roff, cnt - filled);
                        bulk_g2s(&ws.cand[st][filled], spts16 + r.x + roff, take * 16u, &ws.mbar[st]);
                        filled += take;
                        roff += take;
                        if (roff == len) {
                            ri++;
                            roff = 0;
                        }
                    }
                };
                if (lane == 0 && nchunks > 0) {
                    fill(0, 0);
                    if (nchunks > 1) fill(1, 1);
                }
                for (uint32_t chunk = 0; chunk < nchunks; chunk++) {
                    const int st = (int)(chunk & 1u);
                    mbar_wait(&ws.mbar[st], (phase_bits >> st) & 1u);
                    phase_bits ^= 1u << st;
                    const uint32_t cnt = min((uint32_t)KT_CH, total - chunk * KT_CH);
                    const bool last_chunk = chunk + 1 == nchunks;
                    for (uint32_t c = 0; c < cnt; c += 4) {
                        if (c + 4 <= cnt) {
#pragma unroll
                            for (int u = 0; u < 4; u++) {
                                const Point16 cand = ws.cand[st][c + u];
                                const float d2 = dist2(q, cand);
                                if (d2 < tau) {
                                    ws.buf[bcnt][lane] = d2;
                                    bcnt++;
                                }
                            }
                        } else {
                            for (uint32_t u = c; u < cnt; u++) {
                                const float d2 = dist2(q, ws.cand[st][u]);
                                if (d2 < tau) {
                                    ws.buf[bcnt][lane] = d2;
                                    bcnt++;
                                }
                            }
                        }
                        const bool finish = last_chunk && c + 4 >= cnt;
                        if (finish || __any_sync(FULL_MASK, bcnt > (uint32_t)(B - 4))) {
                            float s[B];
#pragma unroll
                            for (int j = 0; j < B; j++) s[j] = ((uint32_t)j < bcnt) ? ws.buf[j][lane] : INFINITY;
                            bitonic_sort_asc<B>(s);
#pragma unroll
                            for (int j = 0; j < B; j++) best[KCAP - 1 - j] = fminf(best[KCAP - 1 - j], s[j]);
                            bitonic_merge_asc<KCAP>(best);
                            bcnt = 0;
                            // the bound stays in force until kk distances are in (best[KCAP-1] is +inf until then)
                            if (live) tau = fminf(tau, best[KCAP - 1]);
                        }
                    }
                    __syncwarp();
                    if (lane == 0 && chunk + 2 < nchunks) fill(st, chunk + 2);
                }
                if (box_done) break;
            }
            if (rejected) {
                const unsigned fm = __ballot_sync(FULL_MASK, live);
                uint32_t slot = 0;
                if (lane == (unsigned)(__ffs(fm) - 1)) slot = atomicAdd(far_count2, (uint32_t)__popc(fm));
                slot = __shfl_sync(FULL_MASK, slot, __ffs(fm) - 1);
                if (live) far_list2[slot + __popc(fm & lt)] = ent;
                continue;
            }

            if (!live) continue;
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < KCAP; j++)
                if (j > extra) sum += sqrt((double)best[j]);
            dist_out[(size_t)(word & idxmask)] = (float)(sum / (double)k);
            if (kth_out) kth_out[(size_t)(word & idxmask)] = best[KCAP - 1];
        }
        __syncwarp();
    }
}

// ---- far pass: queries the main pass could not prove exact, one warp each -----------------------------
// Depth-first search of the table pyramid (an implicit octree: a node of level l is one contiguous
// run of points), nearest child first, pruned by the running (k+1)-th best.  The best list lives
// across the lanes (element e in lane e%32, register e/32) and absorbs 32 new distances at a time
// through warp-shuffle bitonic networks.
constexpr int KF_WARPS = 2;
constexpr int KF_THREADS = KF_WARPS * 32;
constexpr int KNN_MAX_K = 511; // k + 1 distances in at most 16 registers per lane of the tree search

constexpr int KF_STACK = 416; // four nodes are expanded per step: <= 28 * top_level + 32 open nodes with top_level <= 13
static_assert(KF_STACK * 20 >= 16 * 32 * 8 && (KF_STACK * 20) % 16 == 0, "the stack doubles as the buffer of square roots");

struct FarNode { // 20 B (the stack of one warp, KF_STACK of them, also holds the 32 * KPL <= 512 square roots of a finished search)
    uint32_t pb, pe;  // point range
    uint32_t xy;      // node coordinates at its level: x | y << 16
    uint32_t zl;      // z | level << 16
    float mind2;
};

__device__ __forceinline__ float warp_bitonic_sort32(float x, unsigned lane) { // ascending along the lanes
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const float y = __shfl_xor_sync(FULL_MASK, x, j);
            const bool up = (lane & (unsigned)k) == 0u; // k == 32: always ascending
            const bool lower = (lane & (unsigned)j) == 0u;
            x = (lower == up) ? fminf(x, y) : fmaxf(x, y);
        }
    }
    return x;
}
__device__ __forceinline__ float warp_bitonic_merge32(float x, unsigned lane) { // bitonic in, ascending out
#pragma unroll
    for (int j = 16; j > 0; j >>= 1) {
        const float y = __shfl_xor_sync(FULL_MASK, x, j);
        x = ((lane & (unsigned)j) == 0u) ? fminf(x, y) : fmaxf(x, y);
    }
    return x;
}

// The kk nearest squared distances from q to the cloud, ascending along (lane, register): element e
// lives in lane e % 32, register e / 32.  Called by all 32 lanes of a warp with the same arguments.
// One batch of up to 32 candidate distances into the lane-distributed sorted list (element e in lane e % 32,
// register e / 32); returns the new kk-th smallest.
// element e of a lane-distributed list (lane e % 32, register e / 32), e the same in every lane
template <int KPL, class T>
__device__ __forceinline__ T list_element(const T (&v)[KPL], int e) {
    T x = v[0];
#pragma unroll
    for (int j = 1; j < KPL; j++)
        if ((e >> 5) == j) x = v[j];
    return __shfl_sync(FULL_MASK, x, e & 31);
}

template <int KPL>
__device__ __forceinline__ float list_absorb(float (&v)[KPL], float d2, bool pass, unsigned pm, int kk, unsigned lane) {
    if (KPL == 1 && __popc(pm) <= 6) {
        // few survivors: insert them one by one
        while (pm) {
            const int src = __ffs(pm) - 1;
            pm &= pm - 1;
            const float x = __shfl_sync(FULL_MASK, d2, src);
            const float up = __shfl_up_sync(FULL_MASK, v[0], 1);
            if (v[0] > x) v[0] = (lane == 0) ? x : fmaxf(up, x);
        }
    } else {
        float b = warp_bitonic_sort32(pass ? d2 : INFINITY, lane);
        if (KPL == 1) {
            const float r = __shfl_sync(FULL_MASK, b, 31 - (int)lane);
            v[0] = warp_bitonic_merge32(fminf(v[0], r), lane);
        } else if (KPL == 2) {
            const float r = __shfl_sync(FULL_MASK, b, 31 - (int)lane);
            v[KPL - 1] = fminf(v[KPL - 1], r);
            const float lo = fminf(v[0], v[KPL - 1]), hi = fmaxf(v[0], v[KPL - 1]);
            v[0] = warp_bitonic_merge32(lo, lane);
            v[KPL - 1] = warp_bitonic_merge32(hi, lane);
        } else {
            // long lists (kNeighbors > 63): the sorted batch is merged into the registers front to back, each step keeping the 32
            // smallest of (register, carry) and carrying the 32 largest on; registers that lie below the whole carry are skipped
#pragma unroll
            for (int j = 0; j < KPL; j++) {
                if (__shfl_sync(FULL_MASK, b, 0) >= __shfl_sync(FULL_MASK, v[j], 31)) continue;
                const float r = __shfl_sync(FULL_MASK, b, 31 - (int)lane);
                const float lo = fminf(v[j], r), hi = fmaxf(v[j], r);
                v[j] = warp_bitonic_merge32(lo, lane);
                b = warp_bitonic_merge32(hi, lane);
            }
        }
    }
    return list_element<KPL>(v, kk - 1);
}

// Where a search starts: the root (level < 0), or the (at most) 2x2x2 nodes of `level` from (x, y, z) on, which are known to
// hold every point within sqrt(limit) of the query.
struct FarStart {
    int level;
    uint32_t x, y, z;
};

// The kk nearest squared distances from q to the cloud, ascending along (lane, register): element e
// lives in lane e % 32, register e / 32.  Called by all 32 lanes of a warp with the same arguments.
// Every iteration takes the (up to) four nearest open nodes off the stack: the small ones are scanned, the
// others are expanded together, eight lanes per node, one child per lane.
template <int KPL>
__device__ __forceinline__ void dfs_knn(const Point16 q, float limit, const Point16 *__restrict__ spts16, uint32_t n, const GridParams &gp, int kk,
                                        const uint2 *__restrict__ table, uint32_t leaf_points, FarNode *stack, float (&v)[KPL], uint32_t band = 0u,
                                        const FarStart start = FarStart{-1, 0u, 0u, 0u}) {
    const unsigned lane = lane_id();
    const float slack = 0.01f * gp.h;
#pragma unroll
    for (int j = 0; j < KPL; j++) v[j] = INFINITY;
    float tau = INFINITY; // current kk-th smallest
    int sp = 0;

    // Children of open nodes (one per lane) -> stack, nearest on top.  A lane that `want`s its node (cl, chx, chy, chz) reads
    // the node's point range, drops it when empty or farther than `thr`, and the survivors are ranked by (distance, lane).
    auto push_nodes = [&](bool want, int cl, uint32_t chx, uint32_t chy, uint32_t chz, float thr) {
        uint2 r = make_uint2(0u, 0u);
        float mind2 = INFINITY;
        bool admit = false;
        if (want && chx < (uint32_t)level_dim(gp.gdim[0], cl) && chy < (uint32_t)level_dim(gp.gdim[1], cl) && chz < (uint32_t)level_dim(gp.gdim[2], cl) &&
            (gp.bands <= 1 || (chx >> (gp.band_bits - cl)) == band)) { // (children of a band's node stay inside the band; start nodes might not)
            r = table[table_index(gp, cl, chx, chy, chz)];
            if (r.y > r.x) {
                const float pitch = ldexpf(gp.h, cl);
                const uint32_t lx = chx - (band << (gp.band_bits - cl)); // x within the band (band == 0 outside the per-tile mode)
                const float lo[3] = {gp.gmin[0] + (float)lx * pitch, gp.gmin[1] + (float)chy * pitch, gp.gmin[2] + (float)chz * pitch};
                const float qq[3] = {q.x, q.y, q.z};
                mind2 = 0.f;
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    const float d = fmaxf(fmaxf(lo[a] - qq[a], qq[a] - (lo[a] + pitch)) - slack, 0.f);
                    mind2 += d * d;
                }
                admit = mind2 * 0.9999f <= thr;
            }
        }
        const unsigned adm = __ballot_sync(FULL_MASK, admit);
        if (adm == 0u) return;
        const int nadm = __popc(adm);
        FarNode ch;
        ch.pb = r.x; ch.pe = r.y; ch.xy = chx | (chy << 16); ch.zl = chz | ((uint32_t)cl << 16); ch.mind2 = mind2;
        if (nadm <= 12) {
            // few survivors (the usual case once a bound is known): every lane counts the admitted nodes in front of its own
            const uint32_t mine = __float_as_uint(mind2); // non-negative floats: the bit patterns order like the values
            int rank = 0;
            for (unsigned m = adm; m; m &= m - 1u) {
                const int src = __ffs(m) - 1;
                const uint32_t other = __shfl_sync(FULL_MASK, mine, src);
                rank += (other < mine || (other == mine && src < (int)lane)) ? 1 : 0;
            }
            if (admit) stack[sp + nadm - 1 - rank] = ch; // farthest deepest, nearest on top
        } else {
            // many: a 32-lane bitonic sort of (distance, lane) keys
            unsigned long long key = admit ? (((unsigned long long)__float_as_uint(mind2) << 32) | lane) : ~0ull;
#pragma unroll
            for (int k2 = 2; k2 <= 32; k2 <<= 1) {
#pragma unroll
                for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
                    const unsigned long long other = __shfl_xor_sync(FULL_MASK, key, j2);
                    const bool up = (lane & (unsigned)k2) == 0u;
                    const bool lower = (lane & (unsigned)j2) == 0u;
                    key = (lower == up) ? (key < other ? key : other) : (key < other ? other : key);
                }
            }
            // lane i now holds the i-th nearest admitted node's (distance, source lane); fetch that node and store it
            const int src = (int)(key & 31u);
            FarNode sorted_ch;
            sorted_ch.pb = __shfl_sync(FULL_MASK, ch.pb, src);
            sorted_ch.pe = __shfl_sync(FULL_MASK, ch.pe, src);
            sorted_ch.xy = __shfl_sync(FULL_MASK, ch.xy, src);
            sorted_ch.zl = __shfl_sync(FULL_MASK, ch.zl, src);
            sorted_ch.mind2 = __shfl_sync(FULL_MASK, ch.mind2, src);
            if ((int)lane < nadm) stack[sp + nadm - 1 - (int)lane] = sorted_ch;
        }
        sp += nadm;
    };

    bool from_start = start.level >= 0;
    if (!from_start) {
        if (lane == 0) {
            FarNode root;
            root.pb = 0; root.pe = n; root.xy = 0; root.zl = (uint32_t)gp.top_level << 16; root.mind2 = 0.f;
            if (gp.bands > 1) { // per-tile mode: the search never leaves the query's band, the level-band_bits node (band, 0, 0)
                const uint2 r = table[table_index(gp, gp.band_bits, band, 0u, 0u)];
                root.pb = r.x; root.pe = r.y; root.xy = band; root.zl = (uint32_t)gp.band_bits << 16;
            }
            stack[0] = root;
        }
        sp = 1;
    }
    __syncwarp();
    const int group = (int)(lane >> 3);
    while (from_start || sp > 0) {
        if (from_start) { // the first step lists the start nodes instead of the children of open nodes
            from_start = false;
            push_nodes(lane < 8u, start.level, start.x + ((lane >> 2) & 1u), start.y + ((lane >> 1) & 1u), start.z + (lane & 1u), limit);
            __syncwarp();
            continue;
        }
        const int take = min(sp, 4);
        // lane group g looks at the g-th node from the top (g = 0 is the nearest)
        const FarNode node = stack[sp - 1 - min(group, take - 1)];
        const bool have = group < take;
        const uint32_t node_x = node.xy & 0xffffu, node_y = node.xy >> 16, node_z = node.zl & 0xffffu;
        const int node_level = (int)(node.zl >> 16);
        sp -= take;
        __syncwarp();
        // Sparse neighbourhoods (an isolated point among other isolated points: one or two points per node): when none of the
        // nodes taken holds more than eight points they are scanned together, eight lanes per node, in one pass.
        if (__all_sync(FULL_MASK, !have || node.pe - node.pb <= 8u)) {
            const uint32_t c = node.pb + (lane & 7u);
            float d2 = INFINITY;
            if (have && c < node.pe && !(node.mind2 * 0.9999f > fminf(tau, limit))) d2 = dist2(q, spts16[c]);
            const bool pass = d2 < tau && d2 <= limit;
            const unsigned pm = __ballot_sync(FULL_MASK, pass);
            if (pm) tau = list_absorb<KPL>(v, d2, pass, pm, kk, lane);
            continue;
        }
        // small nodes first (nearest first): scanning them tightens the bound for the expansions below
        const bool is_leaf = node_level == 0 || node.pe - node.pb <= leaf_points;
        // the groups' first lanes (0, 8, 16, 24) vote for their nodes: only nodes that are scanned cost anything here
        unsigned todo = __ballot_sync(FULL_MASK, have && is_leaf && !(node.mind2 * 0.9999f > fminf(tau, limit))) & 0x01010101u;
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1u;
            const uint32_t pb = __shfl_sync(FULL_MASK, node.pb, src), pe = __shfl_sync(FULL_MASK, node.pe, src);
            const float nm = __shfl_sync(FULL_MASK, node.mind2, src);
            if (nm * 0.9999f > fminf(tau, limit)) continue; // (the bound may have dropped since the vote)
            for (uint32_t base = pb; base < pe; base += 32) {
                const uint32_t c = base + lane;
                float d2 = INFINITY;
                if (c < pe) d2 = dist2(q, spts16[c]);
                const bool pass = d2 < tau && d2 <= limit;
                const unsigned pm = __ballot_sync(FULL_MASK, pass);
                if (pm) tau = list_absorb<KPL>(v, d2, pass, pm, kk, lane);
            }
        }
        // the others: one child per lane
        const float thr = fminf(tau, limit);
        const bool expand = have && !is_leaf && !(node.mind2 * 0.9999f > thr);
        const int cl = node_level - 1;
        const uint32_t chx = 2u * node_x + ((lane >> 2) & 1u), chy = 2u * node_y + ((lane >> 1) & 1u), chz = 2u * node_z + (lane & 1u);
        push_nodes(expand, cl, chx, chy, chz, thr);
        __syncwarp();
    }
}

// kNeighbors > 63 (lists too long for the main pass's per-lane registers): every query goes to the tree search.
__global__ void __launch_bounds__(256) knn_queue_all_kernel(const uint64_t *__restrict__ sorted, uint32_t n, int idxbits, uint32_t nquery, FarEntry *__restrict__ far_list,
                                                             uint32_t *__restrict__ far_count) {
    const uint64_t idxmask = (1ull << idxbits) - 1ull;
    const unsigned lane = lane_id();
    const uint32_t rounds = (n + blockDim.x * gridDim.x - 1) / (blockDim.x * gridDim.x);
    for (uint32_t r = 0; r < rounds; r++) {
        const uint32_t i = (r * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
        const bool query = i < n && (uint32_t)(sorted[i] & idxmask) < nquery;
        const unsigned m = __ballot_sync(FULL_MASK, query);
        if (m == 0u) continue;
        uint32_t first = 0;
        if (lane == (unsigned)(__ffs(m) - 1)) first = atomicAdd(far_count, (uint32_t)__popc(m));
        first = __shfl_sync(FULL_MASK, first, __ffs(m) - 1);
        if (query) {
            FarEntry e;
            e.q = i;
            e.bound = INFINITY;
            far_list[first + __popc(m & lanemask_lt())] = e;
        }
    }
}

// Start of the search for a query that is a point of the cloud itself (Morton code of its cell: `code`).  The smallest node
// around its cell that holds kk points or more bounds the kk-th distance by the distance to that node's farthest corner
// (one table entry per level, one level per lane); `limit` is lowered to that bound.  Every point within the bound then
// lies in at most 2x2x2 nodes of some level L, and the search starts there instead of at the root: an isolated point
// (what the main pass leaves open on a downsampled frame) no longer descends through the whole pyramid with no bound at all.
__device__ __forceinline__ FarStart far_start(const Point16 q, uint64_t code, const GridParams &gp, int kk, const uint2 *__restrict__ table, uint32_t band, float &limit) {
    const unsigned lane = lane_id();
    const uint32_t cx = compact3(code >> 2), cy = compact3(code >> 1), cz = compact3(code);
    const int root_level = gp.bands > 1 ? gp.band_bits : gp.top_level;
    const float slack = 0.01f * gp.h; // a point may sit this far outside the nominal box of its cell (rounding of cell_u)
    const float qq[3] = {q.x, q.y, q.z};
    bool enough = false;
    float far2 = INFINITY;
    if ((int)lane <= root_level) {
        const int l = (int)lane;
        const uint32_t ax = cx >> l, ay = cy >> l, az = cz >> l;
        const uint2 r = table[table_index(gp, l, ax, ay, az)];
        if (r.y - r.x >= (uint32_t)kk) {
            enough = true;
            const float pitch = ldexpf(gp.h, l);
            const uint32_t lx = ax - (band << (gp.band_bits - l));
            const float lo[3] = {gp.gmin[0] + (float)lx * pitch, gp.gmin[1] + (float)ay * pitch, gp.gmin[2] + (float)az * pitch};
            far2 = 0.f;
#pragma unroll
            for (int a = 0; a < 3; a++) {
                const float d = fmaxf(qq[a] - lo[a], (lo[a] + pitch) - qq[a]) + slack;
                far2 += d * d;
            }
        }
    }
    FarStart st;
    st.level = -1;
    st.x = st.y = st.z = 0u;
    const unsigned m = __ballot_sync(FULL_MASK, enough);
    if (m != 0u) limit = fminf(limit, __shfl_sync(FULL_MASK, far2, __ffs(m) - 1) * 1.0001f);
    if (!(limit < INFINITY)) return st; // fewer than kk points in the band / the cloud and no bound from the main pass: from the root
    // cells that can hold a point within the bound (cell units, 0.02 covers the rounding of cell_u on both sides)
    const float rcells = sqrtf(limit) * gp.inv_h * 1.000001f + 0.02f;
    const float u[3] = {cell_u(q.x, gp.gmin[0], gp.inv_h), cell_u(q.y, gp.gmin[1], gp.inv_h), cell_u(q.z, gp.gmin[2], gp.inv_h)};
    const int dim[3] = {gp.xdim, gp.gdim[1], gp.gdim[2]};
    uint32_t lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; a++) {
        lo[a] = (uint32_t)min(max((int)floorf(u[a] - rcells), 0), dim[a] - 1);
        hi[a] = (uint32_t)min(max((int)floorf(u[a] + rcells), 0), dim[a] - 1);
    }
    lo[0] += band << gp.band_bits;
    hi[0] += band << gp.band_bits;
    for (int l = 0; l < root_level; l++) {
        if ((hi[0] >> l) - (lo[0] >> l) <= 1u && (hi[1] >> l) - (lo[1] >> l) <= 1u && (hi[2] >> l) - (lo[2] >> l) <= 1u) {
            st.level = l;
            st.x = lo[0] >> l;
            st.y = lo[1] >> l;
            st.z = lo[2] >> l;
            break;
        }
    }
    return st;
}

template <int KPL>
__global__ void __launch_bounds__(KF_THREADS) knn_far_kernel(const cwipc_point *__restrict__ spts, const uint64_t *__restrict__ sorted, uint32_t n, const __grid_constant__ GridParams gp, int kk, int k,
                                                              const uint2 *__restrict__ table, float *__restrict__ dist_out, float *__restrict__ kth_out,
                                                              const FarEntry *__restrict__ far_list, const uint32_t *__restrict__ far_count, uint32_t second_from,
                                                              uint32_t leaf_points, bool far_start_enabled) {
    __shared__ __align__(16) FarNode s_stack[KF_WARPS][KF_STACK]; // (also holds 32 * KPL doubles per warp at the end of a search)
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    // when the second scan ran (the main pass queued at least second_from queries) the list it passed on is the one to
    // take: it lies (n + 64) entries behind the main pass's, its counter one word behind
    if (far_count[0] >= second_from) {
        far_list += (size_t)n + 64;
        far_count += 1;
    }
    const uint32_t nentries = *far_count;
    const uint32_t warps_total = (gridDim.x * blockDim.x) >> 5;
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);
    for (uint32_t ei = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; ei < nentries; ei += warps_total) {
        const FarEntry ent = far_list[ei];
        float v[KPL];
        const uint64_t code = sorted[ent.q] >> gp.idxbits;
        const uint32_t band = gp.bands > 1 ? (compact3(code >> 2) >> gp.band_bits) : 0u;
        const Point16 q = spts16[ent.q];
        float limit = ent.bound;
        FarStart start;
        start.level = -1;
        start.x = start.y = start.z = 0u;
        if (far_start_enabled) start = far_start(q, code, gp, kk, table, band, limit);
        dfs_knn<KPL>(q, limit, spts16, n, gp, kk, table, leaf_points, s_stack[warp], v, band, start);
        // sum of sqrt over elements 1..k in ascending order (double), as the reference does
        double sq[KPL];
#pragma unroll
        for (int j = 0; j < KPL; j++) sq[j] = sqrt((double)v[j]);
        // the square roots go through the (now idle) stack memory: every lane adds them up in ascending order from there
        double *s_sq = reinterpret_cast<double *>(s_stack[warp]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < KPL; j++) s_sq[j * 32 + (int)lane] = sq[j];
        __syncwarp();
        double sum = 0.0;
        for (int e = 1; e <= k; e++) sum += s_sq[e];
        const float kth = list_element<KPL>(v, kk - 1);
        __syncwarp(); // the stack is written again by the next search
        if (lane == 0) {
            const size_t orig = (size_t)(sorted[ent.q] & idxmask);
            dist_out[orig] = (float)(sum / (double)k);
            if (kth_out) kth_out[orig] = kth;
        }
    }
}

// External queries (any position, not members of the cloud): the kk smallest squared distances each, ascending.
// Used when a cloud is partitioned over several GPUs: every part answers, the owner merges the lists.
template <int KPL>
__global__ void __launch_bounds__(KF_THREADS) knn_list_kernel(const cwipc_point *__restrict__ spts, uint32_t n, GridParams gp, int kk, const uint2 *__restrict__ table,
                                                               const cwipc_point *__restrict__ queries, const float *__restrict__ limits, uint32_t nq, float *__restrict__ lists,
                                                               uint32_t leaf_points) {
    __shared__ __align__(16) FarNode s_stack[KF_WARPS][KF_STACK]; // (also holds 32 * KPL doubles per warp at the end of a search)
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t warps_total = (gridDim.x * blockDim.x) >> 5;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);
    for (uint32_t qi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; qi < nq; qi += warps_total) {
        float v[KPL];
        dfs_knn<KPL>(ld_point(queries, qi), limits ? limits[qi] : INFINITY, spts16, n, gp, kk, table, leaf_points, s_stack[warp], v);
#pragma unroll
        for (int j = 0; j < KPL; j++) {
            const int e = j * 32 + (int)lane;
            if (e < kk) lists[(size_t)qi * kk + e] = v[j]; // +inf pads when the cloud holds fewer than kk points
        }
    }
}

// Merge `nlists` ascending lists of kk squared distances per query into the mean distance to the k nearest
// (element 0 of the merged list is the query itself).  One thread per query; the lists are tiny.
__global__ void __launch_bounds__(128) knn_merge_lists_kernel(const float *__restrict__ lists, uint32_t nlists, uint32_t nq, int kk, int k, float *__restrict__ mean,
                                                               float *__restrict__ kth_out) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    uint32_t head[16]; // next unread element of each list (nlists <= 16)
    for (uint32_t l = 0; l < nlists; l++) head[l] = 0;
    double sum = 0.0;
    float last = 0.f;
    for (int e = 0; e < kk; e++) {
        float best = INFINITY;
        uint32_t arg = 0;
        for (uint32_t l = 0; l < nlists; l++) {
            if (head[l] < (uint32_t)kk) {
                const float x = lists[((size_t)l * nq + q) * kk + head[l]];
                if (x < best) {
                    best = x;
                    arg = l;
                }
            }
        }
        head[arg]++;
        if (e > 0) sum += sqrt((double)best);
        last = best;
    }
    mean[q] = (float)(sum / (double)k);
    if (kth_out) kth_out[q] = last;
}

// ---- statistics: fixed-order two-level double reduction -------------------------------------------
constexpr int ST_BLOCKS = 256;
constexpr int ST_THREADS = 256;

__global__ void __launch_bounds__(ST_THREADS) stats_kernel(const float *__restrict__ dist, uint32_t n, double *__restrict__ partial) {
    __shared__ double s_sum[ST_THREADS], s_sq[ST_THREADS];
    double sum = 0.0, sq = 0.0;
    for (uint32_t i = blockIdx.x * ST_THREADS + threadIdx.x; i < n; i += ST_BLOCKS * ST_THREADS) {
        const float d = dist[i];
        sum += (double)d;
        sq += (double)__fmul_rn(d, d); // PCL squares in float, accumulates in double
    }
    s_sum[threadIdx.x] = sum;
    s_sq[threadIdx.x] = sq;
    __syncthreads();
    for (int o = ST_THREADS / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            s_sum[threadIdx.x] += s_sum[threadIdx.x + o];
            s_sq[threadIdx.x] += s_sq[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        partial[2 * blockIdx.x] = s_sum[0];
        partial[2 * blockIdx.x + 1] = s_sq[0];
    }
}

// Same reduction, and the block that finishes last adds the 256 partials in index order and derives the threshold
// (mean + mul * unbiased stddev, all in double as pcl::StatisticalOutlierRemoval) on the device, so that the keep
// mask can be taken without a host round trip.
__global__ void __launch_bounds__(ST_THREADS) stats_threshold_kernel(const float *__restrict__ dist, uint32_t n, double *partial, uint32_t *__restrict__ done_counter,
                                                                      double stddev_mul, double *__restrict__ threshold_out) {
    __shared__ double s_sum[ST_THREADS], s_sq[ST_THREADS];
    __shared__ bool s_last;
    double sum = 0.0, sq = 0.0;
    for (uint32_t i = blockIdx.x * ST_THREADS + threadIdx.x; i < n; i += ST_BLOCKS * ST_THREADS) {
        const float d = dist[i];
        sum += (double)d;
        sq += (double)__fmul_rn(d, d);
    }
    s_sum[threadIdx.x] = sum;
    s_sq[threadIdx.x] = sq;
    __syncthreads();
    for (int o = ST_THREADS / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            s_sum[threadIdx.x] += s_sum[threadIdx.x + o];
            s_sq[threadIdx.x] += s_sq[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        __stcg(partial + 2 * blockIdx.x, s_sum[0]);
        __stcg(partial + 2 * blockIdx.x + 1, s_sq[0]);
        __threadfence();
        const uint32_t ticket = atomicAdd(done_counter, 1u);
        s_last = ticket == ST_BLOCKS - 1;
        if (s_last) *done_counter = 0; // clean for the next call
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    static_assert(ST_BLOCKS == ST_THREADS, "one partial per thread");
    s_sum[threadIdx.x] = __ldcg(partial + 2 * threadIdx.x); // parallel fetch, then one thread adds in index order
    s_sq[threadIdx.x] = __ldcg(partial + 2 * threadIdx.x + 1);
    __syncthreads();
    if (threadIdx.x != 0) return;
    double tsum = 0.0, tsq = 0.0;
    for (int b = 0; b < ST_BLOCKS; b++) {
        tsum += s_sum[b];
        tsq += s_sq[b];
    }
    const double dn = (double)n;
    const double mean = tsum / dn;
    const double variance = (tsq - tsum * tsum / dn) / (dn - 1.0);
    *threshold_out = mean + stddev_mul * sqrt(variance);
}

// The same for one tile group of a per-tile outlier removal: only the points whose tile is `tile` count; the group's
// size is counted here too.  A group of at most k points has no statistics: threshold +inf, every point of it is kept.
// partial: 3 * ST_BLOCKS doubles.
__global__ void __launch_bounds__(ST_THREADS) stats_threshold_tile_kernel(const float *__restrict__ dist, const cwipc_point *__restrict__ pts, uint32_t n, uint32_t tile, int k,
                                                                           double *partial, uint32_t *__restrict__ done_counter, double stddev_mul,
                                                                           double *__restrict__ threshold_out, uint32_t *__restrict__ count_out) {
    __shared__ double s_sum[ST_THREADS], s_sq[ST_THREADS], s_cnt[ST_THREADS];
    __shared__ bool s_last;
    double sum = 0.0, sq = 0.0;
    uint32_t cnt = 0;
    const uint32_t *words = reinterpret_cast<const uint32_t *>(pts);
    for (uint32_t i = blockIdx.x * ST_THREADS + threadIdx.x; i < n; i += ST_BLOCKS * ST_THREADS) {
        if ((__ldg(words + 4 * (size_t)i + 3) >> 24) != tile) continue;
        const float d = dist[i];
        sum += (double)d;
        sq += (double)__fmul_rn(d, d);
        cnt++;
    }
    s_sum[threadIdx.x] = sum;
    s_sq[threadIdx.x] = sq;
    s_cnt[threadIdx.x] = (double)cnt;
    __syncthreads();
    for (int o = ST_THREADS / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            s_sum[threadIdx.x] += s_sum[threadIdx.x + o];
            s_sq[threadIdx.x] += s_sq[threadIdx.x + o];
            s_cnt[threadIdx.x] += s_cnt[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        __stcg(partial + 3 * blockIdx.x, s_sum[0]);
        __stcg(partial + 3 * blockIdx.x + 1, s_sq[0]);
        __stcg(partial + 3 * blockIdx.x + 2, s_cnt[0]);
        __threadfence();
        const uint32_t ticket = atomicAdd(done_counter, 1u);
        s_last = ticket == ST_BLOCKS - 1;
        if (s_last) *done_counter = 0; // clean for the next call
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    s_sum[threadIdx.x] = __ldcg(partial + 3 * threadIdx.x);
    s_sq[threadIdx.x] = __ldcg(partial + 3 * threadIdx.x + 1);
    s_cnt[threadIdx.x] = __ldcg(partial + 3 * threadIdx.x + 2);
    __syncthreads();
    if (threadIdx.x != 0) return;
    double tsum = 0.0, tsq = 0.0, dn = 0.0;
    for (int b = 0; b < ST_BLOCKS; b++) {
        tsum += s_sum[b];
        tsq += s_sq[b];
        dn += s_cnt[b];
    }
    *count_out = (uint32_t)dn;
    if (dn <= (double)k) {
        *threshold_out = __longlong_as_double(0x7ff0000000000000ll);
        return;
    }
    const double mean = tsum / dn;
    const double variance = (tsq - tsum * tsum / dn) / (dn - 1.0);
    *threshold_out = mean + stddev_mul * sqrt(variance);
}

// Test hooks of the kNN index (results never depend on them): CWIPC_CUDA_KNN_PITCH scales the pitch relative to the
// expected k-neighbour radius, the others move work between the main pass, the second scan and the tree search.
float env_float(const char *name, float dflt, float lo, float hi) {
    const char *e = getenv(name);
    if (!e || !*e) return dflt;
    const float v = (float)atof(e);
    return (v >= lo && v <= hi) ? v : dflt;
}

struct GridPlan {
    GridParams gp;
    size_t table_entries = 0;
};

// Pitch ~ a fraction of the expected k-neighbour radius of a surface sampled at `spacing`; the main
// pass covers rc = 1 pitch around each query group.  The dense tables bound the number of cells.
GridPlan choose_grid(const float gmin[3], const float gmax[3], size_t n, int k, float hint_spacing, int bands = 1) {
    static const float pitch_factor = env_float("CWIPC_CUDA_KNN_PITCH", 1.0f, 0.05f, 20.f);
    constexpr float rc = 1.0f;
    static const float rc_far = env_float("CWIPC_CUDA_KNN_RC_FAR", 2.0f, 0.f, 8.f); // 0: no second scan
    GridPlan plan;
    GridParams &gp = plan.gp;
    memset(&gp, 0, sizeof(gp));
    const double ext[3] = {(double)gmax[0] - gmin[0], (double)gmax[1] - gmin[1], (double)gmax[2] - gmin[2]};
    double spacing = hint_spacing > 0.f ? (double)hint_spacing : 0.0;
    const double longest = std::max(ext[0], std::max(ext[1], ext[2]));
    if (!(spacing > 0.0)) {
        const double area = 2.0 * (ext[0] * ext[1] + ext[1] * ext[2] + ext[2] * ext[0]);
        const double per_band = std::max(1.0, (double)n / (double)bands); // every tile group is a surface of its own
        if (area > 0.0) spacing = std::sqrt(area / per_band);
        else if (longest > 0.0) spacing = longest / per_band;
        else spacing = 1.0;
    }
    // expected k-neighbour radius on a surface: spacing * sqrt((k+1)/pi); reach of the main pass = rc * h
    double h = spacing * std::sqrt((double)(k + 1) / 3.14159265358979) * (double)pitch_factor;
    gp.idxbits = std::max(1, bit_length((uint64_t)n - 1));
    const int rank_bits = bands > 1 ? bit_length((uint64_t)bands - 1) : 0;
    const int max_axis_bits = std::min(13, (64 - gp.idxbits) / 3) - rank_bits; // per-tile mode: the band number sits above the x cell bits
    if (max_axis_bits < 2) throw CudaError{cudaErrorInvalidValue, "remove_outliers: too many points and tiles for one search index"};
    if (!(h > 0.0) || !std::isfinite(h)) h = 1.0;
    // the bands lie side by side along x, each padded to a power of two of cells (<= 2x on the longest axis)
    // dense tables: 9.1 bytes per cell over all levels.  16 cells per point (146 MB at 1 M points), at most 2^27 cells
    // (1.2 GB, reached from 8 M points on).  Round 1 allowed 4 per point / 2^25: an 8 M-point cloud and the per-tile bands of a
    // 1 M-point cloud then got a pitch 1.6-2x the wanted one, i.e. 2.5-4x the candidates per query (8 M raw: 9.3 -> 6.5 ms).
    const double cell_cap = std::min(std::max(16.0 * (double)n, 65536.0), std::ldexp(1.0, 27)) / (bands > 1 ? 2.0 * (double)bands : 1.0);
    while (true) {
        const double cells = (std::floor(ext[0] / h) + 2) * (std::floor(ext[1] / h) + 2) * (std::floor(ext[2] / h) + 2);
        if (longest / h < (double)((1 << max_axis_bits) - 1) && cells <= cell_cap) break;
        h *= 1.25;
    }
    gp.h = (float)h;
    gp.inv_h = 1.0f / gp.h;
    gp.rc = rc;
    gp.rc_far = rc_far;
    gp.second_min = (int)env_float("CWIPC_CUDA_KNN_SECOND_MIN", 2.f, 1.f, 32.f);
    gp.second_max = (int)env_float("CWIPC_CUDA_KNN_SECOND_MAX", 150.f, 1.f, 1.0e6f);
    int maxdim = 1;
    for (int a = 0; a < 3; a++) {
        gp.gmin[a] = gmin[a];
        gp.gdim[a] = std::max(1, std::min((int)std::floor(ext[a] / (double)gp.h) + 2, 1 << max_axis_bits));
        maxdim = std::max(maxdim, gp.gdim[a]);
    }
    gp.top_level = bit_length((uint64_t)maxdim - 1); // (gdim-1) >> top_level == 0 on every axis
    gp.bands = std::max(1, bands);
    gp.xdim = gp.gdim[0];
    gp.band_bits = gp.top_level;
    if (gp.bands > 1) {
        gp.band_bits = std::max(gp.top_level, KT_GROUP_LEVEL); // a query group (level-KT_GROUP_LEVEL node) never spans two bands
        gp.gdim[0] = ((gp.bands - 1) << gp.band_bits) + gp.xdim;
        gp.top_level = gp.band_bits + rank_bits;
    }
    size_t off = 0;
    for (int l = 0; l <= gp.top_level; l++) {
        gp.table_off[l] = (uint32_t)off;
        off += (size_t)level_dim(gp.gdim[0], l) * level_dim(gp.gdim[1], l) * level_dim(gp.gdim[2], l);
    }
    plan.table_entries = off;
    return plan;
}

// tree search: nodes with at most this many points are scanned directly instead of being expanded
constexpr uint32_t FAR_LEAF_POINTS = 128;

template <int KCAP>
void run_knn(const cwipc_point *spts, const uint64_t *sorted, size_t n, const GridParams &gp, int k, const uint2 *table, float *d_dist, float *d_kth, size_t nquery,
             FarEntry *far_list, uint32_t *far_count, int dev, cudaStream_t s) {
    const int kk = k + 1;
    const size_t smem = sizeof(KnnWarpSmem) * KT_WARPS;
    static std::once_flag once[64];
    std::call_once(once[dev & 63], [&] {
        CWCU_CHECK(cudaFuncSetAttribute(knn_tile_kernel<KCAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CWCU_CHECK(cudaFuncSetAttribute(knn_second_kernel<KCAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    });
    const size_t nitems = div_up(n, (size_t)32);
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min(div_up(nitems, (size_t)KT_WARPS), (size_t)sm_count(dev) * KT_BLOCKS_PER_SM));
    launch("knn_tile_kernel", s, 28 * (size_t)n, [&] {
        knn_tile_kernel<KCAP><<<grid, KT_THREADS, smem, s>>>(spts, sorted, (uint32_t)n, gp, kk, k, table, d_dist, d_kth, (uint32_t)nquery, far_list, far_count);
    });
    if (gp.top_level == 0) return; // one cell spans the cloud: the main pass is exact for every query
    uint32_t second_from = 0xffffffffu; // number of queued queries from which the second scan runs (decided on the device)
    // The second scan pays when the queue is long enough to fill the machine with 32-query warps and the open queries are each
    // other's neighbours (raw, noisy clouds); on a small cloud (a downsampled frame: a few thousand isolated points in the
    // queue) its per-group latency is not bought back.  Measured: 47 K-point frames -2..-5 % throughput, 1 M raw points -23 % time.
    static const float second_from_n = env_float("CWIPC_CUDA_KNN_SECOND_FROM_N", 262144.f, 0.f, 4.0e9f);
    if (gp.rc_far > gp.rc && (double)std::min(nquery, n) >= (double)second_from_n) {
        second_from = 1;
        // open queries with a bound within rc_far pitches: scanned once more, group by group; the rest goes to the second list
        launch("knn_second_kernel", s, (size_t)0, [&] {
            knn_second_kernel<KCAP><<<(unsigned)sm_count(dev) * KT_BLOCKS_PER_SM, KT_THREADS, smem, s>>>(spts, sorted, gp, kk, k, table, d_dist, d_kth, far_list, far_count, second_from,
                                                                                                         far_list + (n + 64), far_count + 1);
        });
    }
    constexpr int KPL = KCAP > 32 ? 2 : 1;
    launch("knn_far_kernel", s, (size_t)0, [&] {
        // CWIPC_CUDA_KNN_FAR_START=0 (tests / A-B only): every search starts at the root with no bound, as in round 1
        static const bool far_start_on = env_float("CWIPC_CUDA_KNN_FAR_START", 1.f, 0.f, 1.f) != 0.f;
        knn_far_kernel<KPL><<<(unsigned)sm_count(dev) * 8, KF_THREADS, 0, s>>>(spts, sorted, (uint32_t)n, gp, kk, k, table, d_dist, d_kth, far_list, far_count, second_from, FAR_LEAF_POINTS,
                                                                               far_start_on);
    });
}

// kNeighbors from 64 to KNN_MAX_K: no main pass, one tree search per query with a list of KPL registers per lane (slow path:
// the reference has no limit on meanK, so large values must work, but no real caller uses them).
template <int KPL>
void run_knn_wide(const cwipc_point *spts, const uint64_t *sorted, size_t n, const GridParams &gp, int k, const uint2 *table, float *d_dist, float *d_kth, size_t nquery,
                  FarEntry *far_list, uint32_t *far_count, int dev, cudaStream_t s) {
    launch("knn_queue_all_kernel", s, 8 * n, [&] {
        knn_queue_all_kernel<<<stream_grid(n, dev), 256, 0, s>>>(sorted, (uint32_t)n, gp.idxbits, (uint32_t)nquery, far_list, far_count);
    });
    launch("knn_far_kernel", s, (size_t)0, [&] {
        static const bool far_start_on = env_float("CWIPC_CUDA_KNN_FAR_START", 1.f, 0.f, 1.f) != 0.f;
        knn_far_kernel<KPL><<<(unsigned)sm_count(dev) * 8, KF_THREADS, 0, s>>>(spts, sorted, (uint32_t)n, gp, k + 1, k, table, d_dist, d_kth, far_list, far_count, 0xffffffffu, FAR_LEAF_POINTS,
                                                                               far_start_on);
    });
}

// The search structure of one cloud: cell-ordered points + table pyramid (scratch lives as long as the object).
struct KnnIndex {
    GridParams gp;
    Scratch keys_a, keys_b, spts, table;
    const uint64_t *sorted = nullptr;
    uint32_t *far_count = nullptr;
};

void build_index(KnnIndex &ix, const cwipc_point *in, size_t n, int k, float hint_spacing, const float *bounds, int dev, cudaStream_t s, const BandLut *lut = nullptr, int bands = 1) {
    float gmin[3], gmax[3];
    if (bounds) {
        for (int a = 0; a < 3; a++) {
            gmin[a] = bounds[a];
            gmax[a] = bounds[3 + a];
        }
    } else {
        global_bbox(in, n, gmin, gmax, dev, s);
    }
    for (int a = 0; a < 3; a++)
        if (!std::isfinite(gmin[a]) || !std::isfinite(gmax[a])) throw CudaError{cudaErrorInvalidValue, "remove_outliers: pointcloud contains non-finite coordinates"};
    const GridPlan plan = choose_grid(gmin, gmax, n, k, hint_spacing, lut ? bands : 1);
    BandLut band_lut;
    if (lut) band_lut = *lut;
    else memset(&band_lut, 0, sizeof(band_lut));
    ix.gp = plan.gp;
    const GridParams &gp = ix.gp;
    int axis_bits = 1;
    for (int a = 0; a < 3; a++) axis_bits = std::max(axis_bits, bit_length((uint64_t)gp.gdim[a] - 1));
    const int keybits = 3 * axis_bits;

    ix.keys_a = Scratch(n * sizeof(uint64_t), s);
    ix.keys_b = Scratch(n * sizeof(uint64_t), s);
    // cell-ordered points, table pyramid, far-query counter (2 extra entries behind the tables)
    ix.spts = Scratch(n * sizeof(cwipc_point), s);
    ix.table = Scratch((plan.table_entries + 2) * sizeof(uint2), s);
    ix.far_count = reinterpret_cast<uint32_t *>(ix.table.as<uint2>() + plan.table_entries);
    launch("knn_keygen_kernel", s, 24 * (size_t)n, [&] {
        knn_keygen_kernel<<<stream_grid(std::max(n, plan.table_entries / 4), dev), 256, 0, s>>>(in, (uint32_t)n, gp, band_lut, ix.keys_a.as<uint64_t>(), ix.table.as<uint2>(),
                                                                                                 (uint32_t)(plan.table_entries + 2));
    });
    ix.sorted = radix_sort_u64(ix.keys_a.as<uint64_t>(), ix.keys_b.as<uint64_t>(), n, gp.idxbits, gp.idxbits + keybits, dev, s);

    launch("knn_layout_kernel", s, 48 * (size_t)n, [&] {
        knn_layout_kernel<<<stream_grid(n, dev), 256, 0, s>>>(ix.sorted, (uint32_t)n, gp, in, ix.spts.as<cwipc_point>(), ix.table.as<uint2>());
    });
}

void check_k(int k, size_t n) {
    if (k < 1) throw CudaError{cudaErrorInvalidValue, "remove_outliers: kNeighbors must be >= 1"};
    if (k > KNN_MAX_K) throw CudaError{cudaErrorInvalidValue, "remove_outliers: kNeighbors > " + std::to_string(KNN_MAX_K) + " is not supported by libcwipc_util_cuda"};
    (void)n;
}

// ---- ICP correspondences (cwipc_cuda_icp): the nearest target point of every moved source point ----------------------
constexpr int ICP_WARPS = 2;
constexpr int ICP_THREADS = ICP_WARPS * 32;
constexpr int ICP_BLOCKS_PER_SM = 8;

struct IcpParams {
    double m[12];      // rows 0..2 of the current source -> target motion
    double origin[3];  // the sums are taken relative to this point (the centre of the target's box)
    float limit;       // (float)(max_correspondence_distance^2): a pair counts iff d2 <= limit
    float slack;       // how far a point may lie outside the nominal box of its node (rounding of cell_u and of the box corners)
    uint32_t check;    // also count the non-finite coordinates of both clouds (first evaluation of a call)
};

// Depth-first search of the table pyramid around q, the search of icp_nearest and icp_neighbours, called by all 32 lanes
// with the same q.  It is dfs_knn's search: the four nearest open nodes per step (8 lanes per node), nodes of at most
// leaf_points points scanned.  It starts at the <= 2x2x2 nodes of the lowest level that cover every cell within sqrt(limit)
// of q, and a node is dropped when its box is farther than tau, the caller's pruning bound (<= limit, the same in every
// lane).  So a query with no target point within the bound only visits the nodes that touch its ball, never a scan of the
// cells around it.  Nodes at exactly tau are kept: an equally near point with a smaller index must still be seen.
// consider(c, valid) is called by every lane at once, with a position c of the cell-ordered target on the lanes where valid
// is true; refresh() (all lanes) follows each batch and may lower tau.  Every target point is offered at most once.
template <class Consider, class Refresh>
__device__ __forceinline__ void pyramid_search(const Point16 q, float limit, float slack, const GridParams &gp, const uint2 *__restrict__ table, uint32_t leaf_points,
                                               FarNode *stack, const float &tau, Consider &&consider, Refresh &&refresh) {
    const unsigned lane = lane_id();
    int sp = 0;
    // Lanes that `want` their node (level cl, (chx, chy, chz)) push it when it holds points and its box is within tau; the
    // pushed nodes are ranked by (distance, lane), the nearest on top.
    auto push_nodes = [&](bool want, int cl, uint32_t chx, uint32_t chy, uint32_t chz) {
        uint2 r = make_uint2(0u, 0u);
        float mind2 = INFINITY;
        bool admit = false;
        if (want && chx < (uint32_t)level_dim(gp.gdim[0], cl) && chy < (uint32_t)level_dim(gp.gdim[1], cl) && chz < (uint32_t)level_dim(gp.gdim[2], cl)) {
            r = table[table_index(gp, cl, chx, chy, chz)];
            if (r.y > r.x) {
                const float pitch = ldexpf(gp.h, cl);
                const float lo[3] = {gp.gmin[0] + (float)chx * pitch, gp.gmin[1] + (float)chy * pitch, gp.gmin[2] + (float)chz * pitch};
                const float qq[3] = {q.x, q.y, q.z};
                mind2 = 0.f;
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    const float d = fmaxf(fmaxf(lo[a] - qq[a], qq[a] - (lo[a] + pitch)) - slack, 0.f);
                    mind2 += d * d;
                }
                admit = !(mind2 * 0.9999f > tau);
            }
        }
        const unsigned adm = __ballot_sync(FULL_MASK, admit);
        if (adm == 0u) return;
        const uint32_t mine = __float_as_uint(mind2);
        int rank = 0;
        for (unsigned m = adm; m; m &= m - 1u) {
            const int src = __ffs(m) - 1;
            const uint32_t other = __shfl_sync(FULL_MASK, mine, src);
            rank += (other < mine || (other == mine && src < (int)lane)) ? 1 : 0;
        }
        const int nadm = __popc(adm);
        if (admit) {
            FarNode ch;
            ch.pb = r.x; ch.pe = r.y; ch.xy = chx | (chy << 16); ch.zl = chz | ((uint32_t)cl << 16); ch.mind2 = mind2;
            stack[sp + nadm - 1 - rank] = ch;
        }
        sp += nadm;
    };

    {
        // the lowest level at which the cells within the bound span at most two nodes per axis (the root at the latest)
        const float rcells = (sqrtf(limit) + slack) * gp.inv_h * 1.000001f + 0.02f;
        const float u[3] = {cell_u(q.x, gp.gmin[0], gp.inv_h), cell_u(q.y, gp.gmin[1], gp.inv_h), cell_u(q.z, gp.gmin[2], gp.inv_h)};
        uint32_t lo[3], hi[3];
#pragma unroll
        for (int a = 0; a < 3; a++) {
            lo[a] = (uint32_t)min(max((int)floorf(u[a] - rcells), 0), gp.gdim[a] - 1);
            hi[a] = (uint32_t)min(max((int)floorf(u[a] + rcells), 0), gp.gdim[a] - 1);
        }
        int level = 0;
        while (level < gp.top_level && !((hi[0] >> level) - (lo[0] >> level) <= 1u && (hi[1] >> level) - (lo[1] >> level) <= 1u && (hi[2] >> level) - (lo[2] >> level) <= 1u)) level++;
        push_nodes(lane < 8u, level, (lo[0] >> level) + ((lane >> 2) & 1u), (lo[1] >> level) + ((lane >> 1) & 1u), (lo[2] >> level) + (lane & 1u));
        __syncwarp();
    }
    const int group = (int)(lane >> 3);
    while (sp > 0) {
        const int take = min(sp, 4);
        const FarNode node = stack[sp - 1 - min(group, take - 1)]; // lane group g looks at the g-th nearest open node
        const bool have = group < take && !(node.mind2 * 0.9999f > tau);
        const int node_level = (int)(node.zl >> 16);
        sp -= take;
        __syncwarp();
        if (__all_sync(FULL_MASK, !have || node.pe - node.pb <= 8u)) { // sparse neighbourhood: every node taken is scanned at once
            const uint32_t c = node.pb + (lane & 7u);
            consider(c, have && c < node.pe);
            refresh();
            continue;
        }
        const bool is_leaf = node_level == 0 || node.pe - node.pb <= leaf_points;
        unsigned todo = __ballot_sync(FULL_MASK, have && is_leaf) & 0x01010101u; // the groups' first lanes vote
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1u;
            const uint32_t pb = __shfl_sync(FULL_MASK, node.pb, src), pe = __shfl_sync(FULL_MASK, node.pe, src);
            if (__shfl_sync(FULL_MASK, node.mind2, src) * 0.9999f > tau) continue; // (the bound may have dropped since the vote)
            for (uint32_t base = pb; base < pe; base += 32)
                consider(base + lane, base + lane < pe);
            refresh();
        }
        const bool expand = have && !is_leaf && !(node.mind2 * 0.9999f > tau);
        push_nodes(expand, node_level - 1, 2u * (node.xy & 0xffffu) + ((lane >> 2) & 1u), 2u * (node.xy >> 16) + ((lane >> 1) & 1u), 2u * (node.zl & 0xffffu) + (lane & 1u));
        __syncwarp();
    }
}

// The nearest target point to q with d2 <= limit, as the key (d2 bits << 32) | (index in the target's input order), or ~0 when
// there is none: the smallest key is the smallest d2 and, among equal ones, the smallest index.  Called by all 32 lanes with
// the same q; the result is the same in every lane.  The pruning bound is min(limit, best d2 so far).
__device__ __forceinline__ uint64_t icp_nearest(const Point16 q, float limit, float slack, const Point16 *__restrict__ spts16, const uint64_t *__restrict__ sorted,
                                                const GridParams &gp, const uint2 *__restrict__ table, uint32_t leaf_points, FarNode *stack) {
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    uint64_t best = ~0ull; // this lane's best key
    float tau = limit;     // pruning bound, the same in every lane
    pyramid_search(
        q, limit, slack, gp, table, leaf_points, stack, tau,
        [&](uint32_t c, bool valid) { // position c of the cell-ordered target
            if (valid) {
                const float d2 = dist2(q, spts16[c]);
                if (d2 <= limit && __float_as_uint(d2) <= (uint32_t)(best >> 32)) best = min(best, ((uint64_t)__float_as_uint(d2) << 32) | (sorted[c] & idxmask));
            }
        },
        [&] {
            const uint32_t hi = __reduce_min_sync(FULL_MASK, (uint32_t)(best >> 32)); // non-negative floats order like their bits
            if (hi != 0xffffffffu) tau = __uint_as_float(hi);
        });
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, (uint64_t)__shfl_xor_sync(FULL_MASK, (unsigned long long)best, o));
    return best;
}

// The kk (1..32) smallest keys (d2 bits << 32) | (index in the target's input order) of the target points with d2 <= limit,
// one per lane: lane j holds the j-th smallest, ~0 where there are fewer.  The set does not depend on the order in which the
// points are met, so it is the same on every run.  The pruning bound is min(limit, the kk-th d2 so far) once kk are held.
__device__ __forceinline__ uint64_t icp_neighbours(const Point16 q, float limit, float slack, int kk, const Point16 *__restrict__ spts16, const uint64_t *__restrict__ sorted,
                                                   const GridParams &gp, const uint2 *__restrict__ table, uint32_t leaf_points, FarNode *stack) {
    const int lane = (int)lane_id();
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    uint64_t mine = ~0ull; // this lane's place in the ascending list
    uint64_t kth = ~0ull;  // the list's last place (kk - 1), the same in every lane
    float tau = limit;
    pyramid_search(
        q, limit, slack, gp, table, leaf_points, stack, tau,
        [&](uint32_t c, bool valid) {
            uint64_t key = ~0ull;
            if (valid) {
                const float d2 = dist2(q, spts16[c]);
                if (d2 <= limit) key = ((uint64_t)__float_as_uint(d2) << 32) | (sorted[c] & idxmask);
            }
            // insert the lanes' keys that beat the list one at a time: place pos = how many listed keys are smaller
            for (unsigned todo = __ballot_sync(FULL_MASK, key < kth); todo; todo &= todo - 1u) {
                const uint64_t x = __shfl_sync(FULL_MASK, (unsigned long long)key, __ffs(todo) - 1);
                if (!(x < kth)) continue;
                const int pos = __popc(__ballot_sync(FULL_MASK, mine < x));
                const uint64_t up = __shfl_up_sync(FULL_MASK, (unsigned long long)mine, 1);
                if (lane == pos) mine = x;
                else if (lane > pos && lane < kk) mine = up;
                kth = __shfl_sync(FULL_MASK, (unsigned long long)mine, kk - 1);
            }
        },
        [&] {
            if (kth != ~0ull) tau = __uint_as_float((uint32_t)(kth >> 32));
        });
    return mine;
}

__device__ __forceinline__ bool finite_point(const Point16 &p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }
__device__ __forceinline__ double pick3(const double (&v)[3], unsigned i) { return i == 0 ? v[0] : (i == 1 ? v[1] : v[2]); }

// One warp per source point (grid-stride): p' = T p with cwipc_cuda_transform's arithmetic, computed on the fly, and its
// nearest target point within the bound.  Lane j of a warp adds up term j of the ICP_NSUMS sums over the warp's
// correspondences, in the warp's (fixed) query order: count, sum d2, sum p' (3), sum q (3), sum p'_a q_b (9, row-major), all in
// double relative to ip.origin; term 17 is the number of non-finite points of both clouds when ip.check is set.  The warp
// stores its sums in partial[warp][ICP_NSUMS]; icp_reduce_kernel adds them up in warp order.
__global__ void __launch_bounds__(ICP_THREADS) icp_match_kernel(const cwipc_point *__restrict__ src, uint32_t ns, const cwipc_point *__restrict__ tgt, uint32_t nt,
                                                                const cwipc_point *__restrict__ spts, const uint64_t *__restrict__ sorted, const __grid_constant__ GridParams gp,
                                                                const uint2 *__restrict__ table, uint32_t leaf_points, const __grid_constant__ IcpParams ip, double *__restrict__ partial) {
    __shared__ __align__(16) FarNode s_stack[ICP_WARPS][KF_STACK];
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, warps_total = (gridDim.x * blockDim.x) >> 5;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);
    double acc = 0.0;
    for (uint32_t qi = gwarp; qi < ns; qi += warps_total) {
        const Point16 p = ld_point(src, qi);
        Point16 q;
        q.x = affine_row(ip.m, p.x, p.y, p.z);
        q.y = affine_row(ip.m + 4, p.x, p.y, p.z);
        q.z = affine_row(ip.m + 8, p.x, p.y, p.z);
        q.rgbt = 0u;
        if (!finite_point(q)) continue; // (a non-finite input point, counted below; or a float overflow of the motion)
        const uint64_t key = icp_nearest(q, ip.limit, ip.slack, spts16, sorted, gp, table, leaf_points, s_stack[warp]);
        if (key == ~0ull) continue;
        const Point16 t = ld_point(tgt, (uint32_t)key);
        const double pr[3] = {(double)q.x - ip.origin[0], (double)q.y - ip.origin[1], (double)q.z - ip.origin[2]};
        const double qr[3] = {(double)t.x - ip.origin[0], (double)t.y - ip.origin[1], (double)t.z - ip.origin[2]};
        double term = 0.0;
        if (lane == 0) term = 1.0;
        else if (lane == 1) term = (double)__uint_as_float((uint32_t)(key >> 32));
        else if (lane < 5) term = pick3(pr, lane - 2);
        else if (lane < 8) term = pick3(qr, lane - 5);
        else if (lane < 17) term = pick3(pr, (lane - 8) / 3) * pick3(qr, (lane - 8) % 3);
        acc += term;
    }
    if (ip.check) {
        uint32_t bad = 0;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) bad += finite_point(ld_point_stream(src, i)) ? 0u : 1u;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nt; i += gridDim.x * blockDim.x) bad += finite_point(ld_point_stream(tgt, i)) ? 0u : 1u;
        bad = warp_sum(bad);
        if (lane == 17) acc = (double)bad;
    }
    if (lane < ICP_NSUMS) partial[(size_t)gwarp * ICP_NSUMS + lane] = acc;
}

// Warp j adds up sum j of every warp's partial sums: lane l the warps l, l + 32, ... in order, then a fixed butterfly.  With
// the per-warp order of icp_match_kernel this is a fixed order: the same bits on every run and with any number of callers.
__global__ void __launch_bounds__(ICP_NSUMS * 32) icp_reduce_kernel(const double *__restrict__ partial, uint32_t nwarps, double *__restrict__ out) {
    const unsigned lane = lane_id(), j = threadIdx.x >> 5;
    double s = 0.0;
    for (uint32_t w = lane; w < nwarps; w += 32) s += partial[(size_t)w * ICP_NSUMS + j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(FULL_MASK, s, o);
    if (lane == 0) out[j] = s;
}

// ---- point-to-plane ICP (cwipc_cuda_icp_point_to_plane, cwipc_cuda_estimate_normals) ----------------------------------------
// One cyclic Jacobi rotation of the symmetric 3x3 A that zeroes A[P][Q], accumulated in the columns of V.
template <int P, int Q>
__device__ __forceinline__ void jacobi3_rotate(double (&A)[3][3], double (&V)[3][3]) {
    if (A[P][Q] == 0.0) return;
    const double theta = (A[Q][Q] - A[P][P]) / (2.0 * A[P][Q]);
    const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
    const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const double a = A[k][P], b = A[k][Q];
        A[k][P] = c * a - s * b;
        A[k][Q] = s * a + c * b;
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const double a = A[P][k], b = A[Q][k];
        A[P][k] = c * a - s * b;
        A[Q][k] = s * a + c * b;
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const double a = V[k][P], b = V[k][Q];
        V[k][P] = c * a - s * b;
        V[k][Q] = s * a + c * b;
    }
}

// The eigen-decomposition of the symmetric 3x3 A by cyclic Jacobi rotations in double (the same rules as icp.cpp's
// horn_rotation: an off-diagonal entry below the rounding of both diagonal entries is dropped): A ends diagonal, holding
// the eigenvalues, and column k of V is the unit eigenvector of A[k][k].
__device__ __forceinline__ void jacobi3_eigen(double (&A)[3][3], double (&V)[3][3]) {
    V[0][0] = 1.0, V[0][1] = 0.0, V[0][2] = 0.0;
    V[1][0] = 0.0, V[1][1] = 1.0, V[1][2] = 0.0;
    V[2][0] = 0.0, V[2][1] = 0.0, V[2][2] = 1.0;
    for (int sweep = 0; sweep < 50 && !(A[0][1] == 0.0 && A[0][2] == 0.0 && A[1][2] == 0.0); sweep++) {
        if (sweep > 3) {
#pragma unroll
            for (int p = 0; p < 2; p++)
#pragma unroll
                for (int q = p + 1; q < 3; q++) {
                    const double g = 100.0 * fabs(A[p][q]);
                    if (fabs(A[p][p]) + g == fabs(A[p][p]) && fabs(A[q][q]) + g == fabs(A[q][q])) A[p][q] = A[q][p] = 0.0;
                }
        }
        jacobi3_rotate<0, 1>(A, V);
        jacobi3_rotate<0, 2>(A, V);
        jacobi3_rotate<1, 2>(A, V);
    }
}

// The unit eigenvector of the smallest eigenvalue of the symmetric 3x3 A.
__device__ __forceinline__ float3 smallest_eigenvector(double (&A)[3][3]) {
    double V[3][3];
    jacobi3_eigen(A, V);
    const int m = A[0][0] <= A[1][1] ? (A[0][0] <= A[2][2] ? 0 : 2) : (A[1][1] <= A[2][2] ? 1 : 2);
    const double x = m == 0 ? V[0][0] : (m == 1 ? V[0][1] : V[0][2]);
    const double y = m == 0 ? V[1][0] : (m == 1 ? V[1][1] : V[1][2]);
    const double z = m == 0 ? V[2][0] : (m == 1 ? V[2][1] : V[2][2]);
    const double inv = 1.0 / sqrt(x * x + y * y + z * z);
    return make_float3((float)(x * inv), (float)(y * inv), (float)(z * inv));
}

// One warp per point of the cloud, in cell order (grid-stride): its neighbourhood is the kk smallest keys (d2, index) of the
// cloud's points with d2 <= limit (itself included), found by icp_neighbours.  The mean and then the covariance relative to
// it are summed in double over the lanes in a fixed butterfly order; the normal is the unit eigenvector of the covariance's
// smallest eigenvalue.  normals[i] (input order) = (nx, ny, nz, 0); (0, 0, 0, 0) for fewer than 3 neighbours or a zero
// covariance; (0, 0, 0, 1) for a point with a non-finite coordinate.
__global__ void __launch_bounds__(ICP_THREADS) icp_normals_kernel(const cwipc_point *__restrict__ pts, uint32_t n, const cwipc_point *__restrict__ spts,
                                                                  const uint64_t *__restrict__ sorted, const __grid_constant__ GridParams gp, const uint2 *__restrict__ table,
                                                                  uint32_t leaf_points, float limit, float slack, int kk, float4 *__restrict__ normals) {
    __shared__ __align__(16) FarNode s_stack[ICP_WARPS][KF_STACK];
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, warps_total = (gridDim.x * blockDim.x) >> 5;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    for (uint32_t c = gwarp; c < n; c += warps_total) {
        const Point16 q = spts16[c];
        const uint32_t self = (uint32_t)(sorted[c] & idxmask);
        float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!finite_point(q)) {
            out.w = 1.f;
        } else {
            const uint64_t key = icp_neighbours(q, limit, slack, kk, spts16, sorted, gp, table, leaf_points, s_stack[warp]);
            const bool have = key != ~0ull;
            const int cnt = __popc(__ballot_sync(FULL_MASK, have));
            if (cnt >= 3) {
                double p[3] = {0.0, 0.0, 0.0};
                if (have) {
                    const Point16 t = ld_point(pts, (uint32_t)(key & idxmask));
                    p[0] = t.x, p[1] = t.y, p[2] = t.z;
                }
                double mean[3];
#pragma unroll
                for (int a = 0; a < 3; a++) mean[a] = warp_sum(p[a]) / (double)cnt;
#pragma unroll
                for (int a = 0; a < 3; a++) p[a] = have ? p[a] - mean[a] : 0.0;
                double A[3][3];
#pragma unroll
                for (int a = 0; a < 3; a++)
#pragma unroll
                    for (int b = a; b < 3; b++) A[a][b] = A[b][a] = warp_sum(p[a] * p[b]);
                if (!(A[0][0] == 0.0 && A[1][1] == 0.0 && A[2][2] == 0.0)) { // (a zero diagonal is a zero covariance)
                    const float3 v = smallest_eigenvector(A);
                    out.x = v.x, out.y = v.y, out.z = v.z;
                }
            }
        }
        if (lane == 0) normals[self] = out;
    }
}

// ---- colored ICP (cwipc_cuda_icp_colored, cwipc_cuda_estimate_color_gradients) ----------------------------------------------
// The intensity of a point: ((double)r + g + b) / 765, an exact integer sum and one division.
__device__ __forceinline__ double pt_intensity(const Point16 &p) { return (double)(pt_r(p) + pt_g(p) + pt_b(p)) / 765.0; }

// One warp per point of the cloud, in cell order (grid-stride), after icp_normals_kernel: the colour gradient g of point i
// (open3d's InitializePointCloudForColoredICP).  Its neighbourhood is the kk smallest keys (d2, index) of the cloud's points
// with d2 <= limit (itself included), found by icp_neighbours, and n = normals[i].  Every neighbour j gives the row
// A_j = d_j - (d_j . n) n with d_j = v_j - v_i and b_j = I_j - I_i; one more row (nn - 1) n with b = 0 keeps g in the tangent
// plane.  The 6 entries of A^T A and the 3 of A^T b are summed in double over the lanes in a fixed butterfly order; g is the
// minimum-norm solution of (A^T A) g = A^T b from jacobi3_eigen, the eigenvalues <= 1e-12 times the largest dropped.
// gradients[i] (input order) = (gx, gy, gz, 0); (0, 0, 0, 0) for fewer than 4 neighbours or a zero normal; (0, 0, 0, 1) for
// a point with a non-finite coordinate.
__global__ void __launch_bounds__(ICP_THREADS) icp_gradients_kernel(const cwipc_point *__restrict__ pts, uint32_t n, const cwipc_point *__restrict__ spts,
                                                                    const uint64_t *__restrict__ sorted, const __grid_constant__ GridParams gp, const uint2 *__restrict__ table,
                                                                    uint32_t leaf_points, float limit, float slack, int kk, const float4 *__restrict__ normals,
                                                                    float4 *__restrict__ gradients) {
    __shared__ __align__(16) FarNode s_stack[ICP_WARPS][KF_STACK];
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, warps_total = (gridDim.x * blockDim.x) >> 5;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);
    const uint64_t idxmask = (1ull << gp.idxbits) - 1ull;
    for (uint32_t c = gwarp; c < n; c += warps_total) {
        const Point16 q = spts16[c]; // (the cell-ordered copy holds the colour too)
        const uint32_t self = (uint32_t)(sorted[c] & idxmask);
        float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!finite_point(q)) {
            out.w = 1.f;
        } else {
            const float4 nf = normals[self];
            const uint64_t key = icp_neighbours(q, limit, slack, kk, spts16, sorted, gp, table, leaf_points, s_stack[warp]);
            const bool have = key != ~0ull;
            const int cnt = __popc(__ballot_sync(FULL_MASK, have));
            if (cnt >= 4 && !(nf.x == 0.f && nf.y == 0.f && nf.z == 0.f)) {
                const double nv[3] = {(double)nf.x, (double)nf.y, (double)nf.z};
                double row[3] = {0.0, 0.0, 0.0}, b = 0.0;
                if (have) {
                    const Point16 t = ld_point(pts, (uint32_t)(key & idxmask));
                    const double d[3] = {(double)t.x - (double)q.x, (double)t.y - (double)q.y, (double)t.z - (double)q.z};
                    const double dn = (d[0] * nv[0] + d[1] * nv[1]) + d[2] * nv[2];
#pragma unroll
                    for (int a = 0; a < 3; a++) row[a] = d[a] - dn * nv[a];
                    b = pt_intensity(t) - pt_intensity(q);
                }
                const double w = (double)(cnt - 1);
                const double cr[3] = {w * nv[0], w * nv[1], w * nv[2]};
                double A[3][3], rhs[3];
#pragma unroll
                for (int a = 0; a < 3; a++) {
#pragma unroll
                    for (int c2 = a; c2 < 3; c2++) A[a][c2] = A[c2][a] = warp_sum(row[a] * row[c2]) + cr[a] * cr[c2];
                    rhs[a] = warp_sum(row[a] * b);
                }
                double V[3][3];
                jacobi3_eigen(A, V);
                const double top = fmax(fmax(A[0][0], A[1][1]), A[2][2]);
                double g[3] = {0.0, 0.0, 0.0};
#pragma unroll
                for (int e = 0; e < 3; e++) {
                    if (!(A[e][e] > 1e-12 * top)) continue;
                    const double vb = (V[0][e] * rhs[0] + V[1][e] * rhs[1]) + V[2][e] * rhs[2];
#pragma unroll
                    for (int k = 0; k < 3; k++) g[k] += V[k][e] * (vb / A[e][e]);
                }
                out.x = (float)g[0], out.y = (float)g[1], out.z = (float)g[2];
            }
        }
        if (lane == 0) gradients[self] = out;
    }
}

__device__ __forceinline__ double pick6(const double (&v)[6], int i) {
    return i == 0 ? v[0] : (i == 1 ? v[1] : (i == 2 ? v[2] : (i == 3 ? v[3] : (i == 4 ? v[4] : v[5]))));
}

// The body of icp_plane_match_kernel and icp_colored_match_kernel.  COLORED scales the point-to-plane row by sg and, when
// sp != 0, adds the photometric row of the pair to the same 30 sums (see icp_colored_match_kernel).
template <bool COLORED>
__device__ __forceinline__ void plane_match(const cwipc_point *__restrict__ src, uint32_t ns, const cwipc_point *__restrict__ tgt, uint32_t nt, const cwipc_point *__restrict__ spts,
                                            const uint64_t *__restrict__ sorted, const GridParams &gp, const uint2 *__restrict__ table, uint32_t leaf_points, const IcpParams &ip,
                                            const float4 *__restrict__ normals, const float4 *__restrict__ gradients, double sg, double sp, double *__restrict__ partial) {
    __shared__ __align__(16) FarNode s_stack[ICP_WARPS][KF_STACK];
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, warps_total = (gridDim.x * blockDim.x) >> 5;
    const Point16 *spts16 = reinterpret_cast<const Point16 *>(spts);
    // the (a, b) of this lane's term: J_a J_b for lanes 2..22, J_a r for lanes 23..28
    int ja = 0, jb = 0;
    if (lane >= 2 && lane < 23) {
        int t = (int)lane - 2;
        while (t >= 6 - ja) t -= 6 - ja++;
        jb = ja + t;
    } else if (lane >= 23 && lane < 29) {
        ja = (int)lane - 23;
    }
    double acc = 0.0;
    for (uint32_t qi = gwarp; qi < ns; qi += warps_total) {
        const Point16 p = ld_point(src, qi);
        Point16 q;
        q.x = affine_row(ip.m, p.x, p.y, p.z);
        q.y = affine_row(ip.m + 4, p.x, p.y, p.z);
        q.z = affine_row(ip.m + 8, p.x, p.y, p.z);
        q.rgbt = 0u;
        if (!finite_point(q)) continue; // (a non-finite input point, counted below; or a float overflow of the motion)
        const uint64_t key = icp_nearest(q, ip.limit, ip.slack, spts16, sorted, gp, table, leaf_points, s_stack[warp]);
        if (key == ~0ull) continue;
        const Point16 t = ld_point(tgt, (uint32_t)key);
        const float4 nf = normals[(uint32_t)key];
        const double nv[3] = {(double)nf.x, (double)nf.y, (double)nf.z};
        const double pr[3] = {(double)q.x - ip.origin[0], (double)q.y - ip.origin[1], (double)q.z - ip.origin[2]};
        const double qr[3] = {(double)t.x - ip.origin[0], (double)t.y - ip.origin[1], (double)t.z - ip.origin[2]};
        const double r = ((pr[0] - qr[0]) * nv[0] + (pr[1] - qr[1]) * nv[1]) + (pr[2] - qr[2]) * nv[2];
        const double J[6] = {pr[1] * nv[2] - pr[2] * nv[1], pr[2] * nv[0] - pr[0] * nv[2], pr[0] * nv[1] - pr[1] * nv[0], nv[0], nv[1], nv[2]};
        if (!COLORED) {
            double term = 0.0;
            if (lane == 0) term = 1.0;
            else if (lane == 1) term = (double)__uint_as_float((uint32_t)(key >> 32));
            else if (lane < 23) term = pick6(J, ja) * pick6(J, jb);
            else if (lane < 29) term = pick6(J, ja) * r;
            acc += term;
        } else {
            const double JG[6] = {sg * J[0], sg * J[1], sg * J[2], sg * J[3], sg * J[4], sg * J[5]}, rG = sg * r;
            double JI[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, rI = 0.0;
            const bool photo = sp != 0.0;
            if (photo) {
                const float4 gf = gradients[(uint32_t)key];
                const double g[3] = {(double)gf.x, (double)gf.y, (double)gf.z};
                const double proj[3] = {(pr[0] - qr[0]) - r * nv[0], (pr[1] - qr[1]) - r * nv[1], (pr[2] - qr[2]) - r * nv[2]}; // p_proj - q
                const double i0 = ((g[0] * proj[0] + g[1] * proj[1]) + g[2] * proj[2]) + pt_intensity(t);
                const double gn = (g[0] * nv[0] + g[1] * nv[1]) + g[2] * nv[2];
                const double d[3] = {-(g[0] - gn * nv[0]), -(g[1] - gn * nv[1]), -(g[2] - gn * nv[2])};
                JI[0] = sp * (pr[1] * d[2] - pr[2] * d[1]), JI[1] = sp * (pr[2] * d[0] - pr[0] * d[2]), JI[2] = sp * (pr[0] * d[1] - pr[1] * d[0]);
                JI[3] = sp * d[0], JI[4] = sp * d[1], JI[5] = sp * d[2];
                rI = sp * (pt_intensity(p) - i0);
            }
            double term = 0.0;
            if (lane == 0) term = 1.0;
            else if (lane == 1) term = (double)__uint_as_float((uint32_t)(key >> 32));
            else if (lane < 23) term = photo ? pick6(JG, ja) * pick6(JG, jb) + pick6(JI, ja) * pick6(JI, jb) : pick6(JG, ja) * pick6(JG, jb);
            else if (lane < 29) term = photo ? pick6(JG, ja) * rG + pick6(JI, ja) * rI : pick6(JG, ja) * rG;
            acc += term;
        }
    }
    if (ip.check) {
        uint32_t bad = 0;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += gridDim.x * blockDim.x) bad += finite_point(ld_point_stream(src, i)) ? 0u : 1u;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nt; i += gridDim.x * blockDim.x) bad += finite_point(ld_point_stream(tgt, i)) ? 0u : 1u;
        bad = warp_sum(bad);
        if (lane == ICP_PLANE_NSUMS - 1) acc = (double)bad;
    }
    if (lane < ICP_PLANE_NSUMS) partial[(size_t)gwarp * ICP_PLANE_NSUMS + lane] = acc;
}

// icp_match_kernel's correspondences (the same search, bound and tie rule) with the point-to-plane sums: for a pair (p', q)
// with target normal n, r = (p' - q) . n and J = [p' x n, n], p' relative to ip.origin, all in double.  Lane j adds up term
// j of ICP_PLANE_NSUMS over the warp's correspondences in the warp's query order: count, sum d2, the 21 entries J_a J_b with
// a <= b (row-major), the 6 entries J_a r; term 29 is the non-finite count of both clouds when ip.check is set.  The warp
// stores them in partial[warp][ICP_PLANE_NSUMS]; icp_plane_reduce_kernel adds them up in warp order.
__global__ void __launch_bounds__(ICP_THREADS) icp_plane_match_kernel(const cwipc_point *__restrict__ src, uint32_t ns, const cwipc_point *__restrict__ tgt, uint32_t nt,
                                                                      const cwipc_point *__restrict__ spts, const uint64_t *__restrict__ sorted, const __grid_constant__ GridParams gp,
                                                                      const uint2 *__restrict__ table, uint32_t leaf_points, const __grid_constant__ IcpParams ip,
                                                                      const float4 *__restrict__ normals, double *__restrict__ partial) {
    plane_match<false>(src, ns, tgt, nt, spts, sorted, gp, table, leaf_points, ip, normals, nullptr, 1.0, 0.0, partial);
}

// icp_plane_match_kernel with the colored-ICP sums (Park, Zhou and Koltun, ICCV 2017; open3d's
// TransformationEstimationForColoredICP): for a pair (p', q) with target normal n, target gradient g = gradients[q] and
// intensities I_s (source point) and I_t (target point), the geometric row J_G = sg [p' x n, n], r_G = sg (p' - q) . n and
// the photometric row J_I = sp [p' x d, d], r_I = sp (I_s - I_0) with p_proj = p' - ((p' - q) . n) n,
// I_0 = g . (p_proj - q) + I_t and d = -(g - (g . n) n).  Lanes 2..28 add J_G J_G^T + J_I J_I^T and J_G r_G + J_I r_I in
// icp_plane_match_kernel's layout, so icp_plane_reduce_kernel adds them up.  sp == 0 (lambda_geometric = 1) skips the
// photometric row, and with sg == 1 the sums are icp_plane_match_kernel's bit for bit.
__global__ void __launch_bounds__(ICP_THREADS) icp_colored_match_kernel(const cwipc_point *__restrict__ src, uint32_t ns, const cwipc_point *__restrict__ tgt, uint32_t nt,
                                                                        const cwipc_point *__restrict__ spts, const uint64_t *__restrict__ sorted, const __grid_constant__ GridParams gp,
                                                                        const uint2 *__restrict__ table, uint32_t leaf_points, const __grid_constant__ IcpParams ip,
                                                                        const float4 *__restrict__ normals, const float4 *__restrict__ gradients, double sg, double sp,
                                                                        double *__restrict__ partial) {
    plane_match<true>(src, ns, tgt, nt, spts, sorted, gp, table, leaf_points, ip, normals, gradients, sg, sp, partial);
}

// icp_reduce_kernel's fixed order for the ICP_PLANE_NSUMS sums of icp_plane_match_kernel.
__global__ void __launch_bounds__(ICP_PLANE_NSUMS * 32) icp_plane_reduce_kernel(const double *__restrict__ partial, uint32_t nwarps, double *__restrict__ out) {
    const unsigned lane = lane_id(), j = threadIdx.x >> 5;
    double s = 0.0;
    for (uint32_t w = lane; w < nwarps; w += 32) s += partial[(size_t)w * ICP_PLANE_NSUMS + j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(FULL_MASK, s, o);
    if (lane == 0) out[j] = s;
}

} // namespace

namespace {
void knn_mean_distances_banded(const cwipc_point *in, size_t n, int k, float hint_spacing, const float *bounds, float *d_dist, int dev, cudaStream_t s, float *d_kth, size_t nquery,
                               const BandLut *lut, int bands) {
    if (n == 0) return;
    check_k(k, n);
    if ((size_t)k >= n) throw CudaError{cudaErrorInvalidValue, "remove_outliers: needs more than kNeighbors points"};
    KnnIndex ix;
    build_index(ix, in, n, k, hint_spacing, bounds, dev, s, lut, bands);
    // a query is queued at most once
    Scratch far_list(2 * (n + 64) * sizeof(FarEntry), s); // the main pass's queue, and what the second scan passes on
    const int kk = k + 1;
    auto go = [&](auto kcap) {
        run_knn<decltype(kcap)::value>(ix.spts.as<cwipc_point>(), ix.sorted, n, ix.gp, k, ix.table.as<uint2>(), d_dist, d_kth, std::min(nquery, n), far_list.as<FarEntry>(),
                                       ix.far_count, dev, s);
    };
    auto go_wide = [&](auto kpl) {
        run_knn_wide<decltype(kpl)::value>(ix.spts.as<cwipc_point>(), ix.sorted, n, ix.gp, k, ix.table.as<uint2>(), d_dist, d_kth, std::min(nquery, n), far_list.as<FarEntry>(), ix.far_count,
                                           dev, s);
    };
    if (kk <= 8) go(std::integral_constant<int, 8>{});
    else if (kk <= 16) go(std::integral_constant<int, 16>{});
    else if (kk <= 32) go(std::integral_constant<int, 32>{});
    else if (kk <= 64) go(std::integral_constant<int, 64>{});
    else if (kk <= 128) go_wide(std::integral_constant<int, 4>{});
    else if (kk <= 256) go_wide(std::integral_constant<int, 8>{});
    else go_wide(std::integral_constant<int, 16>{});
}
} // namespace

void knn_mean_distances(const cwipc_point *in, size_t n, int k, float hint_spacing, const float *bounds, float *d_dist, int dev, cudaStream_t s, float *d_kth, size_t nquery) {
    knn_mean_distances_banded(in, n, k, hint_spacing, bounds, d_dist, dev, s, d_kth, nquery, nullptr, 1);
}

void knn_lists(const cwipc_point *in, size_t n, const cwipc_point *d_queries, const float *d_limits, size_t nq, int k, float hint_spacing, const float *bounds, float *d_lists, int dev,
               cudaStream_t s) {
    check_k(k, n);
    if (nq == 0) return;
    const int kk = k + 1;
    if (n == 0) { // nothing to answer with: every list is all +inf (0x7f800000)
        std::vector<float> inf(nq * (size_t)kk, INFINITY);
        CWCU_CHECK(cudaMemcpyAsync(d_lists, inf.data(), inf.size() * sizeof(float), cudaMemcpyHostToDevice, s));
        stream_sync(s);
        return;
    }
    KnnIndex ix;
    build_index(ix, in, n, k, hint_spacing, bounds, dev, s);
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min(div_up(nq, (size_t)KF_WARPS), (size_t)sm_count(dev) * 8));
    launch("knn_list_kernel", s, (size_t)0, [&] {
        auto go = [&](auto kpl) {
            knn_list_kernel<decltype(kpl)::value><<<grid, KF_THREADS, 0, s>>>(ix.spts.as<cwipc_point>(), (uint32_t)n, ix.gp, kk, ix.table.as<uint2>(), d_queries, d_limits, (uint32_t)nq, d_lists,
                                                                              FAR_LEAF_POINTS);
        };
        if (kk <= 32) go(std::integral_constant<int, 1>{});
        else if (kk <= 64) go(std::integral_constant<int, 2>{});
        else if (kk <= 128) go(std::integral_constant<int, 4>{});
        else if (kk <= 256) go(std::integral_constant<int, 8>{});
        else go(std::integral_constant<int, 16>{});
    });
}

void knn_merge_lists(const float *d_lists, size_t nlists, size_t nq, int k, float *d_mean, float *d_kth, cudaStream_t s) {
    if (nq == 0) return;
    if (nlists == 0 || nlists > 16) throw CudaError{cudaErrorInvalidValue, "knn_merge_lists: between 1 and 16 lists per query"};
    launch("knn_merge_lists_kernel", s, (size_t)0, [&] {
        knn_merge_lists_kernel<<<(unsigned)div_up(nq, 128), 128, 0, s>>>(d_lists, (uint32_t)nlists, (uint32_t)nq, k + 1, k, d_mean, d_kth);
    });
}

void distance_stats(const float *d_dist, size_t n, double out[2], cudaStream_t s) {
    out[0] = out[1] = 0.0;
    if (n == 0) return;
    Scratch partial(2 * ST_BLOCKS * sizeof(double), s);
    launch("stats_kernel", s, 4 * n, [&] { stats_kernel<<<ST_BLOCKS, ST_THREADS, 0, s>>>(d_dist, (uint32_t)n, partial.as<double>()); });
    double *h = static_cast<double *>(thread_pinned(2 * ST_BLOCKS * sizeof(double)));
    CWCU_CHECK(cudaMemcpyAsync(h, partial.p, 2 * ST_BLOCKS * sizeof(double), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
    for (int b = 0; b < ST_BLOCKS; b++) {
        out[0] += h[2 * b];
        out[1] += h[2 * b + 1];
    }
}

namespace {
__global__ void __launch_bounds__(256) mark_open_kernel(const cwipc_point *__restrict__ pts, const float *__restrict__ kth2, uint32_t nquery, float x_lo, float x_hi,
                                                         uint32_t *__restrict__ open_idx, uint32_t *__restrict__ counter) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool open = false;
    if (i < nquery) {
        open = true;
        if (kth2) {
            const double x = (double)ld_point(pts, i).x;
            const double rk = sqrt((double)kth2[i]) * (1.0 + 1e-6);
            open = !(x - rk > (double)x_lo && x + rk < (double)x_hi); // also open when kth2 is +inf or NaN
        }
    }
    const unsigned m = __ballot_sync(FULL_MASK, open);
    if (m == 0u) return;
    const unsigned lane = lane_id();
    uint32_t first = 0;
    if (lane == (unsigned)(__ffs(m) - 1)) first = atomicAdd(counter, (uint32_t)__popc(m));
    first = __shfl_sync(FULL_MASK, first, __ffs(m) - 1);
    if (open) open_idx[first + __popc(m & lanemask_lt())] = i;
}
template <class Index> // uint32_t, or uint64_t words with the index in their low 32 bits
__global__ void __launch_bounds__(256) gather_points_kernel(const cwipc_point *__restrict__ pts, const Index *__restrict__ idx, uint32_t n, cwipc_point *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) st_point(out, i, ld_point(pts, (uint32_t)idx[i]));
}
__global__ void __launch_bounds__(256) gather_floats_kernel(const float *__restrict__ values, const uint32_t *__restrict__ idx, uint32_t n, float *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = values[idx[i]];
}
__global__ void __launch_bounds__(256) scatter_floats_kernel(const float *__restrict__ values, const uint32_t *__restrict__ idx, uint32_t n, float *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[idx[i]] = values[i];
}
} // namespace

size_t mark_open_queries(const cwipc_point *pts, const float *kth2, size_t nquery, float x_lo, float x_hi, uint32_t *open_idx, int dev, cudaStream_t s) {
    (void)dev;
    if (nquery == 0) return 0;
    Scratch counter(sizeof(uint32_t), s);
    CWCU_CHECK(cudaMemsetAsync(counter.p, 0, sizeof(uint32_t), s));
    launch("mark_open_kernel", s, 20 * nquery, [&] {
        mark_open_kernel<<<(unsigned)div_up(nquery, 256), 256, 0, s>>>(pts, kth2, (uint32_t)nquery, x_lo, x_hi, open_idx, counter.as<uint32_t>());
    });
    uint32_t *h = static_cast<uint32_t *>(thread_pinned(sizeof(uint32_t)));
    CWCU_CHECK(cudaMemcpyAsync(h, counter.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
    return *h;
}

size_t knn_open_queries(const cwipc_point *pts, size_t ncomb, size_t nquery, int k, float hint_spacing, const float *bounds, float x_lo, float x_hi, float *d_mean, float *d_kth2,
                        uint32_t *open_idx, int dev, cudaStream_t s) {
    if (ncomb <= (size_t)k) {
        CWCU_CHECK(cudaMemsetAsync(d_kth2, 0x7f, nquery * sizeof(float), s));
        return mark_open_queries(pts, nullptr, nquery, x_lo, x_hi, open_idx, dev, s);
    }
    Scratch d(ncomb * sizeof(float), s), kth2(ncomb * sizeof(float), s);
    knn_mean_distances(pts, ncomb, k, hint_spacing, bounds, d.as<float>(), dev, s, kth2.as<float>(), nquery);
    CWCU_CHECK(cudaMemcpyAsync(d_mean, d.p, nquery * sizeof(float), cudaMemcpyDeviceToDevice, s));
    CWCU_CHECK(cudaMemcpyAsync(d_kth2, kth2.p, nquery * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return mark_open_queries(pts, kth2.as<float>(), nquery, x_lo, x_hi, open_idx, dev, s);
}

void gather_points(const cwipc_point *pts, const uint32_t *idx, size_t n, cwipc_point *out, cudaStream_t s) {
    if (n == 0) return;
    launch("gather_points_kernel", s, 36 * n, [&] { gather_points_kernel<<<(unsigned)div_up(n, 256), 256, 0, s>>>(pts, idx, (uint32_t)n, out); });
}

void gather_points(const cwipc_point *pts, const uint64_t *words, size_t n, cwipc_point *out, cudaStream_t s) {
    if (n == 0) return;
    launch("gather_points_kernel", s, 40 * n, [&] { gather_points_kernel<<<(unsigned)div_up(n, 256), 256, 0, s>>>(pts, words, (uint32_t)n, out); });
}

void gather_floats(const float *values, const uint32_t *idx, size_t n, float *out, cudaStream_t s) {
    if (n == 0) return;
    launch("gather_floats_kernel", s, 12 * n, [&] { gather_floats_kernel<<<(unsigned)div_up(n, 256), 256, 0, s>>>(values, idx, (uint32_t)n, out); });
}

void scatter_floats(const float *values, const uint32_t *idx, size_t n, float *out, cudaStream_t s) {
    if (n == 0) return;
    launch("scatter_floats_kernel", s, 12 * n, [&] { scatter_floats_kernel<<<(unsigned)div_up(n, 256), 256, 0, s>>>(values, idx, (uint32_t)n, out); });
}

// ref: pcl statistical_outlier_removal.hpp -- mean, unbiased variance, threshold in double
double outlier_threshold(double sum, double sq, double n, float stddev_mul) {
    const double mean = sum / n;
    const double variance = (sq - sum * sum / n) / (n - 1.0);
    const double stddev = std::sqrt(variance);
    return mean + (double)stddev_mul * stddev;
}

size_t remove_outliers_points(const cwipc_point *in, size_t n, cwipc_point *out, int k, float stddev_mul, float hint_spacing, const float *bounds, int dev, cudaStream_t s) {
    if (n == 0) return 0;
    if (k < 1 || (size_t)k >= n) {
        // n <= k is undefined behaviour in the reference (PCL reads k+1 results where FLANN returned fewer);
        // defined here as "keep everything" with a warning, and the oracle does the same.
        log(CWIPC_LOG_LEVEL_WARNING, "cwipc_remove_outliers", "fewer points than kNeighbors+1 (" + std::to_string(n) + " <= " + std::to_string(k) + "): keeping all points");
        CWCU_CHECK(cudaMemcpyAsync(out, in, n * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
        return n;
    }
    Scratch dist(n * sizeof(float), s);
    knn_mean_distances(in, n, k, hint_spacing, bounds, dist.as<float>(), dev, s);
    // statistics and threshold stay on the device: the compaction reads the threshold from memory
    Scratch partial((2 * ST_BLOCKS + 1) * sizeof(double), s);
    uint32_t *counter = static_cast<uint32_t *>(thread_zeroed(dev, ZW_HEADER_BYTES, s)) + 6; // word 6 of the zeroed workspace header
    double *d_thr = partial.as<double>() + 2 * ST_BLOCKS;
    launch("stats_kernel", s, 4 * (size_t)n, [&] {
        stats_threshold_kernel<<<ST_BLOCKS, ST_THREADS, 0, s>>>(dist.as<float>(), (uint32_t)n, partial.as<double>(), counter, (double)stddev_mul, d_thr);
    });
    return compact_points(in, n, out, distance_at_most(dist.as<float>(), d_thr), dev, s);
}

size_t remove_outliers_per_tile(const cwipc_point *in, size_t n, cwipc_point *out, const std::vector<int> &tiles, int k, float stddev_mul, float hint_spacing, const float *bounds,
                                int dev, cudaStream_t s) {
    const size_t T = tiles.size();
    if (n == 0 || T == 0) return 0;
    BandLut lut;
    memset(&lut, 0, sizeof(lut));
    for (size_t t = 0; t < T; t++) {
        if (tiles[t] <= 0 || tiles[t] > 255 || T > 255) throw CudaError{cudaErrorInvalidValue, "remove_outliers_per_tile: tile values must be distinct and in 1..255"};
        lut.rank[tiles[t]] = (uint8_t)t;
    }
    Scratch dist(n * sizeof(float), s);
    knn_mean_distances_banded(in, n, k, hint_spacing, bounds, dist.as<float>(), dev, s, nullptr, (size_t)-1, &lut, (int)T);
    // per group: statistics -> threshold (device), then its survivors behind those of the groups before it
    Scratch partial(3 * ST_BLOCKS * sizeof(double), s);
    Scratch thresholds(T * sizeof(double), s);
    Scratch words((2 * T + 1) * sizeof(uint32_t), s); // totals[0..T] (running end positions in `out`), counts[0..T)
    uint32_t *totals = words.as<uint32_t>(), *counts = totals + T + 1;
    CWCU_CHECK(cudaMemsetAsync(totals, 0, sizeof(uint32_t), s));
    uint32_t *done = static_cast<uint32_t *>(thread_zeroed(dev, ZW_HEADER_BYTES, s)) + 6; // word 6 of the zeroed workspace header
    for (size_t t = 0; t < T; t++) {
        launch("stats_kernel", s, 8 * (size_t)n, [&] {
            stats_threshold_tile_kernel<<<ST_BLOCKS, ST_THREADS, 0, s>>>(dist.as<float>(), in, (uint32_t)n, (uint32_t)tiles[t], k, partial.as<double>(), done, (double)stddev_mul,
                                                                         thresholds.as<double>() + t, counts + t);
        });
        compact_tile_group_chained(in, n, out, tiles[t], dist.as<float>(), thresholds.as<double>() + t, totals + t, totals + t + 1, s);
    }
    uint32_t *h = static_cast<uint32_t *>(thread_pinned((2 * T + 1) * sizeof(uint32_t)));
    CWCU_CHECK(cudaMemcpyAsync(h, words.p, (2 * T + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
    for (size_t t = 0; t < T; t++)
        if (h[T + 1 + t] <= (uint32_t)k)
            log(CWIPC_LOG_LEVEL_WARNING, "cwipc_remove_outliers", "fewer points than kNeighbors+1 (" + std::to_string(h[T + 1 + t]) + " <= " + std::to_string(k) + "): keeping all points");
    profile_add_bytes("compact_kernel", 16 * (size_t)h[T]);
    return h[T];
}

struct IcpMatcher::Impl {
    KnnIndex ix;
    const cwipc_point *target;
    size_t nt;
    double origin[3];
    float slack;
    int dev;
    cudaStream_t s;
    uint32_t max_warps;
    Scratch partial; // [max_warps + 1][nsums]: the warps' sums, then the totals
    Scratch normals; // point-to-plane: float4 per target point, input order (icp_normals_kernel)
    Scratch gradients; // colored: float4 per target point, input order (icp_gradients_kernel)
    double sg = 1.0, sp = 0.0; // colored: the weights of the geometric and the photometric row

    Impl(const cwipc_point *target, size_t nt, float hint_spacing, const float *bounds, int k, int nsums, int dev, cudaStream_t s) : target(target), nt(nt), dev(dev), s(s) {
        float box[6];
        if (bounds) {
            memcpy(box, bounds, sizeof(box));
        } else {
            global_bbox(target, nt, box, box + 3, dev, s);
            for (int a = 0; a < 6; a++)
                if (!std::isfinite(box[a])) throw CudaError{cudaErrorInvalidValue, "the target contains non-finite coordinates"};
        }
        float maxabs = 0.f;
        for (int a = 0; a < 3; a++) {
            origin[a] = 0.5 * ((double)box[a] + (double)box[3 + a]);
            maxabs = std::max(maxabs, std::max(std::fabs(box[a]), std::fabs(box[3 + a])));
        }
        build_index(ix, target, nt, k, hint_spacing, box, dev, s);
        // a node's box corners are rounded to float like the points themselves: allow a few units in the last place of the
        // largest coordinate besides the 0.01 pitch of cell_u's rounding
        slack = std::max(0.01f * ix.gp.h, 8.f * std::ldexp(maxabs, -23));
        max_warps = (uint32_t)sm_count(dev) * ICP_BLOCKS_PER_SM * ICP_WARPS;
        partial = Scratch(((size_t)max_warps + 1) * nsums * sizeof(double), s);
    }
    unsigned grid(size_t n) const { return (unsigned)std::max<size_t>(1, std::min(div_up(n, (size_t)ICP_WARPS), (size_t)sm_count(dev) * ICP_BLOCKS_PER_SM)); }
};

IcpMatcher::IcpMatcher(const cwipc_point *target, size_t nt, float hint_spacing, const float *bounds, int dev, cudaStream_t s)
    : m(new Impl(target, nt, hint_spacing, bounds, 1, ICP_NSUMS, dev, s)) {}

IcpMatcher::IcpMatcher(const cwipc_point *target, size_t nt, float hint_spacing, const float *bounds, int dev, cudaStream_t s, double normal_radius, int normal_max_nn)
    : m(new Impl(target, nt, hint_spacing, bounds, normal_max_nn, ICP_PLANE_NSUMS, dev, s)) {
    m->normals = Scratch(nt * sizeof(float4), s);
    const float limit = (float)(normal_radius * normal_radius);
    launch("icp_normals_kernel", s, 16 * nt, [&] {
        icp_normals_kernel<<<m->grid(nt), ICP_THREADS, 0, s>>>(target, (uint32_t)nt, m->ix.spts.as<cwipc_point>(), m->ix.sorted, m->ix.gp, m->ix.table.as<uint2>(), FAR_LEAF_POINTS, limit,
                                                            m->slack, normal_max_nn, m->normals.as<float4>());
    });
}

IcpMatcher::IcpMatcher(const cwipc_point *target, size_t nt, float hint_spacing, const float *bounds, int dev, cudaStream_t s, double normal_radius, int normal_max_nn,
                       double gradient_radius, int gradient_max_nn, double lambda_geometric)
    : IcpMatcher(target, nt, hint_spacing, bounds, dev, s, normal_radius, normal_max_nn) {
    m->gradients = Scratch(nt * sizeof(float4), s);
    m->sg = std::sqrt(lambda_geometric);
    m->sp = std::sqrt(1.0 - lambda_geometric);
    const float limit = (float)(gradient_radius * gradient_radius);
    launch("icp_gradients_kernel", s, 16 * nt, [&] {
        icp_gradients_kernel<<<m->grid(nt), ICP_THREADS, 0, s>>>(target, (uint32_t)nt, m->ix.spts.as<cwipc_point>(), m->ix.sorted, m->ix.gp, m->ix.table.as<uint2>(), FAR_LEAF_POINTS,
                                                              limit, m->slack, gradient_max_nn, m->normals.as<float4>(), m->gradients.as<float4>());
    });
}

IcpMatcher::~IcpMatcher() = default;

const double *IcpMatcher::origin() const { return m->origin; }

int IcpMatcher::nsums() const { return m->normals.p ? ICP_PLANE_NSUMS : ICP_NSUMS; }

void IcpMatcher::evaluate(const cwipc_point *source, size_t ns, const double motion[16], float limit, bool check_finite, double *sums) {
    IcpParams ip;
    memcpy(ip.m, motion, sizeof(ip.m));
    memcpy(ip.origin, m->origin, sizeof(ip.origin));
    ip.limit = limit;
    ip.slack = m->slack;
    ip.check = check_finite ? 1u : 0u;
    const unsigned grid = m->grid(ns);
    const uint32_t nwarps = grid * ICP_WARPS;
    const int nsum = nsums();
    double *partial = m->partial.as<double>(), *d_out = partial + (size_t)m->max_warps * nsum;
    if (!m->normals.p) {
        launch("icp_match_kernel", m->s, 16 * ns, [&] {
            icp_match_kernel<<<grid, ICP_THREADS, 0, m->s>>>(source, (uint32_t)ns, m->target, (uint32_t)m->nt, m->ix.spts.as<cwipc_point>(), m->ix.sorted, m->ix.gp, m->ix.table.as<uint2>(),
                                                            FAR_LEAF_POINTS, ip, partial);
        });
        launch("icp_reduce_kernel", m->s, 8 * (size_t)nwarps * ICP_NSUMS, [&] { icp_reduce_kernel<<<1, ICP_NSUMS * 32, 0, m->s>>>(partial, nwarps, d_out); });
    } else {
        if (!m->gradients.p) {
            launch("icp_plane_match_kernel", m->s, 16 * ns, [&] {
                icp_plane_match_kernel<<<grid, ICP_THREADS, 0, m->s>>>(source, (uint32_t)ns, m->target, (uint32_t)m->nt, m->ix.spts.as<cwipc_point>(), m->ix.sorted, m->ix.gp,
                                                                      m->ix.table.as<uint2>(), FAR_LEAF_POINTS, ip, m->normals.as<float4>(), partial);
            });
        } else {
            launch("icp_colored_match_kernel", m->s, 16 * ns, [&] {
                icp_colored_match_kernel<<<grid, ICP_THREADS, 0, m->s>>>(source, (uint32_t)ns, m->target, (uint32_t)m->nt, m->ix.spts.as<cwipc_point>(), m->ix.sorted, m->ix.gp,
                                                                        m->ix.table.as<uint2>(), FAR_LEAF_POINTS, ip, m->normals.as<float4>(), m->gradients.as<float4>(), m->sg,
                                                                        m->sp, partial);
            });
        }
        launch("icp_plane_reduce_kernel", m->s, 8 * (size_t)nwarps * ICP_PLANE_NSUMS,
               [&] { icp_plane_reduce_kernel<<<1, ICP_PLANE_NSUMS * 32, 0, m->s>>>(partial, nwarps, d_out); });
    }
    double *h = static_cast<double *>(thread_pinned(nsum * sizeof(double)));
    CWCU_CHECK(cudaMemcpyAsync(h, d_out, nsum * sizeof(double), cudaMemcpyDeviceToHost, m->s));
    stream_sync(m->s);
    memcpy(sums, h, nsum * sizeof(double));
}

namespace {
// xyz of n float4 (w: 0, or 1 for a point with a non-finite coordinate) to out[3 n]; false when a w is not 0
bool float4_xyz_to_host(const void *d, size_t n, float *out, cudaStream_t s) {
    float4 *h = static_cast<float4 *>(thread_pinned(n * sizeof(float4)));
    CWCU_CHECK(cudaMemcpyAsync(h, d, n * sizeof(float4), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
    bool finite = true;
    for (size_t i = 0; i < n; i++) {
        out[3 * i] = h[i].x, out[3 * i + 1] = h[i].y, out[3 * i + 2] = h[i].z;
        finite = finite && h[i].w == 0.f;
    }
    return finite;
}
} // namespace

bool IcpMatcher::normals_to_host(float *out) { return float4_xyz_to_host(m->normals.p, m->nt, out, m->s); }

bool IcpMatcher::gradients_to_host(float *out) { return float4_xyz_to_host(m->gradients.p, m->nt, out, m->s); }

} // namespace cwcu
