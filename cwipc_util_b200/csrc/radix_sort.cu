// radix_sort.cu -- stable LSD radix sort of 64-bit words, 8-bit digits, one read + one write of the
// data per digit ("onesweep": the digit histograms of every pass are taken up front in one read; each
// pass ranks a 4096-key tile with warp match_any, chains tiles by decoupled look-back per digit and
// scatters through shared memory so that global stores are run-contiguous).
//
// It replaces boost::sort::spreadsort inside pcl::VoxelGrid (call sites src/cwipc_filters.cpp:52-56,
// 135-140) and provides the uniform-grid ordering for the kNN of cwipc_remove_outliers.
// The words carry the point index in their low bits, below begin_bit, so no separate payload moves.
//
// HBM-bound: per pass 8 B read + 8 B written per key (+ 8 B per key once for the histograms).
#include "radix_sort.hpp"

#include <cooperative_groups.h>
#include <cstring>
#include <mutex>

#include "device_utils.cuh"

namespace cwcu {

namespace {

constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ITEMS = 16;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS; // 4096 keys = 32 KB
constexpr int RS_BINS = 256;
constexpr int RS_MAX_PASSES = 8;

constexpr uint32_t ST_FLAG_SHIFT = 30;
constexpr uint32_t ST_VALUE_MASK = (1u << 30) - 1;
constexpr uint32_t ST_AGGREGATE = 1u << 30, ST_PREFIX = 2u << 30;

__device__ __forceinline__ uint32_t digit_of(uint64_t key, int shift, uint32_t mask) { return (uint32_t)(key >> shift) & mask; }

// Digit histograms of all passes in one read.  Equal digits in neighbouring lanes (the common case for
// the high digits of spatial keys) are merged with one ballot before touching shared memory.
__global__ void __launch_bounds__(RS_THREADS) radix_hist_kernel(const uint64_t *__restrict__ keys, uint32_t n, int begin_bit, int end_bit, int npasses,
                                                                 uint32_t *__restrict__ hist) {
    __shared__ uint32_t s_hist[RS_MAX_PASSES * RS_BINS];
    for (int i = threadIdx.x; i < npasses * RS_BINS; i += RS_THREADS) s_hist[i] = 0;
    __syncthreads();
    const unsigned lane = lane_id();
    const uint32_t stride = gridDim.x * RS_THREADS;
    for (uint32_t base = blockIdx.x * RS_THREADS; base < n; base += stride) {
        const uint32_t idx = base + threadIdx.x;
        const bool valid = idx < n;
        const uint64_t key = valid ? keys[idx] : 0ull;
        for (int p = 0; p < npasses; p++) {
            const int shift = begin_bit + 8 * p;
            const int bits = min(8, end_bit - shift);
            const uint32_t d = valid ? digit_of(key, shift, (1u << bits) - 1u) : 0x100u;
            const uint32_t prev = __shfl_up_sync(FULL_MASK, d, 1);
            const bool head = (lane == 0) || (d != prev);
            const unsigned heads = __ballot_sync(FULL_MASK, head);
            if (head && valid) {
                const unsigned above = heads & ~((2u << lane) - 1u);
                const int next = above ? (__ffs(above) - 1) : 32;
                atomicAdd(&s_hist[p * RS_BINS + d], (uint32_t)(next - (int)lane));
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < npasses * RS_BINS; i += RS_THREADS) {
        const uint32_t v = s_hist[i];
        if (v) atomicAdd(&hist[i], v);
    }
}

// One block per pass: exclusive scan of its 256 digit counts -> first output slot of each digit.
__global__ void __launch_bounds__(RS_BINS) radix_scan_kernel(const uint32_t *__restrict__ hist, uint32_t *__restrict__ binbase) {
    __shared__ uint32_t s_warp[RS_BINS / 32];
    const int p = blockIdx.x;
    const uint32_t v = hist[p * RS_BINS + threadIdx.x];
    const uint32_t incl = warp_inclusive_scan(v);
    if (lane_id() == 31) s_warp[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t offset = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); w++) offset += s_warp[w];
    binbase[p * RS_BINS + threadIdx.x] = offset + incl - v;
}

__global__ void __launch_bounds__(RS_THREADS) radix_onesweep_kernel(const uint64_t *__restrict__ in, uint64_t *__restrict__ out, uint32_t n, int shift, int bits,
                                                                     const uint32_t *__restrict__ binbase, uint32_t *__restrict__ ticket, uint32_t *__restrict__ status) {
    __shared__ uint32_t s_warp_hist[RS_WARPS][RS_BINS]; // counts, then exclusive offsets across warps
    __shared__ uint32_t s_bin_excl[RS_BINS];            // first staging slot of each digit
    __shared__ uint32_t s_bin_out[RS_BINS];             // global slot of staging slot 0 of each digit (biased)
    __shared__ uint32_t s_scan[RS_WARPS];
    __shared__ uint64_t s_keys[RS_TILE];
    __shared__ int s_tile;

    if (threadIdx.x == 0) s_tile = take_ticket(ticket);
#pragma unroll
    for (int w = 0; w < RS_WARPS; w++) s_warp_hist[w][threadIdx.x] = 0;
    __syncthreads();
    const int tile = s_tile;
    const uint32_t tile_base = (uint32_t)tile * RS_TILE;
    if (tile_base >= n) return;
    const uint32_t tile_count = min((uint32_t)RS_TILE, n - tile_base);

    const unsigned warp = threadIdx.x >> 5, lane = lane_id();
    const unsigned lt = lanemask_lt();
    const uint32_t mask = (1u << bits) - 1u;
    const uint32_t warp_base = tile_base + warp * (32 * RS_ITEMS);

    // ---- load (warp-striped: memory order == (item, lane) order inside each warp) ----
    uint64_t key[RS_ITEMS];
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const uint32_t idx = warp_base + i * 32 + lane;
        key[i] = idx < n ? in[idx] : ~0ull;
    }

    // ---- rank inside the warp, digit by digit row ----
    uint32_t rank[RS_ITEMS];
    uint32_t *my_hist = s_warp_hist[warp];
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const uint32_t idx = warp_base + i * 32 + lane;
        const bool valid = idx < n;
        const uint32_t d = valid ? digit_of(key[i], shift, mask) : 0x100u;
        const unsigned peers = __match_any_sync(FULL_MASK, d);
        // every peer reads the running count (one broadcast per digit), the lowest one bumps it: no shuffle on the chain
        const uint32_t before = valid ? my_hist[d] : 0u;
        __syncwarp();
        if (valid && (peers & lt) == 0u) my_hist[d] = before + __popc(peers);
        rank[i] = before + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();

    // ---- per digit (thread == digit): offsets across warps, tile count, chained prefix over tiles ----
    const uint32_t d = threadIdx.x;
    uint32_t count = 0;
#pragma unroll
    for (int w = 0; w < RS_WARPS; w++) {
        const uint32_t c = s_warp_hist[w][d];
        s_warp_hist[w][d] = count;
        count += c;
    }
    uint32_t exclusive = 0;
    {
        uint32_t *mine = status + (size_t)tile * RS_BINS + d;
        if (tile == 0) {
            st_volatile_u32(mine, ST_PREFIX | count);
        } else {
            st_volatile_u32(mine, ST_AGGREGATE | count);
            int t = tile - 1;
            while (true) {
                uint32_t s;
                do {
                    s = ld_volatile_u32(status + (size_t)t * RS_BINS + d);
                } while ((s >> ST_FLAG_SHIFT) == 0u);
                exclusive += s & ST_VALUE_MASK;
                if ((s >> ST_FLAG_SHIFT) == 2u) break;
                --t;
            }
            st_volatile_u32(mine, ST_PREFIX | (exclusive + count));
        }
    }
    // block-wide exclusive scan of the digit counts -> staging layout
    {
        const uint32_t incl = warp_inclusive_scan(count);
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        uint32_t offset = 0;
        for (int w = 0; w < (int)warp; w++) offset += s_scan[w];
        const uint32_t excl_in_tile = offset + incl - count;
        s_bin_excl[d] = excl_in_tile;
        s_bin_out[d] = binbase[d] + exclusive - excl_in_tile;
    }
    __syncthreads();

    // ---- stage: keys land in shared memory grouped by digit, original order inside a digit ----
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const uint32_t idx = warp_base + i * 32 + lane;
        if (idx < n) {
            const uint32_t dd = digit_of(key[i], shift, mask);
            s_keys[s_bin_excl[dd] + my_hist[dd] + rank[i]] = key[i];
        }
    }
    __syncthreads();

    // ---- scatter: consecutive threads write consecutive slots of a digit's run ----
#pragma unroll
    for (int j = 0; j < RS_ITEMS; j++) {
        const uint32_t p = j * RS_THREADS + threadIdx.x;
        if (p < tile_count) {
            const uint64_t k = s_keys[p];
            out[s_bin_out[digit_of(k, shift, mask)] + p] = k;
        }
    }
}

// ---- small inputs: every pass in ONE cooperative launch ------------------------------------------------
// Up to one 4096-key tile per co-resident block.  Per pass: rank the tile (same warp match_any ranking
// as above), publish its 256 digit counts, grid barrier, every block sums the counts of the tiles
// before it and of all tiles (no look-back chain, no per-pass launch), scatter, grid barrier.  A sort
// of a few hundred thousand keys is launch- and latency-bound; this removes 2 + P launches.
constexpr int RF_BITS = 9;                 // digit width of the fused path (per-warp histograms: 8 x 512 x 4 B)
constexpr int RF_BINS = 1 << RF_BITS;
constexpr int RF_DPT = RF_BINS / RS_THREADS; // digits per thread (contiguous)

constexpr size_t RF_SMEM_BYTES = RS_TILE * sizeof(uint64_t) + (size_t)(RS_WARPS + 2) * RF_BINS * sizeof(uint32_t) + 2 * RS_WARPS * sizeof(uint32_t);

// pass widths: as few passes as RF_BITS allows, evenly wide
__host__ __device__ __forceinline__ int fused_passes(int bits) { return (bits + RF_BITS - 1) / RF_BITS; }

// Grid barrier for the cooperative launch (all blocks are co-resident): one arrival per block on a monotonic
// counter, acquire-spin until the k-th multiple of the block count.  Lighter than cg::grid.sync(), which costs
// several microseconds per call here -- more than a whole pass over a 4096-key tile.
__device__ __forceinline__ void grid_barrier(uint32_t *counter, uint32_t target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        uint32_t seen;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
        } while (seen < target);
        __threadfence();
    }
    __syncthreads();
}

__global__ void __launch_bounds__(RS_THREADS) radix_fused_kernel(uint64_t *__restrict__ a, uint64_t *__restrict__ b, uint32_t n, int begin_bit, int end_bit,
                                                                  uint32_t *__restrict__ tile_hist /* [2][ntiles][RF_BINS] */, uint32_t *__restrict__ sync_words /* [2], zero */) {
    uint32_t nbarriers = 0;
    extern __shared__ __align__(16) unsigned char rf_smem[]; // RF_SMEM_BYTES, above the 48 KB static limit
    uint64_t *s_keys = reinterpret_cast<uint64_t *>(rf_smem);                               // [RS_TILE]
    uint32_t(*s_warp_hist)[RF_BINS] = reinterpret_cast<uint32_t(*)[RF_BINS]>(s_keys + RS_TILE); // [RS_WARPS][RF_BINS]
    uint32_t *s_bin_excl = &s_warp_hist[RS_WARPS][0];                                       // [RF_BINS]
    uint32_t *s_bin_out = s_bin_excl + RF_BINS;                                             // [RF_BINS]
    uint32_t(*s_scan)[RS_WARPS] = reinterpret_cast<uint32_t(*)[RS_WARPS]>(s_bin_out + RF_BINS); // [2][RS_WARPS]

    const uint32_t tile = blockIdx.x, ntiles = gridDim.x;
    const uint32_t tile_base = tile * RS_TILE;
    const uint32_t tile_count = tile_base < n ? min((uint32_t)RS_TILE, n - tile_base) : 0u;
    const unsigned warp = threadIdx.x >> 5, lane = lane_id();
    const unsigned lt = lanemask_lt();
    const uint32_t warp_base = tile_base + warp * (32 * RS_ITEMS);
    uint64_t *src = a, *dst = b;
    const int npasses = fused_passes(end_bit - begin_bit);
    int shift = begin_bit;
    for (int pass = 0; pass < npasses; pass++) {
        const int bits = (end_bit - shift + (npasses - pass) - 1) / (npasses - pass);
        const uint32_t mask = (1u << bits) - 1u;
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++)
#pragma unroll
            for (int j = 0; j < RF_DPT; j++) s_warp_hist[w][threadIdx.x * RF_DPT + j] = 0;
        __syncthreads();

        uint64_t key[RS_ITEMS];
#pragma unroll
        for (int i = 0; i < RS_ITEMS; i++) {
            const uint32_t idx = warp_base + i * 32 + lane;
            key[i] = idx < n ? src[idx] : ~0ull;
        }
        uint32_t rank[RS_ITEMS];
        uint32_t *my_hist = s_warp_hist[warp];
#pragma unroll
        for (int i = 0; i < RS_ITEMS; i++) {
            const uint32_t idx = warp_base + i * 32 + lane;
            const bool valid = idx < n;
            const uint32_t dg = valid ? digit_of(key[i], shift, mask) : 0xffffu;
            const unsigned peers = __match_any_sync(FULL_MASK, dg);
            // every peer reads the running count (one broadcast per digit), the lowest one bumps it: no shuffle on the chain
            const uint32_t before = valid ? my_hist[dg] : 0u;
            __syncwarp();
            if (valid && (peers & lt) == 0u) my_hist[dg] = before + __popc(peers);
            rank[i] = before + __popc(peers & lt);
            __syncwarp();
        }
        __syncthreads();

        // my RF_DPT digits: offsets across warps, tile counts
        uint32_t count[RF_DPT];
        uint32_t *hist = tile_hist + (size_t)(pass & 1) * ntiles * RF_BINS;
#pragma unroll
        for (int j = 0; j < RF_DPT; j++) {
            const uint32_t d = threadIdx.x * RF_DPT + j;
            uint32_t c = 0;
#pragma unroll
            for (int w = 0; w < RS_WARPS; w++) {
                const uint32_t v = s_warp_hist[w][d];
                s_warp_hist[w][d] = c;
                c += v;
            }
            count[j] = c;
            hist[(size_t)tile * RF_BINS + d] = c;
        }
        grid_barrier(sync_words, ++nbarriers * ntiles);

        // keys with my digits in earlier tiles and in all tiles
        uint32_t before_tiles[RF_DPT], total[RF_DPT];
#pragma unroll
        for (int j = 0; j < RF_DPT; j++) before_tiles[j] = total[j] = 0;
        for (uint32_t t = 0; t < ntiles; t++) {
#pragma unroll
            for (int j = 0; j < RF_DPT; j++) {
                const uint32_t c = __ldcg(hist + (size_t)t * RF_BINS + threadIdx.x * RF_DPT + j);
                if (t < tile) before_tiles[j] += c;
                total[j] += c;
            }
        }
        {
            // block-wide exclusive scans over the digits: totals (global digit base), tile counts (staging layout)
            uint32_t sum_total = 0, sum_count = 0;
#pragma unroll
            for (int j = 0; j < RF_DPT; j++) {
                sum_total += total[j];
                sum_count += count[j];
            }
            const uint32_t incl_total = warp_inclusive_scan(sum_total);
            const uint32_t incl_count = warp_inclusive_scan(sum_count);
            if (lane == 31) {
                s_scan[0][warp] = incl_total;
                s_scan[1][warp] = incl_count;
            }
            __syncthreads();
            uint32_t run_total = incl_total - sum_total, run_count = incl_count - sum_count;
            for (int w = 0; w < (int)warp; w++) {
                run_total += s_scan[0][w];
                run_count += s_scan[1][w];
            }
#pragma unroll
            for (int j = 0; j < RF_DPT; j++) {
                const uint32_t d = threadIdx.x * RF_DPT + j;
                s_bin_excl[d] = run_count;
                s_bin_out[d] = run_total + before_tiles[j] - run_count;
                run_total += total[j];
                run_count += count[j];
            }
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < RS_ITEMS; i++) {
            const uint32_t idx = warp_base + i * 32 + lane;
            if (idx < n) {
                const uint32_t dd = digit_of(key[i], shift, mask);
                s_keys[s_bin_excl[dd] + my_hist[dd] + rank[i]] = key[i];
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < RS_ITEMS; j++) {
            const uint32_t p = j * RS_THREADS + threadIdx.x;
            if (p < tile_count) {
                const uint64_t k = s_keys[p];
                dst[s_bin_out[digit_of(k, shift, mask)] + p] = k;
            }
        }
        grid_barrier(sync_words, ++nbarriers * ntiles);
        uint64_t *t = src;
        src = dst;
        dst = t;
        shift += bits;
    }
    // leave the two words zero for the next launch: the last block to get here resets them (nobody spins any more)
    if (threadIdx.x == 0 && atomicAdd(sync_words + 1, 1u) == ntiles - 1) {
        sync_words[0] = 0;
        sync_words[1] = 0;
    }
}

// ---- up to ~98 K words: the whole sort inside ONE thread-block cluster, keys in distributed shared memory ---
// A cluster of up to 8 CTAs (one per SM, co-scheduled by the hardware) holds the keys in registers between
// ranking and scatter and in shared memory between passes.  Per pass: warp match_any ranking, per-CTA digit
// counts, cluster barrier, every CTA reads the other CTAs' counts through DSMEM, keys are scattered straight
// into the destination CTA's shared memory (st.shared::cluster), cluster barrier.  No global-memory traffic and
// no grid barrier between passes: a cluster barrier costs a few hundred cycles, and the launch is an ordinary one.
constexpr int RC_THREADS = 512;
constexpr int RC_WARPS = RC_THREADS / 32;
constexpr int RC_BITS = 9;
constexpr int RC_BINS = 1 << RC_BITS; // == RC_THREADS: one digit per thread
constexpr int RC_MAX_CTAS = 8;        // portable cluster size.  16-CTA clusters halve the single-stream latency of a 47 K-word
                                      // sort (31 vs 52 us) but lower the multi-stream throughput: a GPC rarely has 12 idle SMs

template <int IPT>
constexpr size_t rc_smem_bytes() { return (size_t)RC_THREADS * IPT * sizeof(uint64_t) + (size_t)(RC_WARPS + 2) * RC_BINS * sizeof(uint32_t) + RC_WARPS * sizeof(uint32_t); }

template <int IPT>
__global__ void __launch_bounds__(RC_THREADS, 1) radix_cluster_kernel(const uint64_t *__restrict__ in, uint64_t *__restrict__ out, uint32_t n, int begin_bit, int end_bit) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const uint32_t nctas = cluster.num_blocks(), cta = cluster.block_rank();
    constexpr uint32_t CAP = RC_THREADS * IPT; // words per CTA
    extern __shared__ __align__(16) unsigned char rc_smem[];
    uint64_t *buf = reinterpret_cast<uint64_t *>(rc_smem);                                       // [CAP] this CTA's words between passes
    uint32_t(*warp_hist)[RC_BINS] = reinterpret_cast<uint32_t(*)[RC_BINS]>(buf + CAP);           // [RC_WARPS][RC_BINS]
    uint32_t *cta_hist = &warp_hist[RC_WARPS][0];                                                // [RC_BINS] read by the other CTAs
    uint32_t *digit_off = cta_hist + RC_BINS;                                                    // [RC_BINS]
    uint32_t *s_scan = digit_off + RC_BINS;                                                      // [RC_WARPS]

    const unsigned warp = threadIdx.x >> 5, lane = lane_id();
    const unsigned lt = lanemask_lt();
    const uint32_t local_base = warp * (32 * IPT);
    const uint32_t warp_base = cta * CAP + local_base;
    const uint32_t d = threadIdx.x;

    uint64_t key[IPT];
#pragma unroll
    for (int i = 0; i < IPT; i++) {
        const uint32_t idx = warp_base + i * 32 + lane;
        key[i] = idx < n ? in[idx] : ~0ull;
    }
    const int npasses = (end_bit - begin_bit + RC_BITS - 1) / RC_BITS;
    int shift = begin_bit;
    for (int pass = 0; pass < npasses; pass++) {
        const int bits = (end_bit - shift + (npasses - pass) - 1) / (npasses - pass);
        const uint32_t mask = (1u << bits) - 1u;
        const bool last = pass + 1 == npasses;
#pragma unroll
        for (int w = 0; w < RC_WARPS; w++) warp_hist[w][d] = 0;
        __syncthreads();

        uint32_t rank[IPT];
        uint32_t *my_hist = warp_hist[warp];
#pragma unroll
        for (int i = 0; i < IPT; i++) {
            const uint32_t idx = warp_base + i * 32 + lane;
            const bool valid = idx < n;
            const uint32_t dg = valid ? digit_of(key[i], shift, mask) : 0xffffu;
            const unsigned peers = __match_any_sync(FULL_MASK, dg);
            // every peer reads the running count (one broadcast per digit), the lowest one bumps it: no shuffle on the chain
            const uint32_t before = valid ? my_hist[dg] : 0u;
            __syncwarp();
            if (valid && (peers & lt) == 0u) my_hist[dg] = before + __popc(peers);
            rank[i] = before + __popc(peers & lt);
            __syncwarp();
        }
        __syncthreads();

        // digit d: offsets across this CTA's warps, CTA count
        uint32_t count = 0;
#pragma unroll
        for (int w = 0; w < RC_WARPS; w++) {
            const uint32_t v = warp_hist[w][d];
            warp_hist[w][d] = count;
            count += v;
        }
        cta_hist[d] = count;
        cluster.sync();

        // counts of digit d in the CTAs before this one and in all CTAs, read through distributed shared memory
        uint32_t before_ctas = 0, total = 0;
        for (uint32_t cc = 0; cc < nctas; cc++) {
            const uint32_t v = *cluster.map_shared_rank(&cta_hist[d], cc);
            if (cc < cta) before_ctas += v;
            total += v;
        }
        {
            const uint32_t incl = warp_inclusive_scan(total);
            if (lane == 31) s_scan[warp] = incl;
            __syncthreads();
            uint32_t off = incl - total;
            for (int w = 0; w < (int)warp; w++) off += s_scan[w];
            digit_off[d] = off + before_ctas; // position of this CTA's first word with digit d
        }
        __syncthreads();

        // scatter: the last pass goes to global memory, the others into the owning CTA's shared memory
#pragma unroll
        for (int i = 0; i < IPT; i++) {
            const uint32_t idx = warp_base + i * 32 + lane;
            if (idx < n) {
                const uint32_t dg = digit_of(key[i], shift, mask);
                const uint32_t pos = digit_off[dg] + my_hist[dg] + rank[i];
                if (last) {
                    out[pos] = key[i];
                } else {
                    *cluster.map_shared_rank(&buf[pos % CAP], pos / CAP) = key[i];
                }
            }
        }
        cluster.sync(); // remote stores have landed; nobody reads cta_hist any more (and no CTA exits early)
        if (!last) {
#pragma unroll
            for (int i = 0; i < IPT; i++) {
                const uint32_t idx = warp_base + i * 32 + lane;
                key[i] = idx < n ? buf[local_base + i * 32 + lane] : ~0ull;
            }
        }
        shift += bits;
    }
}

template <int IPT>
bool launch_cluster_sort(const uint64_t *in, uint64_t *out, size_t n, int begin_bit, int end_bit, int dev, cudaStream_t s) {
    static int ok[64]; // 0 unknown, 1 usable, -1 not usable on this device
    static std::once_flag once[64];
    std::call_once(once[dev & 63], [&] {
        cudaError_t e = cudaFuncSetAttribute(radix_cluster_kernel<IPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rc_smem_bytes<IPT>());
        ok[dev & 63] = (e == cudaSuccess) ? 1 : -1;
        if (e != cudaSuccess) (void)cudaGetLastError();
    });
    if (ok[dev & 63] != 1) return false;
    const size_t cap = (size_t)RC_THREADS * IPT;
    const unsigned nctas = (unsigned)div_up(n, cap);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(nctas);
    cfg.blockDim = dim3(RC_THREADS);
    cfg.dynamicSmemBytes = rc_smem_bytes<IPT>();
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = nctas;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const uint32_t n32 = (uint32_t)n;
    bool launched = true;
    launch("radix_cluster_kernel", s, 16 * n, [&] {
        cudaError_t e = cudaLaunchKernelEx(&cfg, radix_cluster_kernel<IPT>, in, out, n32, begin_bit, end_bit);
        if (e != cudaSuccess) { // e.g. no GPC with enough free SMs configuration: fall back to the cooperative kernel
            (void)cudaGetLastError();
            launched = false;
        }
    });
    return launched;
}

int fused_tile_limit(int dev) {
    static int limit[64];
    static std::once_flag once[64];
    std::call_once(once[dev & 63], [&] {
        int per_sm = 0, coop = 0;
        CWCU_CHECK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
        CWCU_CHECK(cudaFuncSetAttribute(radix_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RF_SMEM_BYTES));
        CWCU_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, radix_fused_kernel, RS_THREADS, RF_SMEM_BYTES));
        limit[dev & 63] = (coop && per_sm > 0) ? sm_count(dev) : 0; // one tile per SM keeps the barriers cheap
    });
    return limit[dev & 63];
}

} // namespace

uint64_t *radix_sort_u64(uint64_t *a, uint64_t *b, size_t n, int begin_bit, int end_bit, int dev, cudaStream_t s) {
    if (n <= 1 || end_bit <= begin_bit) return a;
    if (n >= (1u << 30)) throw CudaError{cudaErrorInvalidValue, "radix_sort_u64: more than 2^30 points are not supported"};
    const int npasses = (end_bit - begin_bit + 7) / 8;
    if (npasses > RS_MAX_PASSES) throw CudaError{cudaErrorInvalidValue, "radix_sort_u64: bit range too wide"};
    const size_t ntiles = div_up(n, RS_TILE);

    // one cluster of <= 8 CTAs sorts up to 8 x 512 x 24 words entirely in distributed shared memory.  A pass is bound
    // by the shared-memory pipe of each SM (match/LDS/STS per key), so the keys are spread over all 8 CTAs: the
    // smallest per-thread count that fits
    const size_t per_ipt = (size_t)RC_MAX_CTAS * RC_THREADS;
    bool done = false;
    if (n <= per_ipt * 2) done = launch_cluster_sort<2>(a, b, n, begin_bit, end_bit, dev, s);
    else if (n <= per_ipt * 4) done = launch_cluster_sort<4>(a, b, n, begin_bit, end_bit, dev, s);
    else if (n <= per_ipt * 8) done = launch_cluster_sort<8>(a, b, n, begin_bit, end_bit, dev, s);
    else if (n <= per_ipt * 12) done = launch_cluster_sort<12>(a, b, n, begin_bit, end_bit, dev, s);
    else if (n <= per_ipt * 16) done = launch_cluster_sort<16>(a, b, n, begin_bit, end_bit, dev, s);
    else if (n <= per_ipt * 24) done = launch_cluster_sort<24>(a, b, n, begin_bit, end_bit, dev, s);
    if (done) return b;
    if ((int)ntiles <= fused_tile_limit(dev)) {
        const int fpasses = fused_passes(end_bit - begin_bit);
        Scratch hist(2 * ntiles * RF_BINS * sizeof(uint32_t), s);
        uint32_t *tile_hist = hist.as<uint32_t>();
        uint32_t n32 = (uint32_t)n;
        uint32_t *sync_words = static_cast<uint32_t *>(thread_zeroed(dev, ZW_HEADER_BYTES, s)) + 4; // words 4,5 of the zeroed workspace header
        void *args[] = {&a, &b, &n32, &begin_bit, &end_bit, &tile_hist, &sync_words};
        launch("radix_fused_kernel", s, 16 * (size_t)n * fpasses, [&] {
            CWCU_CHECK(cudaLaunchCooperativeKernel((const void *)radix_fused_kernel, dim3((unsigned)ntiles), dim3(RS_THREADS), args, RF_SMEM_BYTES, s));
        });
        return (fpasses & 1) ? b : a;
    }

    // [hist P*256 | binbase P*256 | tickets 8 | status P*ntiles*256] (u32 each)
    const size_t hist_words = (size_t)npasses * RS_BINS;
    const size_t status_words = (size_t)npasses * ntiles * RS_BINS;
    const size_t words = 2 * hist_words + 8 + status_words;
    Scratch scratch(words * sizeof(uint32_t), s);
    CWCU_CHECK(cudaMemsetAsync(scratch.p, 0, words * sizeof(uint32_t), s));
    uint32_t *hist = scratch.as<uint32_t>();
    uint32_t *binbase = hist + hist_words;
    uint32_t *tickets = binbase + hist_words;
    uint32_t *status = tickets + 8;

    const unsigned hist_grid = (unsigned)std::max<size_t>(1, std::min(div_up(n, (size_t)RS_THREADS * 8), (size_t)sm_count(dev) * 8));
    launch("radix_hist_kernel", s, 8 * (size_t)n, [&] { radix_hist_kernel<<<hist_grid, RS_THREADS, 0, s>>>(a, (uint32_t)n, begin_bit, end_bit, npasses, hist); });
    launch("radix_scan_kernel", s, (size_t)2048 * npasses, [&] { radix_scan_kernel<<<npasses, RS_BINS, 0, s>>>(hist, binbase); });

    uint64_t *src = a, *dst = b;
    for (int p = 0; p < npasses; p++) {
        const int shift = begin_bit + 8 * p;
        const int bits = std::min(8, end_bit - shift);
        launch("radix_onesweep_kernel", s, 16 * (size_t)n, [&] {
            radix_onesweep_kernel<<<(unsigned)ntiles, RS_THREADS, 0, s>>>(src, dst, (uint32_t)n, shift, bits, binbase + (size_t)p * RS_BINS, tickets + p,
                                                                           status + (size_t)p * ntiles * RS_BINS);
        });
        std::swap(src, dst);
    }
    return src;
}

} // namespace cwcu
