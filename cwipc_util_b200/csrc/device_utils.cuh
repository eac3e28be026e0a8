// device_utils.cuh -- device-side building blocks shared by the filter kernels (sm_100a):
// 128-bit point loads/stores, warp primitives, and the decoupled look-back prefix used by every
// single-pass scan-shaped kernel (stable compaction, radix scatter, run numbering).
#pragma once

#include <cuda_runtime.h>
#include <cstdint>

#include "cwipc_util_cuda.h"

namespace cwcu {

constexpr unsigned FULL_MASK = 0xffffffffu;

// A cwipc_point viewed as one 128-bit word: x,y,z as raw bits, w = r | g<<8 | b<<16 | tile<<24.
struct __align__(16) Point16 {
    float x, y, z;
    uint32_t rgbt;
};
static_assert(sizeof(Point16) == 16, "Point16 must alias cwipc_point");

__device__ __forceinline__ uint32_t pt_tile(const Point16 &p) { return p.rgbt >> 24; }
__device__ __forceinline__ uint32_t pt_r(const Point16 &p) { return p.rgbt & 0xffu; }
__device__ __forceinline__ uint32_t pt_g(const Point16 &p) { return (p.rgbt >> 8) & 0xffu; }
__device__ __forceinline__ uint32_t pt_b(const Point16 &p) { return (p.rgbt >> 16) & 0xffu; }

// Streaming 128-bit load: read-only path, do not pollute L1 (each point is touched once per pass).
__device__ __forceinline__ Point16 ld_point_stream(const cwipc_point *base, size_t i) {
    Point16 p;
    const void *ptr = reinterpret_cast<const Point16 *>(base) + i;
    uint32_t xi, yi, zi;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(xi), "=r"(yi), "=r"(zi), "=r"(p.rgbt)
                 : "l"(ptr));
    p.x = __uint_as_float(xi);
    p.y = __uint_as_float(yi);
    p.z = __uint_as_float(zi);
    return p;
}

// Cached 128-bit load (gathers that may hit the same line again).
__device__ __forceinline__ Point16 ld_point(const cwipc_point *base, size_t i) {
    return *(reinterpret_cast<const Point16 *>(base) + i);
}

__device__ __forceinline__ void st_point(cwipc_point *base, size_t i, const Point16 &p) {
    *(reinterpret_cast<Point16 *>(base) + i) = p;
}

// One output coordinate of an affine map, the arithmetic cwipc_cuda_transform and cwipc_cuda_icp state:
// (float)(((m[0]*x + m[1]*y) + m[2]*z) + m[3]) in double, every product and sum rounded on its own (never fused), the
// result rounded to the nearest float.  m: one row of a row-major 4x4.
__device__ __forceinline__ float affine_row(const double *m, double x, double y, double z) {
    return __double2float_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[0], x), __dmul_rn(m[1], y)), __dmul_rn(m[2], z)), m[3]));
}

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

template <class T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
    return v;
}

__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(FULL_MASK, v, o);
        if (lane_id() >= (unsigned)o) v += t;
    }
    return v;
}

// ------------------------------------------------------------------------------------------
// Decoupled look-back (single-pass chained scan).
//
// status[t] packs {flag:2 | value:32} in one 64-bit word so that one relaxed 8-byte store publishes
// both.  Tiles are handed out by an atomic ticket (never blockIdx), so every predecessor of a
// running tile has itself started: the spin below always terminates.
// The status array (and the ticket counter) must be zeroed before the launch.
// ------------------------------------------------------------------------------------------
constexpr uint64_t LB_EMPTY = 0, LB_AGGREGATE = 1, LB_PREFIX = 2;

__device__ __forceinline__ uint64_t lb_pack(uint64_t flag, uint32_t value) { return (flag << 32) | value; }
__device__ __forceinline__ uint64_t lb_flag(uint64_t s) { return s >> 32; }
__device__ __forceinline__ uint32_t lb_value(uint64_t s) { return (uint32_t)s; }

__device__ __forceinline__ uint64_t ld_volatile_u64(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u64(uint64_t *p, uint64_t v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Called by ALL 32 lanes of one warp.  Publishes `aggregate` for `tile`, returns the exclusive
// prefix (sum of aggregates of tiles 0..tile-1) in every lane, then publishes the inclusive prefix.
__device__ __forceinline__ uint32_t lookback_exclusive(uint64_t *status, int tile, uint32_t aggregate) {
    const unsigned lane = lane_id();
    if (tile == 0) {
        if (lane == 0) st_volatile_u64(&status[0], lb_pack(LB_PREFIX, aggregate));
        return 0;
    }
    if (lane == 0) st_volatile_u64(&status[tile], lb_pack(LB_AGGREGATE, aggregate));
    uint32_t exclusive = 0;
    int base = tile - 1;
    while (true) {
        const int t = base - (int)lane;
        uint64_t s = lb_pack(LB_PREFIX, 0); // tiles before 0: an empty prefix
        if (t >= 0) {
            do {
                s = ld_volatile_u64(&status[t]);
            } while (lb_flag(s) == LB_EMPTY);
        }
        const unsigned prefix_lanes = __ballot_sync(FULL_MASK, lb_flag(s) == LB_PREFIX);
        const int first = prefix_lanes ? (__ffs(prefix_lanes) - 1) : 32;
        uint32_t v = ((int)lane <= first) ? lb_value(s) : 0u;
        exclusive += warp_sum(v);
        if (prefix_lanes) break;
        base -= 32;
    }
    if (lane == 0) st_volatile_u64(&status[tile], lb_pack(LB_PREFIX, exclusive + aggregate));
    return exclusive;
}

// Ticket: the first `ntickets` callers get 0,1,2,... ; called by one thread per block.
__device__ __forceinline__ int take_ticket(uint32_t *counter) { return (int)atomicAdd(counter, 1u); }

} // namespace cwcu
