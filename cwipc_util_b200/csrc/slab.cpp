// slab.cpp -- one large cloud spread over several GPUs as x-slabs (BASELINE.json configs[3]), inside the library:
// one process (or thread) per GPU, NCCL between them (ncclSend / ncclRecv of device buffers for the points that move,
// small all-gathers / all-reduces for the metadata), everything queued on the calling thread's stream, so that kernels and
// transfers are ordered without host synchronisation in between.  libnccl.so.2 is loaded with dlopen on first use: the
// library does not link against NCCL and single-GPU hosts never load it.
//
// Semantics: the WHOLE cloud is the concatenation of the ranks' parts in rank order, and the results are those of
// cwipc_downsample / cwipc_remove_outliers / cwipc_tilefilter (ref: src/cwipc_filters.cpp:89-172, 181-306) on that cloud,
// left partitioned.
//
// slab_downsample
//   1. one all-gather of (cellsize, count, bounding box) per rank;
//   2. octree box: PCL grows the octree's bounding box while points are inserted IN ORDER, so rank 0 replays its part and
//      broadcasts the box state, then rank 1, ... until the box contains the whole cloud's bounding box (it doubles when
//      it grows: usually after the first part);
//   3. a voxel must be reduced by one rank: voxel columns floorf(x / cellsize) are assigned to ranks from the parts' own x
//      minima, and every point that sits in a column owned by another rank is sent there (only the points of boundary
//      voxels move when the parts are proper x-slabs);
//   4. every rank runs the planned downsample (final octree box, whole-cloud bounds) on what it now holds.  Integer sums
//      make the result bit-identical to the single-GPU one.
// slab_remove_outliers (one group; perTile runs it once per tile value)
//   1. all-gather of (cellsize, count, x extent);  2. halo exchange: every rank receives the points within H of its x extent;
//   3. kNN of the local points against local + halo; queries whose (k+1)-th neighbour sphere leaves the covered interval are
//      "open";  4. open queries (point + current bound) are all-gathered, every rank answers with the k+1 smallest distances
//      among its OWN points, the lists return to the owners (all-to-all), who merge them: exact whatever H was;
//   5. sum d, sum d^2, n all-reduced; every rank thresholds its own points.
// slab_tilefilter: local compaction + all-gather of the counts (the global offset of this rank's piece).
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>

#include "kernels.hpp"
#include "pointcloud.hpp"

using namespace cwcu;

namespace {

// ---- the few NCCL entry points the protocol needs, resolved at run time (declarations restated from nccl.h) --------
typedef struct ncclComm *ncclComm_t;
struct ncclUniqueId {
    char internal[128];
};
enum { NCCL_UINT8 = 1, NCCL_INT32 = 2, NCCL_UINT64 = 5, NCCL_FLOAT32 = 7, NCCL_FLOAT64 = 8 };
enum { NCCL_SUM = 0 };

struct Nccl {
    void *handle = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Send)(const void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    std::string error;
};

Nccl &nccl() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = {getenv("CWIPC_CUDA_NCCL_LIBRARY"), "libnccl.so.2", "libnccl.so"};
        for (const char *name : names) {
            if (!name || !*name) continue;
            n.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (n.handle) break;
        }
        if (!n.handle) {
            n.error = std::string("libnccl.so.2 not found (set CWIPC_CUDA_NCCL_LIBRARY): ") + (dlerror() ? dlerror() : "");
            return;
        }
        auto sym = [&](const char *s) -> void * {
            void *p = dlsym(n.handle, s);
            if (!p && n.error.empty()) n.error = std::string("NCCL symbol missing: ") + s;
            return p;
        };
        n.GetUniqueId = (decltype(n.GetUniqueId))sym("ncclGetUniqueId");
        n.CommInitRank = (decltype(n.CommInitRank))sym("ncclCommInitRank");
        n.CommDestroy = (decltype(n.CommDestroy))sym("ncclCommDestroy");
        n.AllReduce = (decltype(n.AllReduce))sym("ncclAllReduce");
        n.AllGather = (decltype(n.AllGather))sym("ncclAllGather");
        n.Broadcast = (decltype(n.Broadcast))sym("ncclBroadcast");
        n.Send = (decltype(n.Send))sym("ncclSend");
        n.Recv = (decltype(n.Recv))sym("ncclRecv");
        n.GroupStart = (decltype(n.GroupStart))sym("ncclGroupStart");
        n.GroupEnd = (decltype(n.GroupEnd))sym("ncclGroupEnd");
        n.GetErrorString = (decltype(n.GetErrorString))sym("ncclGetErrorString");
    });
    return n;
}

void nccl_check(int rc, const char *what) {
    if (rc != 0) {
        Nccl &n = nccl();
        throw CudaError{cudaErrorUnknown, std::string("NCCL error in ") + what + ": " + (n.GetErrorString ? n.GetErrorString(rc) : std::to_string(rc))};
    }
}
#define NCCL_CHECK(expr) nccl_check((expr), #expr)

} // namespace

struct cwipc_cuda_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, size = 1, dev = 0;
};

namespace {

// ---- small host <-> all ranks helpers (one device round trip each) ---------------------------------------------------
// every rank contributes `count` doubles; all get the size x count matrix
std::vector<double> allgather_doubles(cwipc_cuda_comm *c, const double *mine, size_t count, cudaStream_t s) {
    std::vector<double> all((size_t)c->size * count);
    if (c->size == 1) {
        std::copy(mine, mine + count, all.begin());
        return all;
    }
    Scratch snd(count * sizeof(double), s), rcv(all.size() * sizeof(double), s);
    CWCU_CHECK(cudaMemcpyAsync(snd.p, mine, count * sizeof(double), cudaMemcpyHostToDevice, s));
    NCCL_CHECK(nccl().AllGather(snd.p, rcv.p, count, NCCL_FLOAT64, c->comm, s));
    CWCU_CHECK(cudaMemcpyAsync(all.data(), rcv.p, all.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
    return all;
}

void allreduce_doubles(cwipc_cuda_comm *c, double *values, size_t count, cudaStream_t s) {
    if (c->size == 1) return;
    Scratch buf(count * sizeof(double), s);
    CWCU_CHECK(cudaMemcpyAsync(buf.p, values, count * sizeof(double), cudaMemcpyHostToDevice, s));
    NCCL_CHECK(nccl().AllReduce(buf.p, buf.p, count, NCCL_FLOAT64, NCCL_SUM, c->comm, s));
    CWCU_CHECK(cudaMemcpyAsync(values, buf.p, count * sizeof(double), cudaMemcpyDeviceToHost, s));
    stream_sync(s);
}

// Every rank sends outgoing[q] (device points, may be empty) to rank q; returns what arrived, in rank order, as ONE device
// buffer [from rank 0 | from rank 1 | ...] (own slot empty) with the per-rank counts.  One metadata all-gather, then one
// group of ncclSend / ncclRecv straight between the device buffers.
struct Incoming {
    Scratch buf;
    std::vector<size_t> count, offset; // per source rank, in points
    size_t total = 0;
};
void exchange_points(cwipc_cuda_comm *c, const std::vector<const cwipc_point *> &out_ptr, const std::vector<size_t> &out_count, Incoming &in, cudaStream_t s) {
    const int G = c->size, r = c->rank;
    std::vector<double> row(G);
    for (int q = 0; q < G; q++) row[q] = (double)out_count[q];
    const std::vector<double> table = allgather_doubles(c, row.data(), G, s); // table[p * G + q]: points p sends to q
    in.count.assign(G, 0);
    in.offset.assign(G, 0);
    in.total = 0;
    for (int p = 0; p < G; p++) {
        in.offset[p] = in.total;
        in.count[p] = p == r ? 0 : (size_t)table[(size_t)p * G + r];
        in.total += in.count[p];
    }
    in.buf = Scratch(in.total * sizeof(cwipc_point), s);
    if (G == 1) return;
    NCCL_CHECK(nccl().GroupStart());
    for (int q = 0; q < G; q++) {
        if (q == r) continue;
        if (out_count[q]) NCCL_CHECK(nccl().Send(out_ptr[q], out_count[q] * sizeof(cwipc_point), NCCL_UINT8, q, c->comm, s));
        if (in.count[q]) NCCL_CHECK(nccl().Recv(in.buf.as<cwipc_point>() + in.offset[q], in.count[q] * sizeof(cwipc_point), NCCL_UINT8, q, c->comm, s));
    }
    NCCL_CHECK(nccl().GroupEnd());
}

// Smallest float x with floorf(x * inv) >= v (voxel columns are monotone in x), +-inf passed through.
float column_threshold(double v, float inv) {
    if (!std::isfinite(v)) return (float)v;
    float x = (float)v / inv;
    auto col = [&](float y) { return std::floor(y * inv); };
    for (int it = 0; it < 64 && !(col(x) >= v); it++) x = std::nextafter(x, INFINITY);
    for (int it = 0; it < 64; it++) {
        const float below = std::nextafter(x, -INFINITY);
        if (col(below) < v) break;
        x = below;
    }
    return x;
}

// points of `in` with lo <= x < hi, compacted into a fresh scratch block; returns the count
size_t crop_x(const cwipc_point *in, size_t n, float lo, float hi, Scratch &out, int dev, cudaStream_t s) {
    out = Scratch(n * sizeof(cwipc_point), s);
    if (n == 0) return 0;
    Predicate p;
    p.kind = PredKind::CropBox;
    p.box[0] = lo;
    p.box[1] = hi;
    p.box[2] = p.box[4] = -INFINITY;
    p.box[3] = p.box[5] = INFINITY;
    return compact_points(in, n, out.as<cwipc_point>(), p, dev, s);
}

StoragePtr empty_storage(int dev, cudaStream_t s) {
    auto st = std::make_shared<Storage>(dev, 0, s);
    st->mark_ready();
    return st;
}

// ---- downsample ----------------------------------------------------------------------------------------------------
StoragePtr slab_downsample_storage(const StoragePtr &in, float voxelsize, float pc_cellsize, cwipc_cuda_comm *c, float *cellsize_out, int dev, cudaStream_t s) {
    const int G = c->size, r = c->rank;
    const bool octree = !(voxelsize < 0);
    const size_t n = in->count;
    // 1. what is known locally, one collective
    float bmin[3] = {INFINITY, INFINITY, INFINITY}, bmax[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (n) global_bbox(in->d_pts, n, bmin, bmax, dev, s);
    double row[8] = {(double)pc_cellsize, (double)n, bmin[0], bmin[1], bmin[2], bmax[0], bmax[1], bmax[2]};
    const std::vector<double> info = allgather_doubles(c, row, 8, s);
    float cs = std::fabs(voxelsize);
    bool any = false;
    uint64_t total_points = 0;
    float gmin[3] = {INFINITY, INFINITY, INFINITY}, gmax[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int q = 0; q < G; q++) {
        cs = std::max(cs, (float)info[q * 8 + 0]); // ref: src/cwipc_filters.cpp:103-107 (the cloud's own cellsize wins when larger)
        total_points += (uint64_t)info[q * 8 + 1];
        if (info[q * 8 + 1] > 0) {
            any = true;
            for (int a = 0; a < 3; a++) {
                gmin[a] = std::min(gmin[a], (float)info[q * 8 + 2 + a]);
                gmax[a] = std::max(gmax[a], (float)info[q * 8 + 5 + a]);
            }
        }
    }
    *cellsize_out = cs;
    if (!any) return empty_storage(dev, s); // every part is empty: no leaves, an empty cloud (single-grid mode: the caller reports the reference's error)

    // 2. octree box replay, rank by rank (the box grows with the points IN ORDER).  The box doubles every time it grows, so it
    //    usually contains the whole cloud's bounding box after the first part or two: rank r replays its part and
    //    broadcasts the state; as soon as the box contains the global bounding box no later point can move it, and the
    //    chain stops (every rank takes the same decision from the same data).
    cwipc_cuda_octree_state state{};
    if (octree) {
        Scratch wire(sizeof(state), s);
        for (int q = 0; q < G; q++) {
            if (q == r) {
                float ignored[6];
                octree_replay(in->d_pts, n, cs, state, ignored, dev, s);
                CWCU_CHECK(cudaMemcpyAsync(wire.p, &state, sizeof(state), cudaMemcpyHostToDevice, s));
            }
            if (G > 1) {
                NCCL_CHECK(nccl().Broadcast(wire.p, wire.p, sizeof(state), NCCL_UINT8, q, c->comm, s));
                CWCU_CHECK(cudaMemcpyAsync(&state, wire.p, sizeof(state), cudaMemcpyDeviceToHost, s));
            }
            stream_sync(s);
            bool covers = state.valid != 0;
            for (int a = 0; a < 3 && covers; a++) covers = (double)gmin[a] >= state.min[a] && (double)gmax[a] < state.max[a];
            if (covers) break;
        }
    }
    state.points = total_points; // fixes the fixed-point scale of the centroid sums: the same on every rank as in the one-GPU call

    // 3. voxel columns -> owners; boundary points move to the owner of their column
    const float inv = 1.0f / cs;
    std::vector<double> splits(G + 1, INFINITY); // columns [splits[q], splits[q+1]) belong to rank q
    splits[0] = -INFINITY;
    for (int q = 1; q < G; q++) splits[q] = info[q * 8 + 1] > 0 ? std::floor((float)info[q * 8 + 2] * inv) : INFINITY;
    for (int q = G - 1; q > 0; q--) splits[q] = std::min(splits[q], splits[q + 1]); // an empty part owns nothing; keep the splits monotone
    for (int q = 1; q < G; q++) splits[q] = std::max(splits[q], splits[q - 1]);
    std::vector<float> edges(G + 1);
    for (int q = 0; q <= G; q++) edges[q] = column_threshold(splits[q], inv);
    std::vector<Scratch> pieces(G);
    std::vector<const cwipc_point *> out_ptr(G, nullptr);
    std::vector<size_t> out_count(G, 0);
    Scratch keep_buf;
    const cwipc_point *keep_ptr = in->d_pts;
    size_t keep_count = n;
    if (n > 0 && (bmin[0] < edges[r] || bmax[0] >= edges[r + 1])) {
        keep_count = crop_x(in->d_pts, n, edges[r], edges[r + 1], keep_buf, dev, s);
        keep_ptr = keep_buf.as<cwipc_point>();
        for (int q = 0; q < G; q++) {
            if (q != r && edges[q] < edges[q + 1] && bmax[0] >= edges[q] && bmin[0] < edges[q + 1]) {
                out_count[q] = crop_x(in->d_pts, n, edges[q], edges[q + 1], pieces[q], dev, s);
                out_ptr[q] = pieces[q].as<cwipc_point>();
            }
        }
    }
    Incoming incoming;
    exchange_points(c, out_ptr, out_count, incoming, s);
    StoragePtr mine;
    if (incoming.total == 0 && keep_ptr == in->d_pts) {
        mine = in;
    } else {
        mine = std::make_shared<Storage>(dev, keep_count + incoming.total, s);
        mine->count = keep_count + incoming.total;
        if (keep_count) CWCU_CHECK(cudaMemcpyAsync(mine->d_pts, keep_ptr, keep_count * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
        if (incoming.total) CWCU_CHECK(cudaMemcpyAsync(mine->d_pts + keep_count, incoming.buf.p, incoming.total * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
        mine->mark_ready();
    }
    if (mine->count == 0) return empty_storage(dev, s);

    // 4. the local reduction, with the whole cloud's octree box and bounding box
    const float bounds[6] = {gmin[0], gmin[1], gmin[2], gmax[0], gmax[1], gmax[2]};
    DownsampleResult res = downsample_points_planned(mine, cs, octree, state, bounds, dev, s);
    if (res.failed || !res.out) throw CudaError{cudaErrorUnknown, res.error.empty() ? std::string("downsample failed") : res.error};
    return res.out;
}

// ---- outlier removal of one group -----------------------------------------------------------------------------------
// pts[0..n) is this rank's part of the group.  Survivors are appended to out (capacity >= n); returns their number.
size_t slab_sor_group(const cwipc_point *pts, size_t n, cwipc_point *out, int k, float mul, float pc_cellsize, float halo, cwipc_cuda_comm *c, int dev, cudaStream_t s) {
    const int G = c->size, r = c->rank;
    float bmin[3] = {INFINITY, INFINITY, INFINITY}, bmax[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (n) global_bbox(pts, n, bmin, bmax, dev, s);
    double row[4] = {(double)pc_cellsize, (double)n, n ? (double)bmin[0] : INFINITY, n ? (double)bmax[0] : -INFINITY};
    const std::vector<double> info = allgather_doubles(c, row, 4, s);
    std::vector<double> counts(G), xlo(G), xhi(G);
    double n_total = 0, cs = 0;
    for (int q = 0; q < G; q++) {
        cs = std::max(cs, info[q * 4 + 0]);
        counts[q] = info[q * 4 + 1];
        xlo[q] = info[q * 4 + 2];
        xhi[q] = info[q * 4 + 3];
        n_total += counts[q];
    }
    if (k < 1 || n_total <= (double)k) { // the reference reads past FLANN's results here; defined as keep-all (see outliers.cu)
        if (n) CWCU_CHECK(cudaMemcpyAsync(out, pts, n * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
        return n;
    }
    double H = halo;
    if (!(H > 0)) {
        if (cs > 0) {
            H = 3.0 * cs * std::sqrt((k + 1) / 3.14159265358979);
        } else { // no spacing hint: a third of the mean slab width
            double lo = INFINITY, hi = -INFINITY;
            for (int q = 0; q < G; q++)
                if (counts[q] > 0) {
                    lo = std::min(lo, xlo[q]);
                    hi = std::max(hi, xhi[q]);
                }
            H = std::max(hi - lo, 1e-30) / (3.0 * G);
        }
    }

    // 2. halo exchange: rank q needs every point with x in [xmin_q - H, xmax_q + H]
    std::vector<Scratch> pieces(G);
    std::vector<const cwipc_point *> out_ptr(G, nullptr);
    std::vector<size_t> out_count(G, 0);
    if (n) {
        for (int q = 0; q < G; q++) {
            if (q == r || counts[q] == 0) continue;
            const float lo = std::nextafter((float)(xlo[q] - H), -INFINITY), hi = std::nextafter((float)(xhi[q] + H), INFINITY);
            if (xhi[r] >= lo && xlo[r] < hi) {
                out_count[q] = crop_x(pts, n, lo, hi, pieces[q], dev, s);
                out_ptr[q] = pieces[q].as<cwipc_point>();
            }
        }
    }
    Incoming incoming;
    exchange_points(c, out_ptr, out_count, incoming, s);
    const size_t ncomb = n + incoming.total;
    Scratch combined_buf;
    const cwipc_point *combined = pts;
    if (incoming.total) {
        combined_buf = Scratch(ncomb * sizeof(cwipc_point), s);
        if (n) CWCU_CHECK(cudaMemcpyAsync(combined_buf.p, pts, n * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
        CWCU_CHECK(cudaMemcpyAsync(combined_buf.as<cwipc_point>() + n, incoming.buf.p, incoming.total * sizeof(cwipc_point), cudaMemcpyDeviceToDevice, s));
        combined = combined_buf.as<cwipc_point>();
    }

    // 3. local queries against local + halo points; queries whose neighbourhood leaves the covered interval are open
    bool left = false, right = false;
    for (int q = 0; q < G; q++) {
        if (q == r || counts[q] == 0) continue;
        if (xlo[q] < xlo[r] - H) left = true;
        if (xhi[q] > xhi[r] + H) right = true;
    }
    const float lo_lim = left ? (float)(xlo[r] - H) : -INFINITY, hi_lim = right ? (float)(xhi[r] + H) : INFINITY;
    const int kk = k + 1;
    Scratch dist(std::max<size_t>(n, 1) * sizeof(float), s), kth(std::max<size_t>(ncomb, 1) * sizeof(float), s), open_idx(std::max<size_t>(n, 1) * sizeof(uint32_t), s);
    size_t nopen = 0;
    if (n) {
        if (ncomb > (size_t)k) {
            Scratch dall(ncomb * sizeof(float), s);
            knn_mean_distances(combined, ncomb, k, (float)cs, nullptr, dall.as<float>(), dev, s, kth.as<float>(), n);
            CWCU_CHECK(cudaMemcpyAsync(dist.p, dall.p, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
            nopen = mark_open_queries(combined, kth.as<float>(), n, lo_lim, hi_lim, open_idx.as<uint32_t>(), dev, s);
        } else { // fewer points here than neighbours: every query is open, nothing is known about its neighbourhood
            CWCU_CHECK(cudaMemsetAsync(kth.p, 0x7f, n * sizeof(float), s)); // 0x7f7f7f7f: a huge finite float
            nopen = mark_open_queries(combined, nullptr, n, lo_lim, hi_lim, open_idx.as<uint32_t>(), dev, s);
        }
    }

    // 4. open queries: all-gathered (points + bounds), answered by every rank from its own points, lists returned to the owners
    double my_open = (double)nopen;
    const std::vector<double> opens = allgather_doubles(c, &my_open, 1, s);
    std::vector<size_t> nq(G), qoff(G);
    size_t qtotal = 0;
    for (int q = 0; q < G; q++) {
        qoff[q] = qtotal;
        nq[q] = (size_t)opens[q];
        qtotal += nq[q];
    }
    if (qtotal) {
        Scratch qpts(qtotal * sizeof(cwipc_point), s), qlim(qtotal * sizeof(float), s);
        if (nopen) {
            gather_points(combined, open_idx.as<uint32_t>(), nopen, qpts.as<cwipc_point>() + qoff[r], s);
            gather_floats(kth.as<float>(), open_idx.as<uint32_t>(), nopen, qlim.as<float>() + qoff[r], s);
        }
        if (G > 1) {
            NCCL_CHECK(nccl().GroupStart());
            for (int q = 0; q < G; q++) {
                if (!nq[q]) continue;
                NCCL_CHECK(nccl().Broadcast(qpts.as<cwipc_point>() + qoff[q], qpts.as<cwipc_point>() + qoff[q], nq[q] * sizeof(cwipc_point), NCCL_UINT8, q, c->comm, s));
                NCCL_CHECK(nccl().Broadcast(qlim.as<float>() + qoff[q], qlim.as<float>() + qoff[q], nq[q], NCCL_FLOAT32, q, c->comm, s));
            }
            NCCL_CHECK(nccl().GroupEnd());
        }
        // my answers to everybody's queries: the k+1 smallest distances among my OWN points that lie within the query's bound
        Scratch lists(qtotal * kk * sizeof(float), s);
        knn_lists(pts, n, qpts.as<cwipc_point>(), qlim.as<float>(), qtotal, k, (float)cs, nullptr, lists.as<float>(), dev, s);
        if (nopen) {
            // all-to-all: rank q's answers to MY queries land in mine[q] -- the [nlists][nq][k+1] layout the merge wants
            Scratch mine((size_t)G * nopen * kk * sizeof(float), s), merged(nopen * sizeof(float), s);
            if (G > 1) NCCL_CHECK(nccl().GroupStart());
            for (int q = 0; q < G; q++) {
                if (q == r) {
                    CWCU_CHECK(cudaMemcpyAsync(mine.as<float>() + (size_t)q * nopen * kk, lists.as<float>() + qoff[r] * kk, nopen * kk * sizeof(float), cudaMemcpyDeviceToDevice, s));
                    continue;
                }
                if (nq[q]) NCCL_CHECK(nccl().Send(lists.as<float>() + qoff[q] * kk, nq[q] * kk, NCCL_FLOAT32, q, c->comm, s));
                NCCL_CHECK(nccl().Recv(mine.as<float>() + (size_t)q * nopen * kk, nopen * kk, NCCL_FLOAT32, q, c->comm, s));
            }
            if (G > 1) NCCL_CHECK(nccl().GroupEnd());
            knn_merge_lists(mine.as<float>(), (size_t)G, nopen, k, merged.as<float>(), nullptr, s);
            scatter_floats(merged.as<float>(), open_idx.as<uint32_t>(), nopen, dist.as<float>(), s);
        } else if (G > 1) {
            NCCL_CHECK(nccl().GroupStart());
            for (int q = 0; q < G; q++)
                if (q != r && nq[q]) NCCL_CHECK(nccl().Send(lists.as<float>() + qoff[q] * kk, nq[q] * kk, NCCL_FLOAT32, q, c->comm, s));
            NCCL_CHECK(nccl().GroupEnd());
        }
    }

    // 5. global statistics, local threshold
    double sums[3] = {0.0, 0.0, (double)n};
    if (n) distance_stats(dist.as<float>(), n, sums, s);
    sums[2] = (double)n;
    allreduce_doubles(c, sums, 3, s);
    if (n == 0) return 0;
    Predicate p;
    p.kind = PredKind::DistanceAtMost;
    p.dist = dist.as<float>();
    p.threshold = outlier_threshold(sums[0], sums[1], sums[2], mul);
    return compact_points(pts, n, out, p, dev, s);
}

// what every collective entry point needs of its communicator, for a cloud on `dev`
void check_comm(const cwipc_cuda_comm *comm, int dev) {
    if (comm->size > 1 && !nccl().error.empty()) throw CudaError{cudaErrorUnknown, nccl().error};
    if (dev != comm->dev) throw CudaError{cudaErrorInvalidDevice, "the cloud lives on another device than the communicator"};
}

} // namespace

extern "C" {

int cwipc_cuda_comm_unique_id(void *id128) {
    if (id128 == nullptr) return -1;
    return guarded<int>("cwipc_cuda_comm_unique_id", -1, [&]() -> int {
        if (!nccl().error.empty()) throw CudaError{cudaErrorUnknown, nccl().error};
        ncclUniqueId id;
        NCCL_CHECK(nccl().GetUniqueId(&id));
        memcpy(id128, &id, sizeof(id));
        return 0;
    });
}

cwipc_cuda_comm *cwipc_cuda_comm_create(const void *id128, int nranks, int rank) {
    if (nranks < 1 || rank < 0 || rank >= nranks || (nranks > 1 && id128 == nullptr)) return nullptr;
    return guarded<cwipc_cuda_comm *>("cwipc_cuda_comm_create", nullptr, [&]() -> cwipc_cuda_comm * {
        if (device_count() <= 0) throw CudaError{cudaErrorNoDevice, "libcwipc_util_cuda needs a CUDA device and found none (there is no CPU fallback)"};
        auto *c = new cwipc_cuda_comm();
        c->rank = rank;
        c->size = nranks;
        c->dev = current_device();
        if (nranks > 1) {
            if (!nccl().error.empty()) {
                delete c;
                throw CudaError{cudaErrorUnknown, nccl().error};
            }
            DeviceGuard g(c->dev);
            ncclUniqueId id;
            memcpy(&id, id128, sizeof(id));
            const int rc = nccl().CommInitRank(&c->comm, nranks, id, rank);
            if (rc != 0) {
                delete c;
                nccl_check(rc, "ncclCommInitRank");
            }
        }
        return c;
    });
}

void cwipc_cuda_comm_free(cwipc_cuda_comm *comm) {
    if (comm == nullptr) return;
    if (comm->comm) {
        try {
            DeviceGuard g(comm->dev);
            (void)cudaDeviceSynchronize();
            (void)nccl().CommDestroy(comm->comm);
        } catch (...) {
        }
    }
    delete comm;
}

int cwipc_cuda_comm_rank(cwipc_cuda_comm *comm) { return comm ? comm->rank : -1; }
int cwipc_cuda_comm_size(cwipc_cuda_comm *comm) { return comm ? comm->size : -1; }

// cwipc_downsample of the cloud whose parts are the ranks' `pc` (rank order); this rank's part of the result
cwipc_pointcloud *cwipc_cuda_slab_downsample(cwipc_pointcloud *pc, float voxelsize, cwipc_cuda_comm *comm) {
    if (comm == nullptr) return nullptr;
    return read_entry<cwipc_pointcloud *>("cwipc_cuda_slab_downsample", pc, nullptr, [&](const StoragePtr &in, int dev, cudaStream_t s) -> cwipc_pointcloud * {
        check_comm(comm, dev);
        float cs = 0.f;
        StoragePtr out = slab_downsample_storage(in, voxelsize, pc->cellsize(), comm, &cs, dev, s);
        return new_result(out, pc->timestamp(), cs);
    });
}

// cwipc_remove_outliers of the partitioned cloud; this rank's survivors.  perTile: one pass per tile value, in the order
// of first appearance in the WHOLE cloud (tile 0 = every point), this rank's pieces concatenated in that order.
// halo <= 0: chosen from the cellsize metadata.  ref: src/cwipc_filters.cpp:181-278
cwipc_pointcloud *cwipc_cuda_slab_remove_outliers(cwipc_pointcloud *pc, int kNeighbors, float stddevMulThresh, bool perTile, float halo, cwipc_cuda_comm *comm) {
    if (comm == nullptr) return nullptr;
    return read_entry<cwipc_pointcloud *>("cwipc_cuda_slab_remove_outliers", pc, nullptr, [&](const StoragePtr &in, int dev, cudaStream_t s) -> cwipc_pointcloud * {
        check_comm(comm, dev);
        const size_t n = in->count;
        const float spacing = pc->cellsize();
        if (kNeighbors > 511) throw CudaError{cudaErrorInvalidValue, "remove_outliers: kNeighbors > 511 is not supported by libcwipc_util_cuda"};
        StoragePtr out;
        if (!perTile) {
            out = std::make_shared<Storage>(dev, n, s);
            out->count = slab_sor_group(in->d_pts, n, out->d_pts, kNeighbors, stddevMulThresh, spacing, halo, comm, dev, s);
        } else {
            // distinct tile values in first-appearance order of the whole cloud: the ranks' own lists, concatenated in rank order
            std::vector<int> local = n ? tiles_in_first_appearance_order(in->d_pts, n, s) : std::vector<int>();
            std::vector<double> row(257, -1.0);
            row[0] = (double)local.size();
            for (size_t i = 0; i < local.size(); i++) row[1 + i] = (double)local[i];
            const std::vector<double> all = allgather_doubles(comm, row.data(), 257, s);
            std::vector<int> tiles;
            bool seen[256] = {false};
            for (int q = 0; q < comm->size; q++)
                for (int i = 0; i < (int)all[(size_t)q * 257]; i++) {
                    const int t = (int)all[(size_t)q * 257 + 1 + i];
                    if (!seen[t & 255]) {
                        seen[t & 255] = true;
                        tiles.push_back(t);
                    }
                }
            const bool has_zero = seen[0];
            out = std::make_shared<Storage>(dev, has_zero ? 2 * n : n, s);
            Scratch group(std::max<size_t>(n, 1) * sizeof(cwipc_point), s);
            size_t total = 0;
            for (int tile : tiles) {
                const cwipc_point *src = in->d_pts;
                size_t cnt = n;
                if (tile != 0 && n) {
                    Predicate p;
                    p.kind = PredKind::TileEquals;
                    p.tile = tile;
                    cnt = compact_points(in->d_pts, n, group.as<cwipc_point>(), p, dev, s);
                    src = group.as<cwipc_point>();
                }
                total += slab_sor_group(src, cnt, out->d_pts + total, kNeighbors, stddevMulThresh, spacing, halo, comm, dev, s);
            }
            out->count = total;
        }
        out->mark_ready();
        return new_result(out, pc->timestamp(), pc->cellsize());
    });
}

// cwipc_tilefilter of the partitioned cloud: this rank's piece, and where it sits in the whole result (all-gather of the
// counts).  ref: src/cwipc_filters.cpp:281-306
cwipc_pointcloud *cwipc_cuda_slab_tilefilter(cwipc_pointcloud *pc, int tile, cwipc_cuda_comm *comm, uint64_t *global_offset, uint64_t *global_count) {
    if (comm == nullptr) return nullptr;
    return read_entry<cwipc_pointcloud *>("cwipc_cuda_slab_tilefilter", pc, nullptr, [&](const StoragePtr &, int dev, cudaStream_t s) -> cwipc_pointcloud * {
        check_comm(comm, dev);
        cwipc_pointcloud *rv = cwipc_tilefilter(pc, tile);
        if (!rv) return nullptr;
        double mine = (double)rv->count();
        const std::vector<double> counts = allgather_doubles(comm, &mine, 1, s);
        uint64_t off = 0, tot = 0;
        for (int q = 0; q < comm->size; q++) {
            if (q < comm->rank) off += (uint64_t)counts[q];
            tot += (uint64_t)counts[q];
        }
        if (global_offset) *global_offset = off;
        if (global_count) *global_count = tot;
        return rv;
    });
}

} // extern "C"
