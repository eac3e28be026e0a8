/*
 * cwipc_util_cuda.h -- C ABI of libcwipc_util_cuda, the B200-native drop-in for the filter
 * hot path of cwi-dis/cwipc_util (cwipc_downsample / cwipc_remove_outliers / cwipc_tilefilter
 * plus the cwipc_pointcloud object that carries points between them).
 *
 * Part 1 restates the binary contract of the reference's include/cwipc_util/api.h (struct
 * layouts, vtable order of the abstract C++ classes, the extern "C" entry points that
 * python/cwipc/util.py binds at load time).  Every declaration cites the reference line it
 * replaces as "ref: file:line".  Part 2 declares the cwipc_cuda_* extension entry points
 * (device selection, pinned buffers, async ingest, timers) that the reference does not have.
 *
 * All signatures are plain C: pointers, sizes and scalars.  No torch, no CUDA types.
 */
#ifndef CWIPC_UTIL_CUDA_H
#define CWIPC_UTIL_CUDA_H

#include <stddef.h>
#include <stdint.h>
#include <stdbool.h>

#ifdef __cplusplus
#include <set>
#include <string>
#endif

#ifndef _CWIPC_UTIL_EXPORT
#define _CWIPC_UTIL_EXPORT __attribute__((visibility("default")))
#endif

/* ------------------------------------------------------------------------------------------
 * Part 1a: constants and plain-data records            (ref: include/cwipc_util/api.h:33-162)
 * ---------------------------------------------------------------------------------------- */

#define CWIPC_API_VERSION ((uint64_t)0x20260129)       /* ref: api.h:33 */
#define CWIPC_API_VERSION_OLD ((uint64_t)0x20260129)   /* ref: api.h:39 */
#define CWIPC_CWIPCDUMP_HEADER "cpcd"                  /* ref: api.h:43 */
#define CWIPC_CWIPCDUMP_VERSION ((uint32_t)0x20210208) /* ref: api.h:47 */
#define CWIPC_FLAG_BINARY 1                            /* ref: api.h:51 */
#define CWIPC_POINT_PACKETHEADER_MAGIC 0x20201016      /* ref: api.h:110 */

/* One point, 16 bytes.  This is also the HBM layout: one 128-bit load per point. ref: api.h:88-96 */
struct cwipc_point {
    float x, y, z;
    uint8_t r, g, b;
    uint8_t tile;
};

/* 32-byte header of a .cwipcdump file / of a packet. ref: api.h:59-66 */
struct cwipc_cwipcdump_header {
    char hdr[4];
    uint32_t magic;
    uint64_t timestamp;
    float cellsize;
    uint32_t unused;
    size_t size;
};

struct cwipc_vector { double x, y, z; }; /* ref: api.h:77-81 */

/* ref: api.h:100-106 */
struct cwipc_point_packetheader {
    uint32_t magic;
    uint32_t dataCount;
    uint64_t timestamp;
    float cellsize;
    uint32_t unused;
};

/* ref: api.h:118-127 */
struct cwipc_skeleton_joint {
    uint32_t confidence;
    float x, y, z;
    float q_w, q_x, q_y, q_z;
};

/* ref: api.h:137-141 */
struct cwipc_skeleton_collection {
    uint32_t n_skeletons;
    uint32_t n_joints;
    struct cwipc_skeleton_joint joints[1];
};

/* ref: api.h:150-155 */
struct cwipc_tileinfo {
    struct cwipc_vector normal;
    char *cameraName;
    uint8_t ncamera;
    uint8_t cameraMask;
};

/* ref: api.h:159 */
enum cwipc_log_level {
    CWIPC_LOG_LEVEL_NONE = 0,
    CWIPC_LOG_LEVEL_ERROR = 1,
    CWIPC_LOG_LEVEL_WARNING = 2,
    CWIPC_LOG_LEVEL_TRACE = 3,
    CWIPC_LOG_LEVEL_DEBUG = 4
};

typedef void (*cwipc_log_callback_t)(int level, const char *message); /* ref: api.h:162 */

/* ------------------------------------------------------------------------------------------
 * Part 1b: object handles.  In C++ they are the abstract classes whose vtable order sibling
 * libraries and the apps rely on (apps call pc->free(), generator->get() directly); in C they
 * are opaque.                                         (ref: include/cwipc_util/api.h:164-590)
 * ---------------------------------------------------------------------------------------- */
#ifdef __cplusplus
static_assert(sizeof(struct cwipc_point) == 16, "cwipc_point must be 16 bytes");
static_assert(sizeof(struct cwipc_cwipcdump_header) == 32, "cwipcdump header must be 32 bytes");

class cwipc_metadata;

/* Without PCL the PCL handle is a void* placeholder; this library always returns nullptr for it.
 * ref: api.h:169-172 */
#ifndef _CWIPC_PCL_POINTCLOUD_DEFINED
typedef void *cwipc_pcl_pointcloud;
#define _CWIPC_PCL_POINTCLOUD_PLACEHOLDER_DEFINED
#endif

/* ref: api.h:184-284 -- slot order: dtor, free, _shallowcopy, timestamp, cellsize, _set_cellsize,
 * _set_timestamp, count, get_uncompressed_size, copy_uncompressed, copy_packet,
 * access_pcl_pointcloud, access_metadata. */
class cwipc_pointcloud {
public:
    virtual ~cwipc_pointcloud() {}
    virtual void free() = 0;
    virtual cwipc_pointcloud *_shallowcopy() = 0;
    virtual uint64_t timestamp() = 0;
    virtual float cellsize() = 0;
    virtual void _set_cellsize(float cellsize) = 0;
    virtual void _set_timestamp(uint64_t timestamp) = 0;
    virtual int count() = 0;
    virtual size_t get_uncompressed_size() = 0;
    virtual int copy_uncompressed(struct cwipc_point *pointbuf, size_t size) = 0;
    virtual size_t copy_packet(uint8_t *packet, size_t size) = 0;
    virtual cwipc_pcl_pointcloud access_pcl_pointcloud() = 0;
    virtual cwipc_metadata *access_metadata() = 0;
};

/* ref: api.h:291-335 */
class cwipc_source {
public:
    virtual ~cwipc_source() {}
    virtual void free() = 0;
    virtual bool seek(uint64_t timestamp) = 0;
    virtual bool eof() = 0;
    virtual bool available(bool wait) = 0;
    virtual cwipc_pointcloud *get() = 0;
};

/* ref: api.h:345-444 */
class cwipc_activesource : public cwipc_source {
public:
    virtual ~cwipc_activesource() {}
    virtual bool reload_config(const char *configFile) = 0;
    virtual size_t get_config(char *buffer, size_t size) = 0;
    virtual bool start() = 0;
    virtual void stop() = 0;
    virtual bool seek(uint64_t timestamp) = 0;
    virtual int maxtile() = 0;
    virtual bool get_tileinfo(int tilenum, struct cwipc_tileinfo *tileinfo) = 0;
    virtual void request_metadata(const std::string &name) { metadata_wanted.insert(name); }
    bool is_metadata_requested(const std::string &name) { return metadata_wanted.count(name) != 0; }
    virtual bool auxiliary_operation(const std::string op, const void *inbuf, size_t insize, void *outbuf, size_t outsize) {
        (void)op; (void)inbuf; (void)insize; (void)outbuf; (void)outsize;
        return false;
    }

private:
    std::set<std::string> metadata_wanted;
};

/* ref: api.h:452-500 */
class cwipc_sink {
public:
    virtual ~cwipc_sink() {}
    virtual void free() = 0;
    virtual bool feed(cwipc_pointcloud *pc, bool clear) = 0;
    virtual bool caption(const char *caption) = 0;
    virtual char interact(const char *prompt, const char *responses, int32_t millis) = 0;
};

/* ref: api.h:508-562 */
class cwipc_metadata {
public:
    typedef void (*deallocfunc)(void *);
    virtual ~cwipc_metadata() {}
    virtual int count() = 0;
    virtual const std::string &name(int idx) = 0;
    virtual const std::string &description(int idx) = 0;
    virtual void *pointer(int idx) = 0;
    virtual size_t size(int idx) = 0;
    virtual void _add(const std::string &name, const std::string &description, void *pointer, size_t size, deallocfunc dealloc) = 0;
    virtual void _move(cwipc_metadata *other) = 0;
};

#else /* plain C: opaque handles, ref: api.h:566-588 */
typedef struct _cwipc_pointcloud { int _dummy; } cwipc_pointcloud;
typedef struct _cwipc_pcl_pointcloud { int _dummy; } *cwipc_pcl_pointcloud;
typedef struct _cwipc_source { int _dummy; } cwipc_source;
typedef struct cwipc_activesource { struct _cwipc_source source; } cwipc_activesource;
typedef struct _cwipc_sink { int _dummy; } cwipc_sink;
typedef struct _cwipc_metadata { int _dummy; } cwipc_metadata;
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * Part 1c: entry points bound by python/cwipc/util.py:387-550 and used by the apps.
 * ---------------------------------------------------------------------------------------- */

/* library / logging / leak accounting */
_CWIPC_UTIL_EXPORT const char *cwipc_get_version(void);                                   /* ref: api.h:598, src/cwipc_util.cpp:412 */
_CWIPC_UTIL_EXPORT void cwipc_log_configure(int level, cwipc_log_callback_t callback);    /* ref: api.h:607, src/logging.cpp:74 */
_CWIPC_UTIL_EXPORT void _cwipc_log_emit(int level, const char *module, const char *message); /* ref: api.h:615, src/logging.cpp:131 */
_CWIPC_UTIL_EXPORT int cwipc_dangling_allocations(bool log);                              /* ref: api.h:620, src/cwipc_util.cpp:420 */

/* constructors: host data -> device-resident cloud (one H2D copy) */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_from_points(struct cwipc_point *points, size_t size, int npoint, uint64_t timestamp, char **errorMessage, uint64_t apiVersion); /* ref: api.h:669, src/cwipc_util.cpp:662 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_from_packet(uint8_t *packet, size_t size, char **errorMessage, uint64_t apiVersion); /* ref: api.h:681, src/cwipc_util.cpp:685 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_read_debugdump(const char *filename, char **errorMessage, uint64_t apiVersion);     /* ref: api.h:695, src/cwipc_util.cpp:499 */
_CWIPC_UTIL_EXPORT int cwipc_write_debugdump(const char *filename, cwipc_pointcloud *pc, char **errorMessage);                /* ref: api.h:709, src/cwipc_util.cpp:582 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_read(const char *filename, uint64_t timestamp, char **errorMessage, uint64_t apiVersion); /* ref: api.h:632, src/cwipc_util.cpp:432 */
_CWIPC_UTIL_EXPORT int cwipc_write(const char *filename, cwipc_pointcloud *pc, char **errorMessage);                          /* ref: api.h:643, src/cwipc_util.cpp:461 */
_CWIPC_UTIL_EXPORT int cwipc_write_ext(const char *filename, cwipc_pointcloud *pc, int flag, char **errorMessage);            /* ref: api.h:655, src/cwipc_util.cpp:480 */

/* cwipc_pointcloud methods (thin wrappers over the virtuals) ref: api.h:723-800, src/cwipc_util.cpp:731-773 */
_CWIPC_UTIL_EXPORT void cwipc_pointcloud_free(cwipc_pointcloud *pc);
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_pointcloud__shallowcopy(cwipc_pointcloud *pc);
_CWIPC_UTIL_EXPORT uint64_t cwipc_pointcloud_timestamp(cwipc_pointcloud *pc);
_CWIPC_UTIL_EXPORT float cwipc_pointcloud_cellsize(cwipc_pointcloud *pc);
_CWIPC_UTIL_EXPORT void cwipc_pointcloud__set_cellsize(cwipc_pointcloud *pc, float cellsize);
_CWIPC_UTIL_EXPORT void cwipc_pointcloud__set_timestamp(cwipc_pointcloud *pc, uint64_t timestamp);
_CWIPC_UTIL_EXPORT int cwipc_pointcloud_count(cwipc_pointcloud *pc);
_CWIPC_UTIL_EXPORT size_t cwipc_pointcloud_get_uncompressed_size(cwipc_pointcloud *pc);
_CWIPC_UTIL_EXPORT int cwipc_pointcloud_copy_uncompressed(cwipc_pointcloud *pc, struct cwipc_point *pointbuf, size_t size);
_CWIPC_UTIL_EXPORT size_t cwipc_pointcloud_copy_packet(cwipc_pointcloud *pc, uint8_t *packet, size_t size);
_CWIPC_UTIL_EXPORT cwipc_metadata *cwipc_pointcloud_access_metadata(cwipc_pointcloud *pc);

/* metadata collection ref: api.h:970-1008, src/cwipc_util.cpp:775-797 */
_CWIPC_UTIL_EXPORT void cwipc_metadata__move(cwipc_metadata *src, cwipc_metadata *dest);
_CWIPC_UTIL_EXPORT int cwipc_metadata_count(cwipc_metadata *collection);
_CWIPC_UTIL_EXPORT const char *cwipc_metadata_name(cwipc_metadata *collection, int idx);
_CWIPC_UTIL_EXPORT const char *cwipc_metadata_description(cwipc_metadata *collection, int idx);
_CWIPC_UTIL_EXPORT void *cwipc_metadata_pointer(cwipc_metadata *collection, int idx);
_CWIPC_UTIL_EXPORT size_t cwipc_metadata_size(cwipc_metadata *collection, int idx);

/* sources and sinks (thin wrappers) ref: api.h:807-964, src/cwipc_util.cpp:799-870 */
_CWIPC_UTIL_EXPORT bool cwipc_activesource_start(cwipc_activesource *src);
_CWIPC_UTIL_EXPORT void cwipc_activesource_stop(cwipc_activesource *src);
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_source_get(cwipc_source *src);
_CWIPC_UTIL_EXPORT void cwipc_source_free(cwipc_source *src);
_CWIPC_UTIL_EXPORT bool cwipc_source_eof(cwipc_source *src);
_CWIPC_UTIL_EXPORT bool cwipc_source_available(cwipc_source *src, bool wait);
_CWIPC_UTIL_EXPORT void cwipc_activesource_request_metadata(cwipc_activesource *src, const char *name);
_CWIPC_UTIL_EXPORT bool cwipc_activesource_is_metadata_requested(cwipc_activesource *src, const char *name);
_CWIPC_UTIL_EXPORT bool cwipc_activesource_reload_config(cwipc_activesource *src, const char *configFile);
_CWIPC_UTIL_EXPORT size_t cwipc_activesource_get_config(cwipc_activesource *src, char *buffer, size_t size);
_CWIPC_UTIL_EXPORT bool cwipc_activesource_seek(cwipc_activesource *src, uint64_t timestamp);
_CWIPC_UTIL_EXPORT int cwipc_activesource_maxtile(cwipc_activesource *src);
_CWIPC_UTIL_EXPORT bool cwipc_activesource_get_tileinfo(cwipc_activesource *src, int tilenum, struct cwipc_tileinfo *tileinfo);
_CWIPC_UTIL_EXPORT bool cwipc_activesource_auxiliary_operation(cwipc_activesource *src, const char *op, const void *inbuf, size_t insize, void *outbuf, size_t outsize);
_CWIPC_UTIL_EXPORT void cwipc_sink_free(cwipc_sink *sink);
_CWIPC_UTIL_EXPORT bool cwipc_sink_feed(cwipc_sink *sink, cwipc_pointcloud *pc, bool clear);
_CWIPC_UTIL_EXPORT bool cwipc_sink_caption(cwipc_sink *sink, const char *caption);
_CWIPC_UTIL_EXPORT char cwipc_sink_interact(cwipc_sink *sink, const char *prompt, const char *responses, int32_t millis);

/* factories.  cwipc_synthetic is a host generator feeding cwipc_from_points; capturer, window and
 * proxy are out of scope and return NULL with an error message, like the reference's own
 * no-GUI / unknown-camera paths. */
_CWIPC_UTIL_EXPORT cwipc_activesource *cwipc_synthetic(int fps, int npoints, char **errorMessage, uint64_t apiVersion);   /* ref: api.h:1020, src/cwipc_synthetic.cpp:225 */
_CWIPC_UTIL_EXPORT cwipc_activesource *cwipc_capturer(const char *configFilename, char **errorMessage, uint64_t apiVersion); /* ref: api.h:1035, src/cwipc_capturer.cpp:32 */
_CWIPC_UTIL_EXPORT cwipc_sink *cwipc_window(const char *title, char **errorMessage, uint64_t apiVersion);                 /* ref: api.h:1050, src/cwipc_window.cpp:359 */
_CWIPC_UTIL_EXPORT cwipc_activesource *cwipc_proxy(const char *host, int port, char **errorMessage, uint64_t apiVersion); /* ref: api.h:1143, src/cwipc_proxy.cpp:264 */

/* THE HOT PATH: filters.  Input is borrowed and never modified; the result is a new device-resident
 * cloud owned by the caller.  NULL input gives NULL. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_downsample(cwipc_pointcloud *pc, float voxelsize);  /* ref: api.h:1063, src/cwipc_filters.cpp:30-172 */
/* kNeighbors: 1..63 takes the fast path (lists in registers), 64..511 a slower exact path (one tree search per point); larger
 * values return NULL with an ERROR log (the reference, pcl::StatisticalOutlierRemoval::setMeanK, has no limit). */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_remove_outliers(cwipc_pointcloud *pc, int kNeighbors, float stddevMulThresh, bool perTile); /* ref: api.h:1075, src/cwipc_filters.cpp:181-278 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_tilefilter(cwipc_pointcloud *pc, int tile);         /* ref: api.h:1085, src/cwipc_filters.cpp:281-306 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_tilemap(cwipc_pointcloud *pc, uint8_t map[256]);    /* ref: api.h:1096, src/cwipc_filters.cpp:308-331 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_crop(cwipc_pointcloud *pc, float bbox[6]);          /* ref: api.h:1107, src/cwipc_filters.cpp:333-360 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_colormap(cwipc_pointcloud *pc, uint32_t clearBits, uint32_t setBits); /* ref: api.h:1119, src/cwipc_filters.cpp:362-386 */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_join(cwipc_pointcloud *pc1, cwipc_pointcloud *pc2); /* ref: api.h:1131, src/cwipc_filters.cpp:388-418 */

/* ------------------------------------------------------------------------------------------
 * Part 2: cwipc_cuda_* extensions (no counterpart in the reference).
 * ---------------------------------------------------------------------------------------- */

/* Number of CUDA devices visible (0 if none / no driver). */
_CWIPC_UTIL_EXPORT int cwipc_cuda_device_count(void);
/* Select the device on which the CALLING THREAD creates new clouds (default: $CWIPC_CUDA_DEVICE or 0).
 * Filters always run on the device that holds their input.  Returns 0, or -1 on a bad index. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_set_device(int device);
_CWIPC_UTIL_EXPORT int cwipc_cuda_get_device(void);
/* Block until all work queued by the calling thread on its current device has finished. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_synchronize(void);
/* Page-locked host buffers: cwipc_from_points / copy_uncompressed on such memory run as one DMA. */
_CWIPC_UTIL_EXPORT void *cwipc_cuda_host_alloc(size_t size);
_CWIPC_UTIL_EXPORT void cwipc_cuda_host_free(void *ptr);
/* Like cwipc_from_points, but returns as soon as the copy is queued: the caller promises that
 * `points` is page-locked and stays untouched until cwipc_cuda_synchronize() or until the result
 * (or anything derived from it) has been read back. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_from_points_async(struct cwipc_point *points, size_t size, int npoint, uint64_t timestamp, char **errorMessage, uint64_t apiVersion);
/* Device on which a cloud lives, or -1. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_pointcloud_device(cwipc_pointcloud *pc);
/* Borrow the raw device pointer of a cloud (16-byte points) for interop; valid until free(). */
_CWIPC_UTIL_EXPORT const void *cwipc_cuda_pointcloud_device_ptr(cwipc_pointcloud *pc);
/* cwipc_tilefilter variant used by python/cwipc/registration/util.py:98-112: keep (tile & mask) != 0. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_tilefilter_masked(cwipc_pointcloud *pc, int mask);
/* cwipc_downsample of each camera's points on their own, in one call: the same records, in the same order, as
 *   join(downsample(tilefilter(pc, t1), voxelsize), downsample(tilefilter(pc, t2), voxelsize), ...)
 * over the distinct tile values t1, t2, ... in first-appearance order (src/cwipc_filters.cpp:239-256), tile 0 standing for
 * every point as in cwipc_tilefilter.  This is what python/cwipc/registration/util.py:170-182 (cwipc_downsample_pertile)
 * builds from those filters, so that no voxel mixes the points of two cameras.  voxelsize as in cwipc_downsample (negative:
 * one grid); the result has the input's timestamp and the effective cell size.  Empty input: as cwipc_downsample.  NULL,
 * with an ERROR log naming the tile value, when a group cannot be downsampled. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_downsample_pertile(cwipc_pointcloud *pc, float voxelsize);
/* Each point moved by the 4x4 matrix of its tile value.  matrices: n row-major 4x4 doubles; tiles: n tile values.
 * A point whose tile value equals tiles[i] becomes M_i * (x, y, z, 1); the entry with tile value 0, if any, applies to every
 * point whose value has no entry of its own (tile 0 standing for the whole cloud, as in cwipc_tilefilter); every other point
 * is copied unchanged.  Order, colours and tile bytes are kept; the result has the input's timestamp and cellsize.
 *   Whole cloud: n = 1, tiles = {0}.
 *   Matching is by the exact tile value, as in cwipc_tilefilter, not by bits.  After cwipc_downsample a voxel's tile is the
 *   OR of its cameras' tiles: such a voxel moves only if that exact OR value has an entry, or if there is a tile-0 entry.
 *   Arithmetic: each output coordinate is (float)(((m[r][0]*x + m[r][1]*y) + m[r][2]*z) + m[r][3]), with x, y, z
 *   promoted to double, every product and sum rounded to double (no fused multiply-add) and the result rounded to the
 *   nearest float.  numpy float64 elementwise arithmetic in the same order gives the same bits.  So an identity matrix
 *   returns a listed point bit for bit, except that -0.0 becomes +0.0 (the final + 0.0); unlisted points are copied verbatim.
 *   Errors: n < 1, NULL matrices or tiles, a tile value listed twice (so also n > 256), a non-finite entry, or a last row
 *   other than exactly (0, 0, 0, 1) (only affine maps; singular ones are accepted) give NULL and one ERROR log naming
 *   cwipc_cuda_transform; the input stays usable.  NULL pc: NULL, silently, before any argument check.  An empty cloud
 *   gives an empty cloud.
 *   The cellsize is the input's even when a matrix scales the cloud (set it with _set_cellsize where that matters).  No
 *   metadata is carried over.  The result carries no bounding box: the input's does not bound the moved points. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_transform(cwipc_pointcloud *pc, const double *matrices, const uint8_t *tiles, int n);
/* Per-point mean k-neighbour distance of cwipc_remove_outliers' first pass, copied to host
 * (dist[count]); returns count or -1.  Diagnostic hook used by the parity tests. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_knn_mean_distances(cwipc_pointcloud *pc, int kNeighbors, float *dist, size_t ndist);
/* Voxel keys of cwipc_downsample's key generation (one uint64 per input point, host buffer);
 * returns count or -1.  Diagnostic hook used by the parity tests. */
/* ---- partitioned clouds: one cloud spread over several GPUs as x-slabs (BASELINE configs[3]) ----
 * Building blocks only: every call is local to one GPU; the exchange steps between ranks (NCCL
 * send/recv of boundary and halo points, all-reduce of the statistics) are made by the caller, see
 * cwipc_util_b200/slab.py.  ref for the semantics being partitioned: src/cwipc_filters.cpp:89-278. */
struct cwipc_cuda_octree_state { /* bounding box of pcl::octree::OctreePointCloud while points are inserted */
    double min[3];
    double max[3];
    int32_t depth;
    int32_t valid; /* 0: nothing inserted yet */
    uint64_t points; /* points inserted so far; cwipc_cuda_downsample_planned takes the scale of its fixed-point centroid
                      * sums from the whole cloud's count, so that every part rounds exactly as the one-GPU call does */
};
/* Insert this cloud's points (in order) into the octree box `state` (in/out); bounds = min xyz, max xyz of the cloud. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_octree_replay(cwipc_pointcloud *pc, float cellsize, struct cwipc_cuda_octree_state *state, float bounds[6]);
/* cwipc_downsample of one part, with the octree box and the bounding box of the WHOLE cloud supplied. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_downsample_planned(cwipc_pointcloud *pc, float voxelsize, const struct cwipc_cuda_octree_state *state, const float bounds[6]);
/* New cloud from npoint device-resident 16-byte points (device-to-device copy; e.g. an NCCL receive buffer). */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_from_device_points(const void *dev_points, int npoint, uint64_t timestamp);
/* First pass of cwipc_remove_outliers for the first nquery points against ALL points of the cloud (the rest
 * being halo points): mean distance to the k nearest and the (k+1)-th smallest squared distance, nquery floats each. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_knn_query(cwipc_pointcloud *pc, int kNeighbors, int nquery, float *mean, float *kth2);
/* The same first pass with the result kept on the device: mean distances of the first nquery points, plus the list of
 * "open" queries, i.e. those whose (k+1)-th neighbour sphere is not strictly inside the covered interval (x_lo, x_hi) of
 * this part and therefore have to be completed with the other parts' points.  Only the open queries ever reach the host. */
typedef struct cwipc_cuda_distances cwipc_cuda_distances;
_CWIPC_UTIL_EXPORT cwipc_cuda_distances *cwipc_cuda_knn_query_open(cwipc_pointcloud *pc, int kNeighbors, int nquery, float x_lo, float x_hi, int *nopen);
/* indices, coordinates and current (k+1)-th squared distances of the open queries (nopen entries each, any may be NULL);
 * the distance is an upper bound of the final one: only parts within its reach have to answer the query */
_CWIPC_UTIL_EXPORT int cwipc_cuda_distances_open(cwipc_cuda_distances *d, cwipc_pointcloud *pc, uint32_t *idx, struct cwipc_point *points, float *kth2);
/* overwrite the mean distance of the open queries, in the order cwipc_cuda_distances_open listed them */
_CWIPC_UTIL_EXPORT int cwipc_cuda_distances_patch(cwipc_cuda_distances *d, const float *values, int n);
_CWIPC_UTIL_EXPORT int cwipc_cuda_distances_stats(cwipc_cuda_distances *d, double sums[2]);
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_distances_filter(cwipc_pointcloud *pc, cwipc_cuda_distances *d, double threshold);
_CWIPC_UTIL_EXPORT void cwipc_cuda_distances_free(cwipc_cuda_distances *d);
/* The k+1 smallest squared distances (ascending, +inf padded) from nq arbitrary query points to the cloud: lists[nq][k+1].
 * limits (may be NULL): per query, only distances <= limit are searched for and reported. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_knn_lists(cwipc_pointcloud *pc, const struct cwipc_point *queries, const float *limits, int nq, int kNeighbors, float *lists);
/* Merge lists[nlists][nq][k+1] (one list per part of the cloud) into the mean distance / (k+1)-th squared distance. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_knn_merge_lists(const float *lists, int nlists, int nq, int kNeighbors, float *mean, float *kth2);
/* sums[0] = sum d, sums[1] = sum (float)(d*d), in double: the two numbers the parts all-reduce. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_distance_stats(const float *dist, size_t ndist, double sums[2]);
/* mean + mul * stddev (unbiased) from the all-reduced sums, as pcl::StatisticalOutlierRemoval. */
_CWIPC_UTIL_EXPORT double cwipc_cuda_outlier_threshold(double sum, double sq, double n, float stddevMulThresh);
/* Second pass: keep point i iff !(dist[i] > threshold); order preserved. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_filter_by_distance(cwipc_pointcloud *pc, const float *dist, size_t ndist, double threshold);

/* Diagnostic: stable LSD radix sort of n host words on bits [begin_bit, end_bit), in place (device sort). */
_CWIPC_UTIL_EXPORT int cwipc_cuda_sort_u64(uint64_t *words, size_t n, int begin_bit, int end_bit);
_CWIPC_UTIL_EXPORT int cwipc_cuda_downsample_keys(cwipc_pointcloud *pc, float voxelsize, uint64_t *keys, size_t nkeys);

/* CUDA-event stopwatch on the calling thread's stream. */
_CWIPC_UTIL_EXPORT void *cwipc_cuda_timer_create(void);
_CWIPC_UTIL_EXPORT void cwipc_cuda_timer_destroy(void *timer);
_CWIPC_UTIL_EXPORT void cwipc_cuda_timer_start(void *timer);
_CWIPC_UTIL_EXPORT void cwipc_cuda_timer_stop(void *timer);
/* Waits for the stop event; milliseconds between start and stop, <0 on error. */
_CWIPC_UTIL_EXPORT float cwipc_cuda_timer_elapsed_ms(void *timer);
/* Milliseconds between the start event of `timer_a` and the stop event of `timer_b` (any streams). */
_CWIPC_UTIL_EXPORT float cwipc_cuda_timer_span_ms(void *timer_a, void *timer_b);

/* Kernel accounting.  launches(): kernels launched by this library since load.
 * profile_enable(1): bracket every kernel with events and accumulate per-kernel device time;
 * profile_report(): JSON {"kernel": {"launches": n, "total_ms": t}, ...} into buf, returns length needed. */
_CWIPC_UTIL_EXPORT uint64_t cwipc_cuda_kernel_launches(void);
_CWIPC_UTIL_EXPORT void cwipc_cuda_profile_enable(int on);
_CWIPC_UTIL_EXPORT void cwipc_cuda_profile_reset(void);
_CWIPC_UTIL_EXPORT size_t cwipc_cuda_profile_report(char *buf, size_t size);
/* Overwrite a buffer larger than L2 on the calling thread's stream (bench hygiene). */
/* ---- one cloud partitioned over several GPUs as x-slabs (BASELINE configs[3]) --------------------------------------------
 * One process (or thread) per GPU; the WHOLE cloud is the concatenation of the ranks' parts in rank order, every call below
 * is collective (all ranks call it with their part) and returns this rank's part of what the single-GPU filter returns on
 * the whole cloud.  Points travel with ncclSend / ncclRecv between device buffers, metadata with small all-gathers, all on
 * the calling thread's stream.  libnccl.so.2 is loaded with dlopen on first use ($CWIPC_CUDA_NCCL_LIBRARY overrides).
 * A communicator of size 1 needs no NCCL and no id. */
typedef struct cwipc_cuda_comm cwipc_cuda_comm;
/* 128 bytes (ncclUniqueId) made on one rank, to be handed to every rank by the caller's own means.  0 on success. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_comm_unique_id(void *id128);
/* collective: ncclCommInitRank on the calling thread's current device.  NULL on error. */
_CWIPC_UTIL_EXPORT cwipc_cuda_comm *cwipc_cuda_comm_create(const void *id128, int nranks, int rank);
_CWIPC_UTIL_EXPORT void cwipc_cuda_comm_free(cwipc_cuda_comm *comm);
_CWIPC_UTIL_EXPORT int cwipc_cuda_comm_rank(cwipc_cuda_comm *comm);
_CWIPC_UTIL_EXPORT int cwipc_cuda_comm_size(cwipc_cuda_comm *comm);
/* ref: src/cwipc_filters.cpp:89-172.  Bit-identical (as a set of records) to cwipc_downsample of the whole cloud; rank r
 * holds the voxels of its x-slab, in the reference's order. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_slab_downsample(cwipc_pointcloud *pc, float voxelsize, cwipc_cuda_comm *comm);
/* ref: src/cwipc_filters.cpp:181-278.  halo <= 0: chosen from the cellsize metadata (results never depend on it).  perTile:
 * one pass per tile value in the order of first appearance in the whole cloud; this rank's pieces in that order. */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_slab_remove_outliers(cwipc_pointcloud *pc, int kNeighbors, float stddevMulThresh, bool perTile, float halo, cwipc_cuda_comm *comm);
/* ref: src/cwipc_filters.cpp:281-306.  This rank's piece; *global_offset / *global_count (may be NULL): where it sits in, and
 * the size of, the whole result (all-gather of the counts). */
_CWIPC_UTIL_EXPORT cwipc_pointcloud *cwipc_cuda_slab_tilefilter(cwipc_pointcloud *pc, int tile, cwipc_cuda_comm *comm, uint64_t *global_offset, uint64_t *global_count);

_CWIPC_UTIL_EXPORT void cwipc_cuda_flush_l2(void);
/* Hand cached device memory of the calling thread's current device back to the driver (the library's private memory pool,
 * the calling thread's scratch arena and voxel-table workspace, those of exited threads).  Waits for the device to go idle.
 * Live clouds are not affected.  Returns 0, or -1 on error. */
_CWIPC_UTIL_EXPORT int cwipc_cuda_trim(void);

#ifdef __cplusplus
}
#endif
#endif /* CWIPC_UTIL_CUDA_H */
