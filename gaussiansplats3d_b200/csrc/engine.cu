// engine.cu -- host side of libgsplat_b200.so: the C ABI declared in include/gsplat_b200.h.
//
// One gs_engine = the device-resident state of one sort Worker (src/worker/SortWorker.js) plus one SplatMesh
// (src/splatmesh/SplatMesh.js) on one B200: persistent centres, splat data, scratch, one CUDA stream.
// There is no CPU implementation of any stage in this library: without a device every entry fails.
#include "../../include/gsplat_b200.h"
#include "common.cuh"
#include "sort_kernels.cuh"
#include "raster_kernels.cuh"
#include "shard_kernels.cuh"
#include "ksplat_transform.h"
#include "ksplat_kernels.cuh"
#include "cull_kernels.cuh"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

using namespace gs;

// ---------------------------------------------------------------------------------------------------------------
thread_local char g_gs_err[512] = "";
#define g_err g_gs_err
static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(call)                                                                                                  \
    do {                                                                                                          \
        cudaError_t _e = (call);                                                                                  \
        if (_e != cudaSuccess) return fail(GS_ERR_CUDA, "%s -> %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

extern "C" int gs_abi_version(void) { return GS_ABI_VERSION; }
extern "C" const char *gs_last_error_message(void) { return g_err; }
extern "C" const char *gs_status_string(int s) {
    switch (s) {
        case GS_OK: return "ok";
        case GS_ERR_BAD_ARG: return "bad argument";
        case GS_ERR_NO_DEVICE: return "no CUDA device";
        case GS_ERR_CUDA: return "CUDA error";
        case GS_ERR_DEGENERATE: return "all distances equal";
        case GS_ERR_BUCKET_RANGE: return "bucket index out of range";
        case GS_ERR_NOT_READY: return "not ready";
        case GS_ERR_CAPACITY: return "capacity exceeded";
        default: return "unknown";
    }
}
extern "C" int gs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---------------------------------------------------------------------------------------------------------------
template <typename T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    int ensure(size_t count) {
        if (count <= n) return GS_OK;
        if (p) cudaFree(p);
        p = nullptr; n = 0;
        cudaError_t e = cudaMalloc((void **)&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e != cudaSuccess) return fail(GS_ERR_CUDA, "cudaMalloc(%zu bytes) -> %s", count * sizeof(T), cudaGetErrorString(e));
        n = count;
        return GS_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};
template <typename T> struct PinBuf {
    T *p = nullptr;
    size_t n = 0;
    int ensure(size_t count) {
        if (count <= n) return GS_OK;
        if (p) cudaFreeHost(p);
        p = nullptr; n = 0;
        cudaError_t e = cudaHostAlloc((void **)&p, std::max<size_t>(count, 1) * sizeof(T), cudaHostAllocDefault);
        if (e != cudaSuccess) return fail(GS_ERR_CUDA, "cudaHostAlloc(%zu bytes) -> %s", count * sizeof(T), cudaGetErrorString(e));
        n = count;
        return GS_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; n = 0; }
};

enum { EV_SORT0, EV_DEPTH, EV_BUCKET, EV_SORT1, EV_R0, EV_PROJECT, EV_BIN, EV_R1, EV_H2D0, EV_H2D1, EV_D2H0, EV_D2H1, EV_COUNT };

// one status slot of a pipelined frame: SortControl head (3 words, padded to 4) + RasterControl + slack
constexpr size_t kPipeSlotWords = 4 + (sizeof(RasterControl) + 3) / 4 + 12;   // SortControl head (3 words) + RasterControl
struct gs_engine {
    gs_config cfg{};
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[EV_COUNT]{};
    int sm_count = 148;
    int key_bits = 16;

    // --- sorter state (SortWorker.js:125-178 memory regions, device side) ---
    DevBuf<int4> centers;            // int32x4 or f32x4 per splat
    DevBuf<uint32_t> scene_idx;      // dynamic mode
    DevBuf<uint32_t> indexes;        // indexesToSort
    DevBuf<uint32_t> precomputed;    // precomputedDistances (i32 or f32 bits)
    DevBuf<int32_t> dist;            // mappedDistances
    DevBuf<uint32_t> keys[2];        // radix keys ping/pong (u16 or u32 elements, sized in u32 words)
    DevBuf<uint32_t> vals[2];        // radix values ping/pong
    DevBuf<uint32_t> sorted;         // sortedIndexes
    DevBuf<float> transforms;        // 32 x mat4
    DevBuf<SortControl> ctl;
    DevBuf<DepthParams> depthp;      // per-frame depth parameters (device copy read by k_depth)
    DevBuf<uint32_t> tile_hist;       // radix tile histograms / offsets [pass][digit][tile]
    DevBuf<uint32_t> freq;           // scratch reproduction for gs_sort_indexes
    DevBuf<int32_t> dist_rows_i;     // gs_compute_distances: per-scene integer / float rows
    DevBuf<float> dist_rows_f;
    DevBuf<uint32_t> sub_idx;        // sharded frames: this rank's subset of the sort input (index, distance)
    DevBuf<int32_t> sub_dist;
    uint32_t uploaded_splats = 0;    // 'uploadedSplatCount' SortWorker.js:97
    uint32_t last_render_count = 0;
    bool have_sorted = false;
    bool ctl_dirty = true;           // SortControl needs k_sort_init (first sort / after a failed one); otherwise the sort leaves it clean

    // pinned staging (the shared-memory views of SortWorker.js:180-191)
    PinBuf<uint32_t> h_indexes, h_sorted;
    PinBuf<uint32_t> h_ctl;
    PinBuf<unsigned char> h_frame;

    // --- rasteriser state ---
    RasterState rs;

    gs_timings tm{};
    Profiler prof;
    // CUDA graph of one frame (sort + render), replayed while its shape key is unchanged
    cudaGraphExec_t graph_exec = nullptr;
    cudaStream_t stream2 = nullptr;  // second capture branch (projection beside the depth sort)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    unsigned long long graph_key[8] = {0};
    bool graph_enabled = true;
    bool last_frame_was_graph = false;
    bool no_subset = false;          // gs_frame with sorted_out on a sharded engine needs the full order: replicated sort
    uint32_t graph_launches = 0;
    bool have_prof_begin = false;    // true while a frame's sort already opened the timeline
    bool pending_async = false;
    gs_render_params pending_rp{};
    DevBuf<uint32_t> flush;          // L2 flush scratch (bench hygiene)
    // SplatTree leaves (gs_upload_splat_tree) and the scratch of gs_gather_for_sort
    struct Tree {
        DevBuf<double> center, nmin, nmax;
        DevBuf<uint32_t> offsets, indexes, start;
        DevBuf<unsigned long long> key, total;
        uint32_t count = 0, splats = 0;
    } tree;
    // pipelined frames (gs_frame_begin / gs_frame_end): device frames alternate between two buffers, the D2H copy of frame i runs on
    // copy_stream while frame i+1 computes on `stream`
    cudaStream_t copy_stream = nullptr;
    // ring of per-frame events / host status slots (more entries than frames in flight); the DEVICE frame buffers stay two
    static constexpr int kPipeRing = 4, kPipeMaxInflight = 3;
    cudaEvent_t ev_frame_done[kPipeRing] = {nullptr}, ev_copy_done[kPipeRing] = {nullptr};
    // per-frame parameter blocks are double buffered by frame-buffer parity and uploaded on their own stream, and the frame's status words
    // are snapshotted by the blend kernel into a per-parity device slot that the copy stream reads: a pipelined frame then puts NO copy
    // operation on the compute stream (each small copy there costs a few microseconds of serialisation between two frame graphs)
    cudaStream_t param_stream = nullptr;
    cudaEvent_t ev_params[2] = {nullptr, nullptr};
    bool param_side = false;                       // upload_frame_params goes through param_stream (set by gs_frame_begin)
    bool graph_snapshot[2] = {false, false};       // the captured frame graph of this parity ends in a blend that writes the status snapshot
    DevBuf<uint32_t> status_dev;                   // 2 x kPipeSlotWords
    cudaGraphExec_t graph_exec_alt = nullptr;     // the same frame graph with the alternate frame buffer as target
    unsigned long long graph_key_alt[8] = {0};
    PinBuf<uint32_t> h_pipe;                       // kPipeRing slots x (SortControl head + RasterControl) read back per pipelined frame
    uint64_t pipe_begun = 0, pipe_ended = 0;       // frames begun / ended; in flight = the difference
    uint32_t pipe_inflight() const { return (uint32_t)(pipe_begun - pipe_ended); }

    // --- sort-only sharding by input position (shard_kernels.cuh) ---
    struct Shard {
        DevBuf<unsigned char> block;                 // ShardHeader + runs[R] (exported through CUDA IPC)
        DevBuf<uint32_t> total, ahead, block_total, delta, local_sorted;
        ShardPeers peers{};
        uint32_t *root_out = nullptr;                // rank 0's sortedIndexes as mapped here
        void *opened[kMaxShardRanks + 1] = {nullptr};// IPC mappings to close
        uint32_t world = 0, seq = 0;
        uint32_t pending_render_count = 0;
        bool attached = false, pending = false;
        bool pending_unsplit = false;                // the pending call was below the split threshold: rank 0 sorted alone
    } shard;
};

static int check_engine(gs_engine *e) {
    if (!e) return fail(GS_ERR_BAD_ARG, "null engine");
    cudaError_t ce = cudaSetDevice(e->cfg.device);
    if (ce != cudaSuccess) return fail(GS_ERR_CUDA, "cudaSetDevice(%d) -> %s", e->cfg.device, cudaGetErrorString(ce));
    return GS_OK;
}

extern "C" void gs_destroy(gs_engine *e);
// inside gs_create after the engine object exists: a failing CUDA call must not leak it
#define CUE(call)                                                                                                 \
    do {                                                                                                          \
        cudaError_t _e = (call);                                                                                  \
        if (_e != cudaSuccess) {                                                                                  \
            gs_destroy(e);                                                                                        \
            return fail(GS_ERR_CUDA, "%s -> %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__);      \
        }                                                                                                         \
    } while (0)
extern "C" int gs_create(const gs_config *cfg, gs_engine **out) {
    if (!cfg || !out) return fail(GS_ERR_BAD_ARG, "gs_create: null argument");
    *out = nullptr;
    gs_config c{};
    memcpy(&c, cfg, std::min<size_t>(cfg->struct_size ? cfg->struct_size : sizeof(gs_config), sizeof(gs_config)));
    if (c.distance_map_range == 0) c.distance_map_range = 1u << 16; // Constants.DefaultSplatSortDistanceMapPrecision
    if (c.distance_map_range < 2 || c.distance_map_range > (1u << 24)) return fail(GS_ERR_BAD_ARG, "distance_map_range %u outside [2, 2^24]", c.distance_map_range);
    if (c.world_size == 0) { c.world_size = 1; c.rank = 0; }
    if (c.rank >= c.world_size) return fail(GS_ERR_BAD_ARG, "rank %u >= world_size %u", c.rank, c.world_size);
    if (c.splat_render_mode > GS_RENDER_MODE_2D) return fail(GS_ERR_BAD_ARG, "splat_render_mode %u is neither ThreeD (0) nor TwoD (1)", (unsigned)c.splat_render_mode);
    int ndev = gs_device_count();
    if (ndev <= 0) return fail(GS_ERR_NO_DEVICE, "no CUDA device visible: libgsplat_b200 has no CPU path");
    if (c.device < 0 || c.device >= ndev) return fail(GS_ERR_BAD_ARG, "device %d not in [0,%d)", c.device, ndev);
    CU(cudaSetDevice(c.device));
    gs_engine *e = new (std::nothrow) gs_engine();
    if (!e) return fail(GS_ERR_BAD_ARG, "out of host memory");
    e->cfg = c;
    cudaDeviceProp prop{};
    CUE(cudaGetDeviceProperties(&prop, c.device));
    e->sm_count = prop.multiProcessorCount;
    CUE(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CUE(cudaStreamCreateWithFlags(&e->stream2, cudaStreamNonBlocking));
    CUE(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    CUE(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
    for (int i = 0; i < EV_COUNT; ++i) CUE(cudaEventCreate(&e->ev[i]));
    int kb = 0;
    while ((1u << kb) < c.distance_map_range) ++kb;
    e->key_bits = kb;
    int rc = GS_OK;
    const size_t n = std::max<uint32_t>(c.max_splat_count, 1);
    if ((rc = e->centers.ensure(n)) || (rc = e->indexes.ensure(n)) || (rc = e->dist.ensure(n)) || (rc = e->sorted.ensure(n)) ||
        (rc = e->vals[0].ensure(n)) || (rc = e->vals[1].ensure(n)) || (rc = e->keys[0].ensure(n)) || (rc = e->keys[1].ensure(n)) ||
        (rc = e->ctl.ensure(1)) || (rc = e->depthp.ensure(2)) || (rc = e->transforms.ensure(16 * GS_MAX_SCENES)) || (rc = e->h_ctl.ensure(sizeof(SortControl) / 4 + 64 + sizeof(RasterControl) / 4 + sizeof(ShardHeader) / 4))) {
        gs_destroy(e);
        return rc;
    }
    if (c.dynamic_mode && (rc = e->scene_idx.ensure(n))) { gs_destroy(e); return rc; }
    if (e->scene_idx.p) CUE(cudaMemsetAsync(e->scene_idx.p, 0, e->scene_idx.n * 4, e->stream));
    {   // identity transforms until the caller provides some
        std::vector<float> id(16 * GS_MAX_SCENES, 0.f);
        for (int s = 0; s < GS_MAX_SCENES; ++s) id[16 * s] = id[16 * s + 5] = id[16 * s + 10] = id[16 * s + 15] = 1.f;
        CUE(cudaMemcpy(e->transforms.p, id.data(), id.size() * 4, cudaMemcpyHostToDevice));
    }
    CUE(cudaMemset(e->ctl.p, 0, sizeof(SortControl)));
    rc = raster_init(e->rs, c, e->sm_count);
    if (rc) { gs_destroy(e); return fail(rc, "raster_init failed: %s", g_err); }
    if ((rc = e->status_dev.ensure(2 * kPipeSlotWords))) { gs_destroy(e); return rc; }
    CUE(cudaMemset(e->status_dev.p, 0, 2 * kPipeSlotWords * 4));
    e->rs.snap_base = e->status_dev.p;
    e->rs.snap_stride = (uint32_t)kPipeSlotWords;
    e->rs.snap_sort_ctl = reinterpret_cast<const uint32_t *>(e->ctl.p);
    CUE(cudaStreamSynchronize(e->stream));
    *out = e;
    return GS_OK;
}

#undef CUE

extern "C" void gs_destroy(gs_engine *e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    e->centers.release(); e->scene_idx.release(); e->indexes.release(); e->precomputed.release(); e->dist.release();
    e->keys[0].release(); e->keys[1].release(); e->vals[0].release(); e->vals[1].release(); e->sorted.release();
    e->transforms.release(); e->ctl.release(); e->depthp.release(); e->tile_hist.release(); e->freq.release(); e->dist_rows_i.release(); e->dist_rows_f.release(); e->sub_idx.release(); e->sub_dist.release();
    e->h_indexes.release(); e->h_sorted.release(); e->h_ctl.release(); e->h_frame.release(); e->h_pipe.release();
    e->tree.center.release(); e->tree.nmin.release(); e->tree.nmax.release(); e->tree.offsets.release(); e->tree.indexes.release(); e->tree.start.release(); e->tree.key.release(); e->tree.total.release(); e->flush.release(); e->prof.release();
    e->shard.block.release(); e->shard.total.release(); e->shard.ahead.release(); e->shard.block_total.release(); e->shard.delta.release(); e->shard.local_sorted.release();
    for (void *m : e->shard.opened) if (m) cudaIpcCloseMemHandle(m);
    if (e->rs.peer_attached) { if (e->rs.peer_frame) cudaIpcCloseMemHandle(e->rs.peer_frame); if (e->rs.peer_sync) cudaIpcCloseMemHandle(e->rs.peer_sync); }
    raster_release(e->rs);
    for (int i = 0; i < EV_COUNT; ++i) if (e->ev[i]) cudaEventDestroy(e->ev[i]);
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->stream2) cudaStreamDestroy(e->stream2);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    for (int i = 0; i < gs_engine::kPipeRing; ++i) { if (e->ev_frame_done[i]) cudaEventDestroy(e->ev_frame_done[i]); if (e->ev_copy_done[i]) cudaEventDestroy(e->ev_copy_done[i]); }
    for (int i = 0; i < 2; ++i) if (e->ev_params[i]) cudaEventDestroy(e->ev_params[i]);
    if (e->param_stream) cudaStreamDestroy(e->param_stream);
    e->status_dev.release();
    if (e->graph_exec) cudaGraphExecDestroy(e->graph_exec);
    if (e->graph_exec_alt) cudaGraphExecDestroy(e->graph_exec_alt);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    delete e;
}

extern "C" int gs_upload_centers(gs_engine *e, const void *centers, const uint32_t *sceneIndexes, uint32_t from, uint32_t count) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!centers && count) return fail(GS_ERR_BAD_ARG, "gs_upload_centers: null centers");
    if ((uint64_t)from + count > e->cfg.max_splat_count) return fail(GS_ERR_CAPACITY, "centres [%u,%u) exceed max_splat_count %u", from, from + count, e->cfg.max_splat_count);
    if (count) CU(cudaMemcpyAsync(e->centers.p + from, centers, (size_t)count * 16, cudaMemcpyHostToDevice, e->stream));
    if (e->cfg.dynamic_mode && sceneIndexes && count)
        CU(cudaMemcpyAsync(e->scene_idx.p + from, sceneIndexes, (size_t)count * 4, cudaMemcpyHostToDevice, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->uploaded_splats = from + count; // SortWorker.js:97
    return GS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
template <int MODE>
static void launch_depth(bool identity, int blocks, cudaStream_t st, const uint32_t *idx, const void *centers, const void *pre,
                         const uint32_t *scene, const float *tr, const DepthParams *P, uint32_t s0, uint32_t rc, int32_t *dist, SortControl *ctl) {
    if (identity) gs_launch(k_depth<MODE, true>, blocks, kDepthThreads, 0, st, idx, centers, pre, scene, tr, P, s0, rc, dist, ctl);
    else gs_launch(k_depth<MODE, false>, blocks, kDepthThreads, 0, st, idx, centers, pre, scene, tr, P, s0, rc, dist, ctl);
}

// Distance pass (sorter.cpp:29-140) over positions [lo, hi) of the index list: dist[i] and the running min/max in the control block.
static int enqueue_depth(gs_engine *e, const uint32_t *d_indexes, const float *mvp, bool use_pre, uint32_t lo, uint32_t hi, bool capturing) {
    cudaStream_t st = e->stream;
    const uint32_t n = hi - lo;
    DepthParams P{};
    memcpy(P.mvp, mvp, 64);
    P.irow[0] = (int32_t)((double)mvp[2] * 1000.0);   // sorter.cpp:64 -- f64 product, truncation toward zero
    P.irow[1] = (int32_t)((double)mvp[6] * 1000.0);
    P.irow[2] = (int32_t)((double)mvp[10] * 1000.0);
    P.irow[3] = 1;
    P.frow[0] = mvp[2]; P.frow[1] = mvp[6]; P.frow[2] = mvp[10]; P.frow[3] = 0.f;
    if (!capturing) CU(cudaMemcpyAsync(e->depthp.p + e->rs.frame_parity, &P, sizeof(P), cudaMemcpyHostToDevice, st)); // pageable source: staged before return
    const bool integer = e->cfg.integer_based_sort, dyn = e->cfg.dynamic_mode;
    const int mode = use_pre ? (integer ? kIntPrecomputed : kFloatPrecomputed)
                             : (integer ? (dyn ? kIntDynamic : kIntStatic) : (dyn ? kFloatDynamic : kFloatStatic));
    const int dblocks = (int)std::max<uint64_t>(1, std::min<uint64_t>(((uint64_t)n + kDepthThreads * kDepthItems - 1) / (kDepthThreads * kDepthItems), (uint64_t)e->sm_count * 8));
    const bool identity = (d_indexes == nullptr);
    const void *pre = e->precomputed.p;
    switch (mode) {
        case kIntStatic: launch_depth<kIntStatic>(identity, dblocks, st, d_indexes, e->centers.p, pre, e->scene_idx.p, e->transforms.p, e->depthp.p + e->rs.frame_parity, lo, hi, e->dist.p, e->ctl.p); break;
        case kIntDynamic: launch_depth<kIntDynamic>(identity, dblocks, st, d_indexes, e->centers.p, pre, e->scene_idx.p, e->transforms.p, e->depthp.p + e->rs.frame_parity, lo, hi, e->dist.p, e->ctl.p); break;
        case kIntPrecomputed: launch_depth<kIntPrecomputed>(identity, dblocks, st, d_indexes, e->centers.p, pre, e->scene_idx.p, e->transforms.p, e->depthp.p + e->rs.frame_parity, lo, hi, e->dist.p, e->ctl.p); break;
        case kFloatStatic: launch_depth<kFloatStatic>(identity, dblocks, st, d_indexes, e->centers.p, pre, e->scene_idx.p, e->transforms.p, e->depthp.p + e->rs.frame_parity, lo, hi, e->dist.p, e->ctl.p); break;
        case kFloatDynamic: launch_depth<kFloatDynamic>(identity, dblocks, st, d_indexes, e->centers.p, pre, e->scene_idx.p, e->transforms.p, e->depthp.p + e->rs.frame_parity, lo, hi, e->dist.p, e->ctl.p); break;
        default: launch_depth<kFloatPrecomputed>(identity, dblocks, st, d_indexes, e->centers.p, pre, e->scene_idx.p, e->transforms.p, e->depthp.p + e->rs.frame_parity, lo, hi, e->dist.p, e->ctl.p); break;
    }
    return GS_OK;
}

// The sort proper, everything already on the device.  d_indexes == nullptr: identity.
static int sort_on_device(gs_engine *e, const uint32_t *d_indexes, const float *mvp, uint32_t sort_count, uint32_t render_count,
                          bool use_pre, bool write_buckets, bool capturing = false, bool subset = false, cudaEvent_t wait_for_rects = nullptr) {
    if (sort_count > render_count) return fail(GS_ERR_BAD_ARG, "sortCount %u > renderCount %u", sort_count, render_count);
    if (render_count > e->cfg.max_splat_count) return fail(GS_ERR_CAPACITY, "renderCount %u > max_splat_count %u", render_count, e->cfg.max_splat_count);
    cudaStream_t st = e->stream;
    const uint32_t s0 = render_count - sort_count, n = sort_count;
    const PassPlan pl = make_plan_bits(e->key_bits);
    uint32_t launches = 0;
    uint32_t stride = 0;
    int rc = e->tile_hist.ensure(radix_tile_hist_words(std::max(n, 1u), pl.npasses, &stride));
    if (rc) return rc;
    if (!capturing) CU(cudaEventRecord(e->ev[EV_SORT0], st));
    if (!e->have_prof_begin) e->prof.begin(st);
    if (e->ctl_dirty && !capturing) {   // first sort, or the previous one failed part-way; a completed sort leaves the block clean
        gs_launch(k_sort_init, 1, 256, 0, st, e->ctl.p);
        ++launches;
    }
    if (!capturing) e->ctl_dirty = true;
    if (s0 > 0) { gs_launch(k_copy_head, std::min<uint32_t>((s0 + 255) / 256, e->sm_count * 8), 256, 0, st, d_indexes, e->sorted.p, s0); ++launches; e->prof.mark("k_copy_head", st); }
    if (n > 0) {
        if ((rc = enqueue_depth(e, d_indexes, mvp, use_pre, s0, render_count, capturing))) return rc;
        const bool identity = (d_indexes == nullptr);
        ++launches;
        e->prof.mark("k_depth", st);
        if (!capturing) CU(cudaEventRecord(e->ev[EV_DEPTH], st));
        const uint32_t tiles = (n + kRadixTile - 1) / kRadixTile;
        const uint32_t R = e->cfg.distance_map_range;
        const uint32_t *vsrc = identity ? nullptr : d_indexes + s0;
        int vmode = identity ? kValIotaReversed : kValArrayReversed;
        int32_t *dist_sorted = e->dist.p + s0;
        const unsigned long long *n_dev = nullptr;
        if (subset) {   // this rank sorts only the splats that reach its tiles; bucketed with the GLOBAL min/max found by k_depth above
            if (wait_for_rects) CU(cudaStreamWaitEvent(st, wait_for_rects, 0));
            int rcs = raster_subset(e->rs, e->cfg, d_indexes, render_count, e->dist.p, e->sub_idx.p, e->sub_dist.p, st, e->prof, launches);
            if (rcs) return rcs;
            vsrc = e->sub_idx.p; vmode = kValArrayReversed;
            dist_sorted = e->sub_dist.p;
            n_dev = &e->rs.rctl.p->subset_count;
        }
        static const RadixNames names = {{"k_radix_hist[depth,0]", "k_radix_hist[depth,1]", "k_radix_hist[depth,2]", "k_radix_hist[depth,3]"},
                                         {"k_radix_scan[depth,0]", "k_radix_scan[depth,1]", "k_radix_scan[depth,2]", "k_radix_scan[depth,3]"},
                                         {"k_radix_scatter[depth,0]", "k_radix_scatter[depth,1]", "k_radix_scatter[depth,2]", "k_radix_scatter[depth,3]"}};
        if (e->key_bits <= 16) {
            gs_launch(k_bucket<uint16_t>, tiles, kRadixThreads, 0, st, dist_sorted, (uint16_t *)e->keys[0].p, n, n_dev, R, pl, write_buckets ? 1 : 0, e->ctl.p, e->tile_hist.p, stride);
            ++launches;
            e->prof.mark("k_bucket", st);
            if (!capturing) CU(cudaEventRecord(e->ev[EV_BUCKET], st));
            radix_sort_pairs<uint16_t, uint32_t>((uint16_t *)e->keys[0].p, (uint16_t *)e->keys[1].p, vsrc, render_count - 1u, vmode, e->vals[0].p, e->vals[1].p,
                                       e->sorted.p + s0, n, n_dev, (unsigned long long)n, pl, e->ctl.p, e->tile_hist.p, stride, true, nullptr, st, launches, &e->prof, names, true);
        } else {
            gs_launch(k_bucket<uint32_t>, tiles, kRadixThreads, 0, st, dist_sorted, e->keys[0].p, n, n_dev, R, pl, write_buckets ? 1 : 0, e->ctl.p, e->tile_hist.p, stride);
            ++launches;
            e->prof.mark("k_bucket", st);
            if (!capturing) CU(cudaEventRecord(e->ev[EV_BUCKET], st));
            radix_sort_pairs<uint32_t, uint32_t>(e->keys[0].p, e->keys[1].p, vsrc, render_count - 1u, vmode, e->vals[0].p, e->vals[1].p, e->sorted.p + s0, n,
                                       n_dev, (unsigned long long)n, pl, e->ctl.p, e->tile_hist.p, stride, true, nullptr, st, launches, &e->prof, names, true);
        }
    } else if (!capturing) {
        CU(cudaEventRecord(e->ev[EV_DEPTH], st));
        CU(cudaEventRecord(e->ev[EV_BUCKET], st));
    }
    if (!capturing) CU(cudaEventRecord(e->ev[EV_SORT1], st));
    CU(cudaGetLastError());
    e->tm.kernel_launches = launches;
    e->last_render_count = render_count;
    e->have_sorted = true;
    if (!capturing) e->ctl_dirty = false;
    return GS_OK;
}

// after a stream sync: fold the device-side error bits and stage timings into the engine
static int finish_sort(gs_engine *e, float *sort_time_ms) {
    CU(cudaMemcpyAsync(e->h_ctl.p, e->ctl.p, 12, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    float ms = 0.f;
    if (e->last_frame_was_graph) {   // one graph launch: only the whole-frame time is observable
        e->tm.depth_ms = e->tm.bucket_ms = e->tm.scatter_ms = 0.f;
        cudaEventElapsedTime(&ms, e->ev[EV_SORT0], e->ev[EV_R1]);
    } else {
        cudaEventElapsedTime(&e->tm.depth_ms, e->ev[EV_SORT0], e->ev[EV_DEPTH]);
        cudaEventElapsedTime(&e->tm.bucket_ms, e->ev[EV_DEPTH], e->ev[EV_BUCKET]);
        cudaEventElapsedTime(&e->tm.scatter_ms, e->ev[EV_BUCKET], e->ev[EV_SORT1]);
        cudaEventElapsedTime(&ms, e->ev[EV_SORT0], e->ev[EV_SORT1]);
    }
    e->tm.sort_total_ms = ms;
    if (sort_time_ms) *sort_time_ms = ms;
    const uint32_t err = e->h_ctl.p[2];
    if (err & kErrBucketRange) return fail(GS_ERR_BUCKET_RANGE, "a bucket index fell outside [0,%u): distances overflow the int32/f32 range map", e->cfg.distance_map_range);
    return GS_OK;
}

static int stage_sort_inputs(gs_engine *e, const gs_sort_params *p, const uint32_t **d_indexes) {
    cudaStream_t st = e->stream;
    *d_indexes = nullptr;
    CU(cudaEventRecord(e->ev[EV_H2D0], st));
    if (p->indexes_to_sort_dev) *d_indexes = p->indexes_to_sort_dev;
    else if (p->indexes_to_sort) {
        CU(cudaMemcpyAsync(e->indexes.p, p->indexes_to_sort, (size_t)p->render_count * 4, cudaMemcpyHostToDevice, st));
        *d_indexes = e->indexes.p;
    }
    if (e->cfg.dynamic_mode && p->transforms) CU(cudaMemcpyAsync(e->transforms.p, p->transforms, 16 * GS_MAX_SCENES * 4, cudaMemcpyHostToDevice, st));
    if (p->use_precomputed_distances) {
        if (!p->precomputed_distances) return fail(GS_ERR_BAD_ARG, "use_precomputed_distances without precomputed_distances");
        int rc = e->precomputed.ensure(e->cfg.max_splat_count);
        if (rc) return rc;
        CU(cudaMemcpyAsync(e->precomputed.p, p->precomputed_distances, (size_t)e->uploaded_splats * 4, cudaMemcpyHostToDevice, st));
    }
    CU(cudaEventRecord(e->ev[EV_H2D1], st));
    return GS_OK;
}

extern "C" int gs_sort(gs_engine *e, const gs_sort_params *p, uint32_t *sorted_out, float *sort_time_ms) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!p) return fail(GS_ERR_BAD_ARG, "gs_sort: null params");
    // SortWorker.js:99-100: counts are clamped to what has been uploaded
    gs_sort_params q = *p;
    q.render_count = std::min(q.render_count, e->uploaded_splats);
    q.sort_count = std::min(q.sort_count, e->uploaded_splats);
    if (q.sort_count > q.render_count) return fail(GS_ERR_BAD_ARG, "sortCount %u > renderCount %u", q.sort_count, q.render_count);
    const uint32_t *d_idx = nullptr;
    e->last_frame_was_graph = false;
    if ((rc = stage_sort_inputs(e, &q, &d_idx))) return rc;
    if ((rc = sort_on_device(e, d_idx, q.model_view_proj, q.sort_count, q.render_count, q.use_precomputed_distances != 0, false))) return rc;
    CU(cudaEventRecord(e->ev[EV_D2H0], e->stream));
    if (sorted_out && q.render_count) CU(cudaMemcpyAsync(sorted_out, e->sorted.p, (size_t)q.render_count * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaEventRecord(e->ev[EV_D2H1], e->stream));
    rc = finish_sort(e, sort_time_ms);
    cudaEventElapsedTime(&e->tm.h2d_ms, e->ev[EV_H2D0], e->ev[EV_H2D1]);
    cudaEventElapsedTime(&e->tm.d2h_ms, e->ev[EV_D2H0], e->ev[EV_D2H1]);
    return rc;
}


// ---------------------------------------------------------------------------------------------------------------
// Sort-only on N GPUs (SURVEY.md 8(e) "depth + sort"): rank g sorts the input positions [lo_g, hi_g) of the sort window and the
// ranks assemble the reference's global order in rank 0's sortedIndexes over peer memory.  See shard_kernels.cuh.
static int shard_prepare(gs_engine *e) {
    const uint32_t R = e->cfg.distance_map_range;
    int rc;
    const size_t bytes = sizeof(ShardHeader) + (size_t)R * sizeof(uint2);
    if (e->shard.block.n < bytes) {
        if ((rc = e->shard.block.ensure(bytes))) return rc;
        CU(cudaMemset(e->shard.block.p, 0, bytes));
    }
    const size_t blocks = ((size_t)R + kShardScanThreads - 1) / kShardScanThreads;
    if ((rc = e->shard.total.ensure(R)) || (rc = e->shard.ahead.ensure(R)) || (rc = e->shard.delta.ensure(R)) || (rc = e->shard.block_total.ensure(blocks)) ||
        (rc = e->shard.local_sorted.ensure(e->cfg.max_splat_count)))
        return rc;
    // everything the per-sort path could otherwise grow (cudaFree synchronises the device: not while a peer's wait kernel may be spinning)
    const PassPlan pl = make_plan_bits(e->key_bits);
    if ((rc = e->tile_hist.ensure(radix_tile_hist_words(std::max(e->cfg.max_splat_count, 1u), pl.npasses, nullptr))) || (rc = e->precomputed.ensure(e->cfg.max_splat_count))) return rc;
    return GS_OK;
}
// CUDA loads a kernel's code on its first launch (lazy module loading) and that load can wait for running kernels to finish.  The
// sharded sort keeps bounded spin-wait kernels in flight while the host enqueues the rest of the chain, so every kernel of the chain
// is loaded up front (cudaFuncGetAttributes forces the load); otherwise a first sort could stall on its own wait kernel.
template <typename F> static inline void preload_kernel(F f) { cudaFuncAttributes a; (void)cudaFuncGetAttributes(&a, f); }
template <typename KeyT> static void shard_preload_keyed() {
    preload_kernel(k_bucket<KeyT>);
    preload_kernel(k_radix_hist<KeyT>);
    preload_kernel(k_shard_place<KeyT>);
    preload_kernel(k_radix_scatter<KeyT, uint32_t, kValArray, true, false>);
    preload_kernel(k_radix_scatter<KeyT, uint32_t, kValArrayReversed, true, false>);
    preload_kernel(k_radix_scatter<KeyT, uint32_t, kValIotaReversed, true, false>);
    preload_kernel(k_radix_scatter<KeyT, uint32_t, kValArray, true, true>);
    preload_kernel(k_radix_scatter<KeyT, uint32_t, kValArrayReversed, true, true>);
    preload_kernel(k_radix_scatter<KeyT, uint32_t, kValIotaReversed, true, true>);
}
template <int MODE> static void shard_preload_depth() { preload_kernel(k_depth<MODE, true>); preload_kernel(k_depth<MODE, false>); }
static void shard_preload(gs_engine *e) {
    preload_kernel(k_sort_init); preload_kernel(k_copy_head); preload_kernel(k_radix_scan);
    preload_kernel(k_shard_exchange_minmax); preload_kernel(k_shard_exchange_runs); preload_kernel(k_shard_totals); preload_kernel(k_shard_delta); preload_kernel(k_shard_done);
    shard_preload_depth<kIntStatic>(); shard_preload_depth<kIntDynamic>(); shard_preload_depth<kIntPrecomputed>();
    shard_preload_depth<kFloatStatic>(); shard_preload_depth<kFloatDynamic>(); shard_preload_depth<kFloatPrecomputed>();
    if (e->key_bits <= 16) shard_preload_keyed<uint16_t>(); else shard_preload_keyed<uint32_t>();
    (void)cudaGetLastError();
}
static inline ShardHeader *shard_hdr(void *block) { return (ShardHeader *)block; }
static inline const uint2 *shard_runs(void *block) { return (const uint2 *)((unsigned char *)block + sizeof(ShardHeader)); }

extern "C" int gs_shard_export(gs_engine *e, void *block_handle, void *sorted_handle) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!block_handle || !sorted_handle) return fail(GS_ERR_BAD_ARG, "gs_shard_export: null");
    if ((rc = shard_prepare(e))) return rc;
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, e->shard.block.p));
    memcpy(block_handle, &h, sizeof(h));
    CU(cudaIpcGetMemHandle(&h, e->sorted.p));
    memcpy(sorted_handle, &h, sizeof(h));
    return GS_OK;
}
static int shard_bind(gs_engine *e, uint32_t world, void *const *blocks, uint32_t *root_out) {
    for (uint32_t g = 0; g < world; ++g) {
        e->shard.peers.hdr[g] = shard_hdr(blocks[g]);
        e->shard.peers.runs[g] = shard_runs(blocks[g]);
    }
    shard_preload(e);
    e->shard.root_out = root_out;
    e->shard.world = world;
    e->shard.seq = 0;
    e->shard.attached = true;
    return GS_OK;
}
static int shard_check_group(gs_engine *e, uint32_t world, const char *who) {
    if (world < 1 || world > (uint32_t)kMaxShardRanks) return fail(GS_ERR_BAD_ARG, "%s: world %u outside [1, %d]", who, world, kMaxShardRanks);
    if (e->cfg.world_size != world || e->cfg.rank >= world) return fail(GS_ERR_BAD_ARG, "%s: engine was created as rank %u of %u, not of %u", who, e->cfg.rank, e->cfg.world_size, world);
    return GS_OK;
}
extern "C" int gs_shard_attach(gs_engine *e, uint32_t world, const void *block_handles, const void *root_sorted_handle) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!block_handles || !root_sorted_handle) return fail(GS_ERR_BAD_ARG, "gs_shard_attach: null");
    if ((rc = shard_check_group(e, world, "gs_shard_attach")) || (rc = shard_prepare(e))) return rc;
    void *blocks[kMaxShardRanks] = {nullptr};
    for (uint32_t g = 0; g < world; ++g) {
        if (g == e->cfg.rank) { blocks[g] = e->shard.block.p; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const unsigned char *)block_handles + (size_t)g * GS_IPC_HANDLE_BYTES, sizeof(h));
        CU(cudaIpcOpenMemHandle(&blocks[g], h, cudaIpcMemLazyEnablePeerAccess));
        e->shard.opened[g] = blocks[g];
    }
    uint32_t *root_out = e->sorted.p;
    if (e->cfg.rank != 0) {
        cudaIpcMemHandle_t h;
        void *m = nullptr;
        memcpy(&h, root_sorted_handle, sizeof(h));
        CU(cudaIpcOpenMemHandle(&m, h, cudaIpcMemLazyEnablePeerAccess));
        e->shard.opened[kMaxShardRanks] = m;
        root_out = (uint32_t *)m;
    }
    return shard_bind(e, world, blocks, root_out);
}
// Same process, same device (several engines sharing one GPU, or a test without a second GPU): plain pointers instead of IPC mappings.
extern "C" int gs_shard_attach_local(gs_engine *e, uint32_t world, gs_engine *const *engines) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!engines) return fail(GS_ERR_BAD_ARG, "gs_shard_attach_local: null");
    if ((rc = shard_check_group(e, world, "gs_shard_attach_local"))) return rc;
    void *blocks[kMaxShardRanks] = {nullptr};
    for (uint32_t g = 0; g < world; ++g) {
        gs_engine *pe = engines[g];
        if (!pe || pe->cfg.device != e->cfg.device || pe->cfg.rank != g || pe->cfg.world_size != world ||
            pe->cfg.distance_map_range != e->cfg.distance_map_range)
            return fail(GS_ERR_BAD_ARG, "gs_shard_attach_local: engines[%u] must be rank %u of %u on device %d with the same distance_map_range", g, g, world, e->cfg.device);
        if ((rc = shard_prepare(pe))) return rc;
        blocks[g] = pe->shard.block.p;
    }
    return shard_bind(e, world, blocks, engines[0]->sorted.p);
}

template <typename KeyT>
static int shard_local_sort(gs_engine *e, const uint32_t *d_indexes, uint32_t s0, uint32_t lo, uint32_t hi, uint32_t &launches) {
    cudaStream_t st = e->stream;
    const uint32_t n = hi - lo, R = e->cfg.distance_map_range;
    const PassPlan pl = make_plan_bits(e->key_bits);
    uint32_t stride = 0;
    int rc = e->tile_hist.ensure(radix_tile_hist_words(std::max(n, 1u), pl.npasses, &stride));
    if (rc) return rc;
    const bool identity = (d_indexes == nullptr);
    static const RadixNames names = {{"k_radix_hist[shard,0]", "k_radix_hist[shard,1]", "k_radix_hist[shard,2]", "k_radix_hist[shard,3]"},
                                     {"k_radix_scan[shard,0]", "k_radix_scan[shard,1]", "k_radix_scan[shard,2]", "k_radix_scan[shard,3]"},
                                     {"k_radix_scatter[shard,0]", "k_radix_scatter[shard,1]", "k_radix_scatter[shard,2]", "k_radix_scatter[shard,3]"}};
    const uint32_t me = e->cfg.rank, world = e->shard.world, seq = e->shard.seq;
    uint2 *runs = (uint2 *)shard_runs(e->shard.block.p);
    KeyT *final_keys = nullptr;
    if (n) {   // slice -> keys with the GLOBAL range map -> local order + per-key runs of that order
        const uint32_t tiles = (n + kRadixTile - 1) / kRadixTile;
        gs_launch(k_bucket<KeyT>, tiles, kRadixThreads, 0, st, e->dist.p + lo, (KeyT *)e->keys[0].p, n, nullptr, R, pl, 0, e->ctl.p, e->tile_hist.p, stride);
        ++launches;
        e->prof.mark("k_bucket", st);
        radix_sort_pairs<KeyT, uint32_t>((KeyT *)e->keys[0].p, (KeyT *)e->keys[1].p, identity ? nullptr : d_indexes + lo, hi - 1u,
                                         identity ? kValIotaReversed : kValArrayReversed, e->vals[0].p, e->vals[1].p, e->shard.local_sorted.p, n, nullptr,
                                         (unsigned long long)n, pl, e->ctl.p, e->tile_hist.p, stride, true, runs, st, launches, &e->prof, names, true, true, &final_keys);
    }
    // C2: publish my runs, wait for everybody's, turn them into the offsets of my runs in the global order
    k_shard_exchange_runs<<<1, 32, 0, st>>>(e->shard.peers, me, world, seq);
    ++launches;
    e->prof.mark("k_shard_exchange_runs", st);
    if (n) {
        const uint32_t sblocks = (R + kShardScanThreads - 1) / kShardScanThreads;
        k_shard_totals<<<sblocks, kShardScanThreads, 0, st>>>(e->shard.peers, me, world, R, e->shard.total.p, e->shard.ahead.p, e->shard.block_total.p);
        k_shard_delta<<<sblocks, kShardScanThreads, 0, st>>>(runs, R, e->shard.total.p, e->shard.ahead.p, e->shard.block_total.p, e->shard.delta.p);
        e->prof.mark("k_shard_offsets", st);
        k_shard_place<KeyT><<<std::min<uint32_t>((n + 255) / 256, e->sm_count * 16), 256, 0, st>>>(final_keys, e->shard.local_sorted.p, n, e->shard.delta.p, e->shard.root_out + s0);
        e->prof.mark("k_shard_place", st);
        launches += 3;
    }
    return GS_OK;
}

// Position slice of rank g: [sortStart + n*g/G, sortStart + n*(g+1)/G)
static inline uint32_t shard_bound(uint32_t s0, uint32_t n, uint32_t g, uint32_t world) { return s0 + (uint32_t)(((uint64_t)n * g) / world); }

extern "C" int gs_sort_sharded_async(gs_engine *e, const gs_sort_params *p) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!p) return fail(GS_ERR_BAD_ARG, "gs_sort_sharded: null params");
    if (!e->shard.attached) return fail(GS_ERR_NOT_READY, "gs_sort_sharded: call gs_shard_attach (or gs_shard_attach_local) first");
    if (e->shard.pending) return fail(GS_ERR_NOT_READY, "gs_sort_sharded_async: the previous sharded sort has not been finished");
    gs_sort_params q = *p;
    q.render_count = std::min(q.render_count, e->uploaded_splats);   // SortWorker.js:99-100
    q.sort_count = std::min(q.sort_count, e->uploaded_splats);
    if (q.sort_count > q.render_count) return fail(GS_ERR_BAD_ARG, "sortCount %u > renderCount %u", q.sort_count, q.render_count);
    const uint32_t *d_idx = nullptr;
    e->last_frame_was_graph = false;
    const uint32_t me = e->cfg.rank, world = e->shard.world;
    // The split pays only for large windows (DESIGN.md 6.1: three NVLink handshakes + offsets + placement vs a single sort that is
    // latency bound below ~8 M splats).  Smaller calls are sorted by rank 0 alone; the decision depends only on the call's arguments,
    // so every rank takes the same branch.  GS_SHARD_MIN overrides the threshold (0 = always split).
    uint32_t split_min = 8000000u;
    if (const char *sv = getenv("GS_SHARD_MIN")) split_min = (uint32_t)strtoul(sv, nullptr, 10);
    if (world == 1 || q.sort_count < split_min) {
        e->shard.pending = true;
        e->shard.pending_unsplit = true;
        e->shard.pending_render_count = q.render_count;
        if (me != 0) return GS_OK;
        if ((rc = stage_sort_inputs(e, &q, &d_idx)) ||
            (rc = sort_on_device(e, d_idx, q.model_view_proj, q.sort_count, q.render_count, q.use_precomputed_distances != 0, false))) {
            e->shard.pending = false;
            return rc;
        }
        return GS_OK;
    }
    e->shard.pending_unsplit = false;
    if ((rc = stage_sort_inputs(e, &q, &d_idx))) return rc;
    cudaStream_t st = e->stream;
    const uint32_t s0 = q.render_count - q.sort_count;
    const uint32_t lo = shard_bound(s0, q.sort_count, me, world), hi = shard_bound(s0, q.sort_count, me + 1, world);
    const uint32_t seq = ++e->shard.seq;
    uint32_t launches = 0;
    CU(cudaEventRecord(e->ev[EV_SORT0], st));
    e->prof.begin(st);
    if (e->ctl_dirty) { gs_launch(k_sort_init, 1, 256, 0, st, e->ctl.p); ++launches; }
    e->ctl_dirty = true;
    if (me == 0 && s0 > 0) { gs_launch(k_copy_head, std::min<uint32_t>((s0 + 255) / 256, e->sm_count * 8), 256, 0, st, d_idx, e->sorted.p, s0); ++launches; e->prof.mark("k_copy_head", st); }
    if (hi > lo) {
        if ((rc = enqueue_depth(e, d_idx, q.model_view_proj, q.use_precomputed_distances != 0, lo, hi, false))) return rc;
        ++launches;
        e->prof.mark("k_depth", st);
    }
    // C1: global min/max over peer memory
    k_shard_exchange_minmax<<<1, kShardSyncThreads, 0, st>>>(e->shard.peers, e->ctl.p, me, world, seq, hi > lo ? 0 : 1, (uint2 *)shard_runs(e->shard.block.p),
                                                             e->cfg.distance_map_range);
    ++launches;
    e->prof.mark("k_shard_exchange_minmax", st);
    CU(cudaEventRecord(e->ev[EV_DEPTH], st));
    CU(cudaEventRecord(e->ev[EV_BUCKET], st));
    rc = (e->key_bits <= 16) ? shard_local_sort<uint16_t>(e, d_idx, s0, lo, hi, launches) : shard_local_sort<uint32_t>(e, d_idx, s0, lo, hi, launches);
    if (rc) return rc;
    k_shard_done<<<1, 32, 0, st>>>(e->shard.peers, me, world, seq);
    ++launches;
    e->prof.mark("k_shard_done", st);
    CU(cudaEventRecord(e->ev[EV_SORT1], st));
    CU(cudaGetLastError());
    e->tm.kernel_launches = launches;
    e->last_render_count = q.render_count;
    e->have_sorted = (me == 0);     // the assembled order lives in rank 0's sortedIndexes
    e->ctl_dirty = !(hi > lo);      // an empty slice ran no final radix pass, which is what re-seeds the control block
    e->shard.pending = true;
    e->shard.pending_render_count = q.render_count;
    return GS_OK;
}

extern "C" int gs_sort_sharded_finish(gs_engine *e, uint32_t *sorted_out, float *sort_time_ms) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!e->shard.pending) return fail(GS_ERR_NOT_READY, "gs_sort_sharded_finish: nothing pending");
    e->shard.pending = false;
    const uint32_t rcnt = e->shard.pending_render_count;
    if (e->shard.pending_unsplit && e->cfg.rank != 0) {   // rank 0 sorted alone
        if (sort_time_ms) *sort_time_ms = 0.f;
        return GS_OK;
    }
    CU(cudaEventRecord(e->ev[EV_D2H0], e->stream));
    if (sorted_out && rcnt && e->cfg.rank == 0) CU(cudaMemcpyAsync(sorted_out, e->sorted.p, (size_t)rcnt * 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaEventRecord(e->ev[EV_D2H1], e->stream));
    if (e->shard.pending_unsplit) {
        rc = finish_sort(e, sort_time_ms);
        cudaEventElapsedTime(&e->tm.h2d_ms, e->ev[EV_H2D0], e->ev[EV_H2D1]);
        cudaEventElapsedTime(&e->tm.d2h_ms, e->ev[EV_D2H0], e->ev[EV_D2H1]);
        return rc;
    }
    CU(cudaMemcpyAsync(e->h_ctl.p + 640, e->shard.block.p, sizeof(ShardHeader), cudaMemcpyDeviceToHost, e->stream));
    rc = finish_sort(e, sort_time_ms);
    cudaEventElapsedTime(&e->tm.h2d_ms, e->ev[EV_H2D0], e->ev[EV_H2D1]);
    cudaEventElapsedTime(&e->tm.d2h_ms, e->ev[EV_D2H0], e->ev[EV_D2H1]);
    ShardHeader hd;
    memcpy(&hd, e->h_ctl.p + 640, sizeof(hd));
    if (hd.timeout) {
        cudaMemsetAsync(&shard_hdr(e->shard.block.p)->timeout, 0, 4, e->stream);
        e->ctl_dirty = true;
        return fail(GS_ERR_CUDA, "sharded sort: a peer rank did not reach the exchange within the time limit (are all %u ranks calling gs_sort_sharded?)", e->shard.world);
    }
    return rc;
}

extern "C" int gs_sort_sharded(gs_engine *e, const gs_sort_params *p, uint32_t *sorted_out, float *sort_time_ms) {
    int rc = gs_sort_sharded_async(e, p);
    if (rc) return rc;
    return gs_sort_sharded_finish(e, sorted_out, sort_time_ms);
}

// ---------------------------------------------------------------------------------------------------------------
// Stateless drop-in (sorter.cpp:17-22).  A private engine per (device 0, splatCount, mode, range) is cached so repeated
// calls do not re-allocate; inputs are uploaded on every call like a non-shared-memory worker copies them
// (SortWorker.js:35-51).
static gs_engine *g_dropin = nullptr;
#include <mutex>
static std::mutex g_dropin_mutex;   // the stateless entry shares one cached engine: calls are serialised, not rejected

extern "C" void gs_dropin_release(void) {
    std::lock_guard<std::mutex> lock(g_dropin_mutex);
    if (g_dropin) { gs_destroy(g_dropin); g_dropin = nullptr; }
}

extern "C" int gs_sort_indexes(const uint32_t *indexes, const void *centers, const void *precomputedDistances, int32_t *mappedDistances,
                               uint32_t *frequencies, const float *modelViewProj, uint32_t *indexesOut, const uint32_t *sceneIndexes,
                               const float *transforms, uint32_t distanceMapRange, uint32_t sortCount, uint32_t renderCount,
                               uint32_t splatCount, bool usePrecomputedDistances, bool useIntegerSort, bool dynamicMode) {
    if (!indexes || !modelViewProj || !indexesOut) return fail(GS_ERR_BAD_ARG, "gs_sort_indexes: null indexes/modelViewProj/indexesOut");
    if (!usePrecomputedDistances && !centers) return fail(GS_ERR_BAD_ARG, "gs_sort_indexes: null centers");
    if (usePrecomputedDistances && !precomputedDistances) return fail(GS_ERR_BAD_ARG, "gs_sort_indexes: null precomputedDistances");
    if (dynamicMode && !usePrecomputedDistances && (!sceneIndexes || !transforms)) return fail(GS_ERR_BAD_ARG, "gs_sort_indexes: dynamic mode needs sceneIndexes and transforms");
    if (sortCount > renderCount || renderCount > splatCount) return fail(GS_ERR_BAD_ARG, "need sortCount <= renderCount <= splatCount");
    if (distanceMapRange < 2 || distanceMapRange > (1u << 24)) return fail(GS_ERR_BAD_ARG, "distanceMapRange %u outside [2, 2^24]", distanceMapRange);
    std::lock_guard<std::mutex> lock(g_dropin_mutex);
    int cur_dev = 0;
    if (cudaGetDevice(&cur_dev) != cudaSuccess) { cudaGetLastError(); cur_dev = 0; }     // the caller's current device, like any CUDA library
    gs_engine *e = g_dropin;
    if (!e || e->cfg.device != cur_dev || e->cfg.max_splat_count < splatCount || e->cfg.distance_map_range != distanceMapRange ||
        (bool)e->cfg.integer_based_sort != useIntegerSort || (bool)e->cfg.dynamic_mode != dynamicMode) {
        if (e) gs_destroy(e);
        g_dropin = nullptr;
        gs_config c{};
        c.struct_size = sizeof(c);
        c.device = cur_dev;
        c.max_splat_count = std::max(splatCount, 1u);
        c.distance_map_range = distanceMapRange;
        c.integer_based_sort = useIntegerSort;
        c.dynamic_mode = dynamicMode;
        int rc = gs_create(&c, &e);
        if (rc) return rc;
        g_dropin = e;
    }
    int rc = check_engine(e);
    if (rc) return rc;
    cudaStream_t st = e->stream;
    if (centers && splatCount) CU(cudaMemcpyAsync(e->centers.p, centers, (size_t)splatCount * 16, cudaMemcpyHostToDevice, st));
    if (dynamicMode && sceneIndexes && splatCount) CU(cudaMemcpyAsync(e->scene_idx.p, sceneIndexes, (size_t)splatCount * 4, cudaMemcpyHostToDevice, st));
    if (dynamicMode && transforms) CU(cudaMemcpyAsync(e->transforms.p, transforms, 16 * GS_MAX_SCENES * 4, cudaMemcpyHostToDevice, st));
    if (usePrecomputedDistances) {
        if ((rc = e->precomputed.ensure(e->cfg.max_splat_count))) return rc;
        CU(cudaMemcpyAsync(e->precomputed.p, precomputedDistances, (size_t)splatCount * 4, cudaMemcpyHostToDevice, st));
    }
    if (renderCount) CU(cudaMemcpyAsync(e->indexes.p, indexes, (size_t)renderCount * 4, cudaMemcpyHostToDevice, st));
    e->uploaded_splats = splatCount;
    e->last_frame_was_graph = false;
    const bool want_scratch = (mappedDistances != nullptr) || (frequencies != nullptr);
    if ((rc = sort_on_device(e, e->indexes.p, modelViewProj, sortCount, renderCount, usePrecomputedDistances, want_scratch))) return rc;
    // wasm-trap emulation: results are only written back when the device reported no range error
    if ((rc = finish_sort(e, nullptr))) return rc;
    if (renderCount) CU(cudaMemcpyAsync(indexesOut, e->sorted.p, (size_t)renderCount * 4, cudaMemcpyDeviceToHost, st));
    const uint32_t s0 = renderCount - sortCount;
    if (mappedDistances && sortCount) CU(cudaMemcpyAsync(mappedDistances + s0, e->dist.p + s0, (size_t)sortCount * 4, cudaMemcpyDeviceToHost, st));
    if (frequencies) {
        if ((rc = e->freq.ensure(distanceMapRange))) return rc;
        CU(cudaMemsetAsync(e->freq.p, 0, (size_t)distanceMapRange * 4, st));
        if (sortCount) k_bucket_counts<<<std::min<uint32_t>((sortCount + 255) / 256, e->sm_count * 8), 256, 0, st>>>(e->dist.p, s0, renderCount, e->freq.p);
        k_exclusive_scan_single_block<<<1, 1024, 0, st>>>(e->freq.p, distanceMapRange);
        CU(cudaMemcpyAsync(frequencies, e->freq.p, (size_t)distanceMapRange * 4, cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return GS_OK;
}

extern "C" void sortIndexes(unsigned int *indexes, void *centers, void *precomputedDistances, int *mappedDistances,
                            unsigned int *frequencies, float *modelViewProj, unsigned int *indexesOut, unsigned int *sceneIndexes,
                            float *transforms, unsigned int distanceMapRange, unsigned int sortCount, unsigned int renderCount,
                            unsigned int splatCount, bool usePrecomputedDistances, bool useIntegerSort, bool dynamicMode) {
    (void)gs_sort_indexes(indexes, centers, precomputedDistances, mappedDistances, frequencies, modelViewProj, indexesOut, sceneIndexes,
                          transforms, distanceMapRange, sortCount, renderCount, splatCount, usePrecomputedDistances, useIntegerSort, dynamicMode);
}

// ---------------------------------------------------------------------------------------------------------------
// D1: SplatMesh.computeDistancesOnGPU.  mvp is f64 because three.js Matrix4 elements are JS numbers and the integer rows
// are Math.round(element * 1000) on those doubles (SplatMesh.js:2057-2064).
extern "C" int gs_compute_distances(gs_engine *e, const double *mvp, const double *scene_transforms, uint32_t count, void *out) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!mvp || !out) return fail(GS_ERR_BAD_ARG, "gs_compute_distances: null argument");
    if (count > e->uploaded_splats) return fail(GS_ERR_CAPACITY, "count %u > uploaded splats %u", count, e->uploaded_splats);
    const bool integer = e->cfg.integer_based_sort, dyn = e->cfg.dynamic_mode;
    if (dyn && !scene_transforms) return fail(GS_ERR_BAD_ARG, "dynamic mode needs scene_transforms (f64[16*32])");
    std::vector<int32_t> irows(4 * GS_MAX_SCENES, 0);
    std::vector<float> frows(4 * GS_MAX_SCENES, 0.f);
    auto jsround = [](double v) { return (int32_t)std::floor(v + 0.5); }; // Math.round
    for (int s = 0; s < (dyn ? GS_MAX_SCENES : 1); ++s) {
        double m[16];
        if (dyn) { // tempMatrix = mvp * transform_s (three.js Matrix4.multiply, f64)   SplatMesh.js:1722-1724
            const double *t = scene_transforms + 16 * s;
            for (int c = 0; c < 4; ++c)
                for (int r = 0; r < 4; ++r) m[4 * c + r] = mvp[r] * t[4 * c] + mvp[4 + r] * t[4 * c + 1] + mvp[8 + r] * t[4 * c + 2] + mvp[12 + r] * t[4 * c + 3];
        } else memcpy(m, mvp, sizeof(m));
        for (int k = 0; k < 4; ++k) {
            irows[4 * s + k] = jsround(m[2 + 4 * k] * 1000.0);
            frows[4 * s + k] = (float)m[2 + 4 * k];
        }
    }
    DevBuf<int32_t> &d_ir = e->dist_rows_i;   // engine-owned scratch: an early error return must not leak it
    DevBuf<float> &d_fr = e->dist_rows_f;
    if ((rc = d_ir.ensure(irows.size())) || (rc = d_fr.ensure(frows.size()))) return rc;
    cudaStream_t st = e->stream;
    CU(cudaMemcpyAsync(d_ir.p, irows.data(), irows.size() * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_fr.p, frows.data(), frows.size() * 4, cudaMemcpyHostToDevice, st));
    if ((rc = e->precomputed.ensure(e->cfg.max_splat_count))) return rc;
    const int blocks = std::max(1, (int)std::min<uint32_t>((count + 255) / 256, e->sm_count * 8));
    if (integer && dyn) k_distances_splat_order<true, true><<<blocks, 256, 0, st>>>(e->centers.p, e->scene_idx.p, d_ir.p, d_fr.p, count, e->precomputed.p);
    else if (integer) k_distances_splat_order<true, false><<<blocks, 256, 0, st>>>(e->centers.p, e->scene_idx.p, d_ir.p, d_fr.p, count, e->precomputed.p);
    else if (dyn) k_distances_splat_order<false, true><<<blocks, 256, 0, st>>>(e->centers.p, e->scene_idx.p, d_ir.p, d_fr.p, count, e->precomputed.p);
    else k_distances_splat_order<false, false><<<blocks, 256, 0, st>>>(e->centers.p, e->scene_idx.p, d_ir.p, d_fr.p, count, e->precomputed.p);
    CU(cudaMemcpyAsync(out, e->precomputed.p, (size_t)count * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return GS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
extern "C" int gs_upload_splat_data(gs_engine *e, const gs_splat_data *d) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!d) return fail(GS_ERR_BAD_ARG, "gs_upload_splat_data: null");
    // callers built against the shorter struct (no scale_rotations) are recognised by struct_size; 0 means that older layout
    gs_splat_data dd{};
    const size_t old_size = offsetof(gs_splat_data, scale_rotations);
    memcpy(&dd, d, std::min<size_t>(d->struct_size ? d->struct_size : old_size, sizeof(gs_splat_data)));
    rc = raster_upload(e->rs, e->cfg, dd, e->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(e->stream));
    return GS_OK;
}

static int render_on_device(gs_engine *e, const gs_uniforms *u, const gs_render_params *p, const uint32_t *d_order, bool capturing = false, int phases = 3,
                            const unsigned long long *order_count_dev = nullptr) {
    cudaStream_t st = e->stream;
    if (!capturing && (phases & 1)) CU(cudaEventRecord(e->ev[EV_R0], st));
    if (!e->have_prof_begin) e->prof.begin(st);
    int rc = raster_render(e->rs, e->cfg, *u, *p, d_order, st, e->ev[EV_PROJECT], e->ev[EV_BIN], e->tm, e->prof, !capturing, !capturing, phases, order_count_dev);
    if (rc) return rc;
    if (!capturing && (phases & 2)) CU(cudaEventRecord(e->ev[EV_R1], st));
    CU(cudaGetLastError());
    return GS_OK;
}

static size_t frame_bytes(const gs_render_params *p) { return (size_t)p->width * p->height * (p->frame_format == GS_FRAME_RGBA8 ? 4 : 16); }

static int finish_render(gs_engine *e, const gs_render_params *p, void *frame_out) {
    cudaStream_t st = e->stream;
    CU(cudaEventRecord(e->ev[EV_D2H0], st));
    // world_size > 1: a full-size frame whose pixels outside this rank's coarse tiles are zero
    if (frame_out) CU(cudaMemcpyAsync(frame_out, raster_frame_ptr(e->rs, p->frame_format), frame_bytes(p), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(e->ev[EV_D2H1], st));
    CU(cudaMemcpyAsync(e->h_ctl.p + 16, e->rs.rctl.p, sizeof(RasterControl), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (e->last_frame_was_graph) {
        e->tm.project_ms = e->tm.bin_ms = e->tm.blend_ms = 0.f;
        cudaEventElapsedTime(&e->tm.render_total_ms, e->ev[EV_SORT0], e->ev[EV_R1]);   // whole frame (sort + render) in graph mode
    } else {
        cudaEventElapsedTime(&e->tm.project_ms, e->ev[EV_R0], e->ev[EV_PROJECT]);
        cudaEventElapsedTime(&e->tm.bin_ms, e->ev[EV_PROJECT], e->ev[EV_BIN]);
        cudaEventElapsedTime(&e->tm.blend_ms, e->ev[EV_BIN], e->ev[EV_R1]);
        cudaEventElapsedTime(&e->tm.render_total_ms, e->ev[EV_R0], e->ev[EV_R1]);
    }
    cudaEventElapsedTime(&e->tm.d2h_ms, e->ev[EV_D2H0], e->ev[EV_D2H1]);
    RasterControl rc;
    memcpy(&rc, e->h_ctl.p + 16, sizeof(rc));
    e->tm.tile_instances = rc.total_instances;
    uint32_t vis = 0;
    for (int i = 0; i < kVisibleSlots; ++i) vis += rc.visible_slots[i * 8];
    e->tm.visible_splats = vis;
    if (rc.peer_timeout) return fail(GS_ERR_CUDA, "multi-GPU tile gather: a peer did not arrive within the time limit (ranks must render the same frames)");
    if (rc.overflow) return fail(GS_ERR_CAPACITY, "tile-instance buffer overflow: %llu instances needed, capacity %llu (raise GS_INSTANCE_FACTOR)",
                                 (unsigned long long)rc.total_instances, (unsigned long long)e->rs.instance_capacity);
    return GS_OK;
}

static int stage_order(gs_engine *e, const gs_render_params *p, const uint32_t **d_order) {
    *d_order = nullptr;
    if (p->render_count > e->cfg.max_splat_count) return fail(GS_ERR_CAPACITY, "render_count %u > max_splat_count %u", p->render_count, e->cfg.max_splat_count);
    if (p->sorted_indexes_dev) *d_order = p->sorted_indexes_dev;
    else if (p->sorted_indexes) { // SplatMesh.updateRenderIndexes: upload of the splatIndex attribute
        CU(cudaMemcpyAsync(e->sorted.p, p->sorted_indexes, (size_t)p->render_count * 4, cudaMemcpyHostToDevice, e->stream));
        *d_order = e->sorted.p;
        e->have_sorted = true;
        e->last_render_count = p->render_count;
    } else {
        if (!e->have_sorted || e->last_render_count < p->render_count) return fail(GS_ERR_NOT_READY, "gs_render without sorted indexes: call gs_sort first or pass sorted_indexes");
        *d_order = e->sorted.p;
    }
    return GS_OK;
}

extern "C" int gs_render(gs_engine *e, const gs_uniforms *u, const gs_render_params *p, void *frame_out) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!u || !p) return fail(GS_ERR_BAD_ARG, "gs_render: null argument");
    if (e->pipe_inflight()) return fail(GS_ERR_NOT_READY, "gs_render: pipelined frames are in flight (gs_frame_end first)");
    const uint32_t *d_order = nullptr;
    e->last_frame_was_graph = false;
    if ((rc = stage_order(e, p, &d_order))) return rc;
    if ((rc = render_on_device(e, u, p, d_order))) return rc;
    return finish_render(e, p, frame_out);
}

// host-side parameter blocks of one frame -> device (outside any graph; pageable sources are staged by the driver before return)
static int upload_frame_params(gs_engine *e, const float *mvp, const gs_uniforms &u, const gs_render_params &p) {
    DepthParams P{};
    memcpy(P.mvp, mvp, 64);
    P.irow[0] = (int32_t)((double)mvp[2] * 1000.0);
    P.irow[1] = (int32_t)((double)mvp[6] * 1000.0);
    P.irow[2] = (int32_t)((double)mvp[10] * 1000.0);
    P.irow[3] = 1;
    P.frow[0] = mvp[2]; P.frow[1] = mvp[6]; P.frow[2] = mvp[10]; P.frow[3] = 0.f;
    cudaStream_t st = e->param_side ? e->param_stream : e->stream;
    CU(cudaMemcpyAsync(e->depthp.p + e->rs.frame_parity, &P, sizeof(P), cudaMemcpyHostToDevice, st));
    int rc = raster_upload_params(e->rs, e->cfg, u, p, st);
    if (rc) return rc;
    if (e->param_side) {      // the frame graph (and nothing else on the compute stream) waits for the side upload
        CU(cudaEventRecord(e->ev_params[e->rs.frame_parity], st));
        CU(cudaStreamWaitEvent(e->stream, e->ev_params[e->rs.frame_parity], 0));
    }
    return GS_OK;
}

static int enqueue_frame(gs_engine *e, const gs_sort_params *s, const gs_uniforms *u, const gs_render_params *p, gs_sort_params &q, gs_render_params &rp) {
    q = *s;
    q.render_count = std::min(q.render_count, e->uploaded_splats);
    q.sort_count = std::min(q.sort_count, e->uploaded_splats);
    const uint32_t *d_idx = nullptr;
    int rc;
    if ((rc = stage_sort_inputs(e, &q, &d_idx))) return rc;
    rp = *p;
    rp.sorted_indexes = nullptr; rp.sorted_indexes_dev = nullptr;
    rp.render_count = std::min(rp.render_count, q.render_count);
    cudaStream_t st = e->stream;
    e->last_frame_was_graph = false;
    // sharded frame: sort only this rank's subset (full sorts only; a partial sort keeps the replicated path)
    // The subset path adds two compaction kernels (~35 us at 1M splats) and only shrinks kernels that are already at their latency
    // floor there; it pays off from a few million splats (measured: 1.2M slower, 16M faster).  GS_SUBSET_MIN overrides the threshold.
    const uint32_t subset_min = getenv("GS_SUBSET_MIN") ? (uint32_t)atoll(getenv("GS_SUBSET_MIN")) : 3000000u;
    const bool subset = e->cfg.world_size > 1 && q.sort_count == q.render_count && q.render_count >= subset_min && q.render_count > 0 && !e->no_subset;
    if (subset) {
        if ((rc = e->sub_idx.ensure(e->cfg.max_splat_count)) || (rc = e->sub_dist.ensure(e->cfg.max_splat_count))) return rc;
    }
    const unsigned long long *order_count = subset ? &e->rs.rctl.p->subset_count : nullptr;
    const bool use_graph = e->graph_enabled && !e->prof.on && q.sort_count <= q.render_count && q.render_count <= e->cfg.max_splat_count && e->rs.uploaded;
    if (use_graph) {
        const unsigned long long key[8] = {q.render_count, q.sort_count, ((unsigned long long)rp.width << 32) | rp.height,
                                           ((unsigned long long)rp.frame_format << 8) | (unsigned long long)(rp.flip_y ? 1 : 0) | ((unsigned long long)q.use_precomputed_distances << 4),
                                           (unsigned long long)(uintptr_t)d_idx, ((unsigned long long)e->rs.render_mode << 32) | ((unsigned long long)e->rs.cov_format << 16) | ((unsigned long long)e->rs.sh_format << 8) | e->rs.sh_degree,
                                           e->rs.uploaded, ((unsigned long long)rp.render_count << 1) | (subset ? 1ull : 0ull)};
        if ((rc = upload_frame_params(e, q.model_view_proj, *u, rp))) return rc;
        cudaGraphExec_t &gexec = e->rs.frame_parity ? e->graph_exec_alt : e->graph_exec;      // one instantiated graph per target frame buffer
        unsigned long long *gkey = e->rs.frame_parity ? e->graph_key_alt : e->graph_key;
        if (!gexec || memcmp(key, gkey, sizeof(key)) != 0) {
            if (gexec) { cudaGraphExecDestroy(gexec); gexec = nullptr; }
            // buffers that the enqueue path may grow must be sized BEFORE capture (no allocation inside a capture)
            uint32_t stride = 0;
            const PassPlan pl = make_plan_bits(e->key_bits);
            if ((rc = e->tile_hist.ensure(radix_tile_hist_words(std::max(q.sort_count, 1u), pl.npasses, &stride)))) return rc;
            CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            struct CaptureGuard {   // an early error return must not leave the stream capturing
                cudaStream_t st; bool armed;
                ~CaptureGuard() { if (armed) { cudaGraph_t g = nullptr; cudaStreamEndCapture(st, &g); if (g) cudaGraphDestroy(g); (void)cudaGetLastError(); } }
            } guard{st, true};
            // fork: the projection does not depend on the draw order, so it runs beside the (latency-bound) depth sort
            CU(cudaEventRecord(e->ev_fork, st));
            CU(cudaStreamWaitEvent(e->stream2, e->ev_fork, 0));
            int rc2 = GS_OK;
            uint32_t proj_launches = 0;
            {
                cudaStream_t keep = e->stream;
                e->stream = e->stream2;
                rc2 = render_on_device(e, u, &rp, e->sorted.p, true, 1);
                proj_launches = e->tm.kernel_launches;
                e->stream = keep;
            }
            CU(cudaEventRecord(e->ev_join, e->stream2));
            rc = sort_on_device(e, d_idx, q.model_view_proj, q.sort_count, q.render_count, q.use_precomputed_distances != 0, false, true, subset, e->ev_join);
            const uint32_t sort_launches = e->tm.kernel_launches;
            CU(cudaStreamWaitEvent(st, e->ev_join, 0));
            if (!rc2) rc2 = rc ? rc : render_on_device(e, u, &rp, e->sorted.p, true, 2, order_count);
            e->graph_launches = e->tm.kernel_launches + sort_launches + proj_launches;
            cudaGraph_t g = nullptr;
            guard.armed = false;
            cudaError_t ce = cudaStreamEndCapture(st, &g);
            if (rc2) { if (g) cudaGraphDestroy(g); return rc2; }
            if (ce != cudaSuccess) return fail(GS_ERR_CUDA, "cudaStreamEndCapture -> %s", cudaGetErrorString(ce));
            ce = cudaGraphInstantiate(&gexec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { gexec = nullptr; return fail(GS_ERR_CUDA, "cudaGraphInstantiate -> %s", cudaGetErrorString(ce)); }
            memcpy(gkey, key, sizeof(key));
            e->graph_snapshot[e->rs.frame_parity ? 1 : 0] = e->rs.snapshot_taken;
        }
        if (e->ctl_dirty) gs_launch(k_sort_init, 1, 256, 0, st, e->ctl.p);   // the captured sort assumes (and leaves) a clean control block
        e->ctl_dirty = true;
        CU(cudaEventRecord(e->ev[EV_SORT0], st));
        CU(cudaGraphLaunch(gexec, st));
        e->ctl_dirty = false;
        CU(cudaEventRecord(e->ev[EV_R1], st));
        e->tm.kernel_launches = e->graph_launches;
        e->last_render_count = q.render_count;
        e->have_sorted = !subset;   // a subset order is not a draw order for gs_render
        e->last_frame_was_graph = true;
        return GS_OK;
    }
    if (subset) {   // one stream: projection first (its rects select the subset), then depth + subset sort, then binning + blend
        e->prof.begin(st);
        e->have_prof_begin = true;
        if ((rc = render_on_device(e, u, &rp, e->sorted.p, false, 1))) { e->have_prof_begin = false; return rc; }
        const uint32_t proj_launches = e->tm.kernel_launches;
        if ((rc = sort_on_device(e, d_idx, q.model_view_proj, q.sort_count, q.render_count, q.use_precomputed_distances != 0, false, false, true, nullptr))) { e->have_prof_begin = false; return rc; }
        const uint32_t sort_launches = e->tm.kernel_launches;
        rc = render_on_device(e, u, &rp, e->sorted.p, false, 2, order_count);
        e->have_prof_begin = false;
        if (rc) return rc;
        e->tm.kernel_launches += sort_launches + proj_launches;
        e->have_sorted = false;
        return GS_OK;
    }
    if ((rc = sort_on_device(e, d_idx, q.model_view_proj, q.sort_count, q.render_count, q.use_precomputed_distances != 0, false))) return rc;
    const uint32_t sort_launches = e->tm.kernel_launches;
    e->have_prof_begin = true;
    rc = render_on_device(e, u, &rp, e->sorted.p);
    e->have_prof_begin = false;
    if (rc) return rc;
    e->tm.kernel_launches += sort_launches;
    return GS_OK;
}

extern "C" int gs_frame(gs_engine *e, const gs_sort_params *s, const gs_uniforms *u, const gs_render_params *p, uint32_t *sorted_out, void *frame_out) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!s || !u || !p) return fail(GS_ERR_BAD_ARG, "gs_frame: null argument");
    if (e->pipe_inflight()) return fail(GS_ERR_NOT_READY, "gs_frame: pipelined frames are in flight (gs_frame_end first)");
    e->rs.frame_parity = 0;
    gs_sort_params q; gs_render_params rp;
    e->no_subset = (sorted_out != nullptr);
    rc = enqueue_frame(e, s, u, p, q, rp);
    e->no_subset = false;
    if (rc) return rc;
    if (sorted_out && q.render_count) CU(cudaMemcpyAsync(sorted_out, e->sorted.p, (size_t)q.render_count * 4, cudaMemcpyDeviceToHost, e->stream));
    int rc2 = finish_render(e, &rp, frame_out);
    rc = finish_sort(e, nullptr);
    cudaEventElapsedTime(&e->tm.h2d_ms, e->ev[EV_H2D0], e->ev[EV_H2D1]);
    return rc ? rc : rc2;
}

// Enqueue one frame and return without waiting: the frame stays on the device (gs_buffer_dev(GS_BUF_FRAME)), errors and
// timings are collected by the next gs_synchronize().  Lets a caller keep several frames in flight on the stream.
extern "C" int gs_frame_async(gs_engine *e, const gs_sort_params *s, const gs_uniforms *u, const gs_render_params *p) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!s || !u || !p) return fail(GS_ERR_BAD_ARG, "gs_frame_async: null argument");
    if (e->pipe_inflight()) return fail(GS_ERR_NOT_READY, "gs_frame_async: pipelined frames are in flight (gs_frame_end first): their pictures are still being copied out of the frame buffers");
    gs_sort_params q; gs_render_params rp;
    if ((rc = enqueue_frame(e, s, u, p, q, rp))) return rc;
    e->pending_async = true;
    e->pending_rp = rp;
    return GS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Pipelined frames: gs_frame_begin enqueues frame i (camera H2D, sort, render) and a D2H copy of its picture on a separate copy
// stream; gs_frame_end waits for the OLDEST frame in flight and reports its errors.  Up to three frames may be in flight over TWO
// device frame buffers: frame i+1 renders while frame i's picture crosses PCIe, and frame i+2 is already queued behind it (it
// starts only when frame i's copy has left its buffer), so the GPU never waits for the host between frames
// (begin(0); begin(1); loop { begin(i+2); end(i); }).  Every frame in flight needs its own `frame_out`.  Per-frame latency is that of
// gs_frame; throughput approaches max(compute, copy).  With two buffers a frame graph is the ONLY thing a frame puts on the compute
// stream: the parameter blocks go up on `param_stream` into the block of the frame buffer's parity, and the status words are
// snapshotted by the blend kernel and read back on the copy stream.  Multi-GPU engines that gather tiles into rank 0's exported
// frame keep ONE buffer (the peers store into it), so there the copy only overlaps the host side.
static int pipe_init(gs_engine *e) {
    if (e->copy_stream) return GS_OK;
    CU(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&e->param_stream, cudaStreamNonBlocking));
    for (int i = 0; i < gs_engine::kPipeRing; ++i) {
        CU(cudaEventCreateWithFlags(&e->ev_frame_done[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&e->ev_copy_done[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; ++i) CU(cudaEventCreateWithFlags(&e->ev_params[i], cudaEventDisableTiming));
    int rc = e->h_pipe.ensure(gs_engine::kPipeRing * kPipeSlotWords);
    if (rc) return rc;
    const bool single = e->cfg.world_size > 1;      // (rank 0 of a peer group may hold a double allocation instead: rs.frame_half2)
    if (!single && !e->rs.frame_alt.p) {
        cudaError_t ce = e->rs.frame_alt.ensure(e->rs.frame.n);
        if (ce != cudaSuccess) return fail(GS_ERR_CUDA, "cudaMalloc(second frame buffer) -> %s", cudaGetErrorString(ce));
    }
    return GS_OK;
}

extern "C" int gs_frame_begin(gs_engine *e, const gs_sort_params *s, const gs_uniforms *u, const gs_render_params *p, void *frame_out) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!s || !u || !p) return fail(GS_ERR_BAD_ARG, "gs_frame_begin: null argument");
    if (e->pipe_inflight() >= (uint32_t)gs_engine::kPipeMaxInflight) return fail(GS_ERR_NOT_READY, "gs_frame_begin: %d frames already in flight (call gs_frame_end)", gs_engine::kPipeMaxInflight);
    if (e->pending_async) return fail(GS_ERR_NOT_READY, "gs_frame_begin: an asynchronous frame is pending (gs_synchronize first)");
    if ((rc = pipe_init(e))) return rc;
    constexpr uint64_t R = gs_engine::kPipeRing;
    const uint64_t seq = e->pipe_begun;
    const uint32_t ring = (uint32_t)(seq % R);
    const bool two = raster_second_frame(e->rs) != nullptr;
    // the buffer this frame renders into must have been copied out: frame seq-2 with two buffers, seq-1 with one
    if (two) { if (seq >= 2) CU(cudaStreamWaitEvent(e->stream, e->ev_copy_done[(seq - 2) % R], 0)); }
    else if (seq >= 1) CU(cudaStreamWaitEvent(e->stream, e->ev_copy_done[(seq - 1) % R], 0));
    e->rs.frame_parity = two ? (int)(seq & 1) : 0;
    // parameter blocks of this parity were last read by frame seq-2: its graph must have finished before they are overwritten
    e->param_side = two;
    if (two && seq >= 2) CU(cudaStreamWaitEvent(e->param_stream, e->ev_frame_done[(seq - 2) % R], 0));
    gs_sort_params q; gs_render_params rp;
    rc = enqueue_frame(e, s, u, p, q, rp);
    e->param_side = false;
    if (rc) { e->rs.frame_parity = 0; return rc; }
    cudaStream_t st = e->stream;
    uint32_t *hs = e->h_pipe.p + ring * kPipeSlotWords;
    // (multi-GPU: rank 0's peer_timeout flag is raised AFTER the blend, by k_peer_wait_arrived -- the snapshot would miss it)
    const bool snapshot = two && e->cfg.world_size == 1 && e->last_frame_was_graph && e->graph_snapshot[e->rs.frame_parity];
    if (!snapshot) {      // status read-back in stream order (frames outside a graph, blend generations without the snapshot, one buffer)
        CU(cudaMemcpyAsync(hs, e->ctl.p, 12, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(hs + 4, e->rs.rctl.p, sizeof(RasterControl), cudaMemcpyDeviceToHost, st));
    }
    CU(cudaEventRecord(e->ev_frame_done[ring], st));
    CU(cudaStreamWaitEvent(e->copy_stream, e->ev_frame_done[ring], 0));
    if (snapshot)
        CU(cudaMemcpyAsync(hs, e->status_dev.p + (size_t)e->rs.frame_parity * kPipeSlotWords, (4 + sizeof(RasterControl) / 4) * 4, cudaMemcpyDeviceToHost, e->copy_stream));
    if (frame_out) CU(cudaMemcpyAsync(frame_out, raster_frame_ptr(e->rs, rp.frame_format), frame_bytes(&rp), cudaMemcpyDeviceToHost, e->copy_stream));
    CU(cudaEventRecord(e->ev_copy_done[ring], e->copy_stream));
    ++e->pipe_begun;
    return GS_OK;
}

extern "C" int gs_frame_end(gs_engine *e) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (e->pipe_inflight() == 0) return fail(GS_ERR_NOT_READY, "gs_frame_end: no frame in flight");
    const uint32_t ring = (uint32_t)(e->pipe_ended % (uint64_t)gs_engine::kPipeRing);
    CU(cudaEventSynchronize(e->ev_copy_done[ring]));
    ++e->pipe_ended;
    const uint32_t *hs = e->h_pipe.p + ring * kPipeSlotWords;
    RasterControl rctl;
    memcpy(&rctl, hs + 4, sizeof(rctl));
    e->tm.tile_instances = rctl.total_instances;
    uint32_t vis = 0;
    for (int i = 0; i < kVisibleSlots; ++i) vis += rctl.visible_slots[i * 8];
    e->tm.visible_splats = vis;
    if (hs[2] & kErrBucketRange) return fail(GS_ERR_BUCKET_RANGE, "a bucket index fell outside [0,%u): distances overflow the int32/f32 range map", e->cfg.distance_map_range);
    if (rctl.peer_timeout) return fail(GS_ERR_CUDA, "multi-GPU tile gather: a peer did not arrive within the time limit (ranks must render the same frames)");
    if (rctl.overflow) return fail(GS_ERR_CAPACITY, "tile-instance buffer overflow: %llu instances needed, capacity %llu (raise GS_INSTANCE_FACTOR)",
                                   (unsigned long long)rctl.total_instances, (unsigned long long)e->rs.instance_capacity);
    return GS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// SplatTree leaves -> device, and the per-frame cull + index gather (SURVEY 8(f) N2; cull_kernels.cuh).
extern "C" int gs_upload_splat_tree(gs_engine *e, const double *node_center, const double *node_min, const double *node_max, const uint32_t *node_offsets,
                                    const uint32_t *indexes, uint32_t node_count) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (node_count && (!node_center || !node_min || !node_max || !node_offsets || !indexes)) return fail(GS_ERR_BAD_ARG, "gs_upload_splat_tree: null argument");
    const uint32_t total = node_count ? node_offsets[node_count] : 0;
    if (total > e->cfg.max_splat_count) return fail(GS_ERR_CAPACITY, "the tree's leaves hold %u indexes, engine capacity %u", total, e->cfg.max_splat_count);
    for (uint32_t i = 0; i < node_count; ++i)
        if (node_offsets[i + 1] < node_offsets[i]) return fail(GS_ERR_BAD_ARG, "gs_upload_splat_tree: node_offsets must be non-decreasing");
    auto &t = e->tree;
    const size_t m = std::max<uint32_t>(node_count, 1);
    if ((rc = t.center.ensure(3 * m)) || (rc = t.nmin.ensure(3 * m)) || (rc = t.nmax.ensure(3 * m)) || (rc = t.offsets.ensure(m + 1)) || (rc = t.indexes.ensure(std::max<uint32_t>(total, 1))) ||
        (rc = t.start.ensure(m)) || (rc = t.key.ensure(m)) || (rc = t.total.ensure(1)))
        return rc;
    cudaStream_t st = e->stream;
    if (node_count) {
        CU(cudaMemcpyAsync(t.center.p, node_center, 24 * (size_t)node_count, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(t.nmin.p, node_min, 24 * (size_t)node_count, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(t.nmax.p, node_max, 24 * (size_t)node_count, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(t.offsets.p, node_offsets, 4 * ((size_t)node_count + 1), cudaMemcpyHostToDevice, st));
        if (total) CU(cudaMemcpyAsync(t.indexes.p, indexes, 4 * (size_t)total, cudaMemcpyHostToDevice, st));
    }
    CU(cudaStreamSynchronize(st));
    t.count = node_count; t.splats = total;
    return GS_OK;
}

extern "C" int gs_gather_for_sort(gs_engine *e, const double *model_view, double cos_fov_x_over_2, double cos_fov_y_over_2, int gather_all_nodes,
                                  uint32_t *render_count_out) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!model_view || !render_count_out) return fail(GS_ERR_BAD_ARG, "gs_gather_for_sort: null argument");
    auto &t = e->tree;
    if (!t.count) { *render_count_out = 0; return GS_OK; }
    CullParams P;
    memcpy(P.mv, model_view, sizeof(P.mv));
    P.cos_fov_x_over_2 = cos_fov_x_over_2; P.cos_fov_y_over_2 = cos_fov_y_over_2; P.gather_all = gather_all_nodes;
    cudaStream_t st = e->stream;
    k_tree_cull<<<(t.count + 127) / 128, 128, 0, st>>>(t.center.p, t.nmin.p, t.nmax.p, t.count, P, t.key.p);
    k_tree_layout<<<(t.count + kLayoutThreads - 1) / kLayoutThreads, kLayoutThreads, 0, st>>>(t.key.p, t.offsets.p, t.count, t.start.p, t.total.p);
    k_tree_copy<<<t.count, 128, 0, st>>>(t.start.p, t.offsets.p, t.indexes.p, e->indexes.p);
    CU(cudaMemcpyAsync(e->h_ctl.p + 8, t.total.p, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    unsigned long long total;
    memcpy(&total, e->h_ctl.p + 8, 8);
    *render_count_out = (uint32_t)total;
    e->tm.kernel_launches = 3;
    return GS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// .ksplat -> engine, decoded on the GPU (SURVEY 8f N1).  Header/section parsing is host logic (SplatBuffer.js:819-941).
static uint32_t rd32(const unsigned char *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static uint16_t rd16(const unsigned char *p) { uint16_t v; memcpy(&v, p, 2); return v; }
static float rdf(const unsigned char *p) { float v; memcpy(&v, p, 4); return v; }

extern "C" int gs_upload_ksplat(gs_engine *e, const void *data, size_t bytes, const gs_ksplat_options *opt, gs_ksplat_info *info) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!data || bytes < 4096) return fail(GS_ERR_BAD_ARG, "gs_upload_ksplat: buffer shorter than the 4096-byte header");
    if (!e->cfg.max_width || !e->cfg.max_height) return fail(GS_ERR_NOT_READY, "engine created without a framebuffer (max_width/max_height = 0)");
    gs_ksplat_options o{};
    o.minimum_alpha = 1; o.upload_sort_centers = 1;
    if (opt) memcpy(&o, opt, std::min<size_t>(opt->struct_size ? opt->struct_size : sizeof(o), sizeof(o)));
    const unsigned char *f = (const unsigned char *)data;
    const uint32_t max_sections = rd32(f + 4), max_splats = rd32(f + 12), level = rd16(f + 20);
    if (f[0] == 0 && f[1] < 1) return fail(GS_ERR_BAD_ARG, "unsupported .ksplat version %u.%u", f[0], f[1]);
    if (level > 2) return fail(GS_ERR_BAD_ARG, ".ksplat compression level %u unknown", level);
    if (max_splats > e->cfg.max_splat_count) return fail(GS_ERR_CAPACITY, ".ksplat holds %u splats, engine capacity %u", max_splats, e->cfg.max_splat_count);
    if (4096ull + 1024ull * max_sections > bytes) return fail(GS_ERR_BAD_ARG, ".ksplat truncated (section headers)");
    static const uint32_t kC[3] = {12, 6, 6}, kS[3] = {12, 6, 6}, kR[3] = {16, 8, 8}, kSH[3] = {4, 2, 1}, kRange[3] = {1, 32767, 32767};
    std::vector<KSectionParams> secs;
    std::vector<std::vector<uint32_t>> prefixes;
    unsigned long long base = 4096ull + 1024ull * max_sections;
    uint32_t offset = 0, min_degree = 2;
    for (uint32_t i = 0; i < max_sections; ++i) {
        const unsigned char *h = f + 4096 + 1024ull * i;
        KSectionParams P{};
        P.count = rd32(h + 4);
        P.bucket_size = rd32(h + 8);
        const uint32_t bucket_count = rd32(h + 12);
        const float block = rdf(h + 16);
        const uint32_t storage = rd16(h + 20);
        P.scale_range = rd32(h + 24) ? rd32(h + 24) : kRange[level];
        P.full_bucket_count = rd32(h + 32);
        P.partial_count = rd32(h + 36);
        P.sh_degree_file = rd16(h + 40);
        if (P.sh_degree_file > 2) return fail(GS_ERR_BAD_ARG, ".ksplat section %u: SH degree %d", i, P.sh_degree_file);
        const uint32_t ncomp = P.sh_degree_file == 2 ? 24 : (P.sh_degree_file == 1 ? 9 : 0);
        P.bytes_per_splat = kC[level] + kS[level] + kR[level] + 4 + kSH[level] * ncomp;
        const unsigned long long meta = 4ull * P.partial_count, buckets_bytes = (unsigned long long)storage * bucket_count + meta;
        P.base = base; P.buckets_base = base + meta; P.data_base = base + buckets_bytes;
        P.splat_offset = offset; P.level = (int)level;
        P.scale_factor = ((double)block / 2.0) / (double)P.scale_range;
        if (P.data_base + (unsigned long long)P.bytes_per_splat * P.count > bytes) return fail(GS_ERR_BAD_ARG, ".ksplat truncated (section %u data)", i);
        // an untrusted file must not make the decode kernel read bucket centres or write splats outside its buffers
        if (level >= 1 && P.count) {
            if (P.bucket_size == 0 || storage != 12) return fail(GS_ERR_BAD_ARG, ".ksplat section %u: bucket size %u / bucket storage %u bytes (expected > 0 / 12)", i, P.bucket_size, storage);
            if ((unsigned long long)P.full_bucket_count + P.partial_count > bucket_count) return fail(GS_ERR_BAD_ARG, ".ksplat section %u: %u full + %u partial buckets exceed its %u bucket centres", i, P.full_bucket_count, P.partial_count, bucket_count);
        }
        if (P.data_base > bytes || P.buckets_base > P.data_base) return fail(GS_ERR_BAD_ARG, ".ksplat truncated (section %u buckets)", i);
        std::vector<uint32_t> pre(P.partial_count + 1, 0);
        for (uint32_t k = 0; k < P.partial_count; ++k) {
            const unsigned long long len = rd32(f + P.base + 4ull * k);
            if (len > P.count) return fail(GS_ERR_BAD_ARG, ".ksplat section %u: partial bucket %u claims %llu splats", i, k, len);
            pre[k + 1] = pre[k] + (uint32_t)len;
        }
        if (level >= 1 && (unsigned long long)P.full_bucket_count * P.bucket_size + pre[P.partial_count] < P.count) return fail(GS_ERR_BAD_ARG, ".ksplat section %u: buckets do not cover its splats", i);
        if ((unsigned long long)offset + P.count > max_splats || (unsigned long long)offset + P.count > e->cfg.max_splat_count)
            return fail(GS_ERR_CAPACITY, ".ksplat sections hold more than the %u splats its header declares (engine capacity %u)", max_splats, e->cfg.max_splat_count);
        prefixes.push_back(pre);
        min_degree = std::min<uint32_t>(min_degree, (uint32_t)P.sh_degree_file);
        base += (unsigned long long)P.bytes_per_splat * P.count + buckets_bytes;
        offset += P.count;
        secs.push_back(P);
    }
    if (secs.empty()) min_degree = 0;
    const uint32_t total = offset;
    // storage formats of the "textures" (SplatMesh.js:1064-1066: SH kept at compression level max(1, file level))
    RasterState &rs = e->rs;
    rs.uploaded = 0;
    const bool two_d = rs.render_mode == GS_RENDER_MODE_2D;   // scale/rotation texture instead of covariances (half_covariances unused)
    rs.cov_format = (o.half_covariances && !two_d) ? GS_COV_F16 : GS_COV_F32;
    rs.sh_degree = min_degree;
    rs.sh_format = min_degree ? (level == 2 ? GS_SH_U8 : GS_SH_F16) : GS_SH_NONE;
    const size_t n = e->cfg.max_splat_count, ncomp_out = min_degree == 2 ? 24 : (min_degree == 1 ? 9 : 0);
    cudaError_t ce;
    if (!two_d && (ce = rs.cov.ensure(n * (o.half_covariances ? 12 : 24) + 16)) != cudaSuccess) return fail(GS_ERR_CUDA, "cudaMalloc -> %s", cudaGetErrorString(ce));
    if (ncomp_out && (ce = rs.sh.ensure(n * ncomp_out * (level == 2 ? 1 : 2) + 16)) != cudaSuccess) return fail(GS_ERR_CUDA, "cudaMalloc -> %s", cudaGetErrorString(ce));
    DevBuf<unsigned char> d_file; DevBuf<uint32_t> d_pre; DevBuf<KTransform> d_xf;
    struct Scratch {   // the staged file and the bucket prefixes live for this call only, whichever way it returns
        DevBuf<unsigned char> &a; DevBuf<uint32_t> &b; DevBuf<KTransform> &c;
        ~Scratch() { a.release(); b.release(); c.release(); }
    } scratch{d_file, d_pre, d_xf};
    if ((rc = d_file.ensure(bytes))) return rc;
    cudaStream_t st = e->stream;
    CU(cudaMemcpyAsync(d_file.p, data, bytes, cudaMemcpyHostToDevice, st));
    if (o.has_transform) {
        KTransform K;
        const float lo = rdf(f + 36), hi = rdf(f + 40);
        ksplat_transform_params(o.transform, lo != 0.f ? (double)lo : -1.5, hi != 0.f ? (double)hi : 1.5, K);
        if ((rc = d_xf.ensure(1))) return rc;
        CU(cudaMemcpyAsync(d_xf.p, &K, sizeof(K), cudaMemcpyHostToDevice, st));   // pageable source: staged before return
    }
    size_t pre_words = 0;
    for (auto &p : prefixes) pre_words += p.size();
    if ((rc = d_pre.ensure(pre_words))) return rc;
    size_t at = 0;
    for (size_t i = 0; i < secs.size(); ++i) {
        CU(cudaMemcpyAsync(d_pre.p + at, prefixes[i].data(), prefixes[i].size() * 4, cudaMemcpyHostToDevice, st));
        KSectionParams P = secs[i];
        P.sh_degree_out = (int)min_degree;
        P.minimum_alpha = o.minimum_alpha; P.half_cov = o.half_covariances; P.integer_centers = e->cfg.integer_based_sort; P.write_sort_centers = o.upload_sort_centers;
        if (P.count) {
            const dim3 grid((P.count + 127) / 128);
            if (two_d) {
                if (o.has_transform) k_ksplat_decode<true, true><<<grid, 128, 0, st>>>(d_file.p, P, d_pre.p + at, rs.cc.p, nullptr, rs.sh.p, e->centers.p, d_xf.p, rs.srot.p);
                else k_ksplat_decode<false, true><<<grid, 128, 0, st>>>(d_file.p, P, d_pre.p + at, rs.cc.p, nullptr, rs.sh.p, e->centers.p, nullptr, rs.srot.p);
            } else {
                if (o.has_transform) k_ksplat_decode<true, false><<<grid, 128, 0, st>>>(d_file.p, P, d_pre.p + at, rs.cc.p, rs.cov.p, rs.sh.p, e->centers.p, d_xf.p, nullptr);
                else k_ksplat_decode<false, false><<<grid, 128, 0, st>>>(d_file.p, P, d_pre.p + at, rs.cc.p, rs.cov.p, rs.sh.p, e->centers.p, nullptr, nullptr);
            }
        }
        at += prefixes[i].size();
    }
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    rs.uploaded = total;
    rs.have_scene_idx = false;
    if (o.upload_sort_centers) e->uploaded_splats = total;
    if (info) {
        memset(info, 0, sizeof(*info));
        info->struct_size = sizeof(*info);
        info->splat_count = total; info->sh_degree = min_degree; info->compression_level = level; info->section_count = (uint32_t)secs.size();
        info->scene_center[0] = rdf(f + 24); info->scene_center[1] = rdf(f + 28); info->scene_center[2] = rdf(f + 32);
        const float lo = rdf(f + 36), hi = rdf(f + 40);
        info->min_sh_coeff = lo != 0.f ? lo : -1.5f; info->max_sh_coeff = hi != 0.f ? hi : 1.5f;   // SplatBuffer.js:833-834
    }
    return GS_OK;
}

// Debug / test read-back of an engine buffer (see gs_buffer_id) into host memory.
extern "C" int gs_read_buffer(gs_engine *e, int id, void *out, size_t offset, size_t bytes) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!out) return fail(GS_ERR_BAD_ARG, "gs_read_buffer: null");
    const unsigned char *p = nullptr; size_t cap = 0;
    if (id == GS_BUF_TILE_INFO) {     // host-side values
        const uint64_t info[4] = {e->rs.instance_capacity, e->rs.last_ncoarse, e->rs.last_tile_px, e->rs.last_bin_path};
        if (offset + bytes > sizeof(info)) return fail(GS_ERR_CAPACITY, "gs_read_buffer: [%zu,%zu) outside the %zu-byte buffer", offset, offset + bytes, sizeof(info));
        memcpy(out, (const unsigned char *)info + offset, bytes);
        return GS_OK;
    }
    switch (id) {
        case GS_BUF_TILE_RECTS: p = (const unsigned char *)e->rs.rects.p; cap = e->rs.rects.n * sizeof(ushort4); break;
        case GS_BUF_TILE_RANGES: p = (const unsigned char *)e->rs.ranges.p; cap = e->rs.ranges.n * sizeof(uint2); break;
        case GS_BUF_TILE_LIST: p = (const unsigned char *)e->rs.list.p; cap = std::min<size_t>(e->rs.list.n, e->rs.instance_capacity) * 8; break;
        case GS_BUF_TILE_ORDER: p = (const unsigned char *)e->rs.tile_order.p; cap = e->rs.tile_order.n * 4; break;
        case GS_BUF_CENTERS_COLORS: p = (const unsigned char *)e->rs.cc.p; cap = e->rs.cc.n * 16; break;
        case GS_BUF_COVARIANCES: p = e->rs.cov.p; cap = e->rs.cov.n; break;
        case GS_BUF_SH: p = e->rs.sh.p; cap = e->rs.sh.n; break;
        case GS_BUF_SCALE_ROTATIONS: p = (const unsigned char *)e->rs.srot.p; cap = e->rs.srot.n * 4; break;
        default: { void *q = nullptr; if ((rc = gs_buffer_dev(e, id, &q, &cap))) return rc; p = (const unsigned char *)q; }
    }
    if (!p || offset + bytes > cap) return fail(GS_ERR_CAPACITY, "gs_read_buffer: [%zu,%zu) outside the %zu-byte buffer", offset, offset + bytes, cap);
    CU(cudaMemcpyAsync(out, p + offset, bytes, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return GS_OK;
}

extern "C" int gs_read_projected(gs_engine *e, gs_projected_splat *out, uint32_t count) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!out) return fail(GS_ERR_BAD_ARG, "gs_read_projected: null");
    rc = raster_read_projected(e->rs, out, count, e->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(e->stream));
    return GS_OK;
}

extern "C" int gs_read_projected_2d(gs_engine *e, gs_projected_surfel *out, uint32_t count) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!out) return fail(GS_ERR_BAD_ARG, "gs_read_projected_2d: null");
    if (e->pipe_inflight()) return fail(GS_ERR_NOT_READY, "gs_read_projected_2d: pipelined frames are in flight (gs_frame_end first)");
    rc = raster_read_projected_2d(e->rs, out, count, e->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(e->stream));
    return GS_OK;
}

extern "C" int gs_buffer_dev(gs_engine *e, int id, void **ptr, size_t *bytes) {
    if (!e || !ptr) return fail(GS_ERR_BAD_ARG, "gs_buffer_dev: null");
    size_t b = 0;
    switch (id) {
        case GS_BUF_SORTED_INDEXES: *ptr = e->sorted.p; b = e->sorted.n * 4; break;
        case GS_BUF_FRAME: *ptr = raster_frame_ptr(e->rs, e->rs.last_format); b = e->rs.last_frame_bytes; break;
        case GS_BUF_CENTERS: *ptr = e->centers.p; b = e->centers.n * 16; break;
        case GS_BUF_DISTANCES: *ptr = e->dist.p; b = e->dist.n * 4; break;
        case GS_BUF_SPLAT_RECORDS:
            if (e->rs.render_mode == GS_RENDER_MODE_2D) { *ptr = e->rs.surfels.p; b = e->rs.surfels.n * sizeof(SurfelRecord); }
            else { *ptr = e->rs.records.p; b = e->rs.records.n * sizeof(SplatRecord); }
            break;
        case GS_BUF_INDEXES_TO_SORT: *ptr = e->indexes.p; b = e->indexes.n * 4; break;
        default: return fail(GS_ERR_BAD_ARG, "unknown buffer id %d", id);
    }
    if (bytes) *bytes = b;
    return GS_OK;
}
extern "C" int gs_stream(gs_engine *e, void **s) {
    if (!e || !s) return fail(GS_ERR_BAD_ARG, "gs_stream: null");
    *s = (void *)e->stream;
    return GS_OK;
}
extern "C" int gs_synchronize(gs_engine *e) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (e->pending_async) { // collect errors + timings of the last asynchronous frame
        e->pending_async = false;
        int rc2 = finish_render(e, &e->pending_rp, nullptr);
        rc = finish_sort(e, nullptr);
        return rc ? rc : rc2;
    }
    CU(cudaStreamSynchronize(e->stream));
    return GS_OK;
}

// ---- measurement helpers (bench hygiene; no effect on results) -------------------------------------------------------
__global__ void k_flush_l2(uint32_t *buf, size_t words, uint32_t v) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (size_t)gridDim.x * blockDim.x) buf[i] = v;
}
extern "C" int gs_flush_l2(gs_engine *e) { // overwrite a buffer larger than L2 on the engine's stream
    int rc = check_engine(e);
    if (rc) return rc;
    const size_t words = (size_t)192 * 1024 * 1024 / 4;
    if ((rc = e->flush.ensure(words))) return rc;
    static uint32_t tick = 0;
    k_flush_l2<<<e->sm_count * 8, 512, 0, e->stream>>>(e->flush.p, words, ++tick);
    CU(cudaGetLastError());
    return GS_OK;
}
// ---- fused tile gather: rank 0's frame buffer + handshake block shared with the other ranks through CUDA IPC -------------------------
extern "C" int gs_peer_export(gs_engine *e, void *frame_handle, void *sync_handle) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!frame_handle || !sync_handle) return fail(GS_ERR_BAD_ARG, "gs_peer_export: null");
    if (e->cfg.world_size < 2 || e->cfg.rank != 0) return fail(GS_ERR_BAD_ARG, "gs_peer_export: only rank 0 of a multi-GPU group exports");
    if (!e->rs.frame.p) return fail(GS_ERR_NOT_READY, "engine created without a framebuffer");
    cudaError_t ce = e->rs.peer_sync_local.ensure(1);
    if (ce != cudaSuccess) return fail(GS_ERR_CUDA, "cudaMalloc -> %s", cudaGetErrorString(ce));
    CU(cudaMemset(e->rs.peer_sync_local.p, 0, sizeof(PeerSync)));
    // Double the exported allocation: pipelined frames (gs_frame_begin) then alternate between its halves, so the picture of frame f
    // leaves over PCIe while the peers already store frame f+1 into the other half.  Which half a frame uses travels in the release
    // word.  Every rank sizes its own frame buffer from the same gs_config, so the peers know where the second half starts.
    // GS_PEER_DOUBLE=0 keeps one buffer.
    const char *pd = getenv("GS_PEER_DOUBLE");
    if (!(pd && pd[0] == '0') && e->rs.blend_version >= 2 && !e->rs.frame_half2 && !e->pipe_inflight()) {
        CU(cudaStreamSynchronize(e->stream));
        const size_t half = e->rs.frame.n;
        e->rs.frame.release();
        ce = e->rs.frame.ensure(2 * half);
        if (ce != cudaSuccess) return fail(GS_ERR_CUDA, "cudaMalloc(double frame buffer) -> %s", cudaGetErrorString(ce));
        CU(cudaMemset(e->rs.frame.p, 0, 2 * half));
        e->rs.frame_half2 = e->rs.frame.p + half;
        e->rs.frame_half_bytes = half;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == GS_IPC_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, e->rs.frame.p));
    memcpy(frame_handle, &h, sizeof(h));
    CU(cudaIpcGetMemHandle(&h, e->rs.peer_sync_local.p));
    memcpy(sync_handle, &h, sizeof(h));
    CU(cudaMemset(&e->rs.rctl.p->frame_seq, 0, 4));   // ranks count frames in lockstep from here on
    e->rs.peer_sync = e->rs.peer_sync_local.p;
    e->rs.peer_root = true;
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    if (e->graph_exec_alt) { cudaGraphExecDestroy(e->graph_exec_alt); e->graph_exec_alt = nullptr; }
    return GS_OK;
}
extern "C" int gs_peer_attach(gs_engine *e, const void *frame_handle, const void *sync_handle) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!frame_handle || !sync_handle) return fail(GS_ERR_BAD_ARG, "gs_peer_attach: null");
    if (e->cfg.world_size < 2 || e->cfg.rank == 0) return fail(GS_ERR_BAD_ARG, "gs_peer_attach: only ranks > 0 of a multi-GPU group attach");
    cudaIpcMemHandle_t h;
    void *pf = nullptr, *ps = nullptr;
    memcpy(&h, frame_handle, sizeof(h));
    CU(cudaIpcOpenMemHandle(&pf, h, cudaIpcMemLazyEnablePeerAccess));
    memcpy(&h, sync_handle, sizeof(h));
    CU(cudaIpcOpenMemHandle(&ps, h, cudaIpcMemLazyEnablePeerAccess));
    CU(cudaMemset(&e->rs.rctl.p->frame_seq, 0, 4));
    e->rs.peer_frame = pf;
    e->rs.peer_sync = (PeerSync *)ps;
    e->rs.peer_attached = true;
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    return GS_OK;
}

extern "C" int gs_set_graph_enabled(gs_engine *e, int on) {
    if (!e) return fail(GS_ERR_BAD_ARG, "gs_set_graph_enabled: null");
    e->graph_enabled = on != 0;
    return GS_OK;
}
extern "C" int gs_set_profiling(gs_engine *e, int on) {
    if (!e) return fail(GS_ERR_BAD_ARG, "gs_set_profiling: null");
    e->prof.on = on != 0;
    return GS_OK;
}
// Per-kernel device times of the last sort / render / frame (call after gs_synchronize or a blocking entry).
extern "C" int gs_kernel_timings(gs_engine *e, gs_kernel_time *out, uint32_t capacity, uint32_t *count) {
    int rc = check_engine(e);
    if (rc) return rc;
    if (!count) return fail(GS_ERR_BAD_ARG, "gs_kernel_timings: null");
    CU(cudaStreamSynchronize(e->stream));
    uint32_t n = 0;
    for (size_t i = 1; i < e->prof.used; ++i) {
        if (n < capacity && out) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e->prof.ev[i - 1], e->prof.ev[i]);
            strncpy(out[n].name, e->prof.names[i], sizeof(out[n].name) - 1);
            out[n].name[sizeof(out[n].name) - 1] = 0;
            out[n].ms = ms;
        }
        ++n;
    }
    *count = n;
    return GS_OK;
}
extern "C" int gs_event_create(void **ev) {
    if (!ev) return fail(GS_ERR_BAD_ARG, "gs_event_create: null");
    cudaEvent_t x;
    CU(cudaEventCreate(&x));
    *ev = (void *)x;
    return GS_OK;
}
extern "C" int gs_event_record(gs_engine *e, void *ev) {
    int rc = check_engine(e);
    if (rc) return rc;
    CU(cudaEventRecord((cudaEvent_t)ev, e->stream));
    return GS_OK;
}
extern "C" int gs_event_elapsed_ms(void *ev0, void *ev1, float *ms) {
    if (!ms) return fail(GS_ERR_BAD_ARG, "gs_event_elapsed_ms: null");
    CU(cudaEventSynchronize((cudaEvent_t)ev1));
    CU(cudaEventElapsedTime(ms, (cudaEvent_t)ev0, (cudaEvent_t)ev1));
    return GS_OK;
}
extern "C" int gs_event_destroy(void *ev) {
    if (ev) CU(cudaEventDestroy((cudaEvent_t)ev));
    return GS_OK;
}
extern "C" int gs_last_timings(gs_engine *e, gs_timings *t) {
    if (!e || !t) return fail(GS_ERR_BAD_ARG, "gs_last_timings: null");
    *t = e->tm;
    return GS_OK;
}

// pinned host memory for callers (the SharedArrayBuffer views a shared-memory worker hands out, SortWorker.js:180-191)
extern "C" int gs_host_alloc(void **ptr, size_t bytes) {
    if (!ptr) return fail(GS_ERR_BAD_ARG, "gs_host_alloc: null");
    if (gs_device_count() <= 0) return fail(GS_ERR_NO_DEVICE, "no CUDA device");
    CU(cudaHostAlloc(ptr, std::max<size_t>(bytes, 1), cudaHostAllocDefault));
    return GS_OK;
}
extern "C" int gs_host_free(void *ptr) {
    if (ptr) CU(cudaFreeHost(ptr));
    return GS_OK;
}
