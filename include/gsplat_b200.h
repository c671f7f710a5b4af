/* gsplat_b200.h -- C ABI of libgsplat_b200.so: the B200 (sm_100a) depth -> sort -> rasterise engine that
 * sits behind the GaussianSplats3D sort-worker / SplatMesh boundary.
 *
 * Every entry point cites the reference interface (file:line under mkkellogg/GaussianSplats3D @ v0.4.7)
 * it replaces.  Plain pointers and sizes only; no torch / C++ types.  All functions return 0 (GS_OK) or a
 * gs_status error code unless stated otherwise; nothing in this library falls back to the CPU: without a
 * CUDA device every compute entry returns GS_ERR_NO_DEVICE.
 *
 * Memory kinds: pointers are HOST pointers unless the parameter name ends in `_dev`.
 *
 * Threading: like the reference's worker (one sort in flight, SortWorker.js `sortRunning`), an engine handle is driven by one
 * thread at a time; different handles may be used from different threads.  The stateless drop-in (section 1) keeps one cached
 * private engine; concurrent calls are serialised.  gs_last_error_message() is per thread.
 */
#ifndef GSPLAT_B200_H
#define GSPLAT_B200_H

#include <stdint.h>
#include <stdbool.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GS_API __attribute__((visibility("default")))
#define GS_ABI_VERSION 1
#define GS_MAX_SCENES 32 /* Constants.MaxScenes, src/Constants.js:7 */

typedef enum gs_status {
    GS_OK = 0,
    GS_ERR_BAD_ARG = 1,       /* null pointer, sortCount > renderCount, range < 2, ...                        */
    GS_ERR_NO_DEVICE = 2,     /* no CUDA device / CUDA runtime error at init                                   */
    GS_ERR_CUDA = 3,          /* a CUDA call failed; gs_last_error_message() has the text                      */
    GS_ERR_DEGENERATE = 4,    /* all distances equal (reference: rangeMap = inf -> NaN -> wasm trap)           */
    GS_ERR_BUCKET_RANGE = 5,  /* a bucket index fell outside [0, distanceMapRange) (reference: OOB write)      */
    GS_ERR_NOT_READY = 6,     /* render before upload / sort                                                   */
    GS_ERR_CAPACITY = 7       /* splat range outside the capacity given at create time                         */
} gs_status;

GS_API int gs_abi_version(void);
GS_API const char *gs_status_string(int status);
GS_API const char *gs_last_error_message(void); /* thread-local text of the last failing call */
GS_API int gs_device_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * 1. Stateless drop-in for the reference's only native symbol
 *      extern "C" void sortIndexes(...16 args...)                     src/worker/sorter.cpp:17-22
 *    Same argument order and meaning.  HOST pointers, as the wasm module sees its linear memory
 *    (SortWorker.js:56-60).  The two scratch outputs are reproduced too when their pointers are non-NULL:
 *    `mappedDistances[sortStart..renderCount)` = bucket of each position, `frequencies[b]` = number of
 *    sorted splats in buckets < b (what the reference's in-place counters hold on return).
 *    Every call uploads its inputs, runs the CUDA pipeline and downloads indexesOut: this is the
 *    parity-test boundary; the persistent-state path (section 2) is the fast one.
 * ---------------------------------------------------------------------------------------------------------- */
GS_API int gs_sort_indexes(const uint32_t *indexes, const void *centers, const void *precomputedDistances,
                           int32_t *mappedDistances, uint32_t *frequencies, const float *modelViewProj,
                           uint32_t *indexesOut, const uint32_t *sceneIndexes, const float *transforms,
                           uint32_t distanceMapRange, uint32_t sortCount, uint32_t renderCount, uint32_t splatCount,
                           bool usePrecomputedDistances, bool useIntegerSort, bool dynamicMode);

/* The stateless entry keeps ONE private engine cached (sized for the largest call so far, on the caller's current CUDA device) so that
 * repeated calls do not re-allocate; concurrent callers are serialised by a mutex.  gs_dropin_release() frees it (call it before
 * unloading the library or tearing the CUDA context down; it is re-created on demand). */
GS_API void gs_dropin_release(void);

/* void twin with the reference's exact symbol name and signature; errors are swallowed like a wasm trap
 * would abort the call (indexesOut untouched on failure). */
GS_API void sortIndexes(unsigned int *indexes, void *centers, void *precomputedDistances, int *mappedDistances,
                        unsigned int *frequencies, float *modelViewProj, unsigned int *indexesOut,
                        unsigned int *sceneIndexes, float *transforms, unsigned int distanceMapRange,
                        unsigned int sortCount, unsigned int renderCount, unsigned int splatCount,
                        bool usePrecomputedDistances, bool useIntegerSort, bool dynamicMode);

/* ------------------------------------------------------------------------------------------------------------
 * 2. Engine handle: the state a sort Worker + SplatMesh pair keeps on the device.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct gs_engine gs_engine;

typedef enum gs_render_mode {
    GS_RENDER_MODE_3D = 0,   /* SplatRenderMode.ThreeD: SplatMaterial3D (covariances)                                    */
    GS_RENDER_MODE_2D = 1    /* SplatRenderMode.TwoD: 2D Gaussian surfels, SplatMaterial2D (scale + rotation)            */
} gs_render_mode;

typedef struct gs_config {
    uint32_t struct_size;           /* sizeof(gs_config), for ABI growth                                        */
    int32_t device;                 /* CUDA device ordinal                                                       */
    uint32_t max_splat_count;       /* 'splatCount' of createSortWorker          SortWorker.js:202               */
    uint32_t distance_map_range;    /* 1 << splatSortDistanceMapPrecision        SortWorker.js:243, Constants.js:3 */
    uint8_t integer_based_sort;     /* Viewer option integerBasedSort            Viewer.js:95-98                 */
    uint8_t dynamic_mode;           /* Viewer option dynamicScene                SortWorker.js:120               */
    uint8_t splat_render_mode;      /* Viewer option splatRenderMode (SplatRenderMode.js, Viewer.js:199-202), fixed
                                       for the engine's lifetime like the reference's material: GS_RENDER_MODE_*     */
    uint8_t reserved0;
    uint32_t max_width, max_height; /* largest framebuffer gs_render will be asked for (0,0: sort only)          */
    /* multi-GPU sharding (one engine per process per GPU): this engine rasterises the 128x64-pixel coarse tiles
     * (cx, cy) with (cx + cy) % world_size == rank and leaves every other pixel of its frame zero, so the ranks'
     * frames SUM to the picture (one NCCL all-reduce).  world_size 0 or 1 = everything.                         */
    uint32_t rank, world_size;
} gs_config;

GS_API int gs_create(const gs_config *cfg, gs_engine **out);
GS_API void gs_destroy(gs_engine *e); /* worker.terminate()  Viewer.js:1311 */

/* 'centers' message: persistent sorter centres for splats [from, from+count)      SortWorker.js:84-98
 * centers: int32x4 (integer_based_sort) or f32x4 per splat, exactly what SplatMesh.getIntegerCenters /
 * getFloatCenters(padFour=true) produce (SplatMesh.js:1912-1948).  sceneIndexes may be NULL unless dynamic. */
GS_API int gs_upload_centers(gs_engine *e, const void *centers, const uint32_t *sceneIndexes, uint32_t from,
                             uint32_t count);

typedef struct gs_sort_params {
    uint32_t struct_size;
    float model_view_proj[16];           /* column-major, Viewer.js:1888-1891                                    */
    uint32_t sort_count, render_count;   /* 'splatSortCount' / 'splatRenderCount'    SortWorker.js:99-101         */
    const uint32_t *indexes_to_sort;     /* HOST u32[render_count]; NULL = identity (gatherSceneNodesForSort's
                                            no-tree case, Viewer.js:2061-2074)                                    */
    const uint32_t *indexes_to_sort_dev; /* or DEVICE pointer (takes precedence)                                  */
    const float *transforms;             /* HOST f32[16*GS_MAX_SCENES] when dynamic  SortWorker.js:38-39          */
    const void *precomputed_distances;   /* HOST i32/f32[splat_count] when use_precomputed (SortWorker.js:40-50)  */
    uint8_t use_precomputed_distances;
    uint8_t reserved[3];
} gs_sort_params;

/* 'sort' message -> 'sortDone'.  Runs asynchronously on the engine's stream; the sorted order stays on the
 * device for gs_render.  sorted_out (HOST u32[render_count], may be NULL) receives 'sortedIndexes'
 * (SortWorker.js:68-75); sort_time_ms (may be NULL) the device time of the sort kernels.                       */
GS_API int gs_sort(gs_engine *e, const gs_sort_params *p, uint32_t *sorted_out, float *sort_time_ms);

/* The SplatTree's leaves (`nodesWithIndexes`, src/splattree/SplatTree.js:55-79; built at load on the host like the reference's tree worker)
 * and the per-frame half of Viewer.gatherSceneNodesForSort (src/Viewer.js:1969-2077) on the GPU: every leaf is tested against the view
 * frustum (the two angle tests and the `distance > nodeSize` exemption of Viewer.js:2013-2033, f64), the kept leaves are ordered by their
 * distance to the camera and their index runs are written into the engine's indexesToSort (GS_BUF_INDEXES_TO_SORT) from the END of the
 * window backwards -- nearest leaf last -- exactly the layout the reference builds (Viewer.js:2040-2055).  *render_count = splatRenderCount.
 * Follow with gs_sort(indexes_to_sort_dev = GS_BUF_INDEXES_TO_SORT, render_count, sort_count <= render_count): a partial sort
 * (Viewer.js:1843-1856) re-sorts the nearest sort_count splats and copies the rest through (sorter.cpp:158-160).
 * node_center / node_min / node_max: f64[3 * node_count]; node_offsets: u32[node_count + 1]; indexes: u32[node_offsets[node_count]].
 * model_view: f64[16] column-major = inverse(camera.matrixWorld) [* mesh.matrixWorld]; cos_fov_*: Viewer.js:1990-1995.                 */
GS_API int gs_upload_splat_tree(gs_engine *e, const double *node_center, const double *node_min, const double *node_max,
                                const uint32_t *node_offsets, const uint32_t *indexes, uint32_t node_count);
GS_API int gs_gather_for_sort(gs_engine *e, const double *model_view, double cos_fov_x_over_2, double cos_fov_y_over_2, int gather_all_nodes,
                              uint32_t *render_count);

/* D1: the transform-feedback distance pre-pass, SplatMesh.computeDistancesOnGPU (SplatMesh.js:1701-1814): distances
 * in SPLAT order from the uploaded centres.  model_view_proj is f64 because three.js matrices are JS numbers and the
 * integer rows are Math.round(element * 1000) of those doubles (getIntegerMatrixArray, SplatMesh.js:2057-2064);
 * scene_transforms (f64[16*GS_MAX_SCENES], dynamic mode only, else NULL) are the per-scene matrices multiplied in at
 * SplatMesh.js:1722-1724.  out: HOST i32[count] (integer mode) or f32[count] (float mode, SplatMesh.js:1473-1502).   */
GS_API int gs_compute_distances(gs_engine *e, const double *model_view_proj, const double *scene_transforms,
                                uint32_t count, void *out);

/* ------------------------------------------------------------------------------------------------------------
 * 3. Rasteriser: the data textures SplatMesh uploads (setupDataTextures, SplatMesh.js:637-898) and the uniforms
 *    it sets per frame (updateUniforms :1248-1280, Viewer.updateSplatMesh Viewer.js:651-677, three.js camera
 *    matrices).
 * ---------------------------------------------------------------------------------------------------------- */
typedef enum gs_cov_format { GS_COV_F32 = 0, GS_COV_F16 = 1 } gs_cov_format;
typedef enum gs_sh_format { GS_SH_NONE = 0, GS_SH_F16 = 1, GS_SH_U8 = 2, GS_SH_F32 = 3 } gs_sh_format;

typedef struct gs_splat_data {
    uint32_t struct_size;
    uint32_t from, count;             /* splat range being (re)uploaded                                          */
    const uint32_t *centers_colors;   /* u32x4: {r|g<<8|b<<16|a<<24, bits(x), bits(y), bits(z)}  SplatMesh.js:1143-1153 */
    const void *covariances;          /* 6 x f32 (GS_COV_F32) or 6 x f16 (GS_COV_F16, tightly packed) per splat:
                                         [m00 m01 m02 m11 m12 m22]                     SplatBuffer.js:440-486       */
    int32_t cov_format;
    const void *spherical_harmonics;  /* sh_components values per splat, coefficient-major RGB triples
                                         (sh1.rgb, sh2.rgb, ...)                        SplatBuffer.js:551-734      */
    int32_t sh_format;                /* gs_sh_format                                                             */
    uint32_t sh_degree;               /* 0, 1 (9 values) or 2 (24 values)                                         */
    const uint32_t *scene_indexes;    /* u32 per splat or NULL (single scene)                                     */
    /* appended (callers built against the older, shorter struct are recognised by struct_size):                          */
    const float *scale_rotations;     /* GS_RENDER_MODE_2D engines: 6 x f32 per splat [sx sy sz qx qy qz], qw rebuilt as
                                         sqrt(1 - x^2 - y^2 - z^2) (SplatMesh.updateScaleRotationsPaddedData :1150-1170).
                                         Required there, and `covariances` is then ignored; unused by 3D engines.           */
} gs_splat_data;

GS_API int gs_upload_splat_data(gs_engine *e, const gs_splat_data *d);

/* `.ksplat` buffer (the SplatBuffer container, src/loaders/SplatBuffer.js:819-941, KSplatLoader.loadFromFileData) decoded ON THE
 * GPU into everything above at once: centres+colours, covariances, spherical harmonics AND the sorter's centres
 * (= new SplatBuffer(fileData) + SplatMesh.build + the 'centers' message).  Compression levels 0/1/2, SH degree 0/1/2.
 * A GS_RENDER_MODE_2D engine decodes the scale/rotation texture (fillSplatScaleRotationArray, SplatBuffer.js:349-438, z scale
 * overridden to 1 as SplatMesh.js:1856-1863 does, read at the file's level: 2^-24 for levels 1 and 2) instead of covariances;
 * `half_covariances` has no meaning there.                                                                                       */
typedef struct gs_ksplat_options {
    uint32_t struct_size;
    uint32_t minimum_alpha;          /* splatAlphaRemovalThreshold (Viewer.js), default 1: alpha below it renders as 0            */
    uint8_t half_covariances;        /* halfPrecisionCovariancesOnGPU                                                            */
    uint8_t upload_sort_centers;     /* also fill the sorter's centres (integer or float per gs_config), default 1              */
    uint8_t has_transform;           /* bake `transform` into centres, covariances and SH (static scene: SplatMesh.js:1872-1897)  */
    uint8_t reserved[1];
    double transform[16];            /* column-major Matrix4 of the SplatScene (position, quaternion, scale), JS doubles          */
} gs_ksplat_options;
typedef struct gs_ksplat_info {
    uint32_t struct_size;
    uint32_t splat_count, sh_degree, compression_level, section_count;
    float scene_center[3];
    float min_sh_coeff, max_sh_coeff; /* 8-bit SH range -> gs_uniforms.sh8_min/max                                                */
} gs_ksplat_info;
GS_API int gs_upload_ksplat(gs_engine *e, const void *data, size_t bytes, const gs_ksplat_options *opt, gs_ksplat_info *info);

typedef struct gs_uniforms {
    uint32_t struct_size;
    float model_view[16];             /* three: modelViewMatrix = camera.matrixWorldInverse * mesh.matrixWorld    */
    float projection[16];             /* camera.projectionMatrix                                                  */
    float camera_position[3];         /* cameraPosition uniform (world)                                           */
    float focal[2];                   /* SplatMesh.js:1262                                                        */
    float viewport[2];                /* render dimensions * devicePixelRatio, SplatMesh.js:1257-1259             */
    float inverse_focal_adjustment;   /* SplatMesh.js:1265                                                        */
    float ortho_zoom;                 /* SplatMesh.js:1264                                                        */
    int32_t orthographic_mode;        /* SplatMesh.js:1263                                                        */
    float splat_scale;                /* SplatMaterial.js:469                                                     */
    int32_t point_cloud_mode;         /* SplatMaterial.js:473                                                     */
    int32_t sh_degree;                /* sphericalHarmonicsDegree uniform (<= uploaded degree)                    */
    int32_t antialiased;              /* SplatMaterial3D.js:137-145                                               */
    float kernel_2d_size;             /* default 0.3, SplatMaterial3D.js:21                                       */
    float max_screen_space_splat_size;/* default 1024 (Viewer.js:201), SplatMaterial3D.js:193-194                 */
    float sh8_min[GS_MAX_SCENES];     /* sphericalHarmonics8BitCompressionRangeMin/Max, SplatMaterial.js:402-409  */
    float sh8_max[GS_MAX_SCENES];
    uint32_t scene_count;
    float scene_transforms[16 * GS_MAX_SCENES]; /* dynamic mode `transforms` uniform                              */
    float view_matrix[16];            /* three: viewMatrix (dynamic mode only)                                    */
    float scene_opacity[GS_MAX_SCENES];   /* enableOptionalEffects                                                */
    int32_t scene_visibility[GS_MAX_SCENES];
    int32_t enable_optional_effects;  /* SplatMaterial.js:23-28,124-133; SplatMaterial3D.js:198-202           */
    int32_t dynamic_mode;             /* per-scene transforms in the vertex stage, SplatMaterial.js:136-146       */
    /* fade-in (SplatMaterial.js:347-363) */
    int32_t fade_in_complete;
    float scene_center[3];
    float visible_region_fade_start_radius;
} gs_uniforms;

typedef enum gs_frame_format {
    GS_FRAME_RGBA32F = 0, /* float accumulators, premultiplied colour + coverage alpha                            */
    GS_FRAME_RGBA8 = 1    /* the canvas format: round(clamp(v,0,1)*255) once at the end                           */
} gs_frame_format;

typedef struct gs_render_params {
    uint32_t struct_size;
    uint32_t width, height;
    uint32_t render_count;              /* geometry.instanceCount, SplatMesh.js:1233-1234                         */
    const uint32_t *sorted_indexes;     /* HOST u32[render_count] = the splatIndex attribute
                                           (SplatMesh.updateRenderIndexes :1228-1235); NULL = use the order of
                                           the engine's last gs_sort                                              */
    const uint32_t *sorted_indexes_dev; /* or DEVICE pointer                                                      */
    int32_t frame_format;               /* gs_frame_format                                                        */
    int32_t flip_y;                     /* 0: row 0 = bottom (GL window coords); 1: row 0 = top (image order)     */
} gs_render_params;

/* renderer.render(splatMesh, camera)  Viewer.js:1616.  frame_out: HOST buffer of width*height*4 floats or bytes
 * (may be NULL: the frame stays on the device, see gs_frame_dev).                                               */
GS_API int gs_render(gs_engine *e, const gs_uniforms *u, const gs_render_params *p, void *frame_out);

/* One viewer frame: Viewer.update() -> runSplatSort (full sort) + render  (Viewer.js:1625-1644, 1599-1623).    */
GS_API int gs_frame(gs_engine *e, const gs_sort_params *s, const gs_uniforms *u, const gs_render_params *p,
                    uint32_t *sorted_out, void *frame_out);

/* Same, but only enqueued on the engine's stream: returns without waiting, the frame stays on the device
 * (gs_buffer_dev(GS_BUF_FRAME)); device-side errors and timings are collected by the next gs_synchronize().         */
GS_API int gs_frame_async(gs_engine *e, const gs_sort_params *s, const gs_uniforms *u, const gs_render_params *p);

/* Pipelined frames: the frame loop of Viewer.selfDrivenUpdate (Viewer.js:1543-1555) with up to three frames in flight.  gs_frame_begin
 * enqueues one frame exactly like gs_frame (camera host -> device, full sort, render) plus the copy of its picture into frame_out (HOST,
 * ideally page-locked: gs_host_alloc; every frame in flight needs its own) on a separate copy stream, and returns at once; gs_frame_end
 * waits for the OLDEST frame in flight, after which its frame_out is complete, and returns that frame's status.  Device frames alternate
 * between two buffers, so frame i+1 is computed while frame i crosses PCIe and frame i+2 is already queued behind it:
 *   begin(0); begin(1); for (i...) { begin(i+2); end(i); }       (begin(0); for (i...) { begin(i+1); end(i); } also works)
 * A fourth gs_frame_begin without a gs_frame_end returns GS_ERR_NOT_READY.                                                            */
GS_API int gs_frame_begin(gs_engine *e, const gs_sort_params *s, const gs_uniforms *u, const gs_render_params *p, void *frame_out);
GS_API int gs_frame_end(gs_engine *e);

/* ------------------------------------------------------------------------------------------------------------
 * 4. Device-side access for zero-copy callers and for the multi-GPU plumbing (tile gather over NCCL).
 * ---------------------------------------------------------------------------------------------------------- */
typedef enum gs_buffer_id {
    GS_BUF_SORTED_INDEXES = 0, /* u32[render_count]                                                               */
    GS_BUF_FRAME = 1,          /* last rendered frame in the requested format                                     */
    GS_BUF_CENTERS = 2,
    GS_BUF_DISTANCES = 3,      /* i32[render_count] scratch (= mappedDistances)                                   */
    GS_BUF_SPLAT_RECORDS = 4,  /* per-splat projected records (engine-internal layout: 48 B, 2D engines 96 B)     */
    GS_BUF_INDEXES_TO_SORT = 5,/* u32[max_splat_count] staging for indexesToSort                                  */
    GS_BUF_CENTERS_COLORS = 6, GS_BUF_COVARIANCES = 7, GS_BUF_SH = 8,  /* the uploaded / decoded splat data (gs_read_buffer only) */
    GS_BUF_SCALE_ROTATIONS = 9,/* 2D engines: 6 x f32 per splat, as gs_splat_data.scale_rotations (gs_read_buffer only)          */
    /* Tile binning of the last rendered frame, for tests (gs_read_buffer only).  Coarse tiles are 8 x 4 fine tiles, numbered
     * cy * coarse_x + cx; a list entry is (fine-tile mask << 32) | splat id, bit 8 * fy + fx = fine tile (fx, fy) of the coarse tile.    */
    GS_BUF_TILE_RECTS = 10,    /* u16x4 per uploaded splat: inclusive fine-tile rect {x0, y0, x1, y1}; empty (x1 < x0) = not drawn    */
    GS_BUF_TILE_RANGES = 11,   /* u32x2 per coarse tile: [first, end) of its list; clamped to the instance capacity               */
    GS_BUF_TILE_LIST = 12,     /* u64 list entries, per coarse tile in draw order (up to the instance capacity)                   */
    GS_BUF_TILE_ORDER = 13,    /* u32 per coarse tile: the blend's schedule of coarse tiles                                       */
    GS_BUF_TILE_INFO = 14      /* u64[4]: instance capacity, coarse tiles, fine-tile edge in px, binning path (2 counting, 1 radix) */
} gs_buffer_id;
GS_API int gs_buffer_dev(gs_engine *e, int buffer_id, void **ptr_dev, size_t *bytes);
GS_API int gs_read_buffer(gs_engine *e, int buffer_id, void *out, size_t offset, size_t bytes); /* D2H copy, for tests / tools */
GS_API int gs_stream(gs_engine *e, void **cuda_stream); /* cudaStream_t of the engine */
GS_API int gs_synchronize(gs_engine *e);

/* Fused tile gather (multi-GPU, one process per GPU).  Rank 0 exports CUDA-IPC handles of its frame buffer and of a small handshake
 * block; every other rank attaches, after which its blend kernel stores finished pixels STRAIGHT INTO RANK 0'S FRAME over NVLink
 * and rank 0's frame is complete when gs_frame / gs_synchronize returns -- no NCCL call, no staging copy.  All ranks must render
 * the same sequence of frames.  (Without these calls the ranks' frames are zero outside their own tiles and can be summed.)
 * The exported allocation holds TWO frames (all ranks size it from the same gs_config): rank 0's pipelined frames (gs_frame_begin)
 * alternate between the halves, the half in use travels in the handshake, so frame f+1 is assembled while frame f's picture is
 * copied to the host.  Environment GS_PEER_DOUBLE=0 on rank 0 keeps a single frame.                                                */
#define GS_IPC_HANDLE_BYTES 64
GS_API int gs_peer_export(gs_engine *e, void *frame_handle /*64 B out*/, void *sync_handle /*64 B out*/);      /* rank 0     */
GS_API int gs_peer_attach(gs_engine *e, const void *frame_handle, const void *sync_handle);                    /* ranks > 0  */

/* Sort-only on N GPUs (SURVEY.md 8(e) "depth + sort"): ONE sortIndexes call (sorter.cpp:17-168) split by input position.  Every
 * rank holds all centres; rank g computes distances for, and sorts, positions [sortStart + n*g/N, sortStart + n*(g+1)/N) of the
 * sort window.  Two exchanges over peer memory (NVLink), no NCCL, no host round trip: the global min/max before the range map
 * (8 B per rank pair), and the per-bucket run lengths (8 B per bucket per rank pair) from which every rank derives where its runs
 * sit in the reference's order (buckets descending, inside a bucket higher input positions first = rank N-1 ... 0).  Each rank
 * then stores its 4 B/splat straight into RANK 0's sortedIndexes, which is bit-exact with the single-GPU gs_sort.
 *   setup    every rank: gs_shard_export -> exchange the handles (any transport) -> gs_shard_attach with all N block handles
 *            (index = rank) and rank 0's sorted handle.  gs_shard_attach_local: engines of one process on one device.
 *   per sort every rank calls gs_sort_sharded with the SAME parameters; sorted_out is filled on rank 0 only (may be NULL elsewhere).
 *            _async enqueues and returns; _finish waits, copies, reports errors (a missing peer gives GS_ERR_CUDA after ~2 s).
 *   Windows below 8 M splats (env GS_SHARD_MIN overrides; 0 = always split) are sorted by rank 0 alone -- the single-GPU sort is
 *   latency bound there and the exchange would cost more than it saves; the other ranks' calls then return at once.            */
#define GS_MAX_SHARD_RANKS 8
GS_API int gs_shard_export(gs_engine *e, void *block_handle /*64 B out*/, void *sorted_handle /*64 B out*/);
GS_API int gs_shard_attach(gs_engine *e, uint32_t world, const void *block_handles /* world x 64 B */, const void *root_sorted_handle);
GS_API int gs_shard_attach_local(gs_engine *e, uint32_t world, gs_engine *const *engines /* [world], index = rank */);
GS_API int gs_sort_sharded(gs_engine *e, const gs_sort_params *p, uint32_t *sorted_out /* host, rank 0 */, float *sort_time_ms);
GS_API int gs_sort_sharded_async(gs_engine *e, const gs_sort_params *p);
GS_API int gs_sort_sharded_finish(gs_engine *e, uint32_t *sorted_out /* host, rank 0 */, float *sort_time_ms);

/* Page-locked host memory for callers: the counterpart of the SharedArrayBuffer views a shared-memory sort worker
 * hands to the main thread (SortWorker.js:180-191).  Buffers passed to gs_sort / gs_render from such memory are
 * copied asynchronously without an extra staging copy. */
GS_API int gs_host_alloc(void **ptr, size_t bytes);
GS_API int gs_host_free(void *ptr);

/* Per-splat output of the projection stage (what the vertex shader hands to rasterisation), for parity tests. */
typedef struct gs_projected_splat {
    float cx, cy;        /* quad centre, pixels, GL window coordinates (y up, pixel centres at +0.5)              */
    float b1x, b1y;      /* basisVector1 * inverseFocalAdjustment, pixels    SplatMaterial3D.js:193,206-207        */
    float b2x, b2y;      /* basisVector2 ...                                                                      */
    float r, g, b, a;    /* vColor                                                                                */
    float ndc_z;
    uint32_t valid;      /* 0 = culled / dropped                                                                  */
} gs_projected_splat;
GS_API int gs_read_projected(gs_engine *e, gs_projected_splat *out, uint32_t count); /* splat order */

/* Per-splat output of the 2D (surfel) vertex stage, SplatMaterial2D.js:96-235, for parity tests of GS_RENDER_MODE_2D engines.
 * Re-runs the projection with the parameters of the engine's last frame: the per-splat records and tile rects are rewritten with
 * the same values, and the statistics gs_last_timings reports are left as they are.  gs_read_projected returns GS_ERR_BAD_ARG on a
 * TwoD engine (it has no 3D records), as gs_read_projected_2d does on a ThreeD engine.                                           */
typedef struct gs_projected_surfel {
    float T[9];          /* vT = T = transpose(splat2World) * world2ndc * ndc2pix, column-major: Tu = T[0..2], Tv, Tw     */
    float qcx, qcy;      /* vQuadCenter: NDC units in the eigen branch (as the reference), pixels in the fallback          */
    float cx, cy;        /* quad centre, pixels, GL window coordinates                                                     */
    float h1x, h1y;      /* quad half-edges, pixels: corners = c +- h1 +- h2                                               */
    float h2x, h2y;
    float r, g, b, a;    /* vColor                                                                                         */
    float ndc_z;
    uint32_t branch;     /* 0 = eigen-aligned quad (:199-234), 1 = screen-aligned fallback square (:159-189)               */
    uint32_t valid;      /* 0 = culled / dropped (incl. |distance| < 1e-5, where the reference leaves gl_Position unset)   */
} gs_projected_surfel;
GS_API int gs_read_projected_2d(gs_engine *e, gs_projected_surfel *out, uint32_t count); /* splat order */

typedef struct gs_timings {
    float depth_ms, bucket_ms, scatter_ms, sort_total_ms;
    float project_ms, bin_ms, blend_ms, render_total_ms;
    float h2d_ms, d2h_ms;
    uint64_t tile_instances;   /* (splat, tile) pairs binned in the last render                                   */
    uint32_t kernel_launches;  /* kernels launched by the last gs_sort/gs_render/gs_frame                          */
    uint32_t visible_splats;
} gs_timings;
GS_API int gs_last_timings(gs_engine *e, gs_timings *t);

/* Measurement helpers for bench.py (no effect on results): L2 flush on the engine's stream (writes a 192 MiB scratch
 * buffer) and CUDA events recorded on that stream, so per-step device times can be taken without touching torch.     */
GS_API int gs_flush_l2(gs_engine *e);
/* Per-kernel timeline: when on, a CUDA event is recorded after every kernel the engine launches; gs_kernel_timings
 * returns {kernel name, device ms} for the last gs_sort / gs_render / gs_frame in launch order.                      */
typedef struct gs_kernel_time { char name[40]; float ms; } gs_kernel_time;
GS_API int gs_set_profiling(gs_engine *e, int on);
/* gs_frame / gs_frame_async replay a captured CUDA graph of the frame while its shape is unchanged (default on).      */
GS_API int gs_set_graph_enabled(gs_engine *e, int on);
GS_API int gs_kernel_timings(gs_engine *e, gs_kernel_time *out, uint32_t capacity, uint32_t *count);
GS_API int gs_event_create(void **event);
GS_API int gs_event_record(gs_engine *e, void *event);
GS_API int gs_event_elapsed_ms(void *event0, void *event1, float *ms); /* waits for event1 */
GS_API int gs_event_destroy(void *event);

#ifdef __cplusplus
}
#endif
#endif /* GSPLAT_B200_H */
