// js/gsplat_b200_addon.cc -- N-API glue between Node.js and libgsplat_b200.so.  Binds EVERY entry point of include/gsplat_b200.h (one JS
// function per GS_API symbol, camelCase, same argument order); no arithmetic lives here.  The image this repository is developed in has
// neither Node.js nor node_api.h, so the addon is compile-checked only against js/test/node_api_stub.h (tests/test_abi.py) and has not
// been run; with Node installed it is one `node-gyp rebuild` away (binding.gyp).
//
//   const gs = require('./build/Release/gsplat_b200.node');
//   const h = gs.create({maxSplatCount, distanceMapRange, integerBasedSort, dynamicMode, maxWidth, maxHeight, device, rank, worldSize});
//   gs.uploadCenters(h, centers, sceneIndexesOrNull, from, count);
//   gs.sort(h, {modelViewProj, sortCount, renderCount, indexesToSort, transforms, precomputedDistances, usePrecomputedDistances}, sortedOut);
//   gs.uploadSplatData(h, {...}); gs.frame(h, sortParams, uniforms, renderParams, sortedOutOrNull, frameOutOrNull); ...
// Engine handles are N-API externals whose finalizer calls gs_destroy.  Every failing call throws Error(message) with .code = gs_status.
#ifdef GS_NAPI_STUB
#include "test/node_api_stub.h"
#else
#include <node_api.h>
#endif
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>
#include "../include/gsplat_b200.h"

#define FN(name) static napi_value name(napi_env env, napi_callback_info info)
#define ARGS(n)                                                                  \
    size_t argc = (n); napi_value a[(n) > 0 ? (n) : 1]; memset(a, 0, sizeof(a)); \
    if (napi_get_cb_info(env, info, &argc, a, nullptr, nullptr) != napi_ok) { napi_throw_error(env, nullptr, "napi_get_cb_info failed"); return nullptr; }
#define CHECK(rc) do { int _rc = (rc); if (_rc) return throw_gs(env, _rc); } while (0)

static napi_value throw_gs(napi_env env, int code) {
    char num[16];
    snprintf(num, sizeof(num), "%d", code);
    napi_throw_error(env, num, gs_last_error_message()[0] ? gs_last_error_message() : gs_status_string(code));
    return nullptr;
}
static napi_value undefined(napi_env env) { napi_value v; napi_get_undefined(env, &v); return v; }
static napi_value num(napi_env env, double d) { napi_value v; napi_create_double(env, d, &v); return v; }
static napi_value u32v(napi_env env, uint32_t u) { napi_value v; napi_create_uint32(env, u, &v); return v; }
static napi_value str(napi_env env, const char *s) { napi_value v; napi_create_string_utf8(env, s, NAPI_AUTO_LENGTH, &v); return v; }
static bool is_nullish(napi_env env, napi_value v) {
    if (!v) return true;
    napi_valuetype t; napi_typeof(env, v, &t);
    return t == napi_undefined || t == napi_null;
}
static uint32_t to_u32(napi_env env, napi_value v, uint32_t dflt = 0) {
    if (is_nullish(env, v)) return dflt;
    napi_valuetype t; napi_typeof(env, v, &t);
    if (t == napi_boolean) { bool b = false; napi_get_value_bool(env, v, &b); return b ? 1u : 0u; }
    uint32_t u = dflt; napi_get_value_uint32(env, v, &u); return u;
}
static int32_t to_i32(napi_env env, napi_value v, int32_t dflt = 0) { if (is_nullish(env, v)) return dflt; int32_t i = dflt; napi_get_value_int32(env, v, &i); return i; }
static double to_f64(napi_env env, napi_value v, double dflt = 0) { if (is_nullish(env, v)) return dflt; double d = dflt; napi_get_value_double(env, v, &d); return d; }
static napi_value prop(napi_env env, napi_value obj, const char *key) {
    if (is_nullish(env, obj)) return nullptr;
    bool has = false; napi_value v = nullptr;
    if (napi_has_named_property(env, obj, key, &has) != napi_ok || !has) return nullptr;
    napi_get_named_property(env, obj, key, &v);
    return v;
}
// data pointer of a TypedArray / ArrayBuffer / Buffer (nullptr for null / undefined); *bytes = its length in bytes
static void *typed_ptr(napi_env env, napi_value v, size_t *bytes = nullptr) {
    if (bytes) *bytes = 0;
    if (is_nullish(env, v)) return nullptr;
    bool is_ta = false, is_ab = false, is_dv = false;
    void *data = nullptr; size_t len = 0;
    napi_is_typedarray(env, v, &is_ta);
    if (is_ta) {
        napi_typedarray_type t; napi_value ab; size_t off;
        napi_get_typedarray_info(env, v, &t, &len, &data, &ab, &off);
        static const size_t w[] = {1, 1, 1, 2, 2, 4, 4, 4, 8, 8, 8};
        if (bytes) *bytes = len * w[t];
        return data;
    }
    napi_is_arraybuffer(env, v, &is_ab);
    if (is_ab) { napi_get_arraybuffer_info(env, v, &data, &len); if (bytes) *bytes = len; return data; }
    napi_is_dataview(env, v, &is_dv);
    if (is_dv) { napi_value ab; size_t off; napi_get_dataview_info(env, v, &len, &data, &ab, &off); if (bytes) *bytes = len; return data; }
    return nullptr;
}
static void copy_floats(napi_env env, napi_value v, float *dst, size_t n) {     // Float32Array, Float64Array or plain Array of numbers
    if (is_nullish(env, v)) return;
    bool is_ta = false; napi_is_typedarray(env, v, &is_ta);
    if (is_ta) {
        napi_typedarray_type t; size_t len; void *data; napi_value ab; size_t off;
        napi_get_typedarray_info(env, v, &t, &len, &data, &ab, &off);
        for (size_t i = 0; i < n && i < len; ++i) dst[i] = t == napi_float64_array ? (float)((double *)data)[i] : (t == napi_float32_array ? ((float *)data)[i] : 0.f);
        return;
    }
    for (uint32_t i = 0; i < n; ++i) { napi_value e; if (napi_get_element(env, v, i, &e) != napi_ok) break; dst[i] = (float)to_f64(env, e); }
}
static void copy_doubles(napi_env env, napi_value v, double *dst, size_t n) {
    if (is_nullish(env, v)) return;
    bool is_ta = false; napi_is_typedarray(env, v, &is_ta);
    if (is_ta) {
        napi_typedarray_type t; size_t len; void *data; napi_value ab; size_t off;
        napi_get_typedarray_info(env, v, &t, &len, &data, &ab, &off);
        for (size_t i = 0; i < n && i < len; ++i) dst[i] = t == napi_float64_array ? ((double *)data)[i] : (t == napi_float32_array ? (double)((float *)data)[i] : 0.0);
        return;
    }
    for (uint32_t i = 0; i < n; ++i) { napi_value e; if (napi_get_element(env, v, i, &e) != napi_ok) break; dst[i] = to_f64(env, e); }
}
static gs_engine *engine_of(napi_env env, napi_value v) { void *p = nullptr; if (!is_nullish(env, v)) napi_get_value_external(env, v, &p); return (gs_engine *)p; }
static napi_value ptr_value(napi_env env, const void *p) { napi_value v; napi_create_bigint_uint64(env, (uint64_t)(uintptr_t)p, &v); return v; }
static void *ptr_of(napi_env env, napi_value v) { if (is_nullish(env, v)) return nullptr; uint64_t u = 0; bool lossless = true; napi_get_value_bigint_uint64(env, v, &u, &lossless); return (void *)(uintptr_t)u; }

// ---- struct marshalling (field names = the C struct's, camelCase) ------------------------------------------------------------------
static void fill_sort_params(napi_env env, napi_value o, gs_sort_params *p) {
    memset(p, 0, sizeof(*p));
    p->struct_size = sizeof(*p);
    copy_floats(env, prop(env, o, "modelViewProj"), p->model_view_proj, 16);
    p->sort_count = to_u32(env, prop(env, o, "sortCount"));
    p->render_count = to_u32(env, prop(env, o, "renderCount"));
    p->indexes_to_sort = (const uint32_t *)typed_ptr(env, prop(env, o, "indexesToSort"));
    p->indexes_to_sort_dev = (const uint32_t *)ptr_of(env, prop(env, o, "indexesToSortDev"));
    p->transforms = (const float *)typed_ptr(env, prop(env, o, "transforms"));
    p->precomputed_distances = typed_ptr(env, prop(env, o, "precomputedDistances"));
    p->use_precomputed_distances = (uint8_t)to_u32(env, prop(env, o, "usePrecomputedDistances"));
}
static void fill_uniforms(napi_env env, napi_value o, gs_uniforms *u) {
    memset(u, 0, sizeof(*u));
    u->struct_size = sizeof(*u);
    copy_floats(env, prop(env, o, "modelView"), u->model_view, 16);
    copy_floats(env, prop(env, o, "projection"), u->projection, 16);
    copy_floats(env, prop(env, o, "cameraPosition"), u->camera_position, 3);
    copy_floats(env, prop(env, o, "focal"), u->focal, 2);
    copy_floats(env, prop(env, o, "viewport"), u->viewport, 2);
    u->inverse_focal_adjustment = (float)to_f64(env, prop(env, o, "inverseFocalAdjustment"), 1.0);
    u->ortho_zoom = (float)to_f64(env, prop(env, o, "orthoZoom"), 1.0);
    u->orthographic_mode = to_i32(env, prop(env, o, "orthographicMode"));
    u->splat_scale = (float)to_f64(env, prop(env, o, "splatScale"), 1.0);
    u->point_cloud_mode = to_i32(env, prop(env, o, "pointCloudModeEnabled"));
    u->sh_degree = to_i32(env, prop(env, o, "sphericalHarmonicsDegree"));
    u->antialiased = to_i32(env, prop(env, o, "antialiased"));
    u->kernel_2d_size = (float)to_f64(env, prop(env, o, "kernel2DSize"), 0.3);
    u->max_screen_space_splat_size = (float)to_f64(env, prop(env, o, "maxScreenSpaceSplatSize"), 1024.0);
    for (int i = 0; i < GS_MAX_SCENES; ++i) { u->sh8_min[i] = -1.5f; u->sh8_max[i] = 1.5f; u->scene_opacity[i] = 1.f; u->scene_visibility[i] = 1; }
    copy_floats(env, prop(env, o, "sphericalHarmonics8BitCompressionRangeMin"), u->sh8_min, GS_MAX_SCENES);
    copy_floats(env, prop(env, o, "sphericalHarmonics8BitCompressionRangeMax"), u->sh8_max, GS_MAX_SCENES);
    u->scene_count = to_u32(env, prop(env, o, "sceneCount"), 1);
    for (int s = 0; s < GS_MAX_SCENES; ++s) for (int k = 0; k < 4; ++k) u->scene_transforms[16 * s + 5 * k] = 1.f;
    copy_floats(env, prop(env, o, "transforms"), u->scene_transforms, 16 * GS_MAX_SCENES);
    for (int k = 0; k < 4; ++k) u->view_matrix[5 * k] = 1.f;
    copy_floats(env, prop(env, o, "viewMatrix"), u->view_matrix, 16);
    copy_floats(env, prop(env, o, "sceneOpacity"), u->scene_opacity, GS_MAX_SCENES);
    if (napi_value vis = prop(env, o, "sceneVisibility")) for (uint32_t i = 0; i < GS_MAX_SCENES; ++i) { napi_value e; if (napi_get_element(env, vis, i, &e) != napi_ok || is_nullish(env, e)) break; u->scene_visibility[i] = to_i32(env, e, 1); }
    u->enable_optional_effects = to_i32(env, prop(env, o, "enableOptionalEffects"));
    u->dynamic_mode = to_i32(env, prop(env, o, "dynamicMode"));
    u->fade_in_complete = to_i32(env, prop(env, o, "fadeInComplete"), 1);
    copy_floats(env, prop(env, o, "sceneCenter"), u->scene_center, 3);
    u->visible_region_fade_start_radius = (float)to_f64(env, prop(env, o, "visibleRegionFadeStartRadius"));
}
static void fill_render_params(napi_env env, napi_value o, gs_render_params *p) {
    memset(p, 0, sizeof(*p));
    p->struct_size = sizeof(*p);
    p->width = to_u32(env, prop(env, o, "width"));
    p->height = to_u32(env, prop(env, o, "height"));
    p->render_count = to_u32(env, prop(env, o, "renderCount"));
    p->sorted_indexes = (const uint32_t *)typed_ptr(env, prop(env, o, "sortedIndexes"));
    p->sorted_indexes_dev = (const uint32_t *)ptr_of(env, prop(env, o, "sortedIndexesDev"));
    p->frame_format = to_i32(env, prop(env, o, "frameFormat"), GS_FRAME_RGBA8);
    p->flip_y = to_i32(env, prop(env, o, "flipY"), 1);
}

// ---- library -----------------------------------------------------------------------------------------------------------------------
FN(AbiVersion) { (void)info; return u32v(env, (uint32_t)gs_abi_version()); }
FN(StatusString) { ARGS(1) return str(env, gs_status_string(to_i32(env, a[0]))); }
FN(LastErrorMessage) { (void)info; return str(env, gs_last_error_message()); }
FN(DeviceCount) { (void)info; return u32v(env, (uint32_t)gs_device_count()); }

// sortIndexes(indexes, centers, precomputedDistances, mappedDistances, frequencies, modelViewProj, indexesOut, sceneIndexes, transforms,
//             distanceMapRange, sortCount, renderCount, splatCount, usePrecomputedDistances, useIntegerSort, dynamicMode)   sorter.cpp:17-22
FN(SortIndexes) {
    ARGS(16)
    float mvp[16] = {0};
    copy_floats(env, a[5], mvp, 16);
    CHECK(gs_sort_indexes((const uint32_t *)typed_ptr(env, a[0]), typed_ptr(env, a[1]), typed_ptr(env, a[2]), (int32_t *)typed_ptr(env, a[3]), (uint32_t *)typed_ptr(env, a[4]),
                          mvp, (uint32_t *)typed_ptr(env, a[6]), (const uint32_t *)typed_ptr(env, a[7]), (const float *)typed_ptr(env, a[8]), to_u32(env, a[9]),
                          to_u32(env, a[10]), to_u32(env, a[11]), to_u32(env, a[12]), to_u32(env, a[13]) != 0, to_u32(env, a[14]) != 0, to_u32(env, a[15]) != 0));
    return undefined(env);
}
FN(SortIndexesVoid) {   // the reference's own symbol: errors are swallowed (indexesOut untouched), like a wasm trap aborting the call
    ARGS(16)
    float mvp[16] = {0};
    copy_floats(env, a[5], mvp, 16);
    sortIndexes((unsigned int *)typed_ptr(env, a[0]), typed_ptr(env, a[1]), typed_ptr(env, a[2]), (int *)typed_ptr(env, a[3]), (unsigned int *)typed_ptr(env, a[4]), mvp,
                (unsigned int *)typed_ptr(env, a[6]), (unsigned int *)typed_ptr(env, a[7]), (float *)typed_ptr(env, a[8]), to_u32(env, a[9]), to_u32(env, a[10]), to_u32(env, a[11]),
                to_u32(env, a[12]), to_u32(env, a[13]) != 0, to_u32(env, a[14]) != 0, to_u32(env, a[15]) != 0);
    return undefined(env);
}
FN(DropinRelease) { (void)info; gs_dropin_release(); return undefined(env); }

// ---- engine ------------------------------------------------------------------------------------------------------------------------
FN(Create) {
    ARGS(1)
    gs_config c; memset(&c, 0, sizeof(c)); c.struct_size = sizeof(c);
    c.device = to_i32(env, prop(env, a[0], "device"));
    c.max_splat_count = to_u32(env, prop(env, a[0], "maxSplatCount"));
    c.distance_map_range = to_u32(env, prop(env, a[0], "distanceMapRange"));
    c.integer_based_sort = (uint8_t)to_u32(env, prop(env, a[0], "integerBasedSort"), 1);
    c.dynamic_mode = (uint8_t)to_u32(env, prop(env, a[0], "dynamicMode"));
    c.splat_render_mode = (uint8_t)to_u32(env, prop(env, a[0], "splatRenderMode"));   // SplatRenderMode.ThreeD = 0 / TwoD = 1
    c.max_width = to_u32(env, prop(env, a[0], "maxWidth"));
    c.max_height = to_u32(env, prop(env, a[0], "maxHeight"));
    c.rank = to_u32(env, prop(env, a[0], "rank"));
    c.world_size = to_u32(env, prop(env, a[0], "worldSize"), 1);
    gs_engine *e = nullptr;
    CHECK(gs_create(&c, &e));
    napi_value ext;
    if (napi_create_external(env, e, [](napi_env, void *p, void *) { gs_destroy((gs_engine *)p); }, nullptr, &ext) != napi_ok) { gs_destroy(e); napi_throw_error(env, nullptr, "napi_create_external failed"); return nullptr; }
    return ext;
}
FN(Destroy) { ARGS(1) (void)a; return undefined(env); }   // worker.terminate(): the handle's finalizer calls gs_destroy once the external is collected
FN(UploadCenters) {   // 'centers' message, SortWorker.js:84-98
    ARGS(5)
    CHECK(gs_upload_centers(engine_of(env, a[0]), typed_ptr(env, a[1]), (const uint32_t *)typed_ptr(env, a[2]), to_u32(env, a[3]), to_u32(env, a[4])));
    return undefined(env);
}
FN(Sort) {            // 'sort' message, SortWorker.js:31-81: (engine, sortParams, sortedOutOrNull) -> {sortTime}
    ARGS(3)
    gs_sort_params p; fill_sort_params(env, a[1], &p);
    float ms = 0.f;
    CHECK(gs_sort(engine_of(env, a[0]), &p, (uint32_t *)typed_ptr(env, a[2]), &ms));
    napi_value out; napi_create_object(env, &out); napi_set_named_property(env, out, "sortTime", num(env, ms));
    return out;
}
FN(UploadSplatTree) { // (engine, nodeCenter f64, nodeMin f64, nodeMax f64, nodeOffsets u32, indexes u32, nodeCount)
    ARGS(7)
    CHECK(gs_upload_splat_tree(engine_of(env, a[0]), (const double *)typed_ptr(env, a[1]), (const double *)typed_ptr(env, a[2]), (const double *)typed_ptr(env, a[3]),
                               (const uint32_t *)typed_ptr(env, a[4]), (const uint32_t *)typed_ptr(env, a[5]), to_u32(env, a[6])));
    return undefined(env);
}
FN(GatherForSort) {   // (engine, modelView[16], cosFovXOver2, cosFovYOver2, gatherAllNodes) -> splatRenderCount
    ARGS(5)
    double mv[16] = {0}; copy_doubles(env, a[1], mv, 16);
    uint32_t rc = 0;
    CHECK(gs_gather_for_sort(engine_of(env, a[0]), mv, to_f64(env, a[2]), to_f64(env, a[3]), (int)to_u32(env, a[4]), &rc));
    return u32v(env, rc);
}
FN(ComputeDistances) { // (engine, modelViewProj[16] f64, sceneTransforms f64[512] | null, count, out Int32Array | Float32Array)
    ARGS(5)
    double mvp[16] = {0}; copy_doubles(env, a[1], mvp, 16);
    std::vector<double> tr;
    if (!is_nullish(env, a[2])) { tr.assign(16 * GS_MAX_SCENES, 0.0); for (int s = 0; s < GS_MAX_SCENES; ++s) for (int k = 0; k < 4; ++k) tr[16 * s + 5 * k] = 1.0; copy_doubles(env, a[2], tr.data(), tr.size()); }
    CHECK(gs_compute_distances(engine_of(env, a[0]), mvp, tr.empty() ? nullptr : tr.data(), to_u32(env, a[3]), typed_ptr(env, a[4])));
    return undefined(env);
}
FN(UploadSplatData) { // (engine, {from, count, centersColors, covariances, covFormat, sphericalHarmonics, shFormat, shDegree, sceneIndexes, scaleRotations})
    ARGS(2)
    gs_splat_data d; memset(&d, 0, sizeof(d)); d.struct_size = sizeof(d);
    d.from = to_u32(env, prop(env, a[1], "from"));
    d.count = to_u32(env, prop(env, a[1], "count"));
    d.centers_colors = (const uint32_t *)typed_ptr(env, prop(env, a[1], "centersColors"));
    d.covariances = typed_ptr(env, prop(env, a[1], "covariances"));
    d.cov_format = to_i32(env, prop(env, a[1], "covFormat"));
    d.spherical_harmonics = typed_ptr(env, prop(env, a[1], "sphericalHarmonics"));
    d.sh_format = to_i32(env, prop(env, a[1], "shFormat"));
    d.sh_degree = to_u32(env, prop(env, a[1], "shDegree"));
    d.scene_indexes = (const uint32_t *)typed_ptr(env, prop(env, a[1], "sceneIndexes"));
    d.scale_rotations = (const float *)typed_ptr(env, prop(env, a[1], "scaleRotations"));   // TwoD: the scale/rotation texture
    CHECK(gs_upload_splat_data(engine_of(env, a[0]), &d));
    return undefined(env);
}
FN(UploadKsplat) {    // (engine, ArrayBuffer, {minimumAlpha, halfCovariances, uploadSortCenters, transform}) -> info
    ARGS(3)
    size_t bytes = 0; const void *data = typed_ptr(env, a[1], &bytes);
    gs_ksplat_options o; memset(&o, 0, sizeof(o)); o.struct_size = sizeof(o);
    o.minimum_alpha = to_u32(env, prop(env, a[2], "minimumAlpha"), 1);
    o.half_covariances = (uint8_t)to_u32(env, prop(env, a[2], "halfCovariances"));
    o.upload_sort_centers = (uint8_t)to_u32(env, prop(env, a[2], "uploadSortCenters"), 1);
    if (napi_value t = prop(env, a[2], "transform")) if (!is_nullish(env, t)) { o.has_transform = 1; copy_doubles(env, t, o.transform, 16); }
    gs_ksplat_info inf; memset(&inf, 0, sizeof(inf));
    CHECK(gs_upload_ksplat(engine_of(env, a[0]), data, bytes, &o, &inf));
    napi_value out; napi_create_object(env, &out);
    napi_set_named_property(env, out, "splatCount", u32v(env, inf.splat_count));
    napi_set_named_property(env, out, "sphericalHarmonicsDegree", u32v(env, inf.sh_degree));
    napi_set_named_property(env, out, "compressionLevel", u32v(env, inf.compression_level));
    napi_set_named_property(env, out, "sectionCount", u32v(env, inf.section_count));
    napi_value c; napi_create_array_with_length(env, 3, &c);
    for (uint32_t i = 0; i < 3; ++i) napi_set_element(env, c, i, num(env, inf.scene_center[i]));
    napi_set_named_property(env, out, "sceneCenter", c);
    napi_set_named_property(env, out, "minSphericalHarmonicsCoeff", num(env, inf.min_sh_coeff));
    napi_set_named_property(env, out, "maxSphericalHarmonicsCoeff", num(env, inf.max_sh_coeff));
    return out;
}
FN(Render) {          // (engine, uniforms, renderParams, frameOutOrNull)
    ARGS(4)
    gs_uniforms u; fill_uniforms(env, a[1], &u);
    gs_render_params p; fill_render_params(env, a[2], &p);
    CHECK(gs_render(engine_of(env, a[0]), &u, &p, typed_ptr(env, a[3])));
    return undefined(env);
}
FN(Frame) {           // (engine, sortParams, uniforms, renderParams, sortedOutOrNull, frameOutOrNull)
    ARGS(6)
    gs_sort_params s; fill_sort_params(env, a[1], &s);
    gs_uniforms u; fill_uniforms(env, a[2], &u);
    gs_render_params p; fill_render_params(env, a[3], &p);
    CHECK(gs_frame(engine_of(env, a[0]), &s, &u, &p, (uint32_t *)typed_ptr(env, a[4]), typed_ptr(env, a[5])));
    return undefined(env);
}
FN(FrameAsync) {      // (engine, sortParams, uniforms, renderParams)
    ARGS(4)
    gs_sort_params s; fill_sort_params(env, a[1], &s);
    gs_uniforms u; fill_uniforms(env, a[2], &u);
    gs_render_params p; fill_render_params(env, a[3], &p);
    CHECK(gs_frame_async(engine_of(env, a[0]), &s, &u, &p));
    return undefined(env);
}
FN(FrameBegin) {      // (engine, sortParams, uniforms, renderParams, frameOut from hostAlloc)
    ARGS(5)
    gs_sort_params s; fill_sort_params(env, a[1], &s);
    gs_uniforms u; fill_uniforms(env, a[2], &u);
    gs_render_params p; fill_render_params(env, a[3], &p);
    CHECK(gs_frame_begin(engine_of(env, a[0]), &s, &u, &p, typed_ptr(env, a[4])));
    return undefined(env);
}
FN(FrameEnd) { ARGS(1) CHECK(gs_frame_end(engine_of(env, a[0]))); return undefined(env); }
FN(BufferDev) {       // (engine, bufferId) -> {ptr: BigInt, bytes}
    ARGS(2)
    void *p = nullptr; size_t b = 0;
    CHECK(gs_buffer_dev(engine_of(env, a[0]), to_i32(env, a[1]), &p, &b));
    napi_value out; napi_create_object(env, &out);
    napi_set_named_property(env, out, "ptr", ptr_value(env, p));
    napi_set_named_property(env, out, "bytes", num(env, (double)b));
    return out;
}
FN(ReadBuffer) {      // (engine, bufferId, outTypedArray, offsetBytes)
    ARGS(4)
    size_t bytes = 0; void *out = typed_ptr(env, a[2], &bytes);
    CHECK(gs_read_buffer(engine_of(env, a[0]), to_i32(env, a[1]), out, (size_t)to_f64(env, a[3]), bytes));
    return undefined(env);
}
FN(Stream) { ARGS(1) void *s = nullptr; CHECK(gs_stream(engine_of(env, a[0]), &s)); return ptr_value(env, s); }
FN(Synchronize) { ARGS(1) CHECK(gs_synchronize(engine_of(env, a[0]))); return undefined(env); }
static napi_value handle_pair(napi_env env, const unsigned char *h0, const unsigned char *h1) {
    napi_value out, b0, b1; void *d0, *d1;
    napi_create_object(env, &out);
    napi_create_arraybuffer(env, GS_IPC_HANDLE_BYTES, &d0, &b0); memcpy(d0, h0, GS_IPC_HANDLE_BYTES);
    napi_create_arraybuffer(env, GS_IPC_HANDLE_BYTES, &d1, &b1); memcpy(d1, h1, GS_IPC_HANDLE_BYTES);
    napi_set_named_property(env, out, "first", b0); napi_set_named_property(env, out, "second", b1);
    return out;
}
FN(PeerExport) { ARGS(1) unsigned char f[GS_IPC_HANDLE_BYTES], s[GS_IPC_HANDLE_BYTES]; CHECK(gs_peer_export(engine_of(env, a[0]), f, s)); return handle_pair(env, f, s); }   // {first: frame, second: sync}
FN(PeerAttach) { ARGS(3) CHECK(gs_peer_attach(engine_of(env, a[0]), typed_ptr(env, a[1]), typed_ptr(env, a[2]))); return undefined(env); }
FN(ShardExport) { ARGS(1) unsigned char b[GS_IPC_HANDLE_BYTES], s[GS_IPC_HANDLE_BYTES]; CHECK(gs_shard_export(engine_of(env, a[0]), b, s)); return handle_pair(env, b, s); } // {first: block, second: sorted}
FN(ShardAttach) { ARGS(4) CHECK(gs_shard_attach(engine_of(env, a[0]), to_u32(env, a[1]), typed_ptr(env, a[2]), typed_ptr(env, a[3]))); return undefined(env); }
FN(ShardAttachLocal) {   // (engine, [engines in rank order])
    ARGS(2)
    uint32_t n = 0; napi_get_array_length(env, a[1], &n);
    std::vector<gs_engine *> es(n);
    for (uint32_t i = 0; i < n; ++i) { napi_value e; napi_get_element(env, a[1], i, &e); es[i] = engine_of(env, e); }
    CHECK(gs_shard_attach_local(engine_of(env, a[0]), n, es.data()));
    return undefined(env);
}
FN(SortSharded) {
    ARGS(3)
    gs_sort_params p; fill_sort_params(env, a[1], &p);
    float ms = 0.f;
    CHECK(gs_sort_sharded(engine_of(env, a[0]), &p, (uint32_t *)typed_ptr(env, a[2]), &ms));
    napi_value out; napi_create_object(env, &out); napi_set_named_property(env, out, "sortTime", num(env, ms));
    return out;
}
FN(SortShardedAsync) { ARGS(2) gs_sort_params p; fill_sort_params(env, a[1], &p); CHECK(gs_sort_sharded_async(engine_of(env, a[0]), &p)); return undefined(env); }
FN(SortShardedFinish) {
    ARGS(2)
    float ms = 0.f;
    CHECK(gs_sort_sharded_finish(engine_of(env, a[0]), (uint32_t *)typed_ptr(env, a[1]), &ms));
    napi_value out; napi_create_object(env, &out); napi_set_named_property(env, out, "sortTime", num(env, ms));
    return out;
}
FN(HostAlloc) {       // (bytes) -> ArrayBuffer over page-locked memory (the SharedArrayBuffer views of SortWorker.js:180-191); freed with the buffer
    ARGS(1)
    const size_t bytes = (size_t)to_f64(env, a[0]);
    void *p = nullptr;
    CHECK(gs_host_alloc(&p, bytes));
    napi_value ab;
    if (napi_create_external_arraybuffer(env, p, bytes, [](napi_env, void *data, void *) { gs_host_free(data); }, nullptr, &ab) != napi_ok) { gs_host_free(p); napi_throw_error(env, nullptr, "napi_create_external_arraybuffer failed"); return nullptr; }
    return ab;
}
FN(HostFree) { ARGS(1) (void)a; return undefined(env); }   // host buffers are released by their ArrayBuffer's finalizer
FN(ReadProjected) {   // (engine, count) -> ArrayBuffer of gs_projected_splat records (48 bytes each)
    ARGS(2)
    const uint32_t n = to_u32(env, a[1]);
    void *data = nullptr; napi_value ab;
    napi_create_arraybuffer(env, (size_t)n * sizeof(gs_projected_splat), &data, &ab);
    CHECK(gs_read_projected(engine_of(env, a[0]), (gs_projected_splat *)data, n));
    return ab;
}
FN(ReadProjected2D) { // (engine, count) -> ArrayBuffer of gs_projected_surfel records (TwoD engines)
    ARGS(2)
    const uint32_t n = to_u32(env, a[1]);
    void *data = nullptr; napi_value ab;
    napi_create_arraybuffer(env, (size_t)n * sizeof(gs_projected_surfel), &data, &ab);
    CHECK(gs_read_projected_2d(engine_of(env, a[0]), (gs_projected_surfel *)data, n));
    return ab;
}
FN(LastTimings) {
    ARGS(1)
    gs_timings t; memset(&t, 0, sizeof(t));
    CHECK(gs_last_timings(engine_of(env, a[0]), &t));
    napi_value o; napi_create_object(env, &o);
    const struct { const char *k; double v; } f[] = {{"depthMs", t.depth_ms}, {"bucketMs", t.bucket_ms}, {"scatterMs", t.scatter_ms}, {"sortTotalMs", t.sort_total_ms}, {"projectMs", t.project_ms},
                                                     {"binMs", t.bin_ms}, {"blendMs", t.blend_ms}, {"renderTotalMs", t.render_total_ms}, {"h2dMs", t.h2d_ms}, {"d2hMs", t.d2h_ms},
                                                     {"tileInstances", (double)t.tile_instances}, {"kernelLaunches", (double)t.kernel_launches}, {"visibleSplats", (double)t.visible_splats}};
    for (const auto &kv : f) napi_set_named_property(env, o, kv.k, num(env, kv.v));
    return o;
}
FN(FlushL2) { ARGS(1) CHECK(gs_flush_l2(engine_of(env, a[0]))); return undefined(env); }
FN(SetProfiling) { ARGS(2) CHECK(gs_set_profiling(engine_of(env, a[0]), (int)to_u32(env, a[1]))); return undefined(env); }
FN(SetGraphEnabled) { ARGS(2) CHECK(gs_set_graph_enabled(engine_of(env, a[0]), (int)to_u32(env, a[1]))); return undefined(env); }
FN(KernelTimings) {   // (engine) -> [{name, ms}]
    ARGS(1)
    gs_kernel_time kt[64]; uint32_t n = 0;
    CHECK(gs_kernel_timings(engine_of(env, a[0]), kt, 64, &n));
    napi_value arr; napi_create_array_with_length(env, n < 64 ? n : 64, &arr);
    for (uint32_t i = 0; i < n && i < 64; ++i) {
        napi_value o; napi_create_object(env, &o);
        napi_set_named_property(env, o, "name", str(env, kt[i].name));
        napi_set_named_property(env, o, "ms", num(env, kt[i].ms));
        napi_set_element(env, arr, i, o);
    }
    return arr;
}
FN(EventCreate) { (void)info; void *ev = nullptr; CHECK(gs_event_create(&ev)); return ptr_value(env, ev); }
FN(EventRecord) { ARGS(2) CHECK(gs_event_record(engine_of(env, a[0]), ptr_of(env, a[1]))); return undefined(env); }
FN(EventElapsedMs) { ARGS(2) float ms = 0.f; CHECK(gs_event_elapsed_ms(ptr_of(env, a[0]), ptr_of(env, a[1]), &ms)); return num(env, ms); }
FN(EventDestroy) { ARGS(1) CHECK(gs_event_destroy(ptr_of(env, a[0]))); return undefined(env); }

static napi_value Init(napi_env env, napi_value exports) {
#define EXPORT(js, fn) {js, nullptr, fn, nullptr, nullptr, nullptr, napi_default, nullptr}
    const napi_property_descriptor d[] = {
        EXPORT("abiVersion", AbiVersion), EXPORT("statusString", StatusString), EXPORT("lastErrorMessage", LastErrorMessage), EXPORT("deviceCount", DeviceCount),
        EXPORT("sortIndexesChecked", SortIndexes), EXPORT("sortIndexes", SortIndexesVoid), EXPORT("dropinRelease", DropinRelease),
        EXPORT("create", Create), EXPORT("destroy", Destroy), EXPORT("uploadCenters", UploadCenters), EXPORT("sort", Sort),
        EXPORT("uploadSplatTree", UploadSplatTree), EXPORT("gatherForSort", GatherForSort), EXPORT("computeDistances", ComputeDistances),
        EXPORT("uploadSplatData", UploadSplatData), EXPORT("uploadKsplat", UploadKsplat), EXPORT("render", Render), EXPORT("frame", Frame),
        EXPORT("frameAsync", FrameAsync), EXPORT("frameBegin", FrameBegin), EXPORT("frameEnd", FrameEnd), EXPORT("bufferDev", BufferDev),
        EXPORT("readBuffer", ReadBuffer), EXPORT("stream", Stream), EXPORT("synchronize", Synchronize), EXPORT("peerExport", PeerExport),
        EXPORT("peerAttach", PeerAttach), EXPORT("shardExport", ShardExport), EXPORT("shardAttach", ShardAttach), EXPORT("shardAttachLocal", ShardAttachLocal),
        EXPORT("sortSharded", SortSharded), EXPORT("sortShardedAsync", SortShardedAsync), EXPORT("sortShardedFinish", SortShardedFinish),
        EXPORT("hostAlloc", HostAlloc), EXPORT("hostFree", HostFree), EXPORT("readProjected", ReadProjected), EXPORT("readProjected2D", ReadProjected2D), EXPORT("lastTimings", LastTimings),
        EXPORT("flushL2", FlushL2), EXPORT("setProfiling", SetProfiling), EXPORT("setGraphEnabled", SetGraphEnabled), EXPORT("kernelTimings", KernelTimings),
        EXPORT("eventCreate", EventCreate), EXPORT("eventRecord", EventRecord), EXPORT("eventElapsedMs", EventElapsedMs), EXPORT("eventDestroy", EventDestroy),
    };
#undef EXPORT
    napi_define_properties(env, exports, sizeof(d) / sizeof(d[0]), d);
    return exports;
}
NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
