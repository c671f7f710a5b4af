/* oracle/surfel_oracle.c -- TEST INFRASTRUCTURE ONLY (never linked into or called by the product path).
 *
 * CPU restatement of the reference's 2D Gaussian (surfel) material, SplatRenderMode.TwoD, evaluated per splat in draw order:
 *   vertex base  : src/splatmesh/SplatMaterial.js:112-341 (fetch, transform, cull, colour + SH) -- as raster_oracle.c's 3D path
 *   projection   : src/splatmesh/SplatMaterial2D.js:96-127 (L = R S, T = transpose(splat2World) * world2ndc * ndc2pix)
 *   quad         : SplatMaterial2D.js:199-235 (eigen-aligned parallelogram) and :159-189 (AABB square when a basis vector is < 1 px)
 *   fade-in      : SplatMaterial.js:347-363
 *   fragment     : SplatMaterial2D.js:302-343 (ray-surfel intersection, min(rho3d, rho2d), near test, alpha cut-off)
 *   blend        : NormalBlending, as in 3D
 * GLSL matrices are column-major; `mat3x4` has 3 columns of 4 rows.  Every product below is written out left to right in f32,
 * unfused (-ffp-contract=off).  Coverage: a fragment exists for every pixel whose centre lies inside the rasterised quad; the
 * fragment shader has no discard tied to the quad, so the quad boundary clips the surfel.
 * Pinned by an independent formulation (oracle/surfel_independent.py, tests/test_surfel_oracle.py).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "../include/gsplat_b200.h"

#define GS_ORACLE_API __attribute__((visibility("default")))

static inline float clamp01(float v) { return v < 0.f ? 0.f : (v > 1.f ? 1.f : v); }

static void mat4_mul(const float *a, const float *b, float *o) { /* o = a*b, column-major */
    for (int c = 0; c < 4; ++c)
        for (int r = 0; r < 4; ++r)
            o[4 * c + r] = a[r] * b[4 * c] + a[4 + r] * b[4 * c + 1] + a[8 + r] * b[4 * c + 2] + a[12 + r] * b[4 * c + 3];
}
static void mat4_mul_vec4(const float *m, const float v[4], float out[4]) {
    for (int r = 0; r < 4; ++r) out[r] = m[r] * v[0] + m[4 + r] * v[1] + m[8 + r] * v[2] + m[12 + r] * v[3];
}
static void mat4_inverse(const float *m, float *o) {
    float inv[16];
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const float det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    const float id = 1.0f / det;
    for (int i = 0; i < 16; ++i) o[i] = inv[i] * id;
}
static float half_to_float(uint16_t h) {
    uint32_t s = (uint32_t)(h >> 15) << 31, e = (h >> 10) & 31u, m = h & 1023u, bits;
    if (e == 0) {
        if (m == 0) bits = s;
        else {
            int sh = 0;
            while (!(m & 1024u)) { m <<= 1; ++sh; }
            m &= 1023u;
            bits = s | ((uint32_t)(127 - 15 - sh + 1) << 23) | (m << 13);
        }
    } else if (e == 31) bits = s | 0x7f800000u | (m << 13);
    else bits = s | ((e + 112u) << 23) | (m << 13);
    float f;
    memcpy(&f, &bits, 4);
    return f;
}

static void project_one(const gs_uniforms *u, const gs_splat_data *d, uint32_t s, gs_projected_surfel *o) {
    memset(o, 0, sizeof(*o));
    const uint32_t *cc = d->centers_colors + 4 * (size_t)s;
    float c[3];
    memcpy(c, cc + 1, 12);
    uint32_t scene = 0;
    if (u->scene_count > 1 && d->scene_indexes) scene = d->scene_indexes[s];
    if (u->enable_optional_effects && (u->scene_opacity[scene] <= 0.01f || u->scene_visibility[scene] == 0)) return; /* :129-137 */
    float mv_dyn[16];
    const float *mv = u->model_view; /* transformModelViewMatrix */
    if (u->dynamic_mode) { mat4_mul(u->view_matrix, u->scene_transforms + 16 * scene, mv_dyn); mv = mv_dyn; }
    const float c4[4] = {c[0], c[1], c[2], 1.0f};
    float view[4], clip[4];
    mat4_mul_vec4(mv, c4, view);
    mat4_mul_vec4(u->projection, view, clip);
    const float lim = 1.2f * clip[3]; /* :158-164 */
    if (clip[2] < -lim || clip[0] < -lim || clip[0] > lim || clip[1] < -lim || clip[1] > lim) return;
    const float ndc[3] = {clip[0] / clip[3], clip[1] / clip[3], clip[2] / clip[3]};
    float col[4];
    for (int k = 0; k < 4; ++k) col[k] = (float)((cc[0] >> (8 * k)) & 255u) * (1.0f / 255.0f);
    if (d->sh_degree >= 1 && u->sh_degree >= 1 && d->spherical_harmonics) { /* :173-341 */
        const uint32_t ncomp = d->sh_degree >= 2 ? 24u : 9u;
        float sh[24];
        const float lo = u->sh8_min[scene], range = u->sh8_max[scene] - u->sh8_min[scene];
        for (uint32_t k = 0; k < ncomp; ++k) {
            const size_t at = (size_t)s * ncomp + k;
            if (d->sh_format == GS_SH_F16) sh[k] = half_to_float(((const uint16_t *)d->spherical_harmonics)[at]);
            else if (d->sh_format == GS_SH_U8) sh[k] = ((float)((const uint8_t *)d->spherical_harmonics)[at] / 255.0f) * range + lo;
            else sh[k] = ((const float *)d->spherical_harmonics)[at];
        }
        float cam[3] = {u->camera_position[0], u->camera_position[1], u->camera_position[2]};
        if (u->dynamic_mode) {
            float inv[16], cp[4];
            const float cam4[4] = {cam[0], cam[1], cam[2], 1.0f};
            mat4_inverse(u->scene_transforms + 16 * scene, inv);
            mat4_mul_vec4(inv, cam4, cp);
            cam[0] = cp[0]; cam[1] = cp[1]; cam[2] = cp[2];
        }
        const float dir[3] = {c[0] - cam[0], c[1] - cam[1], c[2] - cam[2]};
        const float il = 1.0f / sqrtf(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
        const float x = dir[0] * il, y = dir[1] * il, z = dir[2] * il;
        const float C1 = 0.4886025119029199f;
        for (int ch = 0; ch < 3; ++ch) col[ch] += C1 * (-sh[0 + ch] * y + sh[3 + ch] * z - sh[6 + ch] * x);
        if (d->sh_degree >= 2 && u->sh_degree >= 2) {
            const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
            for (int ch = 0; ch < 3; ++ch)
                col[ch] += (1.0925484f * xy) * sh[9 + ch] + (-1.0925484f * yz) * sh[12 + ch] + (0.3153916f * (2.0f * zz - xx - yy)) * sh[15 + ch] +
                           (-1.0925484f * xz) * sh[18 + ch] + (0.5462742f * (xx - yy)) * sh[21 + ch];
        }
        for (int ch = 0; ch < 3; ++ch) col[ch] = clamp01(col[ch]);
    }
    /* ---- SplatMaterial2D.js:96-127 ---- */
    const float *sr = d->scale_rotations + 6 * (size_t)s;
    const float qx = sr[3], qy = sr[4], qz = sr[5];
    const float qw = sqrtf(1.0f - qx * qx - qy * qy - qz * qz); /* missingW */
    /* quaternionToRotationMatrix (SplatMaterial.js:64-78): columns */
    const float R[3][3] = {{1.f - 2.f * (qy * qy + qz * qz), 2.f * (qx * qy + qw * qz), 2.f * (qx * qz - qw * qy)},
                           {2.f * (qx * qy - qw * qz), 1.f - 2.f * (qx * qx + qz * qz), 2.f * (qy * qz + qw * qx)},
                           {2.f * (qx * qz + qw * qy), 2.f * (qy * qz - qw * qx), 1.f - 2.f * (qx * qx + qy * qy)}};
    const float S[3] = {sr[0], sr[1], sr[2]};
    float L[3][3]; /* L = R * S: column j = sum_k R[k] * S[j][k] (S diagonal) */
    for (int j = 0; j < 3; ++j)
        for (int r = 0; r < 3; ++r) L[j][r] = R[0][r] * (j == 0 ? S[0] : 0.f) + R[1][r] * (j == 1 ? S[1] : 0.f) + R[2][r] * (j == 2 ? S[2] : 0.f);
    /* world2ndc = transpose(projectionMatrix * transformModelViewMatrix) */
    float PMV[16];
    mat4_mul(u->projection, mv, PMV);
    /* transpose(splat2World) * world2ndc: row i = splat2World column i times world2ndc = (PMV * a_i)^T, a_0 = (L0,0), a_1 = (L1,0),
       a_2 = (centre,1) -- written as the GLSL sum over k of a_i[k] * world2ndc[j][k] with world2ndc[j][k] = PMV[k][j] */
    const float a[3][4] = {{L[0][0], L[0][1], L[0][2], 0.f}, {L[1][0], L[1][1], L[1][2], 0.f}, {c[0], c[1], c[2], 1.f}};
    float SW[3][4];   /* SW[i][j]: row i, column j */
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 4; ++j) SW[i][j] = a[i][0] * PMV[0 * 4 + j] + a[i][1] * PMV[1 * 4 + j] + a[i][2] * PMV[2 * 4 + j] + a[i][3] * PMV[3 * 4 + j];
    const float W = u->viewport[0], H = u->viewport[1];
    /* ndc2pix = mat3x4(vec4(W/2, 0, 0, (W-1)/2), vec4(0, H/2, 0, (H-1)/2), vec4(0, 0, 0, 1)): N[col][row] */
    const float N[3][4] = {{W / 2.0f, 0.f, 0.f, (W - 1.0f) / 2.0f}, {0.f, H / 2.0f, 0.f, (H - 1.0f) / 2.0f}, {0.f, 0.f, 0.f, 1.0f}};
    float T[3][3];    /* T[col][row] (GLSL): T[col j][row i] = sum_k SW[i][k] * N[j][k] */
    for (int j = 0; j < 3; ++j)
        for (int i = 0; i < 3; ++i) T[j][i] = SW[i][0] * N[j][0] + SW[i][1] * N[j][1] + SW[i][2] * N[j][2] + SW[i][3] * N[j][3];
    for (int j = 0; j < 3; ++j)
        for (int i = 0; i < 3; ++i) o->T[3 * j + i] = T[j][i];
    /* ---- eigen quad (:199-235) ---- */
    const float S4[4][4] = {{L[0][0], L[0][1], L[0][2], 0.f}, {L[1][0], L[1][1], L[1][2], 0.f}, {L[2][0], L[2][1], L[2][2], 0.f}, {c[0], c[1], c[2], 1.f}};
    float Tt[16];   /* transpose(transpose(splat2World4) * world2ndc) = PMV * splat2World4 */
    mat4_mul(PMV, &S4[0][0], Tt);
    const float e1[4] = {1.f, 0.f, 0.f, 1.f}, e2[4] = {0.f, 1.f, 0.f, 1.f}, e0[4] = {0.f, 0.f, 0.f, 1.f};
    float t1[4], t2[4], ce[4];
    mat4_mul_vec4(Tt, e1, t1); mat4_mul_vec4(Tt, e2, t2); mat4_mul_vec4(Tt, e0, ce);
    { const float w1 = t1[3], w2 = t2[3], w0 = ce[3]; for (int k = 0; k < 4; ++k) { t1[k] = t1[k] / w1; t2[k] = t2[k] / w2; ce[k] = ce[k] / w0; } }   /* tempPoint /= tempPoint.w */
    const float b1[2] = {t1[0] - ce[0], t1[1] - ce[1]}, b2[2] = {t2[0] - ce[0], t2[1] - ce[1]};
    const float b1s[2] = {b1[0] * 0.5f * W, b1[1] * 0.5f * H}, b2s[2] = {b2[0] * 0.5f * W, b2[1] * 0.5f * H};
    const float minPix = 1.f;
    const float cpx = (ndc[0] * 0.5f + 0.5f) * W, cpy = (ndc[1] * 0.5f + 0.5f) * H;   /* quad centre: ndcCenter in window pixels */
    int drawn = 1;
    if (sqrtf(b1s[0] * b1s[0] + b1s[1] * b1s[1]) < minPix || sqrtf(b2s[0] * b2s[0] + b2s[1] * b2s[1]) < minPix) {
        /* reference-implementation AABB square (:159-189) */
        const float T0[3] = {T[0][0], T[0][1], T[0][2]}, T1[3] = {T[1][0], T[1][1], T[1][2]}, T3[3] = {T[2][0], T[2][1], T[2][2]};
        const float tp[3] = {1.0f, 1.0f, -1.0f};
        const float distance = (T3[0] * T3[0] * tp[0]) + (T3[1] * T3[1] * tp[1]) + (T3[2] * T3[2] * tp[2]);
        const float f[3] = {(1.0f / distance) * tp[0], (1.0f / distance) * tp[1], (1.0f / distance) * tp[2]};
        if (fabsf(distance) < 0.00001f) drawn = 0;   /* `return` with gl_Position unset: dropped */
        const float pix = (T0[0] * T3[0] * f[0]) + (T0[1] * T3[1] * f[1]) + (T0[2] * T3[2] * f[2]);
        const float piy = (T1[0] * T3[0] * f[0]) + (T1[1] * T3[1] * f[1]) + (T1[2] * T3[2] * f[2]);
        const float tx = (T0[0] * T0[0] * f[0]) + (T0[1] * T0[1] * f[1]) + (T0[2] * T0[2] * f[2]);
        const float ty = (T1[0] * T1[0] * f[0]) + (T1[1] * T1[1] * f[1]) + (T1[2] * T1[2] * f[2]);
        const float hx = pix * pix - tx, hy = piy * piy - ty;
        const float ex = sqrtf(hx > 0.0001f ? hx : 0.0001f), ey = sqrtf(hy > 0.0001f ? hy : 0.0001f);
        const float radius = ex > ey ? ex : ey;
        /* ndcOffset = (position * radius * 3) * basisViewport * 2 -> pixels: position * radius * 3 */
        o->h1x = radius * 3.0f; o->h1y = 0.f; o->h2x = 0.f; o->h2y = radius * 3.0f;
        o->qcx = pix; o->qcy = piy;
        o->branch = 1;
    } else {
        /* ndcOffset = (position.x * b1 + position.y * b2) * 3 * inverseFocalAdjustment -> pixels: * viewport / 2 */
        const float k = 3.0f * u->inverse_focal_adjustment;
        o->h1x = b1[0] * k * 0.5f * W; o->h1y = b1[1] * k * 0.5f * H;
        o->h2x = b2[0] * k * 0.5f * W; o->h2y = b2[1] * k * 0.5f * H;
        o->qcx = ce[0]; o->qcy = ce[1];   /* vQuadCenter = center.xy: NDC units */
        o->branch = 0;
    }
    if (!u->fade_in_complete) {
        const float dx = c[0] - u->scene_center[0], dy = c[1] - u->scene_center[1], dz = c[2] - u->scene_center[2];
        const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
        const float st = dist >= u->visible_region_fade_start_radius ? 1.0f : 0.0f;
        col[3] *= (1.0f - st) + (1.0f - clamp01((dist - u->visible_region_fade_start_radius) / 0.75f)) * st;
    }
    o->cx = cpx; o->cy = cpy;
    o->r = col[0]; o->g = col[1]; o->b = col[2]; o->a = col[3];
    o->ndc_z = ndc[2];
    o->valid = (drawn && ndc[2] >= -1.0f && ndc[2] <= 1.0f) ? 1u : 0u;
}

GS_ORACLE_API void gso_project_2d(const gs_uniforms *u, const gs_splat_data *d, gs_projected_surfel *out) {
#pragma omp parallel for schedule(static)
    for (int64_t s = 0; s < (int64_t)d->count; ++s) project_one(u, d, (uint32_t)s, out + s);
}

/* fragment shader (SplatMaterial2D.js:302-343) at pixel centre (fx, fy); returns alpha or -1 for discard */
static float fragment(const gs_projected_surfel *p, float fx, float fy) {
    const float FilterInvSquare = 2.0f, near_n = 0.2f;
    const float *Tu = p->T, *Tv = p->T + 3, *Tw = p->T + 6;
    const float k[3] = {fx * Tw[0] - Tu[0], fx * Tw[1] - Tu[1], fx * Tw[2] - Tu[2]};
    const float l[3] = {fy * Tw[0] - Tv[0], fy * Tw[1] - Tv[1], fy * Tw[2] - Tv[2]};
    const float pp[3] = {k[1] * l[2] - k[2] * l[1], k[2] * l[0] - k[0] * l[2], k[0] * l[1] - k[1] * l[0]};
    if (pp[2] == 0.0f) return -1.f;
    const float sx = pp[0] / pp[2], sy = pp[1] / pp[2];
    const float rho3d = (sx * sx + sy * sy);
    const float dx = p->qcx - fx, dy = p->qcy - fy;
    const float rho2d = FilterInvSquare * (dx * dx + dy * dy);
    const float rho = rho3d < rho2d ? rho3d : rho2d;
    const float depth = (rho3d <= rho2d) ? (sx * Tw[0] + sy * Tw[1]) + Tw[2] : Tw[2];
    if (depth < near_n) return -1.f;
    const float power = -0.5f * rho;
    if (power > 0.0f) return -1.f;
    float alpha = p->a * expf(power);
    if (alpha > 0.99f) alpha = 0.99f;
    if (!(alpha >= 1.0f / 255.0f)) return -1.f;   /* also a NaN alpha (undefined in GLSL: sqrt of a negative missingW) */
    if (1.0f - alpha < 0.0001f) return -1.f;
    return alpha;
}

static void blend_region(const gs_projected_surfel *ps, const uint32_t *order, uint32_t n, uint32_t cx0, uint32_t cy0, uint32_t cw, uint32_t ch, float *frame) {
    memset(frame, 0, (size_t)cw * ch * 4 * sizeof(float));
    const int band = 8, nbands = ((int)ch + band - 1) / band;
#pragma omp parallel for schedule(dynamic, 1)
    for (int bi = 0; bi < nbands; ++bi) {
        const int y0 = (int)cy0 + bi * band, y1 = (y0 + band < (int)(cy0 + ch) ? y0 + band : (int)(cy0 + ch)) - 1;
        for (uint32_t i = 0; i < n; ++i) {
            const gs_projected_surfel *p = ps + order[i];
            if (!p->valid) continue;
            const float ex = fabsf(p->h1x) + fabsf(p->h2x), ey = fabsf(p->h1y) + fabsf(p->h2y);
            float fy0 = floorf(p->cy - ey - 1.0f), fy1 = ceilf(p->cy + ey + 1.0f), fx0 = floorf(p->cx - ex - 1.0f), fx1 = ceilf(p->cx + ex + 1.0f);
            if (fy0 < (float)y0) fy0 = (float)y0;
            if (fy1 > (float)y1) fy1 = (float)y1;
            if (fx0 < (float)cx0) fx0 = (float)cx0;
            if (fx1 > (float)(cx0 + cw) - 1.f) fx1 = (float)(cx0 + cw) - 1.f;
            if (!(fy0 <= fy1) || !(fx0 <= fx1)) continue;
            /* inside test: pixel centre = c + u h1 + v h2 with |u|, |v| <= 1 */
            const float det = p->h1x * p->h2y - p->h2x * p->h1y;
            if (!(det != 0.0f)) continue;
            for (int y = (int)fy0; y <= (int)fy1; ++y) {
                for (int x = (int)fx0; x <= (int)fx1; ++x) {
                    const float fx = (float)x + 0.5f, fy = (float)y + 0.5f;
                    const float dx = fx - p->cx, dy = fy - p->cy;
                    const float uu = (dx * p->h2y - dy * p->h2x) / det, vv = (dy * p->h1x - dx * p->h1y) / det;
                    if (!(fabsf(uu) <= 1.0f && fabsf(vv) <= 1.0f)) continue;
                    const float alpha = fragment(p, fx, fy);
                    if (alpha < 0.f) continue;
                    float *px = frame + ((size_t)(y - (int)cy0) * cw + (size_t)(x - (int)cx0)) * 4;
                    const float om = 1.0f - alpha;
                    px[0] = p->r * alpha + px[0] * om;
                    px[1] = p->g * alpha + px[1] * om;
                    px[2] = p->b * alpha + px[2] * om;
                    px[3] = alpha + px[3] * om;
                }
            }
        }
    }
}

/* Blend in draw order (order[0] first = farthest) into a float RGBA frame, rows bottom-up (GL window coordinates). */
GS_ORACLE_API void gso_blend_2d(const gs_projected_surfel *ps, const uint32_t *order, uint32_t n, uint32_t width, uint32_t height, float *frame) {
    blend_region(ps, order, n, 0, 0, width, height, frame);
}
/* The window [cx0, cx0+cw) x [cy0, cy0+ch) of that frame. */
GS_ORACLE_API void gso_blend_2d_crop(const gs_projected_surfel *ps, const uint32_t *order, uint32_t n, uint32_t width, uint32_t height,
                                     uint32_t cx0, uint32_t cy0, uint32_t cw, uint32_t ch, float *frame) {
    (void)width; (void)height;
    blend_region(ps, order, n, cx0, cy0, cw, ch, frame);
}
