// surfel_kernels.cuh -- the 2D Gaussian (surfel) render mode, SplatRenderMode.TwoD (sm_100a):
//   k_project2d : vertex stage once per splat        SplatMaterial.js:112-341 (shared base), SplatMaterial2D.js:96-235
//   k_blend2d   : fragment stage + blend             SplatMaterial2D.js:302-343, NormalBlending as in 3D
// Everything between the two (depth sort, counting-sort binning, sharded ownership, subset compaction, peer gather) is the 3D
// path unchanged: k_project2d writes the same ushort4 fine-tile rect, from the AABB of the surfel's screen quad.
//
// Per pixel the reference evaluates k = x Tw - Tu, l = y Tw - Tv, p = k x l.  Since Tw x Tw = 0 this is exactly
//   p(x, y) = x (Tv x Tw) + y (Tw x Tu) + (Tu x Tv),
// linear in the pixel.  The record keeps it relative to the quad centre c: p = dx A + dy B + C with A = Tv x Tw, B = Tw x Tu and
// C = k(c) x l(c), so the per-pixel terms stay small (no cancellation of ~1e4-sized products at far-from-origin pixels).
// Included by raster_kernels.cuh ahead of the rasteriser's host side (which launches these kernels).
#pragma once
#include "raster_kernels.cuh"

namespace gs {

struct __align__(16) SurfelRecord {    // 96 bytes, read as 6 x 16 B
    float cx, cy;                      // quad centre, pixels, GL window coordinates
    float m00, m01, m10, m11;          // inverse of the quad's edge map [h1 h2]: (u, v) = m (p - c), inside <=> |u|, |v| <= 1
    float qx, qy;                      // vQuadCenter - c
    float ax, ay, az, bx, by, bz;      // A = Tv x Tw, B = Tw x Tu
    float kx, ky, kz;                  // C = k(c) x l(c)
    float twx, twy, twz;               // Tw: depth = s . Tw.xy + Tw.z
    float r, g, b, a;
};
static_assert(sizeof(SurfelRecord) == 96, "SurfelRecord is staged as six float4");

// column-major o = a * b with GLSL's left-to-right sums, unfused
__device__ __forceinline__ void mat4_mul_rn(const float *a, const float *b, float *o) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int r = 0; r < 4; ++r)
            o[4 * c + r] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a[r], b[4 * c]), __fmul_rn(a[4 + r], b[4 * c + 1])), __fmul_rn(a[8 + r], b[4 * c + 2])),
                                     __fmul_rn(a[12 + r], b[4 * c + 3]));
}

__device__ __forceinline__ void cross3(const float *u, const float *v, float *o) {
    o[0] = u[1] * v[2] - u[2] * v[1];
    o[1] = u[2] * v[0] - u[0] * v[2];
    o[2] = u[0] * v[1] - u[1] * v[0];
}

// ---------------------------------------------------------------------------------------------------------------
// Projection: one thread per splat.  EXPORT additionally writes the ABI's gs_projected_surfel (gs_read_projected_2d).
template <int SHFMT, bool EXPORT>
__global__ void __launch_bounds__(kProjThreads)
k_project2d(const uint4 *__restrict__ cc, const float *__restrict__ srot, const void *__restrict__ sh, int sh_data_degree,
            const uint32_t *__restrict__ scene_idx, const DynamicUniforms *__restrict__ dyn, const ProjParams *__restrict__ Pp, uint32_t count,
            SurfelRecord *__restrict__ rec, ushort4 *__restrict__ rects, RasterControl *rctl, gs_projected_surfel *__restrict__ exp) {
    pdl_enter();
    __shared__ ProjParams s_P;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(Pp);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&s_P);
        for (int i = threadIdx.x; i < (int)(sizeof(ProjParams) / 4); i += kProjThreads) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    const ProjParams &P = s_P;
    const uint32_t s = blockIdx.x * kProjThreads + threadIdx.x;
    uint32_t visible = 0;
    if (s < count) {
        SurfelRecord o;
        float *of = reinterpret_cast<float *>(&o);
#pragma unroll
        for (int k = 0; k < 24; ++k) of[k] = 0.f;
        gs_projected_surfel xo{};
        ushort4 rect = make_ushort4(1, 1, 0, 0);   // empty
        const int4 c4 = ld_nc_v4(cc + s);
        const float2 *sr2 = reinterpret_cast<const float2 *>(srot) + (size_t)s * 3;
        const float2 sr0 = __ldg(sr2), sr1 = __ldg(sr2 + 1), sr3 = __ldg(sr2 + 2);   // sx sy | sz qx | qy qz
        const float cx = __int_as_float(c4.y), cy = __int_as_float(c4.z), cz = __int_as_float(c4.w);
        uint32_t scene = 0;
        if (P.scene_count > 1 && scene_idx) scene = scene_idx[s] & (GS_MAX_SCENES_DEV - 1);
        // SplatMaterial.js:129-137: optional effects cull invisible scenes; scene opacity itself is a 3D-material effect only
        bool alive = true;
        if (P.optional_effects) alive = !(dyn->opacity[scene] <= 0.01f || dyn->visibility[scene] == 0);
        float mvd[16];
        const float *mv = P.mv;
        if (P.dynamic) { mat4_mul_dev(dyn->view, dyn->transforms + 16 * scene, mvd); mv = mvd; }
        float view[4], clip[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) view[r] = mv[r] * cx + mv[4 + r] * cy + mv[8 + r] * cz + mv[12 + r];
#pragma unroll
        for (int r = 0; r < 4; ++r) clip[r] = P.proj[r] * view[0] + P.proj[4 + r] * view[1] + P.proj[8 + r] * view[2] + P.proj[12 + r] * view[3];
        const float lim = 1.2f * clip[3];
        if (clip[2] < -lim || clip[0] < -lim || clip[0] > lim || clip[1] < -lim || clip[1] > lim) alive = false;
        if (alive) {
            const float iw = 1.0f / clip[3];
            const float ndcx = clip[0] * iw, ndcy = clip[1] * iw, ndcz = clip[2] * iw;
            const uint32_t packed = (uint32_t)c4.x;
            float col[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) col[k] = (float)((packed >> (8 * k)) & 255u) * (1.0f / 255.0f);
            if (SHFMT != GS_SH_NONE && sh_data_degree >= 1 && P.sh_degree >= 1) {   // SplatMaterial.js:173-341
                const int ncomp = sh_data_degree >= 2 ? 24 : 9;
                const int nuse = (sh_data_degree >= 2 && P.sh_degree >= 2) ? 24 : 9;
                float shv[24];
                if (SHFMT == GS_SH_F16) {
                    const __half *h = (const __half *)sh + (size_t)s * ncomp;
                    for (int k = 0; k < nuse; ++k) shv[k] = __half2float(h[k]);
                } else if (SHFMT == GS_SH_U8) {
                    const unsigned char *b = (const unsigned char *)sh + (size_t)s * ncomp;
                    const float lo = dyn->sh8_min[scene], range = dyn->sh8_max[scene] - dyn->sh8_min[scene];
                    for (int k = 0; k < nuse; ++k) shv[k] = ((float)b[k] / 255.0f) * range + lo;
                } else {
                    const float *f = (const float *)sh + (size_t)s * ncomp;
                    for (int k = 0; k < nuse; ++k) shv[k] = f[k];
                }
                float camx = P.cam[0], camy = P.cam[1], camz = P.cam[2];
                if (P.dynamic) {
                    float inv[16];
                    mat4_inverse_dev(dyn->transforms + 16 * scene, inv);
                    const float tx = inv[0] * camx + inv[4] * camy + inv[8] * camz + inv[12];
                    const float ty = inv[1] * camx + inv[5] * camy + inv[9] * camz + inv[13];
                    const float tz = inv[2] * camx + inv[6] * camy + inv[10] * camz + inv[14];
                    camx = tx; camy = ty; camz = tz;
                }
                const float dx = cx - camx, dy = cy - camy, dz = cz - camz;
                const float il = rsqrtf(dx * dx + dy * dy + dz * dz);
                const float x = dx * il, y = dy * il, z = dz * il;
                const float C1 = 0.4886025119029199f;
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) col[ch] += C1 * (-shv[ch] * y + shv[3 + ch] * z - shv[6 + ch] * x);
                if (nuse == 24) {
                    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch)
                        col[ch] += (1.0925484f * xy) * shv[9 + ch] + (-1.0925484f * yz) * shv[12 + ch] +
                                   (0.3153916f * (2.0f * zz - xx - yy)) * shv[15 + ch] + (-1.0925484f * xz) * shv[18 + ch] +
                                   (0.5462742f * (xx - yy)) * shv[21 + ch];
                }
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) col[ch] = __saturatef(col[ch]);
            }
            // ---- SplatMaterial2D.js:96-235 in the shader's own f32 operation order, unfused (__f*_rn): the fallback square's
            // pointImage^2 - temp cancels terms of ~1e6 px^2 down to ~1 px^2, so any other rounding of T would move a sub-pixel
            // surfel's square edge by whole percent (and flip the coverage of pixels it clips at high alpha)
            const float qx = sr1.y, qy = sr3.x, qz = sr3.y;
            const float qw = __fsqrt_rn(__fsub_rn(__fsub_rn(__fsub_rn(1.0f, __fmul_rn(qx, qx)), __fmul_rn(qy, qy)), __fmul_rn(qz, qz)));
            float R[3][3];       // quaternionToRotationMatrix (SplatMaterial.js:64-78), R[column][row]
            R[0][0] = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(__fmul_rn(qy, qy), __fmul_rn(qz, qz))));
            R[0][1] = __fmul_rn(2.f, __fadd_rn(__fmul_rn(qx, qy), __fmul_rn(qw, qz)));
            R[0][2] = __fmul_rn(2.f, __fsub_rn(__fmul_rn(qx, qz), __fmul_rn(qw, qy)));
            R[1][0] = __fmul_rn(2.f, __fsub_rn(__fmul_rn(qx, qy), __fmul_rn(qw, qz)));
            R[1][1] = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(__fmul_rn(qx, qx), __fmul_rn(qz, qz))));
            R[1][2] = __fmul_rn(2.f, __fadd_rn(__fmul_rn(qy, qz), __fmul_rn(qw, qx)));
            R[2][0] = __fmul_rn(2.f, __fadd_rn(__fmul_rn(qx, qz), __fmul_rn(qw, qy)));
            R[2][1] = __fmul_rn(2.f, __fsub_rn(__fmul_rn(qy, qz), __fmul_rn(qw, qx)));
            R[2][2] = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(__fmul_rn(qx, qx), __fmul_rn(qy, qy))));
            const float Sd[3] = {sr0.x, sr0.y, sr1.x};
            float L[3][3];       // L = R * S (column j = sum_k R[k] * S[j][k], zero terms included)
#pragma unroll
            for (int j = 0; j < 3; ++j)
#pragma unroll
                for (int r = 0; r < 3; ++r)
                    L[j][r] = __fadd_rn(__fadd_rn(__fmul_rn(R[0][r], j == 0 ? Sd[0] : 0.f), __fmul_rn(R[1][r], j == 1 ? Sd[1] : 0.f)), __fmul_rn(R[2][r], j == 2 ? Sd[2] : 0.f));
            float mvr[16], pmv[16];
            const float *mvx = P.mv;
            if (P.dynamic) { mat4_mul_rn(dyn->view, dyn->transforms + 16 * scene, mvr); mvx = mvr; }
            mat4_mul_rn(P.proj, mvx, pmv);                 // world2ndc = transpose(projectionMatrix * transformModelViewMatrix)
            const float av[3][4] = {{L[0][0], L[0][1], L[0][2], 0.f}, {L[1][0], L[1][1], L[1][2], 0.f}, {cx, cy, cz, 1.f}};
            float SW[3][4];      // transpose(splat2World) * world2ndc
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    SW[i][j] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(av[i][0], pmv[j]), __fmul_rn(av[i][1], pmv[4 + j])), __fmul_rn(av[i][2], pmv[8 + j])), __fmul_rn(av[i][3], pmv[12 + j]));
            const float W = P.viewport[0], H = P.viewport[1];
            const float Nm[3][4] = {{W / 2.0f, 0.f, 0.f, (W - 1.0f) / 2.0f}, {0.f, H / 2.0f, 0.f, (H - 1.0f) / 2.0f}, {0.f, 0.f, 0.f, 1.0f}};
            float T[3][3];       // T[column][row]: Tu = T[0], Tv = T[1], Tw = T[2]
#pragma unroll
            for (int j = 0; j < 3; ++j)
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    T[j][i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(SW[i][0], Nm[j][0]), __fmul_rn(SW[i][1], Nm[j][1])), __fmul_rn(SW[i][2], Nm[j][2])), __fmul_rn(SW[i][3], Nm[j][3]));
            const float *Tu = T[0], *Tv = T[1], *Tw = T[2];
            // eigen quad: Tt = transpose(transpose(splat2World4) * world2ndc) = PMV * splat2World4; tempPoint = Tt * (e, 1) / w
            const float S4[16] = {L[0][0], L[0][1], L[0][2], 0.f, L[1][0], L[1][1], L[1][2], 0.f, L[2][0], L[2][1], L[2][2], 0.f, cx, cy, cz, 1.f};
            float Tt[16];
            mat4_mul_rn(pmv, S4, Tt);
            auto tp = [&](float e0, float e1, int r) {     // (Tt * (e0, e1, 0, 1))[r]
                return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(Tt[r], e0), __fmul_rn(Tt[4 + r], e1)), __fmul_rn(Tt[8 + r], 0.f)), __fmul_rn(Tt[12 + r], 1.f));
            };
            const float w1 = tp(1.f, 0.f, 3), w2 = tp(0.f, 1.f, 3), w0 = tp(0.f, 0.f, 3);
            const float ncx = __fdiv_rn(tp(0.f, 0.f, 0), w0), ncy = __fdiv_rn(tp(0.f, 0.f, 1), w0);
            const float b1x = __fsub_rn(__fdiv_rn(tp(1.f, 0.f, 0), w1), ncx), b1y = __fsub_rn(__fdiv_rn(tp(1.f, 0.f, 1), w1), ncy);
            const float b2x = __fsub_rn(__fdiv_rn(tp(0.f, 1.f, 0), w2), ncx), b2y = __fsub_rn(__fdiv_rn(tp(0.f, 1.f, 1), w2), ncy);
            const float s1x = __fmul_rn(__fmul_rn(b1x, 0.5f), W), s1y = __fmul_rn(__fmul_rn(b1y, 0.5f), H);
            const float s2x = __fmul_rn(__fmul_rn(b2x, 0.5f), W), s2y = __fmul_rn(__fmul_rn(b2y, 0.5f), H);
            const bool fallback = __fsqrt_rn(__fadd_rn(__fmul_rn(s1x, s1x), __fmul_rn(s1y, s1y))) < 1.0f ||
                                  __fsqrt_rn(__fadd_rn(__fmul_rn(s2x, s2x), __fmul_rn(s2y, s2y))) < 1.0f;
            float h1x, h1y, h2x, h2y, qcx, qcy;
            bool drawn = true;
            if (!fallback) {
                const float k3 = __fmul_rn(3.0f, P.inv_focal_adj);
                h1x = __fmul_rn(__fmul_rn(__fmul_rn(b1x, k3), 0.5f), W); h1y = __fmul_rn(__fmul_rn(__fmul_rn(b1y, k3), 0.5f), H);
                h2x = __fmul_rn(__fmul_rn(__fmul_rn(b2x, k3), 0.5f), W); h2y = __fmul_rn(__fmul_rn(__fmul_rn(b2y, k3), 0.5f), H);
                qcx = ncx; qcy = ncy;           // vQuadCenter = center.xy: NDC units, restated as the reference draws it
            } else {
                // the reference-implementation AABB square (:159-189), half side 3 radius px
                const float dist = __fadd_rn(__fadd_rn(__fmul_rn(__fmul_rn(Tw[0], Tw[0]), 1.0f), __fmul_rn(__fmul_rn(Tw[1], Tw[1]), 1.0f)),
                                             __fmul_rn(__fmul_rn(Tw[2], Tw[2]), -1.0f));
                const float id = __fdiv_rn(1.0f, dist);
                const float f0 = __fmul_rn(id, 1.0f), f1 = __fmul_rn(id, 1.0f), f2 = __fmul_rn(id, -1.0f);
                if (fabsf(dist) < 1e-5f) drawn = false;   // gl_Position left unset: dropped (DESIGN.md section 2)
                auto dot3f = [&](const float *a, const float *b) {
                    return __fadd_rn(__fadd_rn(__fmul_rn(__fmul_rn(a[0], b[0]), f0), __fmul_rn(__fmul_rn(a[1], b[1]), f1)), __fmul_rn(__fmul_rn(a[2], b[2]), f2));
                };
                qcx = dot3f(Tu, Tw); qcy = dot3f(Tv, Tw);
                const float hx = __fsub_rn(__fmul_rn(qcx, qcx), dot3f(Tu, Tu)), hy = __fsub_rn(__fmul_rn(qcy, qcy), dot3f(Tv, Tv));
                const float ex = __fsqrt_rn(hx > 0.0001f ? hx : 0.0001f), ey = __fsqrt_rn(hy > 0.0001f ? hy : 0.0001f);
                const float radius = ex > ey ? ex : ey;
                h1x = __fmul_rn(radius, 3.0f); h1y = 0.f; h2x = 0.f; h2y = h1x;
            }
            if (!P.fade_in_complete) {                   // SplatMaterial.js:347-363
                const float ex = cx - P.scene_center[0], ey = cy - P.scene_center[1], ez = cz - P.scene_center[2];
                const float d = sqrtf(ex * ex + ey * ey + ez * ez);
                const float st = d >= P.fade_start ? 1.0f : 0.0f;
                col[3] *= (1.0f - st) + (1.0f - __saturatef((d - P.fade_start) / 0.75f)) * st;
            }
            const float pcx = __fmul_rn(__fadd_rn(__fmul_rn(ndcx, 0.5f), 0.5f), W), pcy = __fmul_rn(__fadd_rn(__fmul_rn(ndcy, 0.5f), 0.5f), H);   // ndcCenter in pixels
            if (EXPORT) {
                xo.T[0] = Tu[0]; xo.T[1] = Tu[1]; xo.T[2] = Tu[2]; xo.T[3] = Tv[0]; xo.T[4] = Tv[1]; xo.T[5] = Tv[2];
                xo.T[6] = Tw[0]; xo.T[7] = Tw[1]; xo.T[8] = Tw[2];
                xo.qcx = qcx; xo.qcy = qcy; xo.cx = pcx; xo.cy = pcy;
                xo.h1x = h1x; xo.h1y = h1y; xo.h2x = h2x; xo.h2y = h2y;
                xo.r = col[0]; xo.g = col[1]; xo.b = col[2]; xo.a = col[3];
                xo.ndc_z = ndcz; xo.branch = fallback ? 1u : 0u;
                xo.valid = (drawn && ndcz >= -1.0f && ndcz <= 1.0f) ? 1u : 0u;
            }
            const float det = h1x * h2y - h2x * h1y;
            const float idet = 1.0f / det;
            if (drawn && ndcz >= -1.0f && ndcz <= 1.0f && det != 0.0f && isfinite(idet) && isfinite(pcx) && isfinite(pcy)) {
                o.cx = pcx; o.cy = pcy;
                o.m00 = h2y * idet; o.m01 = -h2x * idet; o.m10 = -h1y * idet; o.m11 = h1x * idet;
                o.qx = qcx - pcx; o.qy = qcy - pcy;
                float A[3], B[3], Cc[3];
                cross3(Tv, Tw, A);
                cross3(Tw, Tu, B);
                const float k[3] = {pcx * Tw[0] - Tu[0], pcx * Tw[1] - Tu[1], pcx * Tw[2] - Tu[2]};
                const float l[3] = {pcy * Tw[0] - Tv[0], pcy * Tw[1] - Tv[1], pcy * Tw[2] - Tv[2]};
                cross3(k, l, Cc);
                o.ax = A[0]; o.ay = A[1]; o.az = A[2]; o.bx = B[0]; o.by = B[1]; o.bz = B[2];
                o.kx = Cc[0]; o.ky = Cc[1]; o.kz = Cc[2];
                o.twx = Tw[0]; o.twy = Tw[1]; o.twz = Tw[2];
                o.r = col[0]; o.g = col[1]; o.b = col[2]; o.a = col[3];
                // pixel centres (px + 0.5) inside the quad's AABB
                const float hx = (fabsf(h1x) + fabsf(h2x)) * 1.0005f + 0.01f, hy = (fabsf(h1y) + fabsf(h2y)) * 1.0005f + 0.01f;
                const float fx0 = ceilf(pcx - hx - 0.5f), fx1 = floorf(pcx + hx - 0.5f);
                const float fy0 = ceilf(pcy - hy - 0.5f), fy1 = floorf(pcy + hy - 0.5f);
                const float W1 = (float)(P.width - 1), H1 = (float)(P.height - 1);
                if (col[3] > 0.f && fx1 >= 0.f && fy1 >= 0.f && fx0 <= W1 && fy0 <= H1 && fx0 <= fx1 && fy0 <= fy1) {
                    const int px0 = (int)fmaxf(fx0, 0.f), px1 = (int)fminf(fx1, W1);
                    const int py0 = (int)fmaxf(fy0, 0.f), py1 = (int)fminf(fy1, H1);
                    rect = make_ushort4((unsigned short)(px0 >> P.tile_shift), (unsigned short)(py0 >> P.tile_shift),
                                        (unsigned short)(px1 >> P.tile_shift), (unsigned short)(py1 >> P.tile_shift));
                    visible = 1;
                }
            }
        }
        float4 *dst = reinterpret_cast<float4 *>(rec + s);
        const float4 *srcv = reinterpret_cast<const float4 *>(&o);
#pragma unroll
        for (int k = 0; k < 6; ++k) dst[k] = srcv[k];
        rects[s] = rect;
        if (EXPORT) exp[s] = xo;
    }
    const uint32_t nvis = __popc(__ballot_sync(0xffffffffu, visible));
    if (!EXPORT && (threadIdx.x & 31) == 0 && nvis) atomicAdd(&rctl->visible_slots[((blockIdx.x * (kProjThreads / 32) + (threadIdx.x >> 5)) & (kVisibleSlots - 1)) * 8], nvis);
}

// Which of a tile's 8x8-px blocks can hold a pixel centre inside the quad: separating axes x, y (the quad's AABB, from the inverse
// edge map) and the quad's own u, v axes over each block's rectangle of pixel centres -- exact for the parallelogram.
// r0 = cx, cy, m00, m01 ; r1 = m10, m11, ...
template <int NBX, int NBY>
__device__ __noinline__ uint32_t surfel_block_mask(float4 r0, float4 r1, float tile_x0, float tile_y0) {
    const float m00 = r0.z, m01 = r0.w, m10 = r1.x, m11 = r1.y;
    const float ad = 1.0f / fabsf(m00 * m11 - m01 * m10);
    const float hx = (fabsf(m11) + fabsf(m01)) * ad * 1.001f + 0.01f, hy = (fabsf(m10) + fabsf(m00)) * ad * 1.001f + 0.01f;
    if (!(hx < 1e30f) || !(hy < 1e30f)) return 0u;
    const float X0 = tile_x0 - r0.x, Y0 = tile_y0 - r0.y;
    const int ix0 = max(0, (int)ceilf((-hx - X0 - 7.0f) * 0.125f)), ix1 = min(NBX - 1, (int)floorf((hx - X0) * 0.125f));
    const int iy0 = max(0, (int)ceilf((-hy - Y0 - 7.0f) * 0.125f)), iy1 = min(NBY - 1, (int)floorf((hy - Y0) * 0.125f));
    uint32_t bm = 0;
    const float eu = 3.5f * (fabsf(m00) + fabsf(m01)), ev = 3.5f * (fabsf(m10) + fabsf(m11));   // half extents of u, v over a block
#pragma unroll 1
    for (int iy = iy0; iy <= iy1; ++iy) {
        const float my = Y0 + (float)(8 * iy) + 3.5f;
#pragma unroll 1
        for (int ix = ix0; ix <= ix1; ++ix) {
            const float mx = X0 + (float)(8 * ix) + 3.5f;
            const float u = m00 * mx + m01 * my, v = m10 * mx + m11 * my;
            if (fabsf(u) <= 1.001f + eu && fabsf(v) <= 1.001f + ev) bm |= 1u << (iy * NBX + ix);
        }
    }
    return bm;
}

// ---------------------------------------------------------------------------------------------------------------
// Blend: k_blend2's structure (CTA per fine tile, warp = 8x8-px block, lane = 2 vertically adjacent pixels, list filtered by mask
// bit, block masks at staging time, packed f32x2 math, block-level early exit below transmittance 1/512) with the surfel fragment
// shader.  At most 256 records are staged at a time (an 8-bit index per staged record; 96-byte records for 512 threads would not fit
// the static shared memory of the 32-px tile).
template <int FORMAT, int S>
__global__ void __launch_bounds__(128 * S * S, S == 1 ? 6 : 1)   // <= 85 registers: no spills (at 64 it spilled 24 B)
k_blend2d(const uint2 *__restrict__ ranges, const unsigned long long *__restrict__ list, const SurfelRecord *__restrict__ rec, int tiles_x,
          int tiles_y, int coarse_x, uint32_t rank, uint32_t world, int width, int height, int flip_y, void *__restrict__ frame_base,
          const uint32_t *__restrict__ tile_order, StatusSnapshot snap) {
    pdl_enter();
    void *__restrict__ frame = snap.half_src ? (void *)((unsigned char *)frame_base + (size_t)(*snap.half_src & 1u) * snap.half_bytes) : frame_base;
    if (snap.dst && blockIdx.x == 0) {
        if (threadIdx.x < 3) snap.dst[threadIdx.x] = snap.sort_ctl[threadIdx.x];
        for (uint32_t i = threadIdx.x; i < (uint32_t)(sizeof(RasterControl) / 4); i += blockDim.x) snap.dst[4 + i] = snap.raster_ctl[i];
    }
    constexpr int THREADS = 128 * S * S, WARPS = THREADS / 32, NBX = 2 * S, NBY = 2 * S, TILE = 16 * S;
    constexpr int ROUNDS = S == 1 ? 4 : 1, BATCH = ROUNDS * THREADS;
    constexpr int STAGE = THREADS < 256 ? THREADS : 256, SWARPS = STAGE / 32;
    __shared__ float4 s_rec[STAGE][6];
    __shared__ uint32_t s_ids[BATCH];
    __shared__ uint32_t s_cnt[ROUNDS * WARPS + 1];
    __shared__ uint8_t s_list[WARPS][STAGE];
    __shared__ uint8_t s_nlist[WARPS][SWARPS];
    const uint32_t coarse = tile_order[blockIdx.x / kFinePerCoarse], sub = blockIdx.x % kFinePerCoarse;
    const int ccx = (int)(coarse % (uint32_t)coarse_x), ccy = (int)(coarse / (uint32_t)coarse_x);
    const int tx = ccx * kCoarseW + (int)(sub & (kCoarseW - 1)), ty = ccy * kCoarseH + (int)(sub >> kCoarseShiftX);
    if (tx >= tiles_x || ty >= tiles_y) return;
    if (!owns_coarse(ccx, ccy, rank, world)) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = tx * TILE + (warp % NBX) * 8 + (lane & 7), y0 = ty * TILE + (warp / NBX) * 8 + (lane >> 3) * 2;
    const float pxc = (float)x + 0.5f, pyc = (float)y0 + 0.5f;
    const float tile_x0 = (float)(tx * TILE) + 0.5f, tile_y0 = (float)(ty * TILE) + 0.5f;
    f32x2 T = pack2((x < width && y0 < height) ? 1.0f : 0.0f, (x < width && y0 + 1 < height) ? 1.0f : 0.0f);
    f32x2 Rr = pack2(0.f, 0.f), Gg = Rr, Bb = Rr;
    const f32x2 PY = pack2(pyc, pyc + 1.0f);
    bool wdone = !__any_sync(0xffffffffu, fmaxf(lo2(T), hi2(T)) >= kTransmittanceCutoff);
    const uint2 rg = ranges[coarse];
    const uint32_t lt = lanemask_lt();
    const uint32_t nbatch = rg.y > rg.x ? (rg.y - rg.x + BATCH - 1) / BATCH : 0u;     // (0xffffffff, 0): an empty tile of the radix path
    for (uint32_t b = 0; b < nbatch; ++b) {
        const uint32_t base = rg.x + b * (uint32_t)BATCH;
        if (__syncthreads_and(wdone)) break;
        // ---- filter BATCH list entries by this tile's mask bit; order-preserving compaction (order: round, warp, lane) ------------
        uint32_t ids[ROUNDS], bal[ROUNDS];
#pragma unroll
        for (int k = 0; k < ROUNDS; ++k) {
            const uint32_t i = base + (uint32_t)k * THREADS + threadIdx.x;
            bool hit = false;
            ids[k] = 0;
            if (i < rg.y) {
                const unsigned long long e = __ldg(list + i);
                hit = ((uint32_t)(e >> 32) >> sub) & 1u;
                ids[k] = (uint32_t)e;
            }
            bal[k] = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) s_cnt[k * WARPS + warp] = __popc(bal[k]);
        }
        __syncthreads();
        if (warp == 0) {
            uint32_t run = 0;
#pragma unroll
            for (int c = 0; c < ROUNDS * WARPS; c += 32) {
                const uint32_t v = (c + lane < ROUNDS * WARPS) ? s_cnt[c + lane] : 0u;
                const uint32_t inc = warp_inclusive_scan(v);
                if (c + lane < ROUNDS * WARPS) s_cnt[c + lane] = run + inc - v;
                run += __shfl_sync(0xffffffffu, inc, 31);
            }
            if (lane == 0) s_cnt[ROUNDS * WARPS] = run;
        }
        __syncthreads();
        const uint32_t nsurv = s_cnt[ROUNDS * WARPS];
#pragma unroll
        for (int k = 0; k < ROUNDS; ++k)
            if ((bal[k] >> lane) & 1u) s_ids[s_cnt[k * WARPS + warp] + __popc(bal[k] & lt)] = ids[k];
        __syncthreads();
        // ---- stage up to STAGE survivors at a time, then every warp composites the ones that reach its block -----------------------
        for (uint32_t c0 = 0; c0 < nsurv; c0 += STAGE) {
            const uint32_t j = c0 + threadIdx.x;
            uint32_t bm = 0;
            if (threadIdx.x < STAGE && j < nsurv) {
                const float4 *src = reinterpret_cast<const float4 *>(rec + s_ids[j]);
                float4 r[6];
#pragma unroll
                for (int k = 0; k < 6; ++k) r[k] = __ldg(src + k);
                bm = surfel_block_mask<NBX, NBY>(r[0], r[1], tile_x0, tile_y0);
                r[5].w = log2f(r[5].w);            // opacity folded into the exponent
#pragma unroll
                for (int k = 0; k < 6; ++k) s_rec[threadIdx.x][k] = r[k];
            }
            if (warp < SWARPS) {
#pragma unroll
                for (int bk = 0; bk < WARPS; ++bk) {
                    const uint32_t v = __ballot_sync(0xffffffffu, (bm >> bk) & 1u);
                    if ((bm >> bk) & 1u) s_list[bk][warp * 32 + __popc(v & lt)] = (uint8_t)threadIdx.x;
                    if (lane == 0) s_nlist[bk][warp] = (uint8_t)__popc(v);
                }
            }
            __syncthreads();
            if (!wdone) {
#pragma unroll 1
                for (int sw = 0; sw < SWARPS && !wdone; ++sw) {
                    const int cnt = s_nlist[warp][sw];
                    const uint8_t *lst = &s_list[warp][sw * 32];
#pragma unroll 1
                    for (int k = 0; k < cnt; ++k) {
                        const int jj = lst[k];
                        const float4 R0 = s_rec[jj][0], R1 = s_rec[jj][1], R2 = s_rec[jj][2], R3 = s_rec[jj][3], R4 = s_rec[jj][4], R5 = s_rec[jj][5];
                        // R0 = cx cy m00 m01 ; R1 = m10 m11 qx qy ; R2 = Ax Ay Az Bx ; R3 = By Bz Cx Cy ; R4 = Cz Twx Twy Twz ; R5 = r g b log2(a)
                        const float dx = pxc - R0.x;
                        const f32x2 DY = fma2(PY, bcast2(1.0f), bcast2(-R0.y));
                        const f32x2 U = fma2(DY, bcast2(R0.w), bcast2(R0.z * dx)), V = fma2(DY, bcast2(R1.y), bcast2(R1.x * dx));
                        const f32x2 Px = fma2(DY, bcast2(R2.w), bcast2(fmaf(dx, R2.x, R3.z)));
                        const f32x2 Py = fma2(DY, bcast2(R3.x), bcast2(fmaf(dx, R2.y, R3.w)));
                        const f32x2 Pz = fma2(DY, bcast2(R3.y), bcast2(fmaf(dx, R2.z, R4.x)));
                        const f32x2 IZ = pack2(__fdividef(1.0f, lo2(Pz)), __fdividef(1.0f, hi2(Pz)));
                        const f32x2 Sx = mul2(Px, IZ), Sy = mul2(Py, IZ);
                        const f32x2 R3d = fma2(Sx, Sx, mul2(Sy, Sy));
                        const float ex = R1.z - dx;
                        const f32x2 EY = fma2(DY, bcast2(-1.0f), bcast2(R1.w));
                        const f32x2 R2d = mul2(fma2(EY, EY, bcast2(ex * ex)), bcast2(2.0f));
                        const f32x2 Dp = fma2(Sx, bcast2(R4.y), fma2(Sy, bcast2(R4.z), bcast2(R4.w)));
                        float al[2];
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const float r3 = h ? hi2(R3d) : lo2(R3d), r2 = h ? hi2(R2d) : lo2(R2d);
                            const bool near3 = r3 <= r2;
                            const float rho = near3 ? r3 : r2, depth = near3 ? (h ? hi2(Dp) : lo2(Dp)) : R4.w;
                            const float u = h ? hi2(U) : lo2(U), v = h ? hi2(V) : lo2(V), pz = h ? hi2(Pz) : lo2(Pz);
                            // exp(-rho/2) * a = 2^(rho * -log2(e)/2 + log2 a)
                            float a = fminf(0.99f, ex2_approx(fmaf(rho, -0.7213475204444817f, R5.w)));
                            const bool ok = fabsf(u) <= 1.0f && fabsf(v) <= 1.0f && pz != 0.0f && depth >= 0.2f && a >= 1.0f / 255.0f;
                            al[h] = ok ? a : 0.0f;
                        }
                        const f32x2 wgt = mul2(T, pack2(al[0], al[1]));
                        Rr = fma2(wgt, bcast2(R5.x), Rr); Gg = fma2(wgt, bcast2(R5.y), Gg); Bb = fma2(wgt, bcast2(R5.z), Bb);
                        T = fma2(wgt, bcast2(-1.0f), T);
                        if (!__any_sync(0xffffffffu, fmaxf(lo2(T), hi2(T)) >= kTransmittanceCutoff)) { wdone = true; break; }
                    }
                }
            }
            if (__syncthreads_and(wdone)) break;
        }
    }
    const float T0 = lo2(T), T1 = hi2(T), r0 = lo2(Rr), r1 = hi2(Rr), g0 = lo2(Gg), g1 = hi2(Gg), b0 = lo2(Bb), b1 = hi2(Bb);
    if (x < width) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int y = y0 + k;
            if (y < height) {
                const float Tk = k ? T1 : T0, Rk = k ? r1 : r0, Gk = k ? g1 : g0, Bk = k ? b1 : b0;
                const float A = 1.0f - Tk;
                const int out_row = flip_y ? (height - 1 - y) : y;
                const size_t at = (size_t)out_row * width + x;
                if (FORMAT == GS_FRAME_RGBA32F) {
                    reinterpret_cast<float4 *>(frame)[at] = make_float4(Rk, Gk, Bk, A);
                } else {
                    const uint32_t r8 = (uint32_t)(__saturatef(Rk) * 255.0f + 0.5f), g8 = (uint32_t)(__saturatef(Gk) * 255.0f + 0.5f);
                    const uint32_t b8 = (uint32_t)(__saturatef(Bk) * 255.0f + 0.5f), a8 = (uint32_t)(__saturatef(A) * 255.0f + 0.5f);
                    reinterpret_cast<uint32_t *>(frame)[at] = r8 | (g8 << 8) | (b8 << 16) | (a8 << 24);
                }
            }
        }
    }
    if (world > 1) __threadfence_system();
}

} // namespace gs
