// raster_kernels.cuh -- tile-binned forward rasteriser (sm_100a) replacing the reference's WebGL path:
//   k_project     : vertex shader, once per splat (not x4)    SplatMaterial.js:112-341, SplatMaterial3D.js:83-216
//   k_tile_count  : coarse-tile instances per chunk of draw ranks
//   k_tile_emit   : (coarse tile, {fine mask, splat}) instances in DRAW order
//   k_radix_*     : stable sort of the instances by coarse tile id (sort_kernels.cuh) -> per-coarse-tile lists in draw order
//   k_blend       : fragment shader + blend, front-to-back      SplatMaterial3D.js:234-252, :65-75
// Draw order is the reference's (sorted_indexes[0] first = farthest).  We composite front-to-back over the REVERSED
// list with a transmittance accumulator, which is algebraically the same "over" chain (SURVEY.md Appendix C).
#pragma once
#include "common.cuh"
#include "sort_kernels.cuh"
#include "../../include/gsplat_b200.h"
#include <cuda_fp16.h>
#include "ellipse_mask.h"

namespace gs {

constexpr int kTile = 16;              // tile edge in pixels
constexpr int kTileShift = 4;
constexpr float kTransmittanceCutoff = 1.0f / 512.0f;  // stop compositing below this: what is left adds < 0.5/255 (half an RGBA8 step); stated deviation

struct __align__(16) SplatRecord {     // 48 bytes, read as 3 x 16 B
    float cx, cy;                      // quad centre in pixels, GL window coordinates (y up)
    float g1x, g1y;                    // g1 = B1 / |B1|^2 : u = dot(d, g1) is the quad-local coordinate in [-1,1]
    float g2x, g2y;                    // g2 = B2 / |B2|^2
    uint32_t hxhy;                     // half2: half extents of the ellipse's pixel AABB, rounded UP (culling only)
    float a;
    float r, g, b;
    float ndc_z;                       // outside [-1,1] (2.0 for culled splats) <=> not drawn
};

constexpr int kVisibleSlots = 64;
struct RasterControl {
    unsigned long long total_instances;
    uint32_t overflow;
    uint32_t visible;
    uint32_t reserved0;
    uint32_t frame_seq;      // frames rendered so far (never reset): the peer-gather handshake counts in frames
    uint32_t peer_timeout;   // a peer handshake gave up waiting
    uint32_t peer_parity;    // ranks > 0: which half of rank 0's (double) frame buffer this frame's tiles go to (from the release word)
    unsigned long long subset_count;   // sharded frames: splats whose rect touches one of this rank's coarse tiles
    // visible-splat statistic, spread over 64 counters 32 B apart: one counter took ~1.6 ns per same-address atomic, which at one atomic
    // per warp WAS the duration of k_project (16 M splats: 500 K atomics = 0.79 ms; 1.2 M: 26 K = 41 us of a 37 us kernel)
    uint32_t visible_slots[kVisibleSlots * 8];
};

// Block in rank 0's memory that the other ranks map through CUDA IPC: the fused tile gather's handshake.
//   released = 2 f + b : rank 0 has finished with the picture that last occupied half b of its frame allocation; peers may write
//                  frame f's tiles into that half (b = 0 always unless rank 0 pipelines its frames over two halves)
//   arrived      : += 1 by every peer once its tiles of the current frame are in rank 0's buffer
struct PeerSync { uint32_t released; uint32_t arrived; uint32_t pad[2]; };

__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
constexpr long long kPeerTimeoutCycles = 4000000000ll;   // ~2 s: a missing peer must never hang the GPU

// rank 0, start of frame f: the picture of frame f-1 has been consumed (stream order) -> peers may overwrite the buffer
__global__ void k_peer_release(PeerSync *sync, const RasterControl *rctl, uint32_t half) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(&sync->released), "r"(rctl->frame_seq * 2u + (half & 1u)) : "memory");
}
// rank r > 0, before its blend of frame f: wait until rank 0 released frame f
__global__ void k_peer_wait_release(const PeerSync *sync, RasterControl *rctl) {
    // rank 0 cannot release frame f+1 before every peer has signalled frame f, so the word read here is frame f's
    const uint32_t f = rctl->frame_seq;
    const long long t0 = clock64();
    uint32_t v = ld_acquire_sys_u32(&sync->released);
    while ((int32_t)((v >> 1) - f) < 0) {
        if (clock64() - t0 > kPeerTimeoutCycles) { rctl->peer_timeout = 1; v = 0; break; }
        __nanosleep(200);
        v = ld_acquire_sys_u32(&sync->released);
    }
    rctl->peer_parity = v & 1u;
}
// rank r > 0, after its blend: tiles are in rank 0's frame
__global__ void k_peer_signal(PeerSync *sync) {
    __threadfence_system();
    atomicAdd_system(&sync->arrived, 1u);
}
// rank 0, end of frame f: wait for the tiles of all world-1 peers
__global__ void k_peer_wait_arrived(const PeerSync *sync, RasterControl *rctl, uint32_t peers) {
    const uint32_t want = rctl->frame_seq * peers;
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys_u32(&sync->arrived) - want) < 0) {
        if (clock64() - t0 > kPeerTimeoutCycles) { rctl->peer_timeout = 1; break; }
        __nanosleep(200);
    }
    __threadfence_system();
}

struct ProjParams {
    float mv[16], proj[16];
    float cam[3];
    float focal[2], viewport[2];
    float inv_focal_adj, ortho_zoom;
    int orthographic;
    float splat_scale;
    int point_cloud, sh_degree, antialiased;
    float kernel2d, max_size;
    int fade_in_complete;
    float scene_center[3], fade_start;
    int dynamic, optional_effects, scene_count;
    int tiles_x, tiles_y;
    uint32_t rank, world;
    int width, height;
    int tile_shift;                    // log2 of the fine-tile edge in pixels: 4 (16 px) or 5 (32 px, frames beyond ~2048x1024)
};

struct DynamicUniforms {               // only read in dynamic / optional-effects / 8-bit SH modes
    float view[16];
    float transforms[16 * GS_MAX_SCENES_DEV];
    float sh8_min[GS_MAX_SCENES_DEV], sh8_max[GS_MAX_SCENES_DEV];
    float opacity[GS_MAX_SCENES_DEV];
    int visibility[GS_MAX_SCENES_DEV];
};

// Multi-GPU ownership: COARSE tile (cx, cy) belongs to rank (cx + cy) % world -- a diagonal interleave, so every rank gets tiles from
// all over the picture (dense centre and empty border alike) and any `world` horizontally adjacent coarse tiles cover every rank.
__host__ __device__ __forceinline__ bool owns_coarse(int cx, int cy, uint32_t rank, uint32_t world) {
    return world <= 1 || (uint32_t)(cx + cy) % world == rank;
}

__device__ __forceinline__ void mat4_mul_dev(const float *a, const float *b, float *o) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int r = 0; r < 4; ++r)
            o[4 * c + r] = a[r] * b[4 * c] + a[4 + r] * b[4 * c + 1] + a[8 + r] * b[4 * c + 2] + a[12 + r] * b[4 * c + 3];
}
__device__ inline void mat4_inverse_dev(const float *m, float *o) {
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
#pragma unroll
    for (int i = 0; i < 16; ++i) o[i] = inv[i] * id;
}

// ---------------------------------------------------------------------------------------------------------------
// Projection: one thread per splat, splat order (coalesced 16 B + 24 B + SH loads).
//   COVF16: covariances stored as 6 halfs;  SHFMT: gs_sh_format
constexpr int kProjThreads = 128;

template <bool COVF16, int SHFMT>
__global__ void __launch_bounds__(kProjThreads)
k_project(const uint4 *__restrict__ cc, const void *__restrict__ cov, const void *__restrict__ sh, int sh_data_degree,
          const uint32_t *__restrict__ scene_idx, const DynamicUniforms *__restrict__ dyn, const ProjParams *__restrict__ Pp, uint32_t count,
          SplatRecord *__restrict__ rec, ushort4 *__restrict__ rects, RasterControl *rctl) {
    pdl_enter();
    // per-frame parameters: device memory -> shared memory once per CTA (graph-replayable, broadcast reads afterwards)
    __shared__ ProjParams s_P;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(Pp);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&s_P);
        for (int i = threadIdx.x; i < (int)(sizeof(ProjParams) / 4); i += kProjThreads) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    const ProjParams &P = s_P;
    __shared__ float4 s_out[kProjThreads / 32][96];
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * kProjThreads + threadIdx.x;
    uint32_t visible = 0;
    if (s < count) {
        SplatRecord o;
        o.cx = o.cy = o.g1x = o.g1y = o.g2x = o.g2y = o.a = o.r = o.g = o.b = 0.f;
        o.ndc_z = 2.0f;
        o.hxhy = 0;
        ushort4 rect = make_ushort4(1, 1, 0, 0); // empty
        // all of the splat's loads are issued up front (also for splats that turn out to be culled): the kernel is bound by load
        // latency, so memory-level parallelism matters more than the ~30% of bytes that culled splats would not have needed
        const int4 c4 = ld_nc_v4(cc + s);
        float V[6];
        if (COVF16) {
            const uint32_t *h32 = (const uint32_t *)cov + (size_t)s * 3;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const uint32_t w = ld_nc_u32(h32 + k);
                const __half2 hh = *reinterpret_cast<const __half2 *>(&w);
                V[2 * k] = __low2float(hh); V[2 * k + 1] = __high2float(hh);
            }
        } else {
            const float2 *f2 = (const float2 *)cov + (size_t)s * 3;
            const float2 a0 = __ldg(f2), a1 = __ldg(f2 + 1), a2 = __ldg(f2 + 2);
            V[0] = a0.x; V[1] = a0.y; V[2] = a1.x; V[3] = a1.y; V[4] = a2.x; V[5] = a2.y;
        }
        int4 shq[3];
        if (SHFMT == GS_SH_F16 && sh_data_degree >= 2 && P.sh_degree >= 1) {
            const uint4 *h4 = (const uint4 *)((const __half *)sh + (size_t)s * 24);
#pragma unroll
            for (int q = 0; q < 3; ++q) shq[q] = ld_nc_v4(h4 + q);
        }
        const float cx = __int_as_float(c4.y), cy = __int_as_float(c4.z), cz = __int_as_float(c4.w);
        uint32_t scene = 0;
        if (P.scene_count > 1 && scene_idx) scene = scene_idx[s] & (GS_MAX_SCENES_DEV - 1);
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

            if (SHFMT != GS_SH_NONE && sh_data_degree >= 1 && P.sh_degree >= 1) {
                const int ncomp = sh_data_degree >= 2 ? 24 : 9;
                float shv[24];
                const int nuse = (sh_data_degree >= 2 && P.sh_degree >= 2) ? 24 : 9;
                if (SHFMT == GS_SH_F16) {
                    const __half *h = (const __half *)sh + (size_t)s * ncomp;
                    if (ncomp == 24) {
#pragma unroll
                        for (int q = 0; q < 3; ++q) {
                            const int4 v = shq[q];
                            const uint32_t w[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const __half2 hh = *reinterpret_cast<const __half2 *>(&w[k]);
                                shv[q * 8 + 2 * k] = __low2float(hh);
                                shv[q * 8 + 2 * k + 1] = __high2float(hh);
                            }
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < 9; ++k) shv[k] = __half2float(h[k]);
                    }
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
                float dx = cx - camx, dy = cy - camy, dz = cz - camz;
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

            float j00, j02, j11, j12;
            if (P.orthographic == 1) { j00 = P.ortho_zoom; j11 = P.ortho_zoom; j02 = 0.f; j12 = 0.f; }
            else {
                const float iz = 1.0f / view[2], sc = iz * iz;
                j00 = P.focal[0] * iz; j11 = P.focal[1] * iz;
                j02 = -(P.focal[0] * view[0]) * sc; j12 = -(P.focal[1] * view[1]) * sc;
            }
            float T0[3], T1[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float w0 = mv[4 * k + 0], w1 = mv[4 * k + 1], w2 = mv[4 * k + 2];
                T0[k] = w0 * j00 + w2 * j02;
                T1[k] = w1 * j11 + w2 * j12;
            }
            const float VT0x = V[0] * T0[0] + V[1] * T0[1] + V[2] * T0[2];
            const float VT0y = V[1] * T0[0] + V[3] * T0[1] + V[4] * T0[2];
            const float VT0z = V[2] * T0[0] + V[4] * T0[1] + V[5] * T0[2];
            const float VT1x = V[0] * T1[0] + V[1] * T1[1] + V[2] * T1[2];
            const float VT1y = V[1] * T1[0] + V[3] * T1[1] + V[4] * T1[2];
            const float VT1z = V[2] * T1[0] + V[4] * T1[1] + V[5] * T1[2];
            float a = T0[0] * VT0x + T0[1] * VT0y + T0[2] * VT0z;
            const float b = T0[0] * VT1x + T0[1] * VT1y + T0[2] * VT1z;
            float d = T1[0] * VT1x + T1[1] * VT1y + T1[2] * VT1z;
            if (P.antialiased) {
                const float det0 = a * d - b * b;
                a += P.kernel2d; d += P.kernel2d;
                const float det1 = a * d - b * b;
                col[3] *= sqrtf(fmaxf(det0 / det1, 0.0f));
                if (col[3] < 1.0f / 255.0f) alive = false;
            } else { a += P.kernel2d; d += P.kernel2d; }
            const float D = a * d - b * b, half_tr = 0.5f * (a + d);
            const float term2 = sqrtf(fmaxf(0.1f, half_tr * half_tr - D));
            float l1 = half_tr + term2, l2 = half_tr - term2;
            if (P.point_cloud == 1) l1 = l2 = 0.2f;
            if (l2 <= 0.0f) alive = false;
            if (alive) {
                float ex = b, ey = l1 - a;
                const float en = rsqrtf(ex * ex + ey * ey);
                ex *= en; ey *= en;
                const float sqrt8 = 2.8284271247461903f;
                const float s1 = P.splat_scale * fminf(sqrt8 * sqrtf(l1), P.max_size) * P.inv_focal_adj;
                const float s2 = P.splat_scale * fminf(sqrt8 * sqrtf(l2), P.max_size) * P.inv_focal_adj;
                if (P.optional_effects) col[3] *= dyn->opacity[scene];
                if (!P.fade_in_complete) {
                    const float qx = cx - P.scene_center[0], qy = cy - P.scene_center[1], qz = cz - P.scene_center[2];
                    const float dist = sqrtf(qx * qx + qy * qy + qz * qz);
                    const float st = dist >= P.fade_start ? 1.0f : 0.0f;
                    col[3] *= (1.0f - st) + (1.0f - __saturatef((dist - P.fade_start) / 0.75f)) * st;
                }
                // B1 = e1*s1, B2 = (e1.y,-e1.x)*s2 ; g = B/|B|^2 = e/s
                const float is1 = 1.0f / s1, is2 = 1.0f / s2;
                o.cx = (ndcx + 1.0f) * 0.5f * P.viewport[0];
                o.cy = (ndcy + 1.0f) * 0.5f * P.viewport[1];
                o.g1x = ex * is1; o.g1y = ey * is1;
                o.g2x = ey * is2; o.g2y = -ex * is2;
                o.ndc_z = ndcz; o.a = col[3];
                o.r = col[0]; o.g = col[1]; o.b = col[2];
                const bool in_depth = (ndcz >= -1.0f && ndcz <= 1.0f) && isfinite(s1) && isfinite(s2) && s1 > 0.f && s2 > 0.f;
                if (!in_depth && ndcz >= -1.0f && ndcz <= 1.0f) o.ndc_z = 2.0f;
                if (in_depth) {
                    // tight AABB of the ellipse u^2+w^2<=1 : half extents sqrt(B1x^2+B2x^2), sqrt(B1y^2+B2y^2)
                    const float b1x = ex * s1, b1y = ey * s1, b2x = ey * s2, b2y = -ex * s2;
                    const float hx = sqrtf(b1x * b1x + b2x * b2x) * 1.0005f + 0.01f;
                    const float hy = sqrtf(b1y * b1y + b2y * b2y) * 1.0005f + 0.01f;
                    const __half2 hh = __halves2half2(__float2half_ru(fminf(hx, 60000.f)), __float2half_ru(fminf(hy, 60000.f)));
                    o.hxhy = *reinterpret_cast<const uint32_t *>(&hh);
                    // pixel centres (px+0.5) inside [c-h, c+h]
                    const float fx0 = ceilf(o.cx - hx - 0.5f), fx1 = floorf(o.cx + hx - 0.5f);
                    const float fy0 = ceilf(o.cy - hy - 0.5f), fy1 = floorf(o.cy + hy - 0.5f);
                    const float W1 = (float)(P.width - 1), H1 = (float)(P.height - 1);
                    if (fx1 >= 0.f && fy1 >= 0.f && fx0 <= W1 && fy0 <= H1 && fx0 <= fx1 && fy0 <= fy1) {
                        const int px0 = (int)fmaxf(fx0, 0.f), px1 = (int)fminf(fx1, W1);
                        const int py0 = (int)fmaxf(fy0, 0.f), py1 = (int)fminf(fy1, H1);
                        rect = make_ushort4((unsigned short)(px0 >> P.tile_shift), (unsigned short)(py0 >> P.tile_shift),
                                            (unsigned short)(px1 >> P.tile_shift), (unsigned short)(py1 >> P.tile_shift));
                        visible = 1;
                    }
                }
            }
        }
        // stage the 48-byte record so that the warp stores its 1536 contiguous bytes with three fully coalesced 16-byte stores
        float4 *stage = s_out[threadIdx.x >> 5];
        stage[lane * 3 + 0] = make_float4(o.cx, o.cy, o.g1x, o.g1y);
        stage[lane * 3 + 1] = make_float4(o.g2x, o.g2y, __uint_as_float(o.hxhy), o.a);
        stage[lane * 3 + 2] = make_float4(o.r, o.g, o.b, o.ndc_z);
        rects[s] = rect;
    }
    __syncwarp();
    {
        const uint32_t warp_first = blockIdx.x * kProjThreads + (threadIdx.x & ~31u);
        if (warp_first < count) {
            const uint32_t nrec = min(32u, count - warp_first);
            float4 *gdst = reinterpret_cast<float4 *>(rec + warp_first);
            const float4 *stage = s_out[threadIdx.x >> 5];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const uint32_t idx = (uint32_t)k * 32 + lane;
                if (idx < nrec * 3) gdst[idx] = stage[idx];
            }
        }
    }
    const uint32_t nvis = __popc(__ballot_sync(0xffffffffu, visible));
    if ((threadIdx.x & 31) == 0 && nvis) atomicAdd(&rctl->visible_slots[((blockIdx.x * (kProjThreads / 32) + (threadIdx.x >> 5)) & (kVisibleSlots - 1)) * 8], nvis);
}

// ---------------------------------------------------------------------------------------------------------------
// Hierarchical binning.  Splats are binned (in draw order) into COARSE tiles of kCoarseW x kCoarseH fine tiles
// (128 x 64 px: <= 256 coarse tiles at 1920x1080 -> ONE stable radix pass over ~1.1 instances per splat).  Each instance
// carries a 32-bit mask of the fine tiles it touches inside that coarse tile; the blend CTA of a fine tile streams its
// coarse tile's list and keeps the entries whose mask bit is set.  Order inside a list = draw order (stable sort of a
// sequence generated in draw order), so filtering preserves it.
constexpr int kCoarseW = 8, kCoarseH = 4, kCoarseShiftX = 3, kCoarseShiftY = 2;
constexpr int kFinePerCoarse = kCoarseW * kCoarseH;   // 32 = bits of the mask

// Ownership as a bitmask over the diagonal index cx + cy: bit set = this rank's tile.  Avoids integer division by a run-time world
// size in the per-splat binning kernels.  The mask covers diagonals 0..127 only (7680x4320 reaches 62), so raster_render refuses a
// sharded frame whose largest diagonal is 128 or more (kMaxOwnDiag) with GS_ERR_BAD_ARG instead of binning it wrongly.
constexpr int kMaxOwnDiag = 127;
struct OwnMask { unsigned long long lo, hi; };
__host__ __device__ __forceinline__ bool own_diag(const OwnMask &m, int diag) {
    return ((diag < 64 ? m.lo >> diag : m.hi >> (diag - 64)) & 1ull) != 0ull;
}
__device__ __forceinline__ uint32_t own_count_range(const OwnMask &m, int d0, int d1) {   // 0 <= d0 <= d1 < 128
    uint32_t n = 0;
    if (d0 < 64) {
        const int hi = min(d1, 63);
        const unsigned long long w = (m.lo >> d0) & (hi - d0 == 63 ? ~0ull : ((1ull << (hi - d0 + 1)) - 1ull));
        n += __popcll(w);
    }
    if (d1 >= 64) {
        const int lo = max(d0, 64) - 64, hi = d1 - 64;
        const unsigned long long w = (m.hi >> lo) & (hi - lo == 63 ? ~0ull : ((1ull << (hi - lo + 1)) - 1ull));
        n += __popcll(w);
    }
    return n;
}
static inline OwnMask make_own_mask(uint32_t rank, uint32_t world) {
    OwnMask m{~0ull, ~0ull};
    if (world > 1) {
        m.lo = m.hi = 0;
        for (int d = 0; d < 128; ++d)
            if ((uint32_t)d % world == rank) { if (d < 64) m.lo |= 1ull << d; else m.hi |= 1ull << (d - 64); }
    }
    return m;
}

__device__ __forceinline__ uint32_t coarse_instances(ushort4 r, const OwnMask &own, bool sharded) {
    if (r.z < r.x || r.w < r.y) return 0;
    const int cx0 = r.x >> kCoarseShiftX, cx1 = r.z >> kCoarseShiftX, cy0 = r.y >> kCoarseShiftY, cy1 = r.w >> kCoarseShiftY;
    if (!sharded) return (uint32_t)(cx1 - cx0 + 1) * (uint32_t)(cy1 - cy0 + 1);
    if (cx0 == cx1 && cy0 == cy1) return own_diag(own, cx0 + cy0) ? 1u : 0u;
    uint32_t n = 0;   // per coarse row: owned diagonals in [cx0 + cy, cx1 + cy] = population count of a window of the 128-bit mask
    for (int cy = cy0; cy <= cy1; ++cy) n += own_count_range(own, cx0 + cy, cx1 + cy);
    return n;
}

// Does a fine-tile rect reach a coarse tile of this rank?  The coarse tiles of a rect cover EVERY diagonal index cx + cy in
// [cx0 + cy0, cx1 + cy1], and ownership depends on the diagonal only: one window of the 128-bit ownership mask, no loop.
__device__ __forceinline__ bool rect_touches_owned(ushort4 r, const OwnMask &own) {
    if (r.z < r.x || r.w < r.y) return false;
    const int d0 = (r.x >> kCoarseShiftX) + (r.y >> kCoarseShiftY), d1 = (r.z >> kCoarseShiftX) + (r.w >> kCoarseShiftY);
    return own_count_range(own, d0, min(d1, 127)) != 0u;
}

constexpr int kBinThreads = 256;
constexpr int kBinItems = 2;
constexpr int kBinTile = kBinThreads * kBinItems;   // draw ranks per CTA

// This thread's share of "instances of all chunks before mine": whole groups of kBinThreads chunks from the second-level sums,
// the chunks of my own group one per thread.
__device__ __forceinline__ unsigned long long chunk_prefix(const uint32_t *__restrict__ block_sums, const uint32_t *__restrict__ super_sums) {
    const uint32_t grp = blockIdx.x / kBinThreads;
    unsigned long long before = 0;
    for (uint32_t g = threadIdx.x; g < grp; g += kBinThreads) before += super_sums[g];
    const uint32_t b = grp * kBinThreads + threadIdx.x;
    if (b < blockIdx.x) before += block_sums[b];
    return before;
}

// pass 1: instances per warp (256 consecutive draw ranks) and per CTA chunk (rank p = 0 is the NEAREST splat = last in the
// reference's draw order).  Warp-striped like pass 2: warp w of a CTA owns ranks [chunk + 256 w, +256), item k of lane l = +32k + l.
__global__ void __launch_bounds__(kBinThreads)
k_tile_count(const uint32_t *__restrict__ order, uint32_t render_count_host, const unsigned long long *__restrict__ n_dev,
             const ushort4 *__restrict__ rects, uint32_t *__restrict__ block_sums, uint32_t *__restrict__ warp_sums, uint32_t *__restrict__ super_sums,
             OwnMask own, int sharded) {
    pdl_enter();
    const uint32_t render_count = n_dev ? (uint32_t)*n_dev : render_count_host;
    __shared__ uint32_t s_w[kBinThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t run = blockIdx.x * kBinTile + (uint32_t)warp * (32 * kBinItems) + lane;
    uint32_t mine = 0;
#pragma unroll
    for (int k = 0; k < kBinItems; ++k) {
        const uint32_t p = run + (uint32_t)k * 32;
        if (p < render_count) mine += coarse_instances(rects[ld_nc_u32(order + (render_count - 1u - p))], own, sharded != 0);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if (lane == 0) { s_w[warp] = mine; warp_sums[blockIdx.x * (kBinThreads / 32) + warp] = mine; }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t total = 0;
#pragma unroll
        for (int w = 0; w < kBinThreads / 32; ++w) total += s_w[w];
        block_sums[blockIdx.x] = total;
        if (total) atomicAdd(&super_sums[blockIdx.x / kBinThreads], total);   // second level: one counter per kBinThreads chunks
    }
}

// pass 2: write (coarse tile id, {fine mask, splat id}) for every instance, in draw order.  One item at a time (rolled loop, no
// per-thread arrays): the warp's base offset comes from pass 1's sums, the offsets inside an item from a warp scan.
__global__ void __launch_bounds__(kBinThreads)
k_tile_emit(const uint32_t *__restrict__ order, uint32_t render_count_host, const unsigned long long *__restrict__ n_dev,
            const ushort4 *__restrict__ rects, const uint32_t *__restrict__ block_sums, const uint32_t *__restrict__ warp_sums,
            const uint32_t *__restrict__ super_sums, int coarse_x,
            uint16_t *__restrict__ keys, unsigned long long *__restrict__ vals, unsigned long long capacity, RasterControl *rctl, OwnMask own,
            int sharded) {
    pdl_enter();
    const uint32_t render_count = n_dev ? (uint32_t)*n_dev : render_count_host;
    __shared__ unsigned long long s_prefix;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // instances of all earlier chunks
    // two levels (a flat sum over all earlier chunks is quadratic in the chunk count: 16 M splats = 31 K chunks = 0.5 G reads)
    unsigned long long before = chunk_prefix(block_sums, super_sums);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (threadIdx.x == 0) s_prefix = 0;
    __syncthreads();
    if (lane == 0 && before) atomicAdd(&s_prefix, before);
    __syncthreads();
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) rctl->total_instances = s_prefix + block_sums[blockIdx.x];   // read by the tile sort
    unsigned long long w0 = s_prefix;
    for (int w = 0; w < warp; ++w) w0 += warp_sums[blockIdx.x * (kBinThreads / 32) + w];
    const uint32_t run = blockIdx.x * kBinTile + (uint32_t)warp * (32 * kBinItems) + lane;
    bool overflow = false;
#pragma unroll 2
    for (int k = 0; k < kBinItems; ++k) {
        const uint32_t p = run + (uint32_t)k * 32;
        uint32_t sid = 0, cnt = 0;
        ushort4 r = make_ushort4(1, 1, 0, 0);
        if (p < render_count) {
            sid = ld_nc_u32(order + (render_count - 1u - p));
            r = rects[sid];
            cnt = coarse_instances(r, own, sharded != 0);
        }
        const uint32_t inc = warp_inclusive_scan(cnt);
        unsigned long long w = w0 + (inc - cnt);
        w0 += __shfl_sync(0xffffffffu, inc, 31);
        const int cx0 = r.x >> kCoarseShiftX, cx1 = r.z >> kCoarseShiftX, cy0 = r.y >> kCoarseShiftY, cy1 = r.w >> kCoarseShiftY;
        const bool single = (cx0 == cx1 && cy0 == cy1);
        if (cnt && single) {   // the common case: the splat sits inside one coarse tile
            const int fx0 = (int)r.x - cx0 * kCoarseW, fx1 = (int)r.z - cx0 * kCoarseW, fy0 = (int)r.y - cy0 * kCoarseH, fy1 = (int)r.w - cy0 * kCoarseH;
            const uint32_t rowsel = (0x01010101u >> (8 * (kCoarseH - 1 - (fy1 - fy0)))) << (8 * fy0);
            const uint32_t mask = (((1u << (fx1 - fx0 + 1)) - 1u) << fx0) * rowsel;
            if (w < capacity) {
                keys[w] = (uint16_t)(cy0 * coarse_x + cx0);
                vals[w] = ((unsigned long long)mask << 32) | sid;
            } else overflow = true;
        }
        // splats spanning MANY coarse tiles (a few huge ones cover the whole screen): the WARP walks each one's rect together,
        // 32 coarse tiles per step.  Instances of one splat land in different lists, so their mutual order is free.
        const uint32_t area = (uint32_t)(cx1 - cx0 + 1) * (uint32_t)(cy1 - cy0 + 1);
        if (cnt && !single && area <= 32u) {   // a handful of coarse tiles: each lane walks its own rect
#pragma unroll 1
            for (int cy = cy0; cy <= cy1; ++cy) {
                const int fy0 = max((int)r.y, cy * kCoarseH) - cy * kCoarseH, fy1 = min((int)r.w, cy * kCoarseH + kCoarseH - 1) - cy * kCoarseH;
                const uint32_t rowsel = (0x01010101u >> (8 * (kCoarseH - 1 - (fy1 - fy0)))) << (8 * fy0);
#pragma unroll 1
                for (int cx = cx0; cx <= cx1; ++cx) {
                    if (sharded && !own_diag(own, cx + cy)) continue;
                    const int fx0 = max((int)r.x, cx * kCoarseW) - cx * kCoarseW, fx1 = min((int)r.z, cx * kCoarseW + kCoarseW - 1) - cx * kCoarseW;
                    const uint32_t mask = (((1u << (fx1 - fx0 + 1)) - 1u) << fx0) * rowsel;
                    if (w < capacity) {
                        keys[w] = (uint16_t)(cy * coarse_x + cx);
                        vals[w] = ((unsigned long long)mask << 32) | sid;
                    } else overflow = true;
                    ++w;
                }
            }
        }
        uint32_t multi = __ballot_sync(0xffffffffu, cnt != 0u && area > 32u);
        while (multi) {
            const int src = __ffs(multi) - 1;
            multi &= multi - 1;
            const uint32_t bsid = __shfl_sync(0xffffffffu, sid, src);
            unsigned long long bw = __shfl_sync(0xffffffffu, w, src);
            const int bx0 = __shfl_sync(0xffffffffu, (int)r.x, src), by0 = __shfl_sync(0xffffffffu, (int)r.y, src);
            const int bx1 = __shfl_sync(0xffffffffu, (int)r.z, src), by1 = __shfl_sync(0xffffffffu, (int)r.w, src);
            const int ccx0 = bx0 >> kCoarseShiftX, ccy0 = by0 >> kCoarseShiftY;
            const int cw = (bx1 >> kCoarseShiftX) - ccx0 + 1, chh = (by1 >> kCoarseShiftY) - ccy0 + 1;
            const int ntile = cw * chh;
            for (int i0 = 0; i0 < ntile; i0 += 32) {
                const int i = i0 + lane;
                bool mineq = false;
                int cx = 0, cy = 0;
                if (i < ntile) {
                    cy = ccy0 + i / cw; cx = ccx0 + i % cw;
                    mineq = !sharded || own_diag(own, cx + cy);
                }
                const uint32_t bal = __ballot_sync(0xffffffffu, mineq);
                if (mineq) {
                    const unsigned long long at = bw + __popc(bal & lanemask_lt());
                    const int fx0 = max(bx0, cx * kCoarseW) - cx * kCoarseW, fx1 = min(bx1, cx * kCoarseW + kCoarseW - 1) - cx * kCoarseW;
                    const int fy0 = max(by0, cy * kCoarseH) - cy * kCoarseH, fy1 = min(by1, cy * kCoarseH + kCoarseH - 1) - cy * kCoarseH;
                    const uint32_t rowsel = (0x01010101u >> (8 * (kCoarseH - 1 - (fy1 - fy0)))) << (8 * fy0);
                    const uint32_t mask = (((1u << (fx1 - fx0 + 1)) - 1u) << fx0) * rowsel;
                    if (at < capacity) {
                        keys[at] = (uint16_t)(cy * coarse_x + cx);
                        vals[at] = ((unsigned long long)mask << 32) | bsid;
                    } else overflow = true;
                }
                bw += __popc(bal);
            }
        }
    }
    if (overflow) rctl->overflow = 1;
}


// ---------------------------------------------------------------------------------------------------------------
// Binning v2: a COUNTING SORT of the coarse-tile instances straight from the draw order -- count, scan, place -- instead of
// emit + a radix sort of the emitted (key, value) pairs.  One instance is written once (8 B) at its final slot of its coarse tile's
// list.  Up to 1024 coarse tiles in ONE pass (3840x2160 has 1020), so the 4K frame no longer needs a second radix pass.
//   k_bin_count : per chunk of draw ranks, instances per coarse tile            -> hist[tile][chunk], totals[tile]
//   k_bin_scan  : per tile: exclusive scan over chunks + base of the tile's list -> hist becomes offsets, ranges[tile]
//   k_bin_place : per chunk: stable rank of every instance inside the chunk (per-warp lane masks in shared memory: a splat touches a
//                 coarse tile at most once, so the instances of one tile in one warp round ARE a 32-bit lane mask and the rank of lane l
//                 is popc(mask & lanes_below(l))) + the chunk's offset -> list[slot] = {fine mask, splat id}
// Rank order inside a chunk = (warp, round, lane) = draw-rank order (warp-striped, as in the radix kernels).
constexpr int kBinTiles = 256;      // coarse tiles per frame in this path (8-bit bins)
constexpr int kBinRanks = 2048;     // draw ranks per CTA = kWarps * 32 * kItems in every configuration
template <int CFG> struct Bin2Cfg;
template <> struct Bin2Cfg<0> { static constexpr int kWarps = 16, kItems = 4; };     // 32 KB shared in k_bin_place
template <> struct Bin2Cfg<1> { static constexpr int kWarps = 8, kItems = 8; };      // 16 KB shared

__device__ __forceinline__ uint32_t fine_mask_in_coarse(int rx0, int ry0, int rx1, int ry1, int cx, int cy) {
    const int fx0 = max(rx0, cx * kCoarseW) - cx * kCoarseW, fx1 = min(rx1, cx * kCoarseW + kCoarseW - 1) - cx * kCoarseW;
    const int fy0 = max(ry0, cy * kCoarseH) - cy * kCoarseH, fy1 = min(ry1, cy * kCoarseH + kCoarseH - 1) - cy * kCoarseH;
    const uint32_t rowsel = (0x01010101u >> (8 * (kCoarseH - 1 - (fy1 - fy0)))) << (8 * fy0);
    return (((1u << (fx1 - fx0 + 1)) - 1u) << fx0) * rowsel;
}

// Calls f(owner lane, owner's splat id, coarse tile id, fine mask) for every instance of this warp round.  Splats over a handful of
// coarse tiles are walked by their own lane; the few huge ones (> 32 coarse tiles) by the whole warp, 32 tiles per step.
// Must be called by all 32 lanes.  f must not contain warp-synchronous operations.
template <typename F>
__device__ __forceinline__ void round_instances(bool valid, uint32_t sid, ushort4 r, int coarse_x, const OwnMask &own, bool sharded, F f) {
    const int lane = threadIdx.x & 31;
    const bool nonempty = valid && r.z >= r.x && r.w >= r.y;
    const int cx0 = r.x >> kCoarseShiftX, cx1 = r.z >> kCoarseShiftX, cy0 = r.y >> kCoarseShiftY, cy1 = r.w >> kCoarseShiftY;
    const bool big = nonempty && (uint32_t)(cx1 - cx0 + 1) * (uint32_t)(cy1 - cy0 + 1) > 32u;
    if (nonempty && !big) {
#pragma unroll 1
        for (int cy = cy0; cy <= cy1; ++cy)
#pragma unroll 1
            for (int cx = cx0; cx <= cx1; ++cx) {      // one iteration for most splats
                if (sharded && !own_diag(own, cx + cy)) continue;
                f(lane, sid, cy * coarse_x + cx, fine_mask_in_coarse((int)r.x, (int)r.y, (int)r.z, (int)r.w, cx, cy));
            }
    }
    uint32_t multi = __ballot_sync(0xffffffffu, big);
    while (multi) {
        const int src = __ffs(multi) - 1;
        multi &= multi - 1;
        const uint32_t bsid = __shfl_sync(0xffffffffu, sid, src);
        const int bx0 = __shfl_sync(0xffffffffu, (int)r.x, src), by0 = __shfl_sync(0xffffffffu, (int)r.y, src);
        const int bx1 = __shfl_sync(0xffffffffu, (int)r.z, src), by1 = __shfl_sync(0xffffffffu, (int)r.w, src);
        const int ccx0 = bx0 >> kCoarseShiftX, ccy0 = by0 >> kCoarseShiftY;
        const int cw = (bx1 >> kCoarseShiftX) - ccx0 + 1, ntile = cw * ((by1 >> kCoarseShiftY) - ccy0 + 1);
        for (int i = lane; i < ntile; i += 32) {
            const int cy = ccy0 + i / cw, cx = ccx0 + i % cw;
            if (sharded && !own_diag(own, cx + cy)) continue;
            f(src, bsid, cy * coarse_x + cx, fine_mask_in_coarse(bx0, by0, bx1, by1, cx, cy));
        }
    }
}

template <int CFG>
__global__ void __launch_bounds__(Bin2Cfg<CFG>::kWarps * 32)
k_bin_count(const uint32_t *__restrict__ order, uint32_t render_count_host, const unsigned long long *__restrict__ n_dev, const ushort4 *__restrict__ rects,
            int coarse_x, uint32_t nt, uint32_t *__restrict__ hist, uint32_t stride, uint32_t *__restrict__ totals, ushort4 *__restrict__ rect_by_rank,
            OwnMask own, int sharded) {
    pdl_enter();
    constexpr int W = Bin2Cfg<CFG>::kWarps, ITEMS = Bin2Cfg<CFG>::kItems, NT = kBinTiles;
    const uint32_t n = n_dev ? (uint32_t)*n_dev : render_count_host;
    const uint32_t base = blockIdx.x * (uint32_t)(W * 32 * ITEMS);
    if (base >= n) return;
    __shared__ uint32_t s_hist[NT];
    for (uint32_t t = threadIdx.x; t < nt; t += W * 32) s_hist[t] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t run = base + (uint32_t)warp * (32 * ITEMS) + lane;
    uint32_t sid[ITEMS];
    ushort4 rc[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t p = run + (uint32_t)k * 32;
        sid[k] = p < n ? ld_nc_u32(order + (n - 1u - p)) : 0xffffffffu;
    }
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) rc[k] = sid[k] != 0xffffffffu ? rects[sid[k]] : make_ushort4(1, 1, 0, 0);
    // the gathered rects are left in DRAW-RANK order for k_bin_place: its reads are then streams, not a second random gather
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t p = run + (uint32_t)k * 32;
        if (p < n) rect_by_rank[p] = rc[k];
    }
#pragma unroll 1
    for (int k = 0; k < ITEMS; ++k) {
        uint32_t id = 0; ushort4 r = make_ushort4(1, 1, 0, 0);
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) if (j == k) { id = sid[j]; r = rc[j]; }      // register select (no local-memory indexing)
        round_instances(id != 0xffffffffu, id, r, coarse_x, own, sharded != 0, [&](int, uint32_t, int t, uint32_t) { atomicAdd(&s_hist[t], 1u); });
    }
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < nt; t += W * 32) {
        const uint32_t v = s_hist[t];
        hist[(size_t)t * stride + blockIdx.x] = v;
        if (v) atomicAdd(&totals[t], v);
    }
}

// One CTA per coarse tile: where its list starts (all smaller tiles' totals) and the running offset of every chunk inside it.
// On an overflowing frame k_bin_place stores only the slots below `capacity`; slot s holds the same instance either way, so the
// tile ranges are clamped to the capacity and every blend reads written entries only.  total_instances stays UNclamped: it is the
// count the host reports with GS_ERR_CAPACITY.
__global__ void __launch_bounds__(1024)
k_bin_scan(uint32_t *__restrict__ hist, uint32_t stride, uint32_t ranks_per_chunk, uint32_t render_count_host, const unsigned long long *__restrict__ n_dev,
           const uint32_t *__restrict__ totals, uint32_t nt, uint2 *__restrict__ ranges, RasterControl *rctl, uint32_t *__restrict__ tile_order,
           unsigned long long capacity) {
    pdl_enter();
    __shared__ uint32_t s_scan[40];
    __shared__ uint32_t s_carry;
    {   // longest list first: the blend's duration is bounded below by its densest tiles, so their CTAs must start first.
        // rank of this tile among all tiles by list length, descending (ties: lower tile id first)
        const uint32_t mine = totals[blockIdx.x];
        bool ahead = false;
        if (threadIdx.x < nt) { const uint32_t o = totals[threadIdx.x]; ahead = o > mine || (o == mine && threadIdx.x < blockIdx.x); }
        const int rank = __syncthreads_count(ahead);
        if (threadIdx.x == 0) tile_order[rank] = blockIdx.x;
    }
    const uint32_t n = n_dev ? (uint32_t)*n_dev : render_count_host;
    const uint32_t nchunks = (uint32_t)(((uint64_t)n + ranks_per_chunk - 1) / ranks_per_chunk);
    const uint32_t d = blockIdx.x;
    {
        uint32_t total;
        const uint32_t c = threadIdx.x < d ? totals[threadIdx.x] : 0u;
        (void)block_exclusive_scan<1024>(c, s_scan, total);
        if (threadIdx.x == 0) {
            s_carry = total;
            const uint32_t mine = totals[d];
            const uint32_t cap = (uint32_t)min(capacity, 0xffffffffull);
            ranges[d] = make_uint2(min(total, cap), min(total + mine, cap));
            if (d == nt - 1) rctl->total_instances = (unsigned long long)total + mine;
        }
    }
    __syncthreads();
    uint32_t *col = hist + (size_t)d * stride;
    for (uint32_t b = 0; b < nchunks; b += 1024) {
        const uint32_t t = b + threadIdx.x;
        const uint32_t v = t < nchunks ? col[t] : 0u;
        uint32_t total;
        const uint32_t ex = block_exclusive_scan<1024>(v, s_scan, total);
        const uint32_t carry = s_carry;
        if (t < nchunks) col[t] = ex + carry;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
}

template <int CFG>
__global__ void __launch_bounds__(Bin2Cfg<CFG>::kWarps * 32)
k_bin_place(const uint32_t *__restrict__ order, uint32_t render_count_host, const unsigned long long *__restrict__ n_dev, const ushort4 *__restrict__ rect_by_rank,
            int coarse_x, uint32_t nt, const uint32_t *__restrict__ offsets, uint32_t stride, unsigned long long *__restrict__ list, unsigned long long capacity,
            RasterControl *rctl, OwnMask own, int sharded, int pack_ok) {
    pdl_enter();
    constexpr int W = Bin2Cfg<CFG>::kWarps, ITEMS = Bin2Cfg<CFG>::kItems, NT = kBinTiles;
    const uint32_t n = n_dev ? (uint32_t)*n_dev : render_count_host;
    const uint32_t base = blockIdx.x * (uint32_t)(W * 32 * ITEMS);
    if (base >= n) return;
    __shared__ uint32_t s_pre[W][NT];      // instances of this warp per tile, then: END of the slots this warp has handed out in the tile's list
    __shared__ __align__(8) uint32_t s_mask[W][NT];     // lanes of the current round that touch the tile (first: staging of the compaction)
    constexpr bool kCanCompact = NT * 4 >= 32 * ITEMS * 8;   // the mask row of a warp doubles as the staging buffer of its compacted items
    for (uint32_t i = threadIdx.x; i < (uint32_t)(W * NT); i += W * 32) (&s_pre[0][0])[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t run = base + (uint32_t)warp * (32 * ITEMS) + lane;
    uint32_t sid[ITEMS];
    ushort4 rc[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t p = run + (uint32_t)k * 32;
        sid[k] = p < n ? ld_nc_u32(order + (n - 1u - p)) : 0xffffffffu;
        rc[k] = p < n ? rect_by_rank[p] : make_ushort4(1, 1, 0, 0);
    }
    uint32_t *my_pre = s_pre[warp], *my_mask = s_mask[warp];
    // Culled splats (empty rect) and, on a sharded frame, splats that reach none of this rank's tiles leave most lanes idle in the
    // rounds below (ncu: 9-13 of 32 lanes active).  The warp's 32 * ITEMS items are therefore compacted first, order preserved
    // (item k of lane l is draw rank run + 32 k + l, so (k, lane) order is draw order): fewer rounds, full lanes.  A compacted item is
    // 8 bytes, {rect as 4 x u8, splat id}, which needs the frame to be at most 256 tiles wide and high (pack_ok).
    uint32_t nvalid = 32u * ITEMS;
    if (kCanCompact && pack_ok) {
        const uint32_t lt = lanemask_lt();
        unsigned long long *stage = reinterpret_cast<unsigned long long *>(my_mask);
        uint32_t before = 0;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const bool keep = sid[k] != 0xffffffffu && (sharded ? rect_touches_owned(rc[k], own) : (rc[k].z >= rc[k].x && rc[k].w >= rc[k].y));
            const uint32_t bal = __ballot_sync(0xffffffffu, keep);
            if (keep) stage[before + __popc(bal & lt)] = ((unsigned long long)((uint32_t)rc[k].x | ((uint32_t)rc[k].y << 8) | ((uint32_t)rc[k].z << 16) | ((uint32_t)rc[k].w << 24)) << 32) | sid[k];
            before += __popc(bal);
        }
        nvalid = before;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const uint32_t j = (uint32_t)k * 32u + (uint32_t)lane;
            sid[k] = 0xffffffffu;
            rc[k] = make_ushort4(1, 1, 0, 0);
            if (j < nvalid) {
                const unsigned long long v = stage[j];
                const uint32_t pr = (uint32_t)(v >> 32);
                sid[k] = (uint32_t)v;
                rc[k] = make_ushort4((unsigned short)(pr & 255u), (unsigned short)((pr >> 8) & 255u), (unsigned short)((pr >> 16) & 255u), (unsigned short)(pr >> 24));
            }
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < NT / 32; ++i) my_mask[i * 32 + lane] = 0u;      // (rounds clear it again; keeps the buffer's two uses apart)
        __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < ITEMS; ++k)
        if ((uint32_t)k * 32u < nvalid)      // warp-uniform
            round_instances(sid[k] != 0xffffffffu, sid[k], rc[k], coarse_x, own, sharded != 0, [&](int, uint32_t, int t, uint32_t) { atomicAdd(&my_pre[t], 1u); });
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < nt; t += W * 32) {   // counts -> first slot of each warp (chunk offset + earlier warps)
        uint32_t at = offsets[(size_t)t * stride + blockIdx.x];
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const uint32_t c = s_pre[w][t];
            s_pre[w][t] = at;
            at += c;
        }
    }
    __syncthreads();
    bool overflow = false;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        if ((uint32_t)k * 32u >= nvalid) break;      // warp-uniform: the compacted items fill the first rounds
        const bool valid = sid[k] != 0xffffffffu;
        // a round: (1) clear the warp's lane masks, (2) every instance sets its owner's bit in its tile's mask and takes one slot of the
        // tile's list, (3) with all bits in place, the instance of lane l sits popc(mask & lanes below l) after the round's first slot,
        // which is the tile's new end minus the round's population.
#pragma unroll
        for (int i = 0; i < NT / 32; ++i) my_mask[i * 32 + lane] = 0u;
        __syncwarp();
        round_instances(valid, sid[k], rc[k], coarse_x, own, sharded != 0, [&](int owner, uint32_t, int t, uint32_t) {
            atomicOr(&my_mask[t], 1u << owner);
            atomicAdd(&my_pre[t], 1u);
        });
        __syncwarp();
        round_instances(valid, sid[k], rc[k], coarse_x, own, sharded != 0, [&](int owner, uint32_t sid_o, int t, uint32_t fmask) {
            const uint32_t m = my_mask[t];
            const unsigned long long at = (unsigned long long)(my_pre[t] - (uint32_t)__popc(m)) + __popc(m & ((1u << owner) - 1u));
            if (at < capacity) list[at] = ((unsigned long long)fmask << 32) | sid_o;
            else overflow = true;
        });
        __syncwarp();
    }
    if (overflow) rctl->overflow = 1;
}

// ---------------------------------------------------------------------------------------------------------------
// Sharded frames (world_size > 1): the depth sort of a rank covers only the splats whose screen rect touches one of ITS coarse tiles.
// Any subset, bucketed with the GLOBAL min/max and kept in input order, sorts into exactly the global order restricted to that subset
// (ties are broken by input position) -- SURVEY.md 8(e) -- so no keys or splats are exchanged between GPUs.
// pass 1: survivors per warp / chunk of input positions;  pass 2: order-preserving compaction of (index, distance).
__global__ void __launch_bounds__(kBinThreads)
k_subset_count(const uint32_t *__restrict__ indexes, uint32_t count, const ushort4 *__restrict__ rects, OwnMask own,
               uint32_t *__restrict__ block_sums, uint32_t *__restrict__ warp_sums, uint32_t *__restrict__ super_sums) {
    pdl_enter();
    __shared__ uint32_t s_w[kBinThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t run = blockIdx.x * kBinTile + (uint32_t)warp * (32 * kBinItems) + lane;
    uint32_t mine = 0;
#pragma unroll
    for (int k = 0; k < kBinItems; ++k) {
        const uint32_t i = run + (uint32_t)k * 32;
        if (i < count) mine += rect_touches_owned(rects[indexes ? ld_nc_u32(indexes + i) : i], own) ? 1u : 0u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if (lane == 0) { s_w[warp] = mine; warp_sums[blockIdx.x * (kBinThreads / 32) + warp] = mine; }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t total = 0;
#pragma unroll
        for (int w = 0; w < kBinThreads / 32; ++w) total += s_w[w];
        block_sums[blockIdx.x] = total;
        if (total) atomicAdd(&super_sums[blockIdx.x / kBinThreads], total);
    }
}
__global__ void __launch_bounds__(kBinThreads)
k_subset_emit(const uint32_t *__restrict__ indexes, uint32_t count, const ushort4 *__restrict__ rects, OwnMask own,
              const uint32_t *__restrict__ block_sums, const uint32_t *__restrict__ warp_sums, const uint32_t *__restrict__ super_sums,
              const int32_t *__restrict__ dist, uint32_t *__restrict__ sub_idx, int32_t *__restrict__ sub_dist, RasterControl *rctl) {
    pdl_enter();
    __shared__ uint32_t s_prefix;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t before = (uint32_t)chunk_prefix(block_sums, super_sums);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (threadIdx.x == 0) s_prefix = 0;
    __syncthreads();
    if (lane == 0 && before) atomicAdd(&s_prefix, before);
    __syncthreads();
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) rctl->subset_count = (unsigned long long)s_prefix + block_sums[blockIdx.x];   // n of this rank's sort
    uint32_t w0 = s_prefix;
    for (int w = 0; w < warp; ++w) w0 += warp_sums[blockIdx.x * (kBinThreads / 32) + w];
    const uint32_t run = blockIdx.x * kBinTile + (uint32_t)warp * (32 * kBinItems) + lane;
#pragma unroll 2
    for (int k = 0; k < kBinItems; ++k) {
        const uint32_t i = run + (uint32_t)k * 32;
        uint32_t g = 0;
        bool keep = false;
        if (i < count) {
            g = indexes ? ld_nc_u32(indexes + i) : i;
            keep = rect_touches_owned(rects[g], own);
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const uint32_t at = w0 + __popc(bal & lanemask_lt());
            sub_idx[at] = g;
            sub_dist[at] = dist[i];
        }
        w0 += __popc(bal);
    }
}

__global__ void k_raster_init(RasterControl *rctl, SortControl *ctl, uint2 *ranges, uint32_t ntiles, uint32_t *super_sums, uint32_t nsuper, uint32_t *bin_totals, uint32_t *tile_order) {
    pdl_enter();
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    if (tid == 0) {
        rctl->total_instances = 0; rctl->overflow = 0; rctl->visible = 0; rctl->subset_count = 0;
        rctl->frame_seq += 1;
        ctl->error = 0;
    }
    uint32_t *h = &ctl->hist[0][0];
    for (size_t i = tid; i < 4 * kRadix; i += stride) h[i] = 0;
    for (size_t i = tid; i < ntiles; i += stride) ranges[i] = make_uint2(0xffffffffu, 0u); // empty: first > last
    for (size_t i = tid; i < (size_t)kVisibleSlots * 8; i += stride) rctl->visible_slots[i] = 0;
    for (size_t i = tid; i < nsuper; i += stride) super_sums[i] = 0;
    if (bin_totals) for (size_t i = tid; i < 1024; i += stride) bin_totals[i] = 0;
    for (size_t i = tid; i < ntiles; i += stride) tile_order[i] = (uint32_t)i;     // blend schedule: identity unless the counting-sort binning ranks the tiles
}

// ---------------------------------------------------------------------------------------------------------------
// Blend: one 64-thread CTA per fine tile (16x16 px); each thread owns a COLUMN of 4 pixels so that, per splat, the quad-local
// coordinates are evaluated once and stepped down the column with two adds per extra pixel (u += g1.y, w += g2.y).  CTAs of one
// coarse tile are adjacent in the grid so their common list stays in L1/L2.  Per 256 list entries: filter by mask bit (ballot
// compaction keeps draw order), then stage the survivors' records through shared memory 64 at a time and composite front to back.
constexpr int kBlendThreads = 64;
constexpr int kBlendPix = 4;                       // pixels per thread (a column)
constexpr int kBlendScan = 4 * kBlendThreads;      // list entries filtered per batch

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

template <int FORMAT>
__global__ void __launch_bounds__(kBlendThreads)
k_blend(const uint2 *__restrict__ ranges, const unsigned long long *__restrict__ list, const SplatRecord *__restrict__ rec, int tiles_x,
        int tiles_y, int coarse_x, uint32_t rank, uint32_t world, int width, int height, int flip_y, void *__restrict__ frame, const uint32_t *__restrict__ tile_order) {
    pdl_enter();
    __shared__ float4 s_rec[kBlendThreads][3];
    __shared__ uint32_t s_ids[kBlendScan];
    __shared__ uint32_t s_cnt[2][4][2];
    const uint32_t coarse = tile_order[blockIdx.x / kFinePerCoarse], sub = blockIdx.x % kFinePerCoarse;
    const int tx = (int)(coarse % (uint32_t)coarse_x) * kCoarseW + (int)(sub & (kCoarseW - 1));
    const int ty = (int)(coarse / (uint32_t)coarse_x) * kCoarseH + (int)(sub >> kCoarseShiftX);
    if (tx >= tiles_x || ty >= tiles_y) return;
    if (!owns_coarse((int)(coarse % (uint32_t)coarse_x), (int)(coarse / (uint32_t)coarse_x), rank, world)) return;   // another GPU's tile
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lx = lane & 15, ly0 = ((lane >> 4) + 2 * warp) * kBlendPix;     // column lx, rows ly0 .. ly0+3 of the tile
    const int x = tx * kTile + lx, y0 = ty * kTile + ly0;
    const float pxc = (float)x + 0.5f, pyc = (float)y0 + 0.5f;
    const float tile_y0 = (float)(ty * kTile);
    const uint32_t my_bit = 1u << warp;
    const uint2 rg = ranges[coarse];
    float T[kBlendPix], Cr[kBlendPix], Cg[kBlendPix], Cb[kBlendPix];
#pragma unroll
    for (int k = 0; k < kBlendPix; ++k) { T[k] = 1.0f; Cr[k] = Cg[k] = Cb[k] = 0.f; }
    bool done = !(x < width && y0 < height);
    int parity = 0;
    for (uint32_t base = rg.x; base < rg.y; base += kBlendScan) {
        if (__syncthreads_count(done) == kBlendThreads) break;
        // ---- filter 4 x 64 entries, order-preserving compaction (order: round k, warp, lane) ----------------------------------
        uint32_t ids[4], bal[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t i = base + (uint32_t)k * kBlendThreads + threadIdx.x;
            bool hit = false;
            ids[k] = 0;
            if (i < rg.y) {
                const unsigned long long e = __ldg(list + i);
                hit = ((uint32_t)(e >> 32) >> sub) & 1u;
                ids[k] = (uint32_t)e;
            }
            bal[k] = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) s_cnt[parity][k][warp] = __popc(bal[k]);
        }
        __syncthreads();
        uint32_t nsurv = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t c0 = s_cnt[parity][k][0], c1 = s_cnt[parity][k][1];
            const uint32_t off = nsurv + (warp ? c0 : 0u);
            if ((bal[k] >> lane) & 1u) s_ids[off + __popc(bal[k] & lanemask_lt())] = ids[k];
            nsurv += c0 + c1;
        }
        parity ^= 1;
        __syncthreads();
        // ---- composite the survivors, 64 records at a time ------------------------------------------------------------------
        for (uint32_t c0 = 0; c0 < nsurv; c0 += kBlendThreads) {
            const uint32_t j = c0 + threadIdx.x;
            if (j < nsurv) {
                const float4 *src = reinterpret_cast<const float4 *>(rec + s_ids[j]);
                const float4 a0 = __ldg(src);
                float4 a1 = __ldg(src + 1), a2 = __ldg(src + 2);
                // which warps (rows 0-7 / 8-15 of the tile) can the splat's AABB reach?  pixel-row index range of the AABB:
                const uint32_t hb = __float_as_uint(a1.z);
                const float hy = __high2float(*reinterpret_cast<const __half2 *>(&hb));
                const float yl = a0.y - hy - tile_y0 - 0.5f, yh = a0.y + hy - tile_y0 - 0.5f;
                const uint32_t wm = ((yl <= 7.0f && yh >= 0.0f) ? 1u : 0u) | ((yl <= 15.0f && yh >= 8.0f) ? 2u : 0u);
                a1.z = a0.w * a0.w + a1.y * a1.y;     // h = |d(u,w)/dy|^2 : second difference of q down a pixel column is 2h
                a2.w = __uint_as_float(wm);
                s_rec[threadIdx.x][0] = a0;
                s_rec[threadIdx.x][1] = a1;
                s_rec[threadIdx.x][2] = a2;
            }
            __syncthreads();
            const int nb = (int)min((uint32_t)kBlendThreads, nsurv - c0);
            if (!done) {
#pragma unroll 2
                for (int jj = 0; jj < nb; ++jj) {
                    const float4 r2 = s_rec[jj][2];
                    if (!(__float_as_uint(r2.w) & my_bit)) continue;     // warp-uniform: my 8 rows are outside the splat's AABB
                    const float4 r0 = s_rec[jj][0], r1 = s_rec[jj][1];
                    const float dx = pxc - r0.x, dy = pyc - r0.y;
                    const float u = dx * r0.z + dy * r0.w;    // quad-local coordinates of the first pixel of my column
                    const float w = dx * r1.x + dy * r1.y;
                    // q = u^2 + w^2 (A = 8 q; the fragment shader discards A > 8), stepped up the column by forward differences:
                    // q(y+1) - q(y) = 2 (u g1.y + w g2.y) + h,  second difference 2 h
                    float q[kBlendPix];
                    q[0] = u * u + w * w;
                    float dq = 2.0f * (u * r0.w + w * r1.y) + r1.z;
                    const float ddq = r1.z + r1.z;
#pragma unroll
                    for (int k = 1; k < kBlendPix; ++k) { q[k] = q[k - 1] + dq; dq += ddq; }
                    if (fminf(fminf(q[0], q[1]), fminf(q[2], q[3])) > 1.0f) continue;
#pragma unroll
                    for (int k = 0; k < kBlendPix; ++k) {
                        // exp(-0.5 A) * vColor.a with A = 8 q; zero outside the quad's inscribed disc (branch-free)
                        const float alpha = (q[k] <= 1.0f) ? ex2_approx(q[k] * -5.770780163555854f) * r1.w : 0.0f;
                        const float wgt = T[k] * alpha;
                        Cr[k] += wgt * r2.x; Cg[k] += wgt * r2.y; Cb[k] += wgt * r2.z;
                        T[k] -= wgt;                           // T *= (1 - alpha)
                    }
                    if (fmaxf(fmaxf(T[0], T[1]), fmaxf(T[2], T[3])) < kTransmittanceCutoff) { done = true; break; }
                }
            }
            __syncthreads();
        }
    }
    if (x < width) {
#pragma unroll
        for (int k = 0; k < kBlendPix; ++k) {
            const int y = y0 + k;
            if (y >= height) break;
            const float A = 1.0f - T[k]; // alpha accumulates as 1 - prod(1 - alpha_i)
            const int out_row = flip_y ? (height - 1 - y) : y;   // every rank writes its tiles into a full-size frame (others stay 0)
            const size_t at = (size_t)out_row * width + x;
            if (FORMAT == GS_FRAME_RGBA32F) {
                reinterpret_cast<float4 *>(frame)[at] = make_float4(Cr[k], Cg[k], Cb[k], A);
            } else {
                const uint32_t r8 = (uint32_t)(__saturatef(Cr[k]) * 255.0f + 0.5f), g8 = (uint32_t)(__saturatef(Cg[k]) * 255.0f + 0.5f);
                const uint32_t b8 = (uint32_t)(__saturatef(Cb[k]) * 255.0f + 0.5f), a8 = (uint32_t)(__saturatef(A) * 255.0f + 0.5f);
                reinterpret_cast<uint32_t *>(frame)[at] = r8 | (g8 << 8) | (b8 << 16) | (a8 << 24);
            }
        }
    }
    if (world > 1) __threadfence_system();   // the frame may live in a peer GPU's memory (fused tile gather): publish before the signal
}


// ---------------------------------------------------------------------------------------------------------------
// Blend v2: one CTA per fine tile; warp w owns an 8x8-px BLOCK of it, a lane owns two vertically adjacent pixels.  The fine tile is
// 16 px (S = 1: 4 warps) or 32 px (S = 2: 16 warps, frames beyond 256 coarse tiles of 128x64 px).  Differences from round 1's k_blend,
// all aimed at issuing fewer instructions (the blend is FP32-issue bound, not HBM bound):
//   * the thread that stages a splat record into shared memory also decides EXACTLY which of the tile's blocks the ellipse can
//     reach (minimum of the quadratic over the block's rectangle of pixel centres, ellipse_mask.h) -- no AABB-corner work at all;
//   * a warp then walks only the records that touch ITS block (one 32-bit word of touch bits per staging warp), ~45 instructions per
//     record for its 64 pixels, and stops on its own as soon as its 64 pixels are saturated;
//   * opacity is folded into the exponent (ex2(q * k + log2 a)), one multiply less per pixel.
// Same arithmetic otherwise: q = u^2 + w^2 from the inverse quad map, alpha = exp(-4 q) a for q <= 1 (A = 8 q <= 8), front to back.

// ---- 1-D bulk async copy (TMA unit) global -> shared with an mbarrier, used to prefetch the next batch of a coarse-tile list while the
// current batch is being composited (cp.async.bulk needs 16-byte aligned source / destination / size).
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// bounded wait: a protocol error must show up as a wrong picture in a test, never as a hung GPU
__device__ __forceinline__ bool mbar_wait(unsigned long long *bar, uint32_t parity) {
    for (int spin = 0; spin < (1 << 22); ++spin) {
        uint32_t done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) return true;
    }
    return false;
}

// ---- packed 2 x f32 arithmetic (sm_100: FFMA2 / FMUL2, one issue slot for two IEEE fp32 results; scalar operands broadcast for free)
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f32x2 bcast2(float v) { return pack2(v, v); }
__device__ __forceinline__ float lo2(f32x2 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return a; }
__device__ __forceinline__ float hi2(f32x2 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return b; }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

// Which of a tile's 8x8-px blocks can hold a pixel the splat covers: exact minimum of q over each block's rectangle of pixel
// centres (ellipse_mask.h), only for the blocks the ellipse's AABB reaches.  a0 = cx, cy, g1x, g1y; a1 = g2x, g2y, half2(hx, hy), alpha.
// NBX x NBY = blocks per tile row / column.  Not inlined: the caller's composite loop is register-bound and this runs once per staged record.
template <int NBX, int NBY>
__device__ __noinline__ uint32_t block_touch_mask(float4 a0, float4 a1, float tile_x0, float tile_y0) {
    if (!(a1.w > 0.0f)) return 0u;
    const uint32_t hb = __float_as_uint(a1.z);
    const __half2 hh = *reinterpret_cast<const __half2 *>(&hb);
    const float hx = __low2float(hh), hy = __high2float(hh);
    const float qxx = a0.z * a0.z + a1.x * a1.x, qxy = a0.z * a0.w + a1.x * a1.y, qyy = a0.w * a0.w + a1.y * a1.y;
    const float X0 = tile_x0 - a0.x, Y0 = tile_y0 - a0.y;      // first pixel centre of the tile, relative to the splat centre
    // block i spans [X0 + 8 i, X0 + 8 i + 7]; it meets [-hx, hx] iff  (-hx - X0 - 7) / 8 <= i <= (hx - X0) / 8
    const int ix0 = max(0, (int)ceilf((-hx - X0 - 7.0f) * 0.125f)), ix1 = min(NBX - 1, (int)floorf((hx - X0) * 0.125f));
    const int iy0 = max(0, (int)ceilf((-hy - Y0 - 7.0f) * 0.125f)), iy1 = min(NBY - 1, (int)floorf((hy - Y0) * 0.125f));
    // The AABB (exact extents of the ellipse) inside ONE block: that block holds the whole ellipse, nothing to decide.  (A block without
    // a pixel centre inside the ellipse can still pass here; it costs one visit that adds nothing.)
    if (ix0 == ix1 && iy0 == iy1) return 1u << (iy0 * NBX + ix0);
    uint32_t bm = 0;
#pragma unroll 1
    for (int iy = iy0; iy <= iy1; ++iy) {
        const float by0 = Y0 + (float)(8 * iy), by1 = by0 + 7.0f;
#pragma unroll 1
        for (int ix = ix0; ix <= ix1; ++ix) {
            const float bx0 = X0 + (float)(8 * ix), bx1 = bx0 + 7.0f;
            if (ellipse_min_q(bx0, bx1, by0, by1, qxx, qxy, qyy) <= 1.0f + kEllipseSlack) bm |= 1u << (iy * NBX + ix);
        }
    }
    return bm;
}

struct StatusSnapshot {
    const uint32_t *sort_ctl;     // SortControl head: 3 words (dmin, dmax, error)
    const uint32_t *raster_ctl;   // RasterControl
    uint32_t *dst;                // [0, 3) sort head, [4, 4 + sizeof(RasterControl) / 4) raster control; nullptr = no snapshot
    // multi-GPU peers: the frame pointer is rank 0's allocation; *half_src (0 / 1, RasterControl::peer_parity) selects its half
    const uint32_t *half_src;
    unsigned long long half_bytes;
};

template <int FORMAT, int S, int ROUNDS, bool TMA>
__global__ void __launch_bounds__(128 * S * S, S == 1 ? 8 : 2)
k_blend2(const uint2 *__restrict__ ranges, const unsigned long long *__restrict__ list, const SplatRecord *__restrict__ rec, int tiles_x,
         int tiles_y, int coarse_x, uint32_t rank, uint32_t world, int width, int height, int flip_y, void *__restrict__ frame_base, const uint32_t *__restrict__ tile_order,
         StatusSnapshot snap) {
    pdl_enter();
    void *__restrict__ frame = snap.half_src ? (void *)((unsigned char *)frame_base + (size_t)(*snap.half_src & 1u) * snap.half_bytes) : frame_base;
    // Everything the host reads back about a frame (sort error bits, instance / visibility counters, overflow flag) is final before the
    // blend starts; CTA 0 copies it into a per-frame-buffer slot so that the read-back can run on the copy stream, off this stream.
    if (snap.dst && blockIdx.x == 0) {
        if (threadIdx.x < 3) snap.dst[threadIdx.x] = snap.sort_ctl[threadIdx.x];
        for (uint32_t i = threadIdx.x; i < (uint32_t)(sizeof(RasterControl) / 4); i += blockDim.x) snap.dst[4 + i] = snap.raster_ctl[i];
    }
    // (A CTA covering TWO fine tiles side by side -- one scan of the coarse list for 32x16 px -- was measured: fewer instructions, but
    // the per-round barrier then waits for the densest of 8 blocks instead of 4 and the blend got 5-18 % slower.  Not kept.)
    constexpr int THREADS = 128 * S * S, WARPS = THREADS / 32, NBX = 2 * S, NBY = 2 * S, TILE = 16 * S;
    constexpr int BATCH = ROUNDS * THREADS;      // list entries per batch
    __shared__ float4 s_rec[THREADS + 1][3];    // [THREADS] = the null record (alpha 0) that pairs with an odd tail
    __shared__ uint32_t s_ids[BATCH];
    __shared__ uint32_t s_cnt[ROUNDS * WARPS + 1];   // [round][warp] survivors of the filter -> exclusive offsets; last = total
    __shared__ __align__(16) unsigned long long s_chunk[TMA ? 2 : 1][TMA ? BATCH + 2 : 2];   // list batches, double buffered, filled by bulk async copies (TMA)
    __shared__ __align__(8) unsigned long long s_mbar[2];
    __shared__ uint8_t s_list[WARPS][THREADS];  // [block][staging warp * 32 + k] indices of the staged records that reach the block, in order
    __shared__ uint8_t s_nlist[WARPS][WARPS];   // [block][staging warp] how many
    static_assert(THREADS <= 256 || sizeof(uint8_t) == 1, "");
    const uint32_t coarse = tile_order[blockIdx.x / kFinePerCoarse], sub = blockIdx.x % kFinePerCoarse;
    const int ccx = (int)(coarse % (uint32_t)coarse_x), ccy = (int)(coarse / (uint32_t)coarse_x);
    const int tx = ccx * kCoarseW + (int)(sub & (kCoarseW - 1)), ty = ccy * kCoarseH + (int)(sub >> kCoarseShiftX);
    if (tx >= tiles_x || ty >= tiles_y) return;
    if (!owns_coarse(ccx, ccy, rank, world)) return;   // another GPU's tile
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = tx * TILE + (warp % NBX) * 8 + (lane & 7), y0 = ty * TILE + (warp / NBX) * 8 + (lane >> 3) * 2;
    const float pxc = (float)x + 0.5f, pyc = (float)y0 + 0.5f;
    const float tile_x0 = (float)(tx * TILE) + 0.5f, tile_y0 = (float)(ty * TILE) + 0.5f;    // first pixel centre of the tile
    // pixels outside the frame start saturated so that they never keep a warp alive
    f32x2 T = pack2((x < width && y0 < height) ? 1.0f : 0.0f, (x < width && y0 + 1 < height) ? 1.0f : 0.0f);
    f32x2 Rr = pack2(0.f, 0.f), Gg = Rr, Bb = Rr;
    const f32x2 PY = pack2(pyc, pyc + 1.0f);
    bool wdone = !__any_sync(0xffffffffu, fmaxf(lo2(T), hi2(T)) >= kTransmittanceCutoff);
    const uint2 rg = ranges[coarse];
    const uint32_t lt = lanemask_lt();
    if (threadIdx.x < 3) s_rec[THREADS][threadIdx.x] = (threadIdx.x == 1) ? make_float4(0.f, 0.f, 0.f, __int_as_float(0xff800000)) : make_float4(0.f, 0.f, 0.f, 0.f);   // log2(alpha) = -inf
    // The tile's list is consumed in batches of BATCH entries.  Batch b+1 is fetched into the other half of s_chunk by ONE bulk async
    // copy (the TMA unit; completion on an mbarrier) while batch b is filtered, staged and composited, so a dense tile's critical path
    // never waits for list loads.  Copies start at an even entry (16-byte alignment): `skip` = 0 or 1 leading entry to ignore.
    auto issue = [&](uint32_t b) {        // thread 0 only
        const uint32_t start = rg.x + b * (uint32_t)BATCH, cnt = min((uint32_t)BATCH, rg.y - start);
        const uint32_t a0 = start & ~1u, a1 = (start + cnt + 1u) & ~1u, bytes = (a1 - a0) * 8u;
        fence_proxy_async_smem();
        mbar_expect_tx(&s_mbar[b & 1u], bytes);
        bulk_g2s(&s_chunk[b & 1u][0], list + a0, bytes, &s_mbar[b & 1u]);
    };
    // the radix binning path marks an empty tile (0xffffffff, 0): no batch (the u32 difference would wrap to one batch, and a bulk copy
    // would then be issued far outside the list)
    const uint32_t nbatch = rg.y > rg.x ? (rg.y - rg.x + BATCH - 1) / BATCH : 0u;
    if (TMA && threadIdx.x == 0) { mbar_init(&s_mbar[0], 1); mbar_init(&s_mbar[1], 1); mbar_fence_init(); }
    __syncthreads();
    if (TMA && threadIdx.x == 0 && nbatch) issue(0);
    uint32_t pending = (TMA && nbatch) ? 1u : 0u;      // batches issued so far (uniform)
    bool copy_ok = true;
    for (uint32_t b = 0; b < nbatch; ++b) {
        const uint32_t base = rg.x + b * (uint32_t)BATCH;
        if (__syncthreads_and(wdone)) break;
        const unsigned long long *chunk = list + base;
        if (TMA) {
            if (threadIdx.x == 0 && b + 1 < nbatch) issue(b + 1);      // its buffer was last read two barriers ago
            if (b + 1 < nbatch) pending = b + 2;
            copy_ok = mbar_wait(&s_mbar[b & 1u], (b >> 1) & 1u) && copy_ok;
            chunk = &s_chunk[b & 1u][base & 1u];
        }
        // ---- filter 4 x THREADS list entries by this tile's mask bit; order-preserving compaction (order: round, warp, lane) ------
        uint32_t ids[ROUNDS], bal[ROUNDS];
#pragma unroll
        for (int k = 0; k < ROUNDS; ++k) {
            const uint32_t i = base + (uint32_t)k * THREADS + threadIdx.x;
            bool hit = false;
            ids[k] = 0;
            if (i < rg.y) {
                const unsigned long long e = TMA ? chunk[(uint32_t)k * THREADS + threadIdx.x] : __ldg(chunk + (uint32_t)k * THREADS + threadIdx.x);
                hit = ((uint32_t)(e >> 32) >> sub) & 1u;
                ids[k] = (uint32_t)e;
            }
            bal[k] = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) s_cnt[k * WARPS + warp] = __popc(bal[k]);
        }
        __syncthreads();
        if (warp == 0) {      // exclusive scan of the 4 * WARPS counts
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
        // ---- stage up to THREADS survivors at a time, then every warp composites the ones that reach its block -------------------
        for (uint32_t c0 = 0; c0 < nsurv; c0 += THREADS) {
            const uint32_t j = c0 + threadIdx.x;
            uint32_t bm = 0;
            if (j < nsurv) {
                const float4 *src = reinterpret_cast<const float4 *>(rec + s_ids[j]);
                float4 a0 = __ldg(src), a1 = __ldg(src + 1);
                const float4 a2 = __ldg(src + 2);
                // a0 = cx, cy, g1x, g1y ; a1 = g2x, g2y, half2(hx, hy), alpha ; a2 = r, g, b, ndc z
                bm = block_touch_mask<NBX, NBY>(a0, a1, tile_x0, tile_y0);
                // staged form: u(p) = g1 . p + u0, w(p) = g2 . p + w0 at a pixel centre p (two FMAs each in the loop below)
                const float u0 = -fmaf(a0.x, a0.z, a0.y * a0.w), w0 = -fmaf(a0.x, a1.x, a0.y * a1.y);
                a1.z = a0.w * a0.w + a1.y * a1.y;     // h = |d(u,w)/dy|^2
                a1.w = log2f(a1.w);                   // opacity folded into the exponent
                a0.x = u0; a0.y = w0;
                s_rec[threadIdx.x][0] = a0;           // u0, w0, g1x, g1y
                s_rec[threadIdx.x][1] = a1;           // g2x, g2y, h, log2(alpha)
                s_rec[threadIdx.x][2] = a2;
            }
            // per block: the indices of this staging warp's records that reach it, compacted in order
#pragma unroll
            for (int b = 0; b < WARPS; ++b) {
                const uint32_t v = __ballot_sync(0xffffffffu, (bm >> b) & 1u);
                if ((bm >> b) & 1u) s_list[b][warp * 32 + __popc(v & lt)] = (uint8_t)(threadIdx.x & 255);
                if (lane == 0) s_nlist[b][warp] = (uint8_t)__popc(v);
            }
            __syncthreads();
            if (!wdone) {
#pragma unroll 1
                for (int sw = 0; sw < WARPS && !wdone; ++sw) {
                    const int cnt = s_nlist[warp][sw];
                    const uint8_t *lst = &s_list[warp][sw * 32];
                    const int jbase = (THREADS > 256 ? (sw & ~7) * 32 : 0);      // 8-bit index inside the group of 8 staging warps
                    // Two records per iteration: their quad coordinates and exponentials are independent, only the transmittance chain is
                    // serial.  The blend's duration is set by the longest per-warp chain (the densest block), not by issue slots, so the
                    // instruction-level parallelism matters more than the instruction count.  An odd tail pairs with the null record.
#pragma unroll 1
                    for (int k = 0; k < cnt; k += 2) {
                        const int ja = jbase + lst[k];
                        const int jb = (k + 1 < cnt) ? jbase + lst[k + 1] : THREADS;
                        const float4 A = s_rec[ja][0], B = s_rec[ja][1], C = s_rec[ja][2];
                        const float4 D = s_rec[jb][0], E = s_rec[jb][1], F = s_rec[jb][2];
                        // the lane's two pixels ride in the halves of packed f32x2 registers (FFMA2 / FMUL2: one issue slot for both);
                        // per-record scalars enter as broadcast operands
                        const float tua = fmaf(pxc, A.z, A.x), twa = fmaf(pxc, B.x, A.y);
                        const float tub = fmaf(pxc, D.z, D.x), twb = fmaf(pxc, E.x, D.y);
                        const f32x2 Ua = fma2(PY, bcast2(A.w), bcast2(tua)), Wa = fma2(PY, bcast2(B.y), bcast2(twa));
                        const f32x2 Ub = fma2(PY, bcast2(D.w), bcast2(tub)), Wb = fma2(PY, bcast2(E.y), bcast2(twb));
                        const f32x2 Qa = fma2(Wa, Wa, mul2(Ua, Ua)), Qb = fma2(Wb, Wb, mul2(Ub, Ub));
                        // exp(-0.5 A) * vColor.a with A = 8 q, zero outside the quad's inscribed disc
                        const f32x2 Xa = fma2(Qa, bcast2(-5.770780163555854f), bcast2(B.w)), Xb = fma2(Qb, bcast2(-5.770780163555854f), bcast2(E.w));
                        const float ea0 = (lo2(Qa) <= 1.0f) ? ex2_approx(lo2(Xa)) : 0.0f, ea1 = (hi2(Qa) <= 1.0f) ? ex2_approx(hi2(Xa)) : 0.0f;
                        const float eb0 = (lo2(Qb) <= 1.0f) ? ex2_approx(lo2(Xb)) : 0.0f, eb1 = (hi2(Qb) <= 1.0f) ? ex2_approx(hi2(Xb)) : 0.0f;
                        f32x2 wgt = mul2(T, pack2(ea0, ea1));
                        Rr = fma2(wgt, bcast2(C.x), Rr); Gg = fma2(wgt, bcast2(C.y), Gg); Bb = fma2(wgt, bcast2(C.z), Bb);
                        T = fma2(wgt, bcast2(-1.0f), T);                                   // T *= (1 - alpha)
                        wgt = mul2(T, pack2(eb0, eb1));
                        Rr = fma2(wgt, bcast2(F.x), Rr); Gg = fma2(wgt, bcast2(F.y), Gg); Bb = fma2(wgt, bcast2(F.z), Bb);
                        T = fma2(wgt, bcast2(-1.0f), T);
                        if (!__any_sync(0xffffffffu, fmaxf(lo2(T), hi2(T)) >= kTransmittanceCutoff)) { wdone = true; break; }
                    }
                }
            }
            if (__syncthreads_and(wdone)) break;      // every pixel of the tile is saturated: the rest of the batch cannot change it
        }
    }
    // a CTA must not retire while a bulk copy into its shared memory is in flight: wait for the last batch issued (if it was not consumed)
    if (TMA) {
        __syncthreads();
        const uint32_t last = pending ? pending - 1u : 0u;
        if (pending && threadIdx.x == 0) copy_ok = mbar_wait(&s_mbar[last & 1u], (last >> 1) & 1u) && copy_ok;
        // (a batch that WAS consumed has completed its phase already: the wait returns at once)
    }
    float T0 = lo2(T), T1 = hi2(T), r0 = lo2(Rr), r1 = hi2(Rr), g0 = lo2(Gg), g1 = hi2(Gg), b0 = lo2(Bb), b1 = hi2(Bb);
    if (!copy_ok) { T0 = T1 = 0.5f; r0 = r1 = 1.0f; g0 = g1 = 0.0f; b0 = b1 = 1.0f; }      // protocol failure: paint the pixels magenta so that every comparison fails
    if (x < width) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int y = y0 + k;
            if (y < height) {
                const float Tk = k ? T1 : T0, Rk = k ? r1 : r0, Gk = k ? g1 : g0, Bk = k ? b1 : b0;
                const float A = 1.0f - Tk;      // alpha accumulates as 1 - prod(1 - alpha_i)
                const int out_row = flip_y ? (height - 1 - y) : y;   // every rank writes its tiles into a full-size frame
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
    if (world > 1) __threadfence_system();   // the frame may live in a peer GPU's memory (fused tile gather): publish before the signal
}

// records -> the ABI's gs_projected_splat (basis vectors recovered from g = B/|B|^2)
__global__ void k_export_projected(const SplatRecord *__restrict__ rec, const ushort4 *__restrict__ rects, uint32_t count, gs_projected_splat *out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= count) return;
    const SplatRecord r = rec[s];
    gs_projected_splat o;
    o.cx = r.cx; o.cy = r.cy;
    const float n1 = r.g1x * r.g1x + r.g1y * r.g1y, n2 = r.g2x * r.g2x + r.g2y * r.g2y;
    o.b1x = n1 > 0.f ? r.g1x / n1 : 0.f; o.b1y = n1 > 0.f ? r.g1y / n1 : 0.f;
    o.b2x = n2 > 0.f ? r.g2x / n2 : 0.f; o.b2y = n2 > 0.f ? r.g2y / n2 : 0.f;
    o.r = r.r; o.g = r.g; o.b = r.b; o.a = r.a;
    o.ndc_z = r.ndc_z;
    o.valid = (r.ndc_z >= -1.0f && r.ndc_z <= 1.0f) ? 1u : 0u;
    if (!o.valid) o.ndc_z = 0.f;
    out[s] = o;
}

} // namespace gs
#include "surfel_kernels.cuh"   // the 2D (surfel) render mode's projection and blend
namespace gs {

// ---------------------------------------------------------------------------------------------------------------
// Host side of the rasteriser
template <typename T> struct RBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaError_t ensure(size_t count) {
        if (count <= n) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; n = 0;
        cudaError_t e = cudaMalloc((void **)&p, (count ? count : 1) * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

struct RasterState {
    int render_mode = GS_RENDER_MODE_3D;   // gs_config.splat_render_mode, fixed at create time
    RBuf<uint4> cc;
    RBuf<unsigned char> cov, sh;
    RBuf<uint32_t> scene_idx;
    int cov_format = GS_COV_F32, sh_format = GS_SH_NONE;
    uint32_t sh_degree = 0, uploaded = 0;
    bool have_scene_idx = false;
    RBuf<SplatRecord> records;
    RBuf<float> srot;           // 2D: scale/rotation texture, 6 x f32 per splat
    RBuf<SurfelRecord> surfels; // 2D: projected records (instead of `records`)
    RBuf<gs_projected_surfel> exported2d;
    RBuf<ushort4> rects;
    RBuf<uint32_t> block_sums; // coarse instances per chunk of draw ranks
    RBuf<uint32_t> warp_sums;  // ... and per warp (256 draw ranks) inside the chunk
    RBuf<uint32_t> super_sums; // ... and per group of kBinThreads chunks: [0, S) binning, [S, 2S) subset compaction
    uint32_t super_stride = 0;
    RBuf<uint16_t> ikeys[2];   // instance keys ping/pong (coarse tile ids)
    RBuf<unsigned long long> ivals[2];   // instance values ping/pong: {fine-tile mask, splat id}
    RBuf<unsigned long long> list;       // final per-coarse-tile lists
    RBuf<uint2> ranges;
    RBuf<RasterControl> rctl;
    RBuf<SortControl> sctl;
    RBuf<uint32_t> tile_hist;   // radix tile histograms
    RBuf<uint32_t> bin_hist;    // binning v2: [coarse tile][chunk] instance counts -> offsets
    RBuf<ushort4> rect_by_rank; // binning v2: the rects gathered in draw-rank order by k_bin_count
    RBuf<uint32_t> tile_order;  // blend schedule: coarse tiles by list length, longest first
    RBuf<uint32_t> bin_totals;  // binning v2: instances per coarse tile (1024 words, zeroed by k_raster_init)
    uint32_t bin_stride = 0;
    int bin_cfg = 0;
    int bin_compact = 1;        // GS_BIN_COMPACT=0: k_bin_place without the warp-level compaction of culled splats (A/B)
    int bin_version = 2, blend_version = 2;   // GS_BIN / GS_BLEND = 1 selects the round-1 kernels (A/B measurements)
    int blend_tma = 0, blend_rounds = 4;      // GS_BLEND_TMA = 1: bulk-async list prefetch; GS_BLEND_ROUNDS = 2 / 4 (16-px tiles)
    RBuf<DynamicUniforms> dyn;
    RBuf<ProjParams> projp;     // per-frame projection parameters (device copy read by k_project)
    RBuf<unsigned char> frame;
    RBuf<unsigned char> frame_alt;   // second device frame: pipelined frames (gs_frame_begin) alternate so a D2H copy can overlap the next frame
    unsigned char *frame_half2 = nullptr;   // multi-GPU rank 0 with a double-size exported frame allocation: its second half (instead of frame_alt)
    size_t frame_half_bytes = 0;
    int frame_parity = 0;
    // status snapshot taken by the blend kernel (see StatusSnapshot): destination slots [parity * snap_stride], source sort control
    uint32_t *snap_base = nullptr;
    uint32_t snap_stride = 0;
    const uint32_t *snap_sort_ctl = nullptr;
    bool snapshot_taken = false;   // the last raster_render launched a blend that wrote the snapshot
    RBuf<gs_projected_splat> exported;
    // fused tile gather over NVLink peer memory (world_size > 1)
    RBuf<PeerSync> peer_sync_local;      // rank 0 owns the block
    PeerSync *peer_sync = nullptr;       // rank 0: local block; others: rank 0's block mapped through CUDA IPC
    void *peer_frame = nullptr;          // others: rank 0's frame buffer mapped through CUDA IPC
    bool peer_root = false, peer_attached = false;
    unsigned long long instance_capacity = 0;
    // binning of the last frame (GS_BUF_TILE_INFO): coarse tiles, fine-tile edge in px, path (2 = counting sort, 1 = radix sort)
    uint32_t last_ncoarse = 0, last_tile_px = 0, last_bin_path = 0;
    uint32_t hist_stride = 0;
    int sm_count = 148;
    int last_format = GS_FRAME_RGBA32F;
    size_t last_frame_bytes = 0;
};

#define RCU(call)                                                                                                 \
    do {                                                                                                          \
        cudaError_t _e = (call);                                                                                  \
        if (_e != cudaSuccess) { snprintf(raster_err(), 512, "%s -> %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); return GS_ERR_CUDA; } \
    } while (0)

static inline char *raster_err() { return g_gs_err; }

static int raster_init(RasterState &rs, const gs_config &c, int sm_count) {
    rs.sm_count = sm_count;
    rs.render_mode = c.splat_render_mode;
    const size_t n = c.max_splat_count ? c.max_splat_count : 1;
    RCU(rs.rctl.ensure(1));
    RCU(cudaMemset(rs.rctl.p, 0, sizeof(RasterControl)));   // k_raster_init resets the per-frame fields only (peer flags, frame count)
    RCU(rs.sctl.ensure(1));
    RCU(rs.dyn.ensure(2));          // per-frame parameter blocks: one per frame-buffer parity (pipelined frames upload them off-stream)
    RCU(rs.projp.ensure(2));
    RCU(cudaMemset(rs.dyn.p, 0, 2 * sizeof(DynamicUniforms)));
    if (c.max_width && c.max_height) {
        RCU(rs.cc.ensure(n));
        if (rs.render_mode == GS_RENDER_MODE_2D) { RCU(rs.surfels.ensure(n)); RCU(rs.srot.ensure(6 * n)); }
        else RCU(rs.records.ensure(n));
        RCU(rs.rects.ensure(n));
        RCU(rs.block_sums.ensure((n + kBinTile - 1) / kBinTile + 1));
        RCU(rs.warp_sums.ensure(((n + kBinTile - 1) / kBinTile + 1) * (kBinThreads / 32)));
        rs.super_stride = (uint32_t)(((n + kBinTile - 1) / kBinTile) / kBinThreads + 2);
        RCU(rs.super_sums.ensure(2 * (size_t)rs.super_stride));
        const char *f = getenv("GS_INSTANCE_FACTOR");
        const double factor = f ? atof(f) : 4.0;
        const size_t tiles = (size_t)((c.max_width + kTile - 1) / kTile) * ((c.max_height + kTile - 1) / kTile);
        rs.instance_capacity = (unsigned long long)(factor * (double)n) + 4ull * tiles + 65536ull;
        if (rs.instance_capacity > 0xfffffff0ull) rs.instance_capacity = 0xfffffff0ull;
        for (int i = 0; i < 2; ++i) { RCU(rs.ikeys[i].ensure(rs.instance_capacity)); RCU(rs.ivals[i].ensure(rs.instance_capacity)); }
        // +2: k_blend2's bulk list copies start and end on an even entry, so a list ending at the capacity may read one entry beyond it
        RCU(rs.list.ensure(rs.instance_capacity + 2));
        RCU(rs.ranges.ensure(65536));
        RCU(rs.tile_order.ensure(65536));
        RCU(rs.frame.ensure((size_t)c.max_width * (c.max_height + kTile) * 16));
        RCU(rs.tile_hist.ensure(radix_tile_hist_words(rs.instance_capacity, 2, &rs.hist_stride)));
        if (const char *v = getenv("GS_BIN")) rs.bin_version = atoi(v);
        if (const char *v = getenv("GS_BLEND")) rs.blend_version = atoi(v);
        if (const char *v = getenv("GS_BIN_COMPACT")) rs.bin_compact = atoi(v);
        if (const char *v = getenv("GS_BLEND_TMA")) rs.blend_tma = atoi(v);
        if (const char *v = getenv("GS_BLEND_ROUNDS")) rs.blend_rounds = atoi(v);
        if (const char *v = getenv("GS_BINCFG")) rs.bin_cfg = atoi(v);
        {   // binning v2: one column of chunk counts per coarse tile (2048 draw ranks per chunk in both configurations)
            const size_t coarse = (size_t)((c.max_width + kTile * kCoarseW - 1) / (kTile * kCoarseW)) * ((c.max_height + kTile * kCoarseH - 1) / (kTile * kCoarseH));
            const size_t chunks = (n + 2047) / 2048 + 1;
            rs.bin_stride = (uint32_t)((chunks + 31) & ~(size_t)31);
            RCU(rs.bin_hist.ensure(std::max<size_t>(coarse, 1) * rs.bin_stride));
            RCU(rs.rect_by_rank.ensure(n));
            RCU(rs.bin_totals.ensure(1024));
            RCU(cudaMemset(rs.bin_totals.p, 0, 1024 * 4));
        }
    }
    return GS_OK;
}

static void raster_release(RasterState &rs) {
    rs.cc.release(); rs.cov.release(); rs.sh.release(); rs.scene_idx.release(); rs.records.release(); rs.rects.release();
    rs.srot.release(); rs.surfels.release(); rs.exported2d.release();
    rs.block_sums.release(); rs.warp_sums.release(); rs.super_sums.release(); rs.ikeys[0].release(); rs.ikeys[1].release(); rs.ivals[0].release(); rs.ivals[1].release();
    rs.list.release(); rs.ranges.release(); rs.rctl.release(); rs.sctl.release(); rs.tile_hist.release(); rs.bin_hist.release(); rs.bin_totals.release(); rs.rect_by_rank.release(); rs.tile_order.release();
    rs.dyn.release(); rs.projp.release(); rs.frame.release(); rs.frame_alt.release(); rs.peer_sync_local.release(); rs.exported.release();
}

static int raster_upload(RasterState &rs, const gs_config &c, const gs_splat_data &d, cudaStream_t st) {
    if (!c.max_width || !c.max_height) { snprintf(raster_err(), 512, "engine created without a framebuffer (max_width/max_height = 0)"); return GS_ERR_NOT_READY; }
    if ((uint64_t)d.from + d.count > c.max_splat_count) { snprintf(raster_err(), 512, "splat data [%u,%u) exceeds max_splat_count %u", d.from, d.from + d.count, c.max_splat_count); return GS_ERR_CAPACITY; }
    const bool two_d = rs.render_mode == GS_RENDER_MODE_2D;
    if (!d.centers_colors) { snprintf(raster_err(), 512, "gs_upload_splat_data: null centers_colors"); return GS_ERR_BAD_ARG; }
    if (!two_d && !d.covariances) { snprintf(raster_err(), 512, "gs_upload_splat_data: null covariances"); return GS_ERR_BAD_ARG; }
    if (two_d && !d.scale_rotations) { snprintf(raster_err(), 512, "gs_upload_splat_data: a TwoD (surfel) engine needs scale_rotations (6 floats per splat)"); return GS_ERR_BAD_ARG; }
    if (d.sh_degree > 2) { snprintf(raster_err(), 512, "sh_degree %u > 2", d.sh_degree); return GS_ERR_BAD_ARG; }
    const size_t n = c.max_splat_count;
    const size_t cov_elt = d.cov_format == GS_COV_F16 ? 12 : 24;
    const size_t ncomp = d.sh_degree == 2 ? 24 : (d.sh_degree == 1 ? 9 : 0);
    const size_t sh_elt = ncomp * (d.sh_format == GS_SH_F16 ? 2 : (d.sh_format == GS_SH_U8 ? 1 : 4));
    if (d.from == 0) rs.uploaded = 0; // a (re)upload from splat 0 may change the storage formats
    if (rs.uploaded && (rs.cov_format != d.cov_format || (rs.sh_degree != d.sh_degree) || (ncomp && rs.sh_format != d.sh_format))) {
        snprintf(raster_err(), 512, "splat data format changed between partial uploads"); return GS_ERR_BAD_ARG;
    }
    rs.cov_format = d.cov_format;
    rs.sh_degree = d.sh_degree;
    rs.sh_format = ncomp ? d.sh_format : GS_SH_NONE;
    if (!two_d) RCU(rs.cov.ensure(n * cov_elt + 16));
    if (ncomp) {
        if (!d.spherical_harmonics) { snprintf(raster_err(), 512, "sh_degree %u without spherical_harmonics", d.sh_degree); return GS_ERR_BAD_ARG; }
        RCU(rs.sh.ensure(n * sh_elt + 16));
    }
    RCU(cudaMemcpyAsync(rs.cc.p + d.from, d.centers_colors, (size_t)d.count * 16, cudaMemcpyHostToDevice, st));
    if (two_d) RCU(cudaMemcpyAsync(rs.srot.p + (size_t)d.from * 6, d.scale_rotations, (size_t)d.count * 24, cudaMemcpyHostToDevice, st));
    else RCU(cudaMemcpyAsync(rs.cov.p + (size_t)d.from * cov_elt, d.covariances, (size_t)d.count * cov_elt, cudaMemcpyHostToDevice, st));
    if (ncomp) RCU(cudaMemcpyAsync(rs.sh.p + (size_t)d.from * sh_elt, d.spherical_harmonics, (size_t)d.count * sh_elt, cudaMemcpyHostToDevice, st));
    if (d.scene_indexes) {
        RCU(rs.scene_idx.ensure(n));
        RCU(cudaMemcpyAsync(rs.scene_idx.p + d.from, d.scene_indexes, (size_t)d.count * 4, cudaMemcpyHostToDevice, st));
        rs.have_scene_idx = true;
    }
    rs.uploaded = std::max<uint32_t>(rs.uploaded, d.from + d.count);
    return GS_OK;
}

static unsigned char *raster_second_frame(RasterState &rs) { return rs.frame_alt.p ? rs.frame_alt.p : rs.frame_half2; }
static void *raster_frame_ptr(RasterState &rs, int) { return (rs.frame_parity && raster_second_frame(rs)) ? raster_second_frame(rs) : rs.frame.p; }

template <bool COVF16>
static void launch_project(RasterState &rs, uint32_t count, cudaStream_t st) {
    const int blocks = (int)((count + kProjThreads - 1) / kProjThreads);
    const uint32_t *sc = rs.have_scene_idx ? rs.scene_idx.p : nullptr;
#define GS_PROJ(FMT) gs_launch(k_project<COVF16, FMT>, blocks, kProjThreads, 0, st, rs.cc.p, rs.cov.p, rs.sh.p, (int)rs.sh_degree, sc, rs.dyn.p + rs.frame_parity, rs.projp.p + rs.frame_parity, count, rs.records.p, rs.rects.p, rs.rctl.p)
    switch (rs.sh_format) {
        case GS_SH_F16: GS_PROJ(GS_SH_F16); break;
        case GS_SH_U8: GS_PROJ(GS_SH_U8); break;
        case GS_SH_F32: GS_PROJ(GS_SH_F32); break;
        default: GS_PROJ(GS_SH_NONE); break;
    }
#undef GS_PROJ
}

template <bool EXPORT>
static void launch_project2d(RasterState &rs, uint32_t count, cudaStream_t st, gs_projected_surfel *exp) {
    const int blocks = (int)((count + kProjThreads - 1) / kProjThreads);
    const uint32_t *sc = rs.have_scene_idx ? rs.scene_idx.p : nullptr;
#define GS_PROJ2D(FMT) gs_launch(k_project2d<FMT, EXPORT>, blocks, kProjThreads, 0, st, rs.cc.p, rs.srot.p, rs.sh.p, (int)rs.sh_degree, sc, rs.dyn.p + rs.frame_parity, rs.projp.p + rs.frame_parity, count, rs.surfels.p, rs.rects.p, rs.rctl.p, exp)
    switch (rs.sh_format) {
        case GS_SH_F16: GS_PROJ2D(GS_SH_F16); break;
        case GS_SH_U8: GS_PROJ2D(GS_SH_U8); break;
        case GS_SH_F32: GS_PROJ2D(GS_SH_F32); break;
        default: GS_PROJ2D(GS_SH_NONE); break;
    }
#undef GS_PROJ2D
}

// Fine-tile edge for a frame: 16 px while that gives at most 256 coarse tiles (8 x 4 fine tiles each: one counting-sort pass with 8-bit
// bins, 1920x1080 = 255), else 32 px (3840x2160 = 255 coarse tiles of 256 x 128 px).  Larger frames keep 32 px and the multi-pass path.
static inline int frame_tile_shift(uint32_t width, uint32_t height) {
    const uint32_t cx = (width + kTile * kCoarseW - 1) / (kTile * kCoarseW), cy = (height + kTile * kCoarseH - 1) / (kTile * kCoarseH);
    return (cx * cy <= 256u) ? kTileShift : kTileShift + 1;
}

static int raster_upload_params(RasterState &rs, const gs_config &c, const gs_uniforms &u, const gs_render_params &p, cudaStream_t st) {
    const int tshift = frame_tile_shift(p.width, p.height), tpx = 1 << tshift;
    const int tiles_x = (p.width + tpx - 1) / tpx, tiles_y = (p.height + tpx - 1) / tpx;
    const uint32_t world = c.world_size, rank = c.rank;
    const bool upload_params = true;
    ProjParams P{};
    memcpy(P.mv, u.model_view, 64); memcpy(P.proj, u.projection, 64);
    memcpy(P.cam, u.camera_position, 12);
    P.focal[0] = u.focal[0]; P.focal[1] = u.focal[1]; P.viewport[0] = u.viewport[0]; P.viewport[1] = u.viewport[1];
    P.inv_focal_adj = u.inverse_focal_adjustment; P.ortho_zoom = u.ortho_zoom; P.orthographic = u.orthographic_mode;
    P.splat_scale = u.splat_scale; P.point_cloud = u.point_cloud_mode; P.sh_degree = u.sh_degree; P.antialiased = u.antialiased;
    P.kernel2d = u.kernel_2d_size; P.max_size = u.max_screen_space_splat_size; P.fade_in_complete = u.fade_in_complete;
    memcpy(P.scene_center, u.scene_center, 12); P.fade_start = u.visible_region_fade_start_radius;
    P.dynamic = u.dynamic_mode; P.optional_effects = u.enable_optional_effects; P.scene_count = (int)u.scene_count;
    P.tiles_x = tiles_x; P.tiles_y = tiles_y; P.rank = rank; P.world = world; P.width = (int)p.width; P.height = (int)p.height;
    P.tile_shift = tshift;
    if (upload_params) RCU(cudaMemcpyAsync(rs.projp.p + rs.frame_parity, &P, sizeof(P), cudaMemcpyHostToDevice, st)); // pageable source: staged before return
    if (upload_params && (u.dynamic_mode || u.enable_optional_effects || rs.sh_format == GS_SH_U8)) {
        DynamicUniforms du;
        memcpy(du.view, u.view_matrix, 64);
        memcpy(du.transforms, u.scene_transforms, sizeof(du.transforms));
        memcpy(du.sh8_min, u.sh8_min, sizeof(du.sh8_min)); memcpy(du.sh8_max, u.sh8_max, sizeof(du.sh8_max));
        memcpy(du.opacity, u.scene_opacity, sizeof(du.opacity)); memcpy(du.visibility, u.scene_visibility, sizeof(du.visibility));
        RCU(cudaMemcpyAsync(rs.dyn.p + rs.frame_parity, &du, sizeof(du), cudaMemcpyHostToDevice, st)); // pageable source: staged before return
    }

    return GS_OK;
}

static int raster_render(RasterState &rs, const gs_config &c, const gs_uniforms &u, const gs_render_params &p, const uint32_t *d_order,
                         cudaStream_t st, cudaEvent_t ev_project, cudaEvent_t ev_bin, gs_timings &tm, Profiler &prof, bool upload_params, bool record_events,
                         int phases = 3, const unsigned long long *order_count_dev = nullptr) {
    if (!rs.uploaded) { snprintf(raster_err(), 512, "gs_render before gs_upload_splat_data"); return GS_ERR_NOT_READY; }
    if (p.width == 0 || p.height == 0 || p.width > c.max_width || p.height > c.max_height) {
        snprintf(raster_err(), 512, "frame %ux%u outside the engine's %ux%u", p.width, p.height, c.max_width, c.max_height); return GS_ERR_BAD_ARG;
    }
    if (p.render_count > rs.uploaded) { snprintf(raster_err(), 512, "render_count %u > uploaded splats %u", p.render_count, rs.uploaded); return GS_ERR_CAPACITY; }
    const int tshift = frame_tile_shift(p.width, p.height), tpx = 1 << tshift;
    const int tiles_x = (p.width + tpx - 1) / tpx, tiles_y = (p.height + tpx - 1) / tpx;
    const uint32_t world = c.world_size, rank = c.rank;
    const uint32_t local_tiles = (uint32_t)tiles_x * (uint32_t)tiles_y;
    uint32_t launches = 0;

    if (upload_params) { int prc = raster_upload_params(rs, c, u, p, st); if (prc) return prc; }
    const int coarse_x = (tiles_x + kCoarseW - 1) / kCoarseW, coarse_y = (tiles_y + kCoarseH - 1) / kCoarseH;
    const uint32_t ncoarse = (uint32_t)coarse_x * (uint32_t)coarse_y;
    if (ncoarse > 65536u) { snprintf(raster_err(), 512, "frame %ux%u needs %u coarse tiles (> 65536)", p.width, p.height, ncoarse); return GS_ERR_BAD_ARG; }
    if (world > 1 && coarse_x - 1 + coarse_y - 1 > kMaxOwnDiag) {
        snprintf(raster_err(), 512, "frame %ux%u is too long for sharded rendering: its coarse-tile diagonal cx + cy reaches %d (at most %d with world_size > 1)",
                 p.width, p.height, coarse_x - 1 + coarse_y - 1, kMaxOwnDiag);
        return GS_ERR_BAD_ARG;
    }
    int tile_bits = 1;
    while ((1u << tile_bits) < std::max(ncoarse, 2u)) ++tile_bits;
    const PassPlan pl = make_plan_bits(tile_bits);
    if (phases & 1) {
        gs_launch(k_raster_init, 8, 256, 0, st, rs.rctl.p, rs.sctl.p, rs.ranges.p, ncoarse, rs.super_sums.p, 2 * rs.super_stride, rs.bin_totals.p, rs.tile_order.p);
        ++launches;
        prof.mark("k_raster_init", st);
        // rank 0 frees its frame buffer for the peers' stores right at the START of the frame (everything that consumed the previous
        // picture is earlier in stream order), so their blends never wait for rank 0's own sort + binning
        if (world > 1 && rs.peer_root) { k_peer_release<<<1, 1, 0, st>>>(rs.peer_sync, rs.rctl.p, (uint32_t)(rs.frame_parity && rs.frame_half2)); ++launches; }
        const uint32_t count = rs.uploaded;
        if (rs.render_mode == GS_RENDER_MODE_2D) {
            launch_project2d<false>(rs, count, st, nullptr);
            ++launches;
            prof.mark("k_project2d", st);
        } else {
            if (rs.cov_format == GS_COV_F16) launch_project<true>(rs, count, st); else launch_project<false>(rs, count, st);
            ++launches;
            prof.mark("k_project", st);
        }
        if (record_events) RCU(cudaEventRecord(ev_project, st));
    }
    if (!(phases & 2)) { tm.kernel_launches = launches; return GS_OK; }
    rs.snapshot_taken = false;
    const bool bin2 = rs.bin_version >= 2 && ncoarse <= 256u;
    rs.last_ncoarse = ncoarse; rs.last_tile_px = (uint32_t)tpx; rs.last_bin_path = bin2 ? 2u : 1u;
    if (p.render_count && local_tiles && bin2) {
        const OwnMask own = make_own_mask(rank, world);
        const int sharded = world > 1 ? 1 : 0;
        const uint32_t chunks = (p.render_count + kBinRanks - 1u) / kBinRanks;
#define GS_BIN_COUNT(C) gs_launch(k_bin_count<C>, chunks, Bin2Cfg<C>::kWarps * 32, 0, st, d_order, p.render_count, order_count_dev, rs.rects.p, coarse_x, ncoarse, rs.bin_hist.p, rs.bin_stride, rs.bin_totals.p, rs.rect_by_rank.p, own, sharded)
#define GS_BIN_PLACE(C) gs_launch(k_bin_place<C>, chunks, Bin2Cfg<C>::kWarps * 32, 0, st, d_order, p.render_count, order_count_dev, rs.rect_by_rank.p, coarse_x, ncoarse, rs.bin_hist.p, rs.bin_stride, rs.list.p, rs.instance_capacity, rs.rctl.p, own, sharded, (rs.bin_compact && tiles_x <= 256 && tiles_y <= 256) ? 1 : 0)
        if (rs.bin_cfg == 0) GS_BIN_COUNT(0); else GS_BIN_COUNT(1);
        ++launches;
        prof.mark("k_bin_count", st);
        gs_launch(k_bin_scan, ncoarse, 1024, 0, st, rs.bin_hist.p, rs.bin_stride, (uint32_t)kBinRanks, p.render_count, order_count_dev, rs.bin_totals.p, ncoarse, rs.ranges.p, rs.rctl.p, rs.tile_order.p,
                  rs.instance_capacity);
        ++launches;
        prof.mark("k_bin_scan", st);
        if (rs.bin_cfg == 0) GS_BIN_PLACE(0); else GS_BIN_PLACE(1);
#undef GS_BIN_COUNT
#undef GS_BIN_PLACE
        ++launches;
        prof.mark("k_bin_place", st);
    }
    if (p.render_count && local_tiles && !bin2) {
        const uint32_t chunks = (p.render_count + kBinTile - 1) / kBinTile;
        gs_launch(k_tile_count, chunks, kBinThreads, 0, st, d_order, p.render_count, order_count_dev, rs.rects.p, rs.block_sums.p, rs.warp_sums.p, rs.super_sums.p, make_own_mask(rank, world), world > 1 ? 1 : 0);
        ++launches;
        prof.mark("k_tile_count", st);
        gs_launch(k_tile_emit, chunks, kBinThreads, 0, st, d_order, p.render_count, order_count_dev, rs.rects.p, rs.block_sums.p, rs.warp_sums.p, rs.super_sums.p, coarse_x, rs.ikeys[0].p,
                                                    rs.ivals[0].p, rs.instance_capacity, rs.rctl.p, make_own_mask(rank, world), world > 1 ? 1 : 0);
        ++launches;
        prof.mark("k_tile_emit", st);
        static const RadixNames names = {{"k_radix_hist[tile,0]", "k_radix_hist[tile,1]", "k_radix_hist[tile,2]", "k_radix_hist[tile,3]"},
                                         {"k_radix_scan[tile,0]", "k_radix_scan[tile,1]", "k_radix_scan[tile,2]", "k_radix_scan[tile,3]"},
                                         {"k_radix_scatter[tile,0]", "k_radix_scatter[tile,1]", "k_radix_scatter[tile,2]", "k_radix_scatter[tile,3]"}};
        // The instance count lives on the device only: the radix grids are sized for the capacity and surplus CTAs exit.
        const unsigned long long *n_dev = &rs.rctl.p->total_instances;
        radix_sort_pairs<uint16_t, unsigned long long>(rs.ikeys[0].p, rs.ikeys[1].p, rs.ivals[0].p, 0u, kValArray, rs.ivals[1].p, rs.ivals[0].p, rs.list.p, 0u,
                                                       n_dev, rs.instance_capacity, pl, rs.sctl.p, rs.tile_hist.p, rs.hist_stride, false, rs.ranges.p, st, launches,
                                                       &prof, names);
    }
    if (record_events) RCU(cudaEventRecord(ev_bin, st));
    if (local_tiles) {
        const bool peer_mode = world > 1 && (rs.peer_root || rs.peer_attached);
        // multi-GPU without the peer path: pixels of other ranks' tiles must be zero so that the frames can be summed (all-reduce)
        void *target = raster_frame_ptr(rs, p.frame_format);
        if (world > 1 && !peer_mode) RCU(cudaMemsetAsync(target, 0, (size_t)p.width * p.height * (p.frame_format == GS_FRAME_RGBA8 ? 4 : 16), st));
        if (peer_mode && rs.peer_attached) {   // fused tile gather: blend straight into rank 0's frame over NVLink
            k_peer_wait_release<<<1, 1, 0, st>>>(rs.peer_sync, rs.rctl.p);
            ++launches;
            target = rs.peer_frame;
        }
        const uint32_t grid = ncoarse * kFinePerCoarse;
        if (rs.render_mode == GS_RENDER_MODE_2D) {
            const bool to_peer = peer_mode && rs.peer_attached;
            const StatusSnapshot snap{rs.snap_sort_ctl, reinterpret_cast<const uint32_t *>(rs.rctl.p),
                                      (rs.snap_base && rs.snap_sort_ctl) ? rs.snap_base + (size_t)rs.frame_parity * rs.snap_stride : nullptr,
                                      to_peer ? &rs.rctl.p->peer_parity : nullptr, to_peer ? (unsigned long long)rs.frame.n : 0ull};
            rs.snapshot_taken = snap.dst != nullptr;
#define GS_BLEND2D(FMT, SC) gs_launch(k_blend2d<FMT, SC>, grid, 128 * SC * SC, 0, st, rs.ranges.p, rs.list.p, rs.surfels.p, tiles_x, tiles_y, coarse_x, rank, world, (int)p.width, (int)p.height, p.flip_y, target, rs.tile_order.p, snap)
            if (tshift == kTileShift) { if (p.frame_format == GS_FRAME_RGBA8) GS_BLEND2D(GS_FRAME_RGBA8, 1); else GS_BLEND2D(GS_FRAME_RGBA32F, 1); }
            else { if (p.frame_format == GS_FRAME_RGBA8) GS_BLEND2D(GS_FRAME_RGBA8, 2); else GS_BLEND2D(GS_FRAME_RGBA32F, 2); }
#undef GS_BLEND2D
            ++launches;
            prof.mark("k_blend2d", st);
        } else if (rs.blend_version >= 2 || tshift != kTileShift) {
            const bool to_peer = peer_mode && rs.peer_attached;
            const StatusSnapshot snap{rs.snap_sort_ctl, reinterpret_cast<const uint32_t *>(rs.rctl.p),
                                      (rs.snap_base && rs.snap_sort_ctl) ? rs.snap_base + (size_t)rs.frame_parity * rs.snap_stride : nullptr,
                                      to_peer ? &rs.rctl.p->peer_parity : nullptr, to_peer ? (unsigned long long)rs.frame.n : 0ull};
            rs.snapshot_taken = snap.dst != nullptr;
#define GS_BLEND2(FMT, SC, RD, TM) gs_launch(k_blend2<FMT, SC, RD, TM>, grid, 128 * SC * SC, 0, st, rs.ranges.p, rs.list.p, rs.records.p, tiles_x, tiles_y, coarse_x, rank, world, (int)p.width, (int)p.height, p.flip_y, target, rs.tile_order.p, snap)
#define GS_BLEND2F(SC, RD, TM) do { if (p.frame_format == GS_FRAME_RGBA8) GS_BLEND2(GS_FRAME_RGBA8, SC, RD, TM); else GS_BLEND2(GS_FRAME_RGBA32F, SC, RD, TM); } while (0)
            // list batches: plain loads; GS_BLEND_TMA=1 prefetches them with bulk async copies instead (measured: no gain, DESIGN.md)
            const bool tma = rs.blend_tma > 0;
            if (tshift == kTileShift) {
                if (rs.blend_rounds == 2) { if (tma) GS_BLEND2F(1, 2, true); else GS_BLEND2F(1, 2, false); }
                else { if (tma) GS_BLEND2F(1, 4, true); else GS_BLEND2F(1, 4, false); }
            } else { if (tma) GS_BLEND2F(2, 1, true); else GS_BLEND2F(2, 1, false); }
#undef GS_BLEND2F
#undef GS_BLEND2
        } else if (p.frame_format == GS_FRAME_RGBA8)
            gs_launch(k_blend<GS_FRAME_RGBA8>, grid, kBlendThreads, 0, st, rs.ranges.p, rs.list.p, rs.records.p, tiles_x, tiles_y, coarse_x, rank, world, (int)p.width, (int)p.height, p.flip_y, target, rs.tile_order.p);
        else
            gs_launch(k_blend<GS_FRAME_RGBA32F>, grid, kBlendThreads, 0, st, rs.ranges.p, rs.list.p, rs.records.p, tiles_x, tiles_y, coarse_x, rank, world, (int)p.width, (int)p.height, p.flip_y, target, rs.tile_order.p);
        if (rs.render_mode != GS_RENDER_MODE_2D) {
            ++launches;
            prof.mark("k_blend", st);
        }
        if (peer_mode && rs.peer_attached) { k_peer_signal<<<1, 1, 0, st>>>(rs.peer_sync); ++launches; }
        if (peer_mode && rs.peer_root) { k_peer_wait_arrived<<<1, 1, 0, st>>>(rs.peer_sync, rs.rctl.p, world - 1); ++launches; prof.mark("k_peer_wait_arrived", st); }
    }
    rs.last_format = p.frame_format;
    const size_t rows = p.height;
    rs.last_frame_bytes = rows * p.width * (p.frame_format == GS_FRAME_RGBA8 ? 4 : 16);
    tm.kernel_launches = launches;
    return GS_OK;
}

// order-preserving compaction of the sort input to this rank's splats (needs k_project's rects of THIS frame)
static int raster_subset(RasterState &rs, const gs_config &c, const uint32_t *d_indexes, uint32_t count, const int32_t *dist, uint32_t *sub_idx,
                         int32_t *sub_dist, cudaStream_t st, Profiler &prof, uint32_t &launches) {
    const uint32_t chunks = (count + kBinTile - 1) / kBinTile;
    const OwnMask own = make_own_mask(c.rank, c.world_size);
    gs_launch(k_subset_count, chunks, kBinThreads, 0, st, d_indexes, count, rs.rects.p, own, rs.block_sums.p, rs.warp_sums.p, rs.super_sums.p + rs.super_stride);
    ++launches;
    prof.mark("k_subset_count", st);
    gs_launch(k_subset_emit, chunks, kBinThreads, 0, st, d_indexes, count, rs.rects.p, own, rs.block_sums.p, rs.warp_sums.p, rs.super_sums.p + rs.super_stride, dist, sub_idx, sub_dist, rs.rctl.p);
    ++launches;
    prof.mark("k_subset_emit", st);
    return GS_OK;
}

// 2D: re-run the projection with the last frame's parameters, exporting the vertex-stage outputs
static int raster_read_projected_2d(RasterState &rs, gs_projected_surfel *out, uint32_t count, cudaStream_t st) {
    if (rs.render_mode != GS_RENDER_MODE_2D) { snprintf(raster_err(), 512, "gs_read_projected_2d on a ThreeD engine (splat_render_mode 0)"); return GS_ERR_BAD_ARG; }
    if (!rs.uploaded) { snprintf(raster_err(), 512, "gs_read_projected_2d before gs_upload_splat_data"); return GS_ERR_NOT_READY; }
    if (count > rs.uploaded) { snprintf(raster_err(), 512, "count %u > uploaded %u", count, rs.uploaded); return GS_ERR_CAPACITY; }
    RCU(rs.exported2d.ensure(rs.uploaded));
    launch_project2d<true>(rs, rs.uploaded, st, rs.exported2d.p);
    RCU(cudaGetLastError());
    RCU(cudaMemcpyAsync(out, rs.exported2d.p, (size_t)count * sizeof(gs_projected_surfel), cudaMemcpyDeviceToHost, st));
    return GS_OK;
}

static int raster_read_projected(RasterState &rs, gs_projected_splat *out, uint32_t count, cudaStream_t st) {
    if (rs.render_mode == GS_RENDER_MODE_2D) { snprintf(raster_err(), 512, "gs_read_projected on a TwoD (surfel) engine: use gs_read_projected_2d"); return GS_ERR_BAD_ARG; }
    if (count > rs.uploaded) { snprintf(raster_err(), 512, "count %u > uploaded %u", count, rs.uploaded); return GS_ERR_CAPACITY; }
    RCU(rs.exported.ensure(count));
    if (count) k_export_projected<<<(count + 255) / 256, 256, 0, st>>>(rs.records.p, rs.rects.p, count, rs.exported.p);
    RCU(cudaMemcpyAsync(out, rs.exported.p, (size_t)count * sizeof(gs_projected_splat), cudaMemcpyDeviceToHost, st));
    return GS_OK;
}

} // namespace gs
