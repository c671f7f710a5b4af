// ksplat_kernels.cuh -- decode a `.ksplat` buffer (src/loaders/SplatBuffer.js) straight into the arrays the engine consumes.
// Replaces the reference's slowest load-time loop (per-splat JS DataView reads):
//   centres   SplatBuffer.fillSplatCenterArray :307-347, bucket lookup getBucketIndex :199-219
//   cov       fillSplatCovarianceArray :488-520 -> computeCovariance :440-486  (float64, stored f32 or f16)
//   colour    fillSplatColorArray :522-549 ; texel packing SplatMesh.updateCenterColorsPaddedData (SplatMesh.js:1143-1153)
//   SH        fillSphericalHarmonicsArray :551-734 (channel-major file order -> coefficient-major RGB triples, stored at level max(1, file))
//   sorter    SplatMesh.getIntegerCenters / getFloatCenters (SplatMesh.js:1912-1948)
// float64 steps use explicit __dmul_rn/__dadd_rn so that no FMA contraction changes the JavaScript (unfused) results.
#pragma once
#include "common.cuh"
#include <cuda_fp16.h>
#include "ksplat_transform.h"   // KTransform

namespace gs {

struct KSectionParams {
    unsigned long long base, buckets_base, data_base;   // byte offsets into the file image
    uint32_t count, splat_offset, bytes_per_splat;
    uint32_t bucket_size, full_bucket_count, partial_count;
    uint32_t scale_range;
    double scale_factor;                                // (bucketBlockSize / 2) / compressionScaleRange   (:924)
    int level, sh_degree_file, sh_degree_out;
    uint32_t minimum_alpha;
    int half_cov, integer_centers, write_sort_centers;
};

template <typename T> __device__ __forceinline__ T load_unaligned(const unsigned char *p) {
    T v;
    unsigned char *d = reinterpret_cast<unsigned char *>(&v);
#pragma unroll
    for (int i = 0; i < (int)sizeof(T); ++i) d[i] = p[i];
    return v;
}
__device__ __forceinline__ float half_bits_to_float(uint16_t h) { return __half2float(__ushort_as_half(h)); }

// THREE.DataUtils.toHalfFloat (three r160): table-driven conversion that TRUNCATES the mantissa (base[e] + (mantissa >> shift[e])),
// after clamping to +-65504.  Restated arithmetically.
__device__ __forceinline__ uint16_t to_half_three(float val) {
    val = fminf(fmaxf(val, -65504.0f), 65504.0f);
    const uint32_t f = __float_as_uint(val);
    const uint32_t sign = (f >> 16) & 0x8000u, mant = f & 0x007fffffu;
    const int ex = (int)((f >> 23) & 0xffu) - 127;
    uint32_t base;
    int shift;
    if (ex < -27) { base = 0; shift = 24; }
    else if (ex < -14) { base = 0x0400u >> (-ex - 14); shift = -ex - 1; }
    else if (ex <= 15) { base = (uint32_t)(ex + 15) << 10; shift = 13; }
    else if (ex < 128) { base = 0x7c00u; shift = 24; }
    else { base = 0x7c00u; shift = 13; }
    return (uint16_t)((base | sign) + (mant >> shift));
}

// TwoD render mode: SplatBuffer.fillSplatScaleRotationArray (SplatBuffer.js:349-438) for one splat, in float64 with three.js's operation
// order (unfused): quaternion.normalize(); with a scene transform, transform * R * S (Matrix4.multiplyMatrices: the R*S and S*I products
// are exact, the zero fourth-row terms add exact zeros) -> Matrix4.decompose -> normalize; ensurePositiveW.  sz is the SplatMesh
// override (1 read at the file's compression level, SplatMesh.js:1856-1863).  Out: f32 [sx sy sz qx qy qz].
__device__ __forceinline__ void ksplat_scale_rotation(const double *T, double sx, double sy, double sz, double x, double y, double z, double w,
                                                      float *out) {
    auto normalize = [](double &x, double &y, double &z, double &w) {
        const double ln = __dsqrt_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)), __dmul_rn(w, w)));
        if (ln == 0.0) { x = y = z = 0.0; w = 1.0; return; }
        const double il = __ddiv_rn(1.0, ln);
        x = __dmul_rn(x, il); y = __dmul_rn(y, il); z = __dmul_rn(z, il); w = __dmul_rn(w, il);
    };
    normalize(x, y, z, w);
    if (T) {
        const double x2 = __dadd_rn(x, x), y2 = __dadd_rn(y, y), z2 = __dadd_rn(z, z);
        const double xx = __dmul_rn(x, x2), xy = __dmul_rn(x, y2), xz = __dmul_rn(x, z2), yy = __dmul_rn(y, y2), yz = __dmul_rn(y, z2), zz = __dmul_rn(z, z2);
        const double wx = __dmul_rn(w, x2), wy = __dmul_rn(w, y2), wz = __dmul_rn(w, z2);
        const double R[3][3] = {{__dsub_rn(1.0, __dadd_rn(yy, zz)), __dsub_rn(xy, wz), __dadd_rn(xz, wy)},
                                {__dadd_rn(xy, wz), __dsub_rn(1.0, __dadd_rn(xx, zz)), __dsub_rn(yz, wx)},
                                {__dsub_rn(xz, wy), __dadd_rn(yz, wx), __dsub_rn(1.0, __dadd_rn(xx, yy))}};
        const double sc[3] = {sx, sy, sz};
        double RS[3][3], m[3][3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) RS[i][j] = __dmul_rn(R[i][j], sc[j]);
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j)
                m[i][j] = __dadd_rn(__dadd_rn(__dmul_rn(T[i], RS[0][j]), __dmul_rn(T[4 + i], RS[1][j])), __dmul_rn(T[8 + i], RS[2][j]));
        double dsx = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[0][0], m[0][0]), __dmul_rn(m[1][0], m[1][0])), __dmul_rn(m[2][0], m[2][0])));
        const double dsy = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[0][1], m[0][1]), __dmul_rn(m[1][1], m[1][1])), __dmul_rn(m[2][1], m[2][1])));
        const double dsz = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[0][2], m[0][2]), __dmul_rn(m[1][2], m[1][2])), __dmul_rn(m[2][2], m[2][2])));
        // Matrix4.determinant: only its sign is used (the affine fourth row leaves the n44 term)
        const double det = m[0][0] * (m[1][1] * m[2][2] - m[1][2] * m[2][1]) - m[0][1] * (m[1][0] * m[2][2] - m[1][2] * m[2][0]) +
                           m[0][2] * (m[1][0] * m[2][1] - m[1][1] * m[2][0]);
        if (det < 0) dsx = -dsx;
        const double is[3] = {__ddiv_rn(1.0, dsx), __ddiv_rn(1.0, dsy), __ddiv_rn(1.0, dsz)};
        double r[3][3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) r[i][j] = __dmul_rn(m[i][j], is[j]);
        const double t = __dadd_rn(__dadd_rn(r[0][0], r[1][1]), r[2][2]);   // Quaternion.setFromRotationMatrix
        if (t > 0) {
            const double k = __ddiv_rn(0.5, __dsqrt_rn(__dadd_rn(t, 1.0)));
            w = __ddiv_rn(0.25, k); x = __dmul_rn(__dsub_rn(r[2][1], r[1][2]), k); y = __dmul_rn(__dsub_rn(r[0][2], r[2][0]), k); z = __dmul_rn(__dsub_rn(r[1][0], r[0][1]), k);
        } else if (r[0][0] > r[1][1] && r[0][0] > r[2][2]) {
            const double k = __dmul_rn(2.0, __dsqrt_rn(__dsub_rn(__dsub_rn(__dadd_rn(1.0, r[0][0]), r[1][1]), r[2][2])));
            w = __ddiv_rn(__dsub_rn(r[2][1], r[1][2]), k); x = __dmul_rn(0.25, k); y = __ddiv_rn(__dadd_rn(r[0][1], r[1][0]), k); z = __ddiv_rn(__dadd_rn(r[0][2], r[2][0]), k);
        } else if (r[1][1] > r[2][2]) {
            const double k = __dmul_rn(2.0, __dsqrt_rn(__dsub_rn(__dsub_rn(__dadd_rn(1.0, r[1][1]), r[0][0]), r[2][2])));
            w = __ddiv_rn(__dsub_rn(r[0][2], r[2][0]), k); x = __ddiv_rn(__dadd_rn(r[0][1], r[1][0]), k); y = __dmul_rn(0.25, k); z = __ddiv_rn(__dadd_rn(r[1][2], r[2][1]), k);
        } else {
            const double k = __dmul_rn(2.0, __dsqrt_rn(__dsub_rn(__dsub_rn(__dadd_rn(1.0, r[2][2]), r[0][0]), r[1][1])));
            w = __ddiv_rn(__dsub_rn(r[1][0], r[0][1]), k); x = __ddiv_rn(__dadd_rn(r[0][2], r[2][0]), k); y = __ddiv_rn(__dadd_rn(r[1][2], r[2][1]), k); z = __dmul_rn(0.25, k);
        }
        normalize(x, y, z, w);
        sx = dsx; sy = dsy; sz = dsz;
    }
    const double flip = w < 0 ? -1.0 : 1.0;   // ensurePositiveW
    out[0] = (float)sx; out[1] = (float)sy; out[2] = (float)sz;
    out[3] = (float)(x * flip); out[4] = (float)(y * flip); out[5] = (float)(z * flip);
}

// XF: bake the scene transform (centre.applyMatrix4 :340-342, T3 (M M^T) T3^T :461-466, SH decode -> rotate -> re-encode :663-716).
// SR (TwoD engines): write the scale/rotation texture `srot` (6 x f32 per splat) instead of covariances.
template <bool XF, bool SR>
__global__ void __launch_bounds__(128)
k_ksplat_decode(const unsigned char *__restrict__ file, KSectionParams P, const uint32_t *__restrict__ partial_prefix,
                uint4 *__restrict__ cc, void *__restrict__ cov, void *__restrict__ sh_out, int4 *__restrict__ sort_centers,
                const KTransform *__restrict__ xf, float *__restrict__ srot) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.count) return;
    const unsigned char *rec = file + P.data_base + (size_t)i * P.bytes_per_splat;
    float c[3], s[3], qw, qx, qy, qz;
    uchar4 rgba;
    const unsigned char *shp;
    if (P.level == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { c[k] = load_unaligned<float>(rec + 4 * k); s[k] = load_unaligned<float>(rec + 12 + 4 * k); }
        qw = load_unaligned<float>(rec + 24); qx = load_unaligned<float>(rec + 28); qy = load_unaligned<float>(rec + 32); qz = load_unaligned<float>(rec + 36);
        rgba = load_unaligned<uchar4>(rec + 40);
        shp = rec + 44;
    } else {
        // bucket of this splat: full buckets first, then the partially filled ones with explicit lengths (:199-219)
        uint32_t b;
        const uint32_t in_full = P.full_bucket_count * P.bucket_size;
        if (i < in_full) b = i / P.bucket_size;
        else {
            const uint32_t r = i - in_full;      // partial_prefix[k] = splats in partial buckets < k ; find last k with prefix <= r
            uint32_t lo = 0, hi = P.partial_count;
            while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (partial_prefix[mid] <= r) lo = mid; else hi = mid; }
            b = P.full_bucket_count + lo;
        }
        const unsigned char *bc = file + P.buckets_base + (size_t)b * 12;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double u = (double)load_unaligned<uint16_t>(rec + 2 * k) - (double)P.scale_range;
            c[k] = (float)__dadd_rn(__dmul_rn(u, P.scale_factor), (double)load_unaligned<float>(bc + 4 * k));   // (x - sr) * sf + bucket, f64 -> f32
            s[k] = half_bits_to_float(load_unaligned<uint16_t>(rec + 6 + 2 * k));
        }
        qw = half_bits_to_float(load_unaligned<uint16_t>(rec + 12)); qx = half_bits_to_float(load_unaligned<uint16_t>(rec + 14));
        qy = half_bits_to_float(load_unaligned<uint16_t>(rec + 16)); qz = half_bits_to_float(load_unaligned<uint16_t>(rec + 18));
        rgba = load_unaligned<uchar4>(rec + 20);
        shp = rec + 24;
    }
    const uint32_t g = P.splat_offset + i;
    if (XF) {   // Vector3.applyMatrix4 in f64 on the decoded f32 centre, stored back as f32
        const double *T = xf->t;
        const double x = c[0], y = c[1], z = c[2];
        const double w = __ddiv_rn(1.0, __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[3], x), __dmul_rn(T[7], y)), __dmul_rn(T[11], z)), T[15]));
        c[0] = (float)__dmul_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[0], x), __dmul_rn(T[4], y)), __dmul_rn(T[8], z)), T[12]), w);
        c[1] = (float)__dmul_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[1], x), __dmul_rn(T[5], y)), __dmul_rn(T[9], z)), T[13]), w);
        c[2] = (float)__dmul_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[2], x), __dmul_rn(T[6], y)), __dmul_rn(T[10], z)), T[14]), w);
    }
    // ---- centres + colours texel ----------------------------------------------------------------------------------------
    const uint32_t a = rgba.w >= P.minimum_alpha ? rgba.w : 0u;
    cc[g] = make_uint4((uint32_t)rgba.x | ((uint32_t)rgba.y << 8) | ((uint32_t)rgba.z << 16) | (a << 24), __float_as_uint(c[0]), __float_as_uint(c[1]),
                       __float_as_uint(c[2]));
    // ---- sorter centres ---------------------------------------------------------------------------------------------------
    if (P.write_sort_centers) {
        if (P.integer_centers) {   // Math.round(f32 * 1000.0) on the f64 product, w = 1000
            sort_centers[g] = make_int4((int)floor(__dmul_rn((double)c[0], 1000.0) + 0.5), (int)floor(__dmul_rn((double)c[1], 1000.0) + 0.5),
                                        (int)floor(__dmul_rn((double)c[2], 1000.0) + 0.5), 1000);
        } else sort_centers[g] = make_int4(__float_as_int(c[0]), __float_as_int(c[1]), __float_as_int(c[2]), __float_as_int(1.0f));
    }
    if (SR) {
        // the z scale override 1 goes through toUncompressedFloat at the file's level: fromHalfFloat(1) = 2^-24 at levels 1 and 2
        const double sz = P.level == 0 ? 1.0 : 5.9604644775390625e-08;
        float o[6];
        ksplat_scale_rotation(XF ? xf->t : nullptr, (double)s[0], (double)s[1], sz, (double)qx, (double)qy, (double)qz, (double)qw, o);
        float2 *d = reinterpret_cast<float2 *>(srot + (size_t)g * 6);
        d[0] = make_float2(o[0], o[1]); d[1] = make_float2(o[2], o[3]); d[2] = make_float2(o[4], o[5]);
    }
    // ---- covariance = (R S)(R S)^T in float64, three.js operation order ---------------------------------------------------
    if (!SR) {
        const double x = qx, y = qy, z = qz, w = qw;
        const double x2 = __dadd_rn(x, x), y2 = __dadd_rn(y, y), z2 = __dadd_rn(z, z);
        const double xx = __dmul_rn(x, x2), xy = __dmul_rn(x, y2), xz = __dmul_rn(x, z2), yy = __dmul_rn(y, y2), yz = __dmul_rn(y, z2), zz = __dmul_rn(z, z2);
        const double wx = __dmul_rn(w, x2), wy = __dmul_rn(w, y2), wz = __dmul_rn(w, z2);
        double R[3][3];
        R[0][0] = __dsub_rn(1.0, __dadd_rn(yy, zz)); R[0][1] = __dsub_rn(xy, wz); R[0][2] = __dadd_rn(xz, wy);
        R[1][0] = __dadd_rn(xy, wz); R[1][1] = __dsub_rn(1.0, __dadd_rn(xx, zz)); R[1][2] = __dsub_rn(yz, wx);
        R[2][0] = __dsub_rn(xz, wy); R[2][1] = __dadd_rn(yz, wx); R[2][2] = __dsub_rn(1.0, __dadd_rn(xx, yy));
        double M[3][3];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int k = 0; k < 3; ++k) M[r][k] = __dmul_rn(R[r][k], (double)s[k]);
        auto dot = [&](int r0, int r1) { return __dadd_rn(__dadd_rn(__dmul_rn(M[r0][0], M[r1][0]), __dmul_rn(M[r0][1], M[r1][1])), __dmul_rn(M[r0][2], M[r1][2])); };
        double v[6] = {dot(0, 0), dot(0, 1), dot(0, 2), dot(1, 1), dot(1, 2), dot(2, 2)};
        if (XF) {   // X = S T3^T, Y = T3 X with Matrix3.multiplyMatrices' left-to-right sums
            const double *T = xf->t;
            const double t3[3][3] = {{T[0], T[4], T[8]}, {T[1], T[5], T[9]}, {T[2], T[6], T[10]}};
            const double S[3][3] = {{v[0], v[1], v[2]}, {v[1], v[3], v[4]}, {v[2], v[4], v[5]}};
            double X[3][3];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    X[r][k] = __dadd_rn(__dadd_rn(__dmul_rn(S[r][0], t3[k][0]), __dmul_rn(S[r][1], t3[k][1])), __dmul_rn(S[r][2], t3[k][2]));
            auto Y = [&](int r, int k) { return __dadd_rn(__dadd_rn(__dmul_rn(t3[r][0], X[0][k]), __dmul_rn(t3[r][1], X[1][k])), __dmul_rn(t3[r][2], X[2][k])); };
            v[0] = Y(0, 0); v[1] = Y(0, 1); v[2] = Y(0, 2); v[3] = Y(1, 1); v[4] = Y(1, 2); v[5] = Y(2, 2);
        }
        if (P.half_cov) {
            uint16_t *o = reinterpret_cast<uint16_t *>(cov) + (size_t)g * 6;
#pragma unroll
            for (int k = 0; k < 6; ++k) o[k] = to_half_three((float)v[k]);
        } else {
            float *o = reinterpret_cast<float *>(cov) + (size_t)g * 6;
#pragma unroll
            for (int k = 0; k < 6; ++k) o[k] = (float)v[k];
        }
    }
    // ---- spherical harmonics: file [band][channel][coef] -> GPU [coef][channel] ------------------------------------------------
    if (P.sh_degree_out >= 1) {
        const int ncomp = P.sh_degree_out >= 2 ? 24 : 9;
        auto src_of = [](int o) {
            if (o < 9) { const int coef = o / 3, ch = o % 3; return ch * 3 + coef; }
            const int coef = (o - 9) / 3, ch = (o - 9) % 3;
            return 9 + ch * 5 + coef;
        };
        if (!XF) {
            for (int o = 0; o < ncomp; ++o) {
                const int src = src_of(o);
                if (P.level == 2) reinterpret_cast<unsigned char *>(sh_out)[(size_t)g * ncomp + o] = shp[src];
                else if (P.level == 1) reinterpret_cast<uint16_t *>(sh_out)[(size_t)g * ncomp + o] = load_unaligned<uint16_t>(shp + 2 * src);
                else reinterpret_cast<uint16_t *>(sh_out)[(size_t)g * ncomp + o] = to_half_three(load_unaligned<float>(shp + 4 * src));
            }
        } else {
            // decode to JS numbers (toUncompressedFloat :12-20), rotate band by band (dot3 / dot5: sums in coefficient order), re-encode
            const double lo = xf->sh_lo, range = __dsub_rn(xf->sh_hi, xf->sh_lo);
            auto value = [&](int o) -> double {
                const int src = src_of(o);
                if (P.level == 2) return __dadd_rn(__dmul_rn(__ddiv_rn((double)shp[src], 255.0), range), lo);   // fromUint8: v / 255 * range + min
                if (P.level == 1) return (double)half_bits_to_float(load_unaligned<uint16_t>(shp + 2 * src));
                return (double)load_unaligned<float>(shp + 4 * src);
            };
            auto store = [&](int o, double r) {
                if (P.level == 2) {   // toUint8 (:21-25)
                    const double cl = fmin(fmax(r, lo), xf->sh_hi);
                    const double q = floor(__dmul_rn(__ddiv_rn(__dsub_rn(cl, lo), range), 255.0));
                    reinterpret_cast<unsigned char *>(sh_out)[(size_t)g * ncomp + o] = (unsigned char)fmin(fmax(q, 0.0), 255.0);
                } else reinterpret_cast<uint16_t *>(sh_out)[(size_t)g * ncomp + o] = to_half_three((float)r);
            };
#pragma unroll 1
            for (int ch = 0; ch < 3; ++ch) {
                const double i0 = value(0 + ch), i1 = value(3 + ch), i2 = value(6 + ch);
#pragma unroll
                for (int l = 0; l < 3; ++l)
                    store(3 * l + ch, __dadd_rn(__dadd_rn(__dmul_rn(i0, xf->m1[l][0]), __dmul_rn(i1, xf->m1[l][1])), __dmul_rn(i2, xf->m1[l][2])));
                if (ncomp == 24) {
                    double in[5];
#pragma unroll
                    for (int k = 0; k < 5; ++k) in[k] = value(9 + 3 * k + ch);
#pragma unroll
                    for (int l = 0; l < 5; ++l) {
                        double acc = __dmul_rn(in[0], xf->m2[l][0]);
#pragma unroll
                        for (int k = 1; k < 5; ++k) acc = __dadd_rn(acc, __dmul_rn(in[k], xf->m2[l][k]));
                        store(9 + 3 * l + ch, acc);
                    }
                }
            }
        }
    }
}

} // namespace gs
