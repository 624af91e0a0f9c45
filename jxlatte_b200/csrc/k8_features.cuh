// k8_features.cuh -- image features between stage 2 and the colour transform (SURVEY.md 8f-4): k x k upsampling.
//
// k8_upsample replaces Frame.performUpsampling (J/frame/Frame.java:217-260): per output phase (ky, kx) a 5x5 kernel over the
// mirrored neighbourhood, accumulated in (iy, ix) order with uncontracted multiply-adds, clamped to the window's range with
// the Java's initial min / max (Float.MAX_VALUE / Float.MIN_VALUE -- the smallest positive float, a reference quirk kept).
#pragma once
#include "common.cuh"
#include "k2_restore.cuh"
#include "k7_blend.cuh"

__device__ __forceinline__ int mirror_coord(int c, int size) {      // MathHelper.mirrorCoordinate (J/util/MathHelper.java:323-329)
    while (c < 0 || c >= size) {
        const int tc = ~c;
        c = tc >= 0 ? tc : (size << 1) + tc;
    }
    return c;
}

// one thread per INPUT pixel: the 25 samples are loaded once and feed the k * k output phases; weights in shared memory
__global__ void k8_upsample(const float *__restrict__ in, int h, int w, int k, const float *__restrict__ weights, float *__restrict__ out) {
    extern __shared__ float s_w[];
    for (int i = threadIdx.x; i < k * k * 25; i += blockDim.x) s_w[i] = weights[i];
    __syncthreads();
    const long long n = (long long)h * w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(i / w), x = (int)(i - (long long)y * w);
        float s[25];
        float mn = 3.4028234663852886e38f, mx = 1.401298464324817e-45f;
#pragma unroll
        for (int iy = 0; iy < 5; iy++) {
            const int yy = mirror_coord(y + iy - 2, h);
#pragma unroll
            for (int ix = 0; ix < 5; ix++) {
                const int xx = mirror_coord(x + ix - 2, w);
                const float v = in[(size_t)yy * w + xx];
                s[iy * 5 + ix] = v;
                if (v < mn) mn = v;
                if (v > mx) mx = v;
            }
        }
        for (int ky = 0; ky < k; ky++)
            for (int kx = 0; kx < k; kx++) {
                const float *wt = s_w + (ky * k + kx) * 25;
                float total = 0.0f;
#pragma unroll
                for (int t = 0; t < 25; t++) total = __fadd_rn(total, __fmul_rn(wt[t], s[t]));
                out[(size_t)(y * k + ky) * w * k + x * k + kx] = total < mn ? mn : (total > mx ? mx : total);
            }
    }
}

// ---- noise: XorShiro (J/frame/features/XorShiro.java), Frame.initializeNoise / synthesizeNoise (J/frame/Frame.java:748-835) ----
__host__ __device__ __forceinline__ unsigned long long split_mix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}

struct NoiseArgs {
    float *local[3];          // uniform [1, 2) samples
    float *plane[3];          // X, Y, B in / out
    int h, w, group_dim, log_dim, group_cols, num_groups;
    unsigned long long seed0;
    float lut[8];
    float base_x, base_b;
};

// XorShiro is eight independent xorshift128+ lanes; lane i supplies ints 2i and 2i+1 of every batch of 16.  One thread per
// (group, lane) walks its lane through the group's 3 * rows * ceil(cols / 16) batches.
__global__ void k8_noise_rng(NoiseArgs A) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int group = t >> 3, lane = t & 7;
    if (group >= A.num_groups) return;
    const int y0 = (group / A.group_cols) << A.log_dim, x0 = (group % A.group_cols) << A.log_dim;
    const unsigned long long seed1 = ((unsigned long long)(unsigned)x0 << 32) | (unsigned long long)(unsigned)y0;
    unsigned long long s0 = split_mix64(A.seed0 + 0x9e3779b97f4a7c15ULL), s1 = split_mix64(seed1 + 0x9e3779b97f4a7c15ULL);
    for (int i = 0; i < lane; i++) { s0 = split_mix64(s0); s1 = split_mix64(s1); }
    const int ys = min(A.group_dim, A.h - y0), xs = min(A.group_dim, A.w - x0);
    for (int c = 0; c < 3; c++)
        for (int y = 0; y < ys; y++) {
            float *row = A.local[c] + (size_t)(y0 + y) * A.w + x0;
            for (int x = 0; x < xs; x += 16) {
                const unsigned long long a = s1;
                unsigned long long b = s0;
                const unsigned long long sum = a + b;
                s0 = a;
                b ^= b << 23;
                s1 = b ^ a ^ (b >> 18) ^ (a >> 5);
                const int p = x + 2 * lane;
                if (p < xs) row[p] = __uint_as_float(((unsigned)(sum & 0xffffffffULL) >> 9) | 0x3f800000u);
                if (p + 1 < xs) row[p + 1] = __uint_as_float(((unsigned)(sum >> 32) >> 9) | 0x3f800000u);
            }
        }
}

// Laplacian-filtered noise of the three channels at one pixel, then the intensity-dependent mix into X, Y, B
__global__ void k8_noise_apply(NoiseArgs A) {
    const long long n = (long long)A.h * A.w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(i / A.w), x = (int)(i - (long long)y * A.w);
        float nz[3];
        for (int c = 0; c < 3; c++) {
            float acc = 0.0f;
            for (int iy = 0; iy < 5; iy++) {
                const int cy = mirror_coord(y + iy - 2, A.h);
                for (int ix = 0; ix < 5; ix++) {
                    const int cx = mirror_coord(x + ix - 2, A.w);
                    const float lap = (iy == 2 && ix == 2) ? -3.84f : 0.16f;
                    acc = __fadd_rn(acc, __fmul_rn(A.local[c][(size_t)cy * A.w + cx], lap));
                }
            }
            nz[c] = acc;
        }
        const float X = A.plane[0][i], Y = A.plane[1][i], B = A.plane[2][i];
        float in_r = __fadd_rn(Y, X);
        in_r = in_r < 0.0f ? 0.0f : __fmul_rn(3.0f, in_r);
        float in_g = __fsub_rn(Y, X);
        in_g = in_g < 0.0f ? 0.0f : __fmul_rn(3.0f, in_g);
        int ir, ig;
        float fr, fg;
        if (in_r >= 7.0f) { ir = 6; fr = 1.0f; } else { ir = (int)in_r; fr = __fsub_rn(in_r, (float)ir); }
        if (in_g >= 7.0f) { ig = 6; fg = 1.0f; } else { ig = (int)in_g; fg = __fsub_rn(in_g, (float)ig); }
        float sr = __fadd_rn(__fmul_rn(__fsub_rn(A.lut[ir + 1], A.lut[ir]), fr), A.lut[ir]);
        float sg = __fadd_rn(__fmul_rn(__fsub_rn(A.lut[ig + 1], A.lut[ig]), fg), A.lut[ig]);
        sr = clamp01(sr);
        sg = clamp01(sg);
        const float nr = __fmul_rn(sr, __fadd_rn(__fmul_rn(0.00171875f, nz[0]), __fmul_rn(0.21828125f, nz[2])));
        const float ng = __fmul_rn(sg, __fadd_rn(__fmul_rn(0.00171875f, nz[1]), __fmul_rn(0.21828125f, nz[2])));
        const float nrg = __fadd_rn(nr, ng);
        A.plane[1][i] = __fadd_rn(Y, nrg);
        A.plane[0][i] = __fadd_rn(X, __fsub_rn(__fadd_rn(__fmul_rn(A.base_x, nrg), nr), ng));
        A.plane[2][i] = __fadd_rn(B, __fmul_rn(A.base_b, nrg));
    }
}

// ---- splines: Spline.renderSpline's pixel loop (J/frame/features/spline/Spline.java:170-199) ----
// The arcs (position, colour values, sigma, bounding box) are prepared on the host (splines_host.cuh); here every pixel walks
// the arcs in order and adds the contributions of those whose box covers it, which is the order the Java adds them in.
struct SplineArcDev {
    float y, x, sigma, inv_sigma;
    float value[3];
    int x0, x1, y0, y1;     // inclusive box
};

__device__ __forceinline__ float erf_ref(float z) {      // MathHelper.erf (J/util/MathHelper.java:40-66): float polynomial, double exp
    const float az = fabsf(z);
    float r;
    if (az > 1e-4f) {
        const float t = __fdiv_rn(1.0f, __fadd_rn(__fmul_rn(az, 0.5f), 1.0f));
        float u = __fsub_rn(__fmul_rn(t, 0.17087277f), 0.82215223f);
        u = __fadd_rn(__fmul_rn(t, u), 1.48851587f);
        u = __fsub_rn(__fmul_rn(t, u), 1.13520398f);
        u = __fadd_rn(__fmul_rn(t, u), 0.27886807f);
        u = __fsub_rn(__fmul_rn(t, u), 0.18628806f);
        u = __fadd_rn(__fmul_rn(t, u), 0.09678418f);
        u = __fadd_rn(__fmul_rn(t, u), 0.37409196f);
        u = __fadd_rn(__fmul_rn(t, u), 1.00002368f);
        u = __fsub_rn(__fmul_rn(t, u), 1.26551223f);
        const float e = (float)exp((double)__fadd_rn(__fmul_rn(-z, z), u));
        r = __fsub_rn(1.0f, __fmul_rn(t, e));
    } else {
        const float t = __fdiv_rn(1.0f, __fadd_rn(__fmul_rn(az, 0.47047f), 1.0f));
        float u = __fsub_rn(__fmul_rn(t, 0.7478556f), 0.0958798f);
        u = __fadd_rn(__fmul_rn(t, u), 0.3480242f);
        u = __fmul_rn(t, u);
        const float e = (float)exp((double)__fmul_rn(-z, z));
        r = __fsub_rn(1.0f, __fmul_rn(u, e));
    }
    return z < 0.0f ? -r : r;
}

#define K8_ARC_CHUNK 128
__global__ void k8_splines(float *p0, float *p1, float *p2, int h, int w, const SplineArcDev *__restrict__ arcs, int n, float sqrt_f) {
    __shared__ SplineArcDev s_arc[K8_ARC_CHUNK];
    const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int tx0 = blockIdx.x * 32, ty0 = blockIdx.y * 8;
    const bool inside = x < w && y < h;
    float acc[3] = {0.0f, 0.0f, 0.0f};
    if (inside) { acc[0] = p0[(size_t)y * w + x]; acc[1] = p1[(size_t)y * w + x]; acc[2] = p2[(size_t)y * w + x]; }
    for (int base = 0; base < n; base += K8_ARC_CHUNK) {
        const int cnt = min(K8_ARC_CHUNK, n - base);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) s_arc[i] = arcs[base + i];
        __syncthreads();
        for (int i = 0; i < cnt; i++) {
            const SplineArcDev &a = s_arc[i];
            if (a.x1 < tx0 || a.x0 > tx0 + 31 || a.y1 < ty0 || a.y0 > ty0 + 7) continue;      // whole tile outside: uniform skip
            if (!inside || x < a.x0 || x > a.x1 || y < a.y0 || y > a.y1) continue;
            const float dy = __fsub_rn((float)y, a.y), dx = __fsub_rn((float)x, a.x);
            const float dist = __fsqrt_rn(__fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dx, dx)));
            const float half = __fmul_rn(0.5f, dist);
            float factor = erf_ref(__fmul_rn(__fadd_rn(half, sqrt_f), a.inv_sigma));
            factor = __fsub_rn(factor, erf_ref(__fmul_rn(__fsub_rn(half, sqrt_f), a.inv_sigma)));
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const float extra = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(0.25f, a.value[c]), a.sigma), factor), factor);
                acc[c] = __fadd_rn(acc[c], extra);
            }
        }
    }
    if (inside) { p0[(size_t)y * w + x] = acc[0]; p1[(size_t)y * w + x] = acc[1]; p2[(size_t)y * w + x] = acc[2]; }
}

// ---- PNG-ready samples: JXLImage.transfer (TF_SRGB.fromLinearF, J/color/TransferFunction.java:39-43) + ImageBuffer
// castToIntWithMax / clamp (J/util/ImageBuffer.java:129-160) + PNGWriter's sample interleave (J/io/PNGWriter.java:191-203) ----
struct PackArgs {
    const void *plane[8];
    int is_int[8], depth[8];
    int n_channels, n_color, linear, h, w, bits;
    int layout;                 // 0: interleaved PNG bytes (big-endian 16 bit); 1: planar [C][h][w] uint8 / native-endian uint16
    unsigned char *out;
};

__device__ __forceinline__ int java_f2i(float v) {        // (int) cast of the JVM: NaN -> 0, saturating
    if (v != v) return 0;
    if (v >= 2147483648.0f) return 2147483647;
    if (v <= -2147483648.0f) return -2147483647 - 1;
    return (int)v;
}

// One sample of the pipeline: channel c of plane[] at i (int32 when is_int[c], else float32) -> its `bits`-bit value, clamped to
// [0, maxv].  An int channel whose depth is `bits` is only clamped; TF_SRGB.fromLinearF comes first when `oetf` (a colour channel of
// a linear image).  The per-channel arrays are read where the reference reads them, so k8_pack_samples keeps its instructions.
__device__ __forceinline__ int pack_sample(const void *const *plane, const int *is_int, const int *depth, int c, long long i, int bits, int maxv,
                                           bool oetf) {
    int q;
    if (is_int[c] && depth[c] == bits) {
        q = ((const int *)plane[c])[i];
    } else {
        float v;
        if (is_int[c]) v = __fmul_rn((float)((const int *)plane[c])[i], __fdiv_rn(1.0f, (float)((1 << depth[c]) - 1)));
        else v = ((const float *)plane[c])[i];
        if (oetf) {
            if (v < 0.00313066844250063f) v = __fmul_rn(v, 12.92f);
            else v = __fadd_rn(__fmul_rn(1.055f, (float)pow((double)v, 0.4166666666666667)), -0.055f);
        }
        q = java_f2i(__fadd_rn(__fmul_rn(v, (float)maxv), 0.5f));
    }
    return q < 0 ? 0 : (q > maxv ? maxv : q);
}

__global__ void k8_pack_samples(PackArgs A) {
    const long long n = (long long)A.h * A.w;
    const int maxv = (1 << A.bits) - 1, bytes = A.bits > 8 ? 2 : 1;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        unsigned char *o = A.out + i * A.n_channels * bytes;
        for (int c = 0; c < A.n_channels; c++) {
            const int q = pack_sample(A.plane, A.is_int, A.depth, c, i, A.bits, maxv, A.linear && c < A.n_color);
            if (A.layout == 1) {
                if (bytes == 2) reinterpret_cast<unsigned short *>(A.out)[c * n + i] = (unsigned short)q;
                else A.out[c * n + i] = (unsigned char)q;
            } else if (bytes == 2) { o[2 * c] = (unsigned char)(q >> 8); o[2 * c + 1] = (unsigned char)(q & 255); }
            else o[c] = (unsigned char)q;
        }
    }
}

// ---- the same conversion for the three colour planes of a VarDCT frame, rows [r0, r1) x columns [0, cw) of planes with
// pitch `pitch`, straight after stage 2 on the device: what the pipelined host entry point sends back instead of 12 bytes of
// float per pixel (jxlb200_vardct_reconstruct_packed).  Four pixels per thread: three 128-bit loads, 12 or 24 bytes out.
//
// The reference's sample pipeline -- TF_SRGB.fromLinearF with (float)Math.pow(double) (J/color/TransferFunction.java:39-43), then
// (int)(v * max + 0.5f) and a clamp (J/util/ImageBuffer.java:129-145) -- is a MONOTONE step function of the float v: every stage
// is non-decreasing in float arithmetic.  So it is exactly a table of thresholds, thr[k] = the smallest float whose sample is
// >= k, built once on the host by bisection over float bit patterns WITH the reference's formula (pack_sample_ref below), and the
// device only counts thresholds <= v (binary search): bit-identical to evaluating the formula, without a double-precision pow
// per sample (which made this kernel, not PCIe, the limit of the packed call: 100 M pows per 8K frame).
static inline int pack_sample_ref(float v, int linear, int maxv) {
    if (v != v) return 0;
    if (linear) {
        if (v < 0.00313066844250063f) v = v * 12.92f;
        else v = 1.055f * (float)pow((double)v, 0.4166666666666667) + -0.055f;
    }
    const float f = v * (float)maxv + 0.5f;
    if (f != f) return 0;
    long long q = f >= 2147483648.0f ? 2147483647ll : (f <= -2147483648.0f ? -2147483648ll : (long long)f);   // the JVM's (int) cast
    return q < 0 ? 0 : (q > maxv ? maxv : (int)q);
}
// floats ordered as integers: key(v) increases with v over all non-NaN floats
static inline uint32_t float_key(float v) { uint32_t u; memcpy(&u, &v, 4); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
static inline float key_float(uint32_t k) { uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k; float v; memcpy(&v, &u, 4); return v; }
// thr[k - 1], k = 1 .. maxv: the smallest float v with pack_sample_ref(v) >= k (+inf when no float reaches k)
static inline void pack_thresholds(int bits, int linear, std::vector<float> &thr) {
    const int maxv = (1 << bits) - 1;
    thr.resize(maxv);
    const uint32_t kmin = float_key(-INFINITY), kmax = float_key(INFINITY);
    uint32_t from = kmin;
    for (int k = 1; k <= maxv; k++) {
        uint32_t lo = from, hi = kmax;                      // invariant: sample(lo) < k or lo == from; answer in (lo, hi]
        if (pack_sample_ref(key_float(hi), linear, maxv) < k) { thr[k - 1] = INFINITY; continue; }
        if (pack_sample_ref(key_float(lo), linear, maxv) >= k) { thr[k - 1] = key_float(lo); continue; }
        while (hi - lo > 1) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (pack_sample_ref(key_float(mid), linear, maxv) >= k) hi = mid; else lo = mid;
        }
        thr[k - 1] = key_float(hi);
        from = hi;
    }
}

// number of thresholds <= v = the sample; NaN compares false everywhere -> 0, like the JVM's (int) cast
template <int BITS> __device__ __forceinline__ int pack_search(const float *__restrict__ coarse, const float *__restrict__ thr, float v) {
    constexpr int MAXV = (1 << BITS) - 1;
    if (BITS == 8) {
        int lo = 0;                                         // thresholds [0, 255) in shared memory
#pragma unroll
        for (int step = 128; step >= 1; step >>= 1)
            if (lo + step <= MAXV && coarse[lo + step - 1] <= v) lo += step;
        return lo;
    } else {
        // coarse[j] = thr[256 j + 255] (shared memory): first the 256-sample segment, then inside it (global, one or two lines)
        int seg = 0;
#pragma unroll
        for (int step = 128; step >= 1; step >>= 1)
            if (seg + step <= 255 && coarse[seg + step - 1] <= v) seg += step;
        // seg = number of coarse thresholds <= v: the answer lies in [256 seg, 256 seg + 255]
        const float *t = thr + 256 * seg;
        int lo = 0;
#pragma unroll
        for (int step = 128; step >= 1; step >>= 1)
            if (256 * seg + lo + step <= MAXV && __ldg(t + lo + step - 1) <= v) lo += step;
        return 256 * seg + lo;
    }
}

template <int BITS>
__global__ void k8_pack_rgb(const float *__restrict__ p0, const float *__restrict__ p1, const float *__restrict__ p2, long long pitch,
                            int r0, int r1, int cw, const float *__restrict__ thr, unsigned char *__restrict__ out) {
    __shared__ float coarse[256];
    if (BITS == 8) { for (int i = threadIdx.x; i < 255; i += blockDim.x) coarse[i] = thr[i]; }
    else { for (int i = threadIdx.x; i < 255; i += blockDim.x) coarse[i] = thr[256 * i + 255]; }
    __syncthreads();
    const int quads = (cw + 3) >> 2;
    const long long n = (long long)(r1 - r0) * quads;
    constexpr int bytes = BITS > 8 ? 2 : 1;
    const bool vec = (pitch & 3) == 0 && ((((size_t)p0 | (size_t)p1 | (size_t)p2) & 15) == 0);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int r = r0 + (int)(i / quads), x = 4 * (int)(i % quads);
        const long long o = (long long)r * pitch + x;
        float a[4], b[4], c[4];
        const int nv = min(4, cw - x);
        if (vec && x + 4 <= pitch) {
            const float4 va = *reinterpret_cast<const float4 *>(p0 + o), vb = *reinterpret_cast<const float4 *>(p1 + o), vc = *reinterpret_cast<const float4 *>(p2 + o);
            a[0] = va.x; a[1] = va.y; a[2] = va.z; a[3] = va.w; b[0] = vb.x; b[1] = vb.y; b[2] = vb.z; b[3] = vb.w;
            c[0] = vc.x; c[1] = vc.y; c[2] = vc.z; c[3] = vc.w;
        } else {
            for (int k = 0; k < 4; k++) { const bool in = k < nv; a[k] = in ? p0[o + k] : 0.0f; b[k] = in ? p1[o + k] : 0.0f; c[k] = in ? p2[o + k] : 0.0f; }
        }
        unsigned char *dst = out + ((long long)r * cw + x) * 3 * bytes;
        for (int k = 0; k < nv; k++) {
            const int q[3] = {pack_search<BITS>(coarse, thr, a[k]), pack_search<BITS>(coarse, thr, b[k]), pack_search<BITS>(coarse, thr, c[k])};
            for (int ch = 0; ch < 3; ch++) {
                if (bytes == 2) { dst[(3 * k + ch) * 2] = (unsigned char)(q[ch] >> 8); dst[(3 * k + ch) * 2 + 1] = (unsigned char)(q[ch] & 255); }   // PNG is big endian
                else dst[3 * k + ch] = (unsigned char)q[ch];
            }
        }
    }
}

// ---- LF coefficients (SURVEY.md 8f-1: "the one front-end piece worth a tiny kernel"): dequantisation, LF chroma-from-luma and the
// adaptive smoothing of LFCoefficients (J/frame/vardct/LFCoefficients.java:61-103, adaptiveSmooth :113-179), one thread per LF sample.
// Smoothing never leaves an LF group (256 x 256 blocks): a sample on the border of its group is copied.  Operand order as in the Java.
struct LfArgs {
    const int32_t *q[3];        // quantised LF, frame order X, Y, B, hb x wb
    const uint8_t *ep;          // extraPrecision per LF group
    float *out[3];
    int hb, wb, gcols, cfl, smooth;
    float sd[3], kx, kb;
};
__device__ __forceinline__ void lf_value(const LfArgs &A, size_t o, const float (&sdg)[3], float (&v)[3]) {
    v[0] = __fmul_rn((float)A.q[0][o], sdg[0]);
    v[1] = __fmul_rn((float)A.q[1][o], sdg[1]);
    v[2] = __fmul_rn((float)A.q[2][o], sdg[2]);
    if (A.cfl) {
        v[0] = __fadd_rn(v[0], __fmul_rn(A.kx, v[1]));
        v[2] = __fadd_rn(v[2], __fmul_rn(A.kb, v[1]));
    }
}
// the value of LF sample i (row-major over hb x wb): dequantised, LF chroma-from-luma, adaptively smoothed inside its LF group
__device__ __forceinline__ void lf_sample(const LfArgs &A, long long i, float (&c)[3]) {
    const int y = (int)(i / A.wb), x = (int)(i - (long long)y * A.wb);
    const int gy = y >> 8, gx = x >> 8, ly = y & 255, lx = x & 255;
    const int h = min(256, A.hb - (gy << 8)), w = min(256, A.wb - (gx << 8));
    const float div = (float)(1 << A.ep[gy * A.gcols + gx]);
    const float sdg[3] = {__fdiv_rn(A.sd[0], div), __fdiv_rn(A.sd[1], div), __fdiv_rn(A.sd[2], div)};
    lf_value(A, (size_t)i, sdg, c);
    const bool interior = A.smooth && h >= 3 && w >= 3 && ly >= 1 && ly + 1 < h && lx >= 1 && lx + 1 < w;
    if (interior) {
        float nb[8][3];     // W, E, N, S, NW, NE, SW, SE
        const long long wb = A.wb;
        lf_value(A, (size_t)(i - 1), sdg, nb[0]); lf_value(A, (size_t)(i + 1), sdg, nb[1]);
        lf_value(A, (size_t)(i - wb), sdg, nb[2]); lf_value(A, (size_t)(i + wb), sdg, nb[3]);
        lf_value(A, (size_t)(i - wb - 1), sdg, nb[4]); lf_value(A, (size_t)(i - wb + 1), sdg, nb[5]);
        lf_value(A, (size_t)(i + wb - 1), sdg, nb[6]); lf_value(A, (size_t)(i + wb + 1), sdg, nb[7]);
        float wv[3], gap = 0.5f;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const float adjacent = __fadd_rn(__fadd_rn(__fadd_rn(nb[0][k], nb[1][k]), nb[2][k]), nb[3][k]);
            const float diag = __fadd_rn(__fadd_rn(__fadd_rn(nb[4][k], nb[5][k]), nb[6][k]), nb[7][k]);
            wv[k] = __fadd_rn(__fadd_rn(__fmul_rn(0.05226273532324128f, c[k]), __fmul_rn(0.20345139757231578f, adjacent)),
                              __fmul_rn(0.0334829185968739f, diag));
            const float g = __fmul_rn(fabsf(__fsub_rn(c[k], wv[k])), A.sd[k]);
            if (g > gap) gap = g;
        }
        gap = __fsub_rn(3.0f, __fmul_rn(4.0f, gap));
        gap = gap > 0.0f ? gap : 0.0f;
#pragma unroll
        for (int k = 0; k < 3; k++) c[k] = __fadd_rn(__fmul_rn(__fsub_rn(c[k], wv[k]), gap), wv[k]);
    }
}
__global__ void k8_lf_dequant(LfArgs A) {
    const long long n = (long long)A.hb * A.wb;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float c[3];
        lf_sample(A, i, c);
        A.out[0][i] = c[0]; A.out[1][i] = c[1]; A.out[2][i] = c[2];
    }
}
