// k10_preview.cuh -- 1:8 previews of a frame.
//
// k10_lf_preview renders a VarDCT frame from its LF image alone: each LF sample is the DC of one 8x8 block, and a block whose only
// coefficient is the DC inverts to that constant, so the LF image is the frame at 1:8.  One thread per output sample of the cropped
// ceil(h/8) x ceil(w/8) frame, in one launch:
//   * 4:4:4: the sample k8_lf_dequant computes (dequantisation by the LF group's extraPrecision, LF chroma-from-luma, adaptive
//     smoothing inside the 256 x 256-block LF group), through the same lf_sample;
//   * chroma-subsampled: dequantisation only (LFCoefficients applies no chroma-from-luma there, and smoothing with subsampling is a
//     stream error), then Frame.invertSubsampling's 0.75 / 0.25 doubling on each subsampled axis, evaluated from the reduced-grid
//     neighbours in registers: horizontal first, then vertical on the horizontally doubled values, with the rounded operations of
//     k6_upsample_h / _v (double_px), so the result equals the two-pass form bit for bit;
//   * then the frame's colour transform (color_px: XYB -> linear, YCbCr -> RGB, or none).
//
// k10_area_mean8 is the 1:8 preview of a finished canvas: the mean of each 8 x 8 area (fewer pixels on the right and bottom edge).
// Int32 channels are first cast as ImageBuffer.castToFloat does (k9_cast_to_float: one rounded multiply by 1f / ((1 << depth) - 1)).
// The sum starts at 0 and adds the area's samples in row-major order with __fadd_rn; it is divided once with __fdiv_rn by the number
// of pixels the area covers, so a float32 loop in numpy reproduces it exactly.
#pragma once
#include "common.cuh"
#include "k2_restore.cuh"
#include "k6_subsample.cuh"
#include "k8_features.cuh"

struct PreviewArgs {
    LfArgs lf;                  // q[], ep, hb, wb (the full LF grid), gcols, cfl, smooth, sd, kx, kb; lf.out is not used
    int sy[3], sx[3], subsampled;
    int out_h, out_w;
    float *out[3];
    K2Params P;                 // the colour transform (color_mode, m, ob, cob)
};

// channel c's dequantised LF at (ry, rx) of its reduced (hb >> sy) x (wb >> sx) grid, without chroma-from-luma
__device__ __forceinline__ float lf_reduced(const PreviewArgs &A, int c, int ry, int rx) {
    const int sy = A.sy[c], sx = A.sx[c], wc = A.lf.wb >> sx;
    const int g = ((ry << sy) >> 8) * A.lf.gcols + ((rx << sx) >> 8);
    const float sdg = __fdiv_rn(A.lf.sd[c], (float)(1 << A.lf.ep[g]));
    return __fmul_rn((float)A.lf.q[c][(size_t)ry * wc + rx], sdg);
}

// channel c's reduced grid doubled horizontally (when sx), at reduced row ry and full-grid column x
__device__ __forceinline__ float lf_row_doubled(const PreviewArgs &A, int c, int ry, int x) {
    if (!A.sx[c]) return lf_reduced(A, c, ry, x);
    const int wc = A.lf.wb >> 1, rx = x >> 1;
    const int side = (x & 1) ? min(rx + 1, wc - 1) : max(rx - 1, 0);
    return double_px(__fmul_rn(0.75f, lf_reduced(A, c, ry, rx)), lf_reduced(A, c, ry, side));
}

__global__ void k10_lf_preview(PreviewArgs A) {
    const long long n = (long long)A.out_h * A.out_w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(i / A.out_w), x = (int)(i - (long long)y * A.out_w);
        float v[3];
        if (!A.subsampled) {
            lf_sample(A.lf, (long long)y * A.lf.wb + x, v);
        } else {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                if (!A.sy[c]) {
                    v[c] = lf_row_doubled(A, c, y, x);
                } else {
                    const int hc = A.lf.hb >> 1, ry = y >> 1;
                    const int side = (y & 1) ? min(ry + 1, hc - 1) : max(ry - 1, 0);
                    v[c] = double_px(__fmul_rn(0.75f, lf_row_doubled(A, c, ry, x)), lf_row_doubled(A, c, side, x));
                }
            }
        }
        color_px(A.P, v[0], v[1], v[2]);
        A.out[0][i] = v[0]; A.out[1][i] = v[1]; A.out[2][i] = v[2];
    }
}

constexpr int kAreaChannels = 8;        // channels per k10_area_mean8 launch
struct AreaArgs {
    const void *plane[kAreaChannels];   // h x w, int32 when is_int[c], else float32
    int is_int[kAreaChannels];
    float scale[kAreaChannels];         // 1f / ((1 << depth) - 1) for int32 channels
    float *out[kAreaChannels];          // ceil(h / 8) x ceil(w / 8)
    int h, w, oh, ow;
};

// blockIdx.y = channel
__global__ void k10_area_mean8(AreaArgs A) {
    const int c = blockIdx.y;
    const long long n = (long long)A.oh * A.ow;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int oy = (int)(i / A.ow), ox = (int)(i - (long long)oy * A.ow);
        const int y0 = oy << 3, x0 = ox << 3, bh = min(8, A.h - y0), bw = min(8, A.w - x0);
        float s = 0.0f;
        if (A.is_int[c]) {
            const int32_t *p = (const int32_t *)A.plane[c];
            for (int y = 0; y < bh; y++)
                for (int x = 0; x < bw; x++) s = __fadd_rn(s, __fmul_rn((float)p[(size_t)(y0 + y) * A.w + x0 + x], A.scale[c]));
        } else {
            const float *p = (const float *)A.plane[c];
            for (int y = 0; y < bh; y++)
                for (int x = 0; x < bw; x++) s = __fadd_rn(s, p[(size_t)(y0 + y) * A.w + x0 + x]);
        }
        A.out[c][i] = __fdiv_rn(s, (float)(bh * bw));
    }
}
