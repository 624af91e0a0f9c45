// k6_subsample.cuh -- chroma-subsampled VarDCT frames (JPEG recompression: jpegUpsamplingY/X != 0, SURVEY.md 8f-2).
//
// Replaces Frame.invertSubsampling (J/frame/Frame.java:681-723) and the shifted block positions of
// HFCoefficients.dequantizeHFCoefficients / finalizeLLF (J/frame/vardct/HFCoefficients.java:290-303, :205-222) and
// PassGroup.invertVarDCT (J/frame/group/PassGroup.java:217-226): a varblock at luma block (by, bx) takes part in
// channel c only when by, bx are multiples of the channel's subsampling factor, and then sits at (by >> sy, bx >> sx) of
// the channel's smaller plane with the same TransformType and hf multiplier.  When every varblock is 8x8 (what JPEG
// recompression produces) channel c is therefore an ordinary 4:4:4 problem on strided block maps: k6_submap builds the
// maps, stage 1 runs once per channel, k6_upsample_* restores the plane size.
#pragma once
#include "common.cuh"

// flag[0] |= 1 when a subsampled channel meets a varblock larger than 8x8 (overlapping writes in the reference; unsupported)
__global__ void k6_submap(const uint8_t *__restrict__ ds, const int32_t *__restrict__ hf, int wb, int hbc, int wbc, int sy, int sx,
                          uint8_t *__restrict__ ds_c, uint8_t *__restrict__ bo_c, int32_t *__restrict__ hf_c, int *__restrict__ flag) {
    const int n = hbc * wbc;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int y = i / wbc, x = i - y * wbc;
        const size_t src = (size_t)(y << sy) * wb + (x << sx);
        const uint8_t t = ds[src];
        if ((sy | sx) && !(t <= 3 || (t >= 12 && t <= 17)) && t <= 26) *flag = 1;
        ds_c[i] = t;
        bo_c[i] = 1;
        hf_c[i] = hf[src];
    }
}

// one output sample of a doubling: .75 of the input sample it lies on (c75 = __fmul_rn(0.75f, centre), shared by the two outputs of
// that sample) + .25 of the input neighbour on its side (clamped at the edge)
__device__ __forceinline__ float double_px(float c75, float side) { return __fadd_rn(c75, __fmul_rn(0.25f, side)); }

// one horizontal doubling: out[y][2x] = .75 in[y][x] + .25 in[y][max(x-1,0)], out[y][2x+1] = .75 in[y][x] + .25 in[y][min(x+1,w-1)]
__global__ void k6_upsample_h(const float *__restrict__ in, int h, int w, float *__restrict__ out) {
    const long long n = (long long)h * w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(i / w), x = (int)(i - (long long)y * w);
        const float *row = in + (size_t)y * w;
        const float b75 = __fmul_rn(0.75f, row[x]);
        const float l = double_px(b75, row[x == 0 ? 0 : x - 1]);
        const float r = double_px(b75, row[x + 1 == w ? w - 1 : x + 1]);
        *reinterpret_cast<float2 *>(out + (size_t)y * 2 * w + 2 * x) = make_float2(l, r);
    }
}

// one vertical doubling
__global__ void k6_upsample_v(const float *__restrict__ in, int h, int w, float *__restrict__ out) {
    const long long n = (long long)h * w;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(i / w), x = (int)(i - (long long)y * w);
        const float b75 = __fmul_rn(0.75f, in[(size_t)y * w + x]);
        const float up = in[(size_t)(y == 0 ? 0 : y - 1) * w + x], dn = in[(size_t)(y + 1 == h ? h - 1 : y + 1) * w + x];
        out[(size_t)(2 * y) * w + x] = double_px(b75, up);
        out[(size_t)(2 * y + 1) * w + x] = double_px(b75, dn);
    }
}
