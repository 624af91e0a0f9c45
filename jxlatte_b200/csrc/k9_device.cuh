// k9_device.cuh -- per-pixel glue of the frame loop that the host path does in numpy, for device-resident decoding: a caller that
// keeps its channel buffers on the device (jxlatte_b200.decoder.DeviceEngine) would otherwise have to bring them back for these.
//
// k9_cast_to_float replaces ImageBuffer.castToFloat (J/util/ImageBuffer.java) on an int32 channel: (float)v * scale with
// scale = 1f / ((1 << depth) - 1) computed once on the host; one rounded multiply, never contracted.
// k9_modular_xyb replaces the lossy-Modular lines of Frame.decodeFrame (J/frame/Frame.java:429-447): the integer channels Y, X, B - Y
// scaled by LFGlobal.lfDequant into float X, Y, B, with the int32 sum Y + (B - Y) wrapping as Java's int addition does.
#pragma once
#include "common.cuh"

__global__ void k9_cast_to_float(const int32_t *__restrict__ in, long long n, float scale, float *__restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = __fmul_rn((float)in[i], scale);
}

struct XybArgs {
    const int32_t *y, *x, *b;       // Modular channels 0, 1, 2: Y, X, B - Y
    float *out[3];                  // X, Y, B
    long long n;
    float dq[3];                    // LFGlobal.lfDequant in X, Y, B order
};
__global__ void k9_modular_xyb(XybArgs A) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < A.n; i += (long long)gridDim.x * blockDim.x) {
        const int32_t y = A.y[i];
        const int32_t yb = (int32_t)((uint32_t)y + (uint32_t)A.b[i]);          // wrapping int32 add
        A.out[0][i] = __fmul_rn(A.dq[0], (float)A.x[i]);
        A.out[1][i] = __fmul_rn(A.dq[1], (float)y);
        A.out[2][i] = __fmul_rn(A.dq[2], (float)yb);
    }
}
