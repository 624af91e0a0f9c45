// k11_batch.cuh -- the output of a batch decode: every image of the batch oriented, converted to 8 / 16-bit samples and written
// into its slot of one [n][c][out_h][out_w] tensor, in one launch (jxlb200_pack_batch_dev).
#pragma once
#include <type_traits>

// Output (y, x) of an image shown with orientation o -> the stored (pre-orientation) sample it shows; h x w is the stored size.
// JXLCodestreamDecoder.transposeBuffer (J/JXLCodestreamDecoder.java:43-112): 2 mirrors the columns, 3 turns by 180 degrees,
// 4 mirrors the rows, 5 transposes, 6 / 8 turn by 90 degrees clockwise / counter-clockwise, 7 transposes across the other diagonal.
__device__ __forceinline__ void orient_source(int o, int h, int w, int y, int x, int &sy, int &sx) {
    switch (o) {
    case 2: sy = y; sx = w - 1 - x; break;
    case 3: sy = h - 1 - y; sx = w - 1 - x; break;
    case 4: sy = h - 1 - y; sx = x; break;
    case 5: sy = x; sx = y; break;
    case 6: sy = h - 1 - x; sx = y; break;
    case 7: sy = h - 1 - x; sx = w - 1 - y; break;
    case 8: sy = x; sx = w - 1 - y; break;
    default: sy = y; sx = x; break;
    }
}

// blockIdx.z walks the items; each (32 x 8)-thread block covers a tile of 32 * P columns by 8 rows of the slot, where P = 16 bytes of
// output samples (16 px at 8 bits, 8 px at 16).  vec: every slot row starts 16-byte aligned, so a thread's P samples of a channel
// leave in one 128-bit store.
template <int BITS>
__global__ void __launch_bounds__(256) k11_pack_batch(const jxlb200_batch_item *__restrict__ items, int n, int c_out, int out_h, int out_w,
                                                      int vec, void *out) {
    typedef typename std::conditional<BITS == 8, uint8_t, uint16_t>::type T;
    constexpr int P = 16 / sizeof(T), MAXV = (1 << BITS) - 1;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * P;
    if (y >= out_h || x0 >= out_w) return;
    const int ncolor = c_out < 3 ? c_out : 3;
    for (int it = blockIdx.z; it < n; it += gridDim.z) {
        const jxlb200_batch_item &I = items[it];
        const int o = I.orientation, h = I.h, w = I.w;
        const int oh = o >= 5 ? w : h, ow = o >= 5 ? h : w;
        for (int c = 0; c < c_out; c++) {
            const bool fill = I.plane[c] == nullptr;
            const int pitch = I.pitch[c];
            const bool oetf = I.linear && c < ncolor;
            union { uint4 v; T s[P]; } q;
#pragma unroll
            for (int k = 0; k < P; k++) {
                const int x = x0 + k;
                q.s[k] = 0;
                if (y < oh && x < ow) {
                    if (fill) {
                        q.s[k] = (T)MAXV;
                    } else {
                        int sy, sx;
                        orient_source(o, h, w, y, x, sy, sx);
                        q.s[k] = (T)pack_sample(I.plane, I.is_int, I.depth, c, (long long)sy * pitch + sx, BITS, MAXV, oetf);
                    }
                }
            }
            T *dst = reinterpret_cast<T *>(out) + (((size_t)it * c_out + c) * out_h + y) * out_w + x0;
            if (vec) {
                *reinterpret_cast<uint4 *>(dst) = q.v;
            } else {
#pragma unroll
                for (int k = 0; k < P; k++)
                    if (x0 + k < out_w) dst[k] = q.s[k];
            }
        }
    }
}
