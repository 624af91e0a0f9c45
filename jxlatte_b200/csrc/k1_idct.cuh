// k1_idct.cuh -- K1: HF dequantisation + chroma-from-luma + LLF-from-LF + inverse transform, fused per varblock.
//
// Replaces (J/ = java/com/traneptora/jxlatte/ in the reference):
//   HFCoefficients.dequantizeHFCoefficients  J/frame/vardct/HFCoefficients.java:267-319
//   HFCoefficients.chromaFromLuma            :146-192
//   HFCoefficients.finalizeLLF               :194-229  (+ MathHelper.forwardDCT2D, J/util/MathHelper.java:124-136)
//   PassGroup.invertVarDCT                   J/frame/group/PassGroup.java:170-331 (all 27 TransformTypes)
//
// Three kernel families, each persistent over the K0 work lists:
//   k1_small   8x8-class (DCT8, Hornuss, DCT2, DCT4, DCT4x8, DCT8x4, AFV0-3): one thread per varblock-channel, 64
//              coefficients in registers, staged through shared memory so global traffic stays row-coalesced.
//   k1_medium  16/32-class (8 shapes): tile in shared memory, one thread per line, IDCT in registers.
//   k1_big     any side >= 64: two passes (columns, then rows) over 32-line strips, lane = line, each warp owning 32
//              outputs of 32 lines; the intermediate lives in the output plane (L2-resident between the passes).
// Every float operation is an explicit round-to-nearest mul/add/sub/div in the Java's order (Java never contracts to
// FMA), so the XYB planes this stage writes are bit-identical to the reference's (see transforms.cuh for why).
#pragma once
#include "common.cuh"
#include "k0_lists.cuh"
#include "transforms.cuh"

__constant__ float c_afv[256];        // PassGroup.AFV_BASIS (J/frame/group/PassGroup.java:19-58)
__constant__ float c_cos[1302];       // MathHelper.cosineLut levels 1..5 (lengths 2..32), [n][k], J/util/MathHelper.java:17-30
__constant__ int c_cos_off[6];        // offset of level l
__constant__ float c_llf_scale[32];   // LLFScale.SCALE_F (J/frame/vardct/LLFScale.java:7-23)
__constant__ DevTables c_tab;

struct CosLut {   // packed MathHelper.cosineLut, constant-bank operand once the index is a compile-time constant
    __device__ __forceinline__ float operator()(int i) const { return c_cos[i]; }
};

__device__ __forceinline__ int ilog2_pow2(int v) { return 31 - __clz(v); }

// HFCoefficients.dequantizeHFCoefficients :310-314, one coefficient (not in the LLF corner)
__device__ __forceinline__ float dequant_one(int coeff, float qb, float qbn, float sfc, float w) {
    float quant;
    if (coeff > -2 && coeff < 2) quant = coeff == 0 ? 0.0f : (coeff > 0 ? qb : -qb);
    else quant = __fsub_rn((float)coeff, __fdiv_rn(qbn, (float)coeff));
    return __fmul_rn(__fmul_rn(quant, sfc), w);
}

// Per-varblock constants shared by the three families
struct VB {
    int by, bx, type, H, W;     // origin in cells, TransformType, pixel size
    int dsH, dsW;               // LLF corner size
    float sfc[3];               // scaleFactor[c] / hfMultiplier  (:299)
    int origin;                 // raster index of the origin cell (blockList order key)
    const float *w[3];          // weights in storage orientation
};

__device__ __forceinline__ VB make_vb(const K1Params &P, int item, int type) {
    VB v;
    v.by = item >> 16;
    v.bx = item & 0xffff;
    v.type = type;
    const TTInfo tt = c_tt[type];
    v.dsH = tt.bh; v.dsW = tt.bw;
    v.H = tt.bh * 8; v.W = tt.bw * 8;
    v.origin = v.by * P.wb + v.bx;
    const float hm = (float)P.hf_mul[v.origin];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        v.sfc[c] = __fdiv_rn(P.sf[c], hm);
        v.w[c] = P.wexp + c_tab.wexp_off[type] + c * v.H * v.W;
    }
    return v;
}

// ------------------------------------------------------------------------------------------------------------
// k1_small: 8x8-class
// ------------------------------------------------------------------------------------------------------------
#define SMALL_PITCH 100   // 96 varblock-channels + 4: bank = (4 * elem + slot) mod 32, conflict-free for both phases

struct SmemOut {
    float *base;
    __device__ __forceinline__ void operator()(int y, int x, float val) const { base[(y * 8 + x) * SMALL_PITCH] = val; }
};
struct AfvBasis {
    __device__ __forceinline__ float operator()(int j, int i) const { return c_afv[j * 16 + i]; }
};

__global__ void __launch_bounds__(128) k1_small(K1Params P, const Sched *__restrict__ S, const int *__restrict__ items) {
    __shared__ float tile[64 * SMALL_PITCH];
    const int total = S->small_cum[N_SMALL];
    const int tid = threadIdx.x;
    for (int b = blockIdx.x; b < total; b += gridDim.x) {
        int ti = 0;
        while (b >= S->small_cum[ti + 1]) ti++;
        const int type = c_small_types[ti];
        const int first = (b - S->small_cum[ti]) * SMALL_BATCH;
        const int nvb = min(SMALL_BATCH, S->cnt[type] - first);
        const int *it = items + S->start[type] + first;

        // load + dequant + CfL: lane = (varblock, row y): one 32-byte row of each coefficient plane and of each weight table per
        // thread as two 128-bit loads (rows of a varblock are 32-byte aligned when the planes are; P.vec says so), instead of
        // 48 scalar loads with their address arithmetic -- this phase, not the transform, was most of the kernel's instructions
        // lane -> (varblock, row): sixteen varblocks side by side, two rows per warp.  The staging index is (y * 8 + x) * 100 +
        // 3 * varblock + c, so rows fall on the same bank (800 = 0 mod 32) and varblocks on distinct ones: eight rows per warp
        // (the earlier mapping) made every staging access an 8-way bank conflict, two rows make it 2-way
        const int y = tid >> 4;
        for (int pass = 0; pass < 2; pass++) {
            const int vbi = (tid & 15) + 16 * pass;
            if (vbi < nvb) {
                const VB v = make_vb(P, it[vbi], type);
                const int py = v.by * 8 + y, px = v.bx * 8;
                const size_t gi = (size_t)py * P.W + px;
                int q[3][8];
                float w[3][8];
#pragma unroll
                for (int c = 0; c < 3; c++) {
                    const int32_t *qp = (c == 0 ? P.q[0] : (c == 1 ? P.q[1] : P.q[2])) + gi;
                    if (P.vec) {
                        const int4 a = __ldg(reinterpret_cast<const int4 *>(qp)), b4 = __ldg(reinterpret_cast<const int4 *>(qp) + 1);
                        q[c][0] = a.x; q[c][1] = a.y; q[c][2] = a.z; q[c][3] = a.w; q[c][4] = b4.x; q[c][5] = b4.y; q[c][6] = b4.z; q[c][7] = b4.w;
                    } else {
#pragma unroll
                        for (int x = 0; x < 8; x++) q[c][x] = __ldg(qp + x);
                    }
                    const float4 wa = __ldg(reinterpret_cast<const float4 *>(v.w[c] + y * 8)), wb4 = __ldg(reinterpret_cast<const float4 *>(v.w[c] + y * 8) + 1);
                    w[c][0] = wa.x; w[c][1] = wa.y; w[c][2] = wa.z; w[c][3] = wa.w; w[c][4] = wb4.x; w[c][5] = wb4.y; w[c][6] = wb4.z; w[c][7] = wb4.w;
                }
                // chromaFromLuma factors of this row's 64x64 tile (MedVB has the story of the gate)
                const int tile_i = (py >> 6) * P.tw + (px >> 6);
                float kX = 0.0f, kB = 0.0f;
                {
                    // the three loads leave together (one round trip instead of gate -> factors): this kernel is latency-bound
                    const int gate = __ldg(P.cfl_gate + tile_i), fx = __ldg(P.xfy + tile_i), fb = __ldg(P.bfy + tile_i);
                    if (gate <= v.origin) {
                        kX = __fadd_rn(P.base_x, __fdiv_rn((float)fx, P.color_factor));
                        kB = __fadd_rn(P.base_b, __fdiv_rn((float)fb, P.color_factor));
                    }
                }
                float lf3[3] = {0.0f, 0.0f, 0.0f};
                if (y == 0) { lf3[0] = __ldg(P.lf[0] + v.origin); lf3[1] = __ldg(P.lf[1] + v.origin); lf3[2] = __ldg(P.lf[2] + v.origin); }
#pragma unroll
                for (int x = 0; x < 8; x++) {
                    float X, Y, B;
                    if (y == 0 && x == 0) {   // LLF of a 1x1 corner is the LF sample itself (scale 1)
                        X = lf3[0]; Y = lf3[1]; B = lf3[2];
                    } else {
                        X = dequant_one(q[0][x], P.qb[0], P.qbn, v.sfc[0], w[0][x]);
                        Y = dequant_one(q[1][x], P.qb[1], P.qbn, v.sfc[1], w[1][x]);
                        B = dequant_one(q[2][x], P.qb[2], P.qbn, v.sfc[2], w[2][x]);
                        X = __fadd_rn(X, __fmul_rn(kX, Y));
                        B = __fadd_rn(B, __fmul_rn(kB, Y));
                    }
                    float *d = tile + (y * 8 + x) * SMALL_PITCH + vbi * 3;
                    d[0] = X; d[1] = Y; d[2] = B;
                }
            }
        }
        __syncthreads();
        // transform: one thread per varblock-channel
        if (tid < nvb * 3) {
            float v[64];
#pragma unroll
            for (int e = 0; e < 64; e++) v[e] = tile[e * SMALL_PITCH + tid];
            SmemOut out{tile + tid};
            switch (type) {
            case 0: inv_dct8x8(v, CosLut(), out); break;
            case 1: inv_hornuss(v, out); break;
            case 2: inv_dct2(v, out); break;
            case 3: inv_dct4(v, CosLut(), out); break;
            case 12: inv_dct4x8<false>(v, CosLut(), out); break;
            case 13: inv_dct4x8<true>(v, CosLut(), out); break;
            default: inv_afv(v, (type == 16 || type == 17) ? 1 : 0, (type == 15 || type == 17) ? 1 : 0, AfvBasis(), CosLut(), out); break;
            }
        }
        __syncthreads();
        for (int pass = 0; pass < 2; pass++) {
            const int vbi = (tid & 15) + 16 * pass;
            if (vbi < nvb) {
                const int item = it[vbi];
                const int by = item >> 16, bx = item & 0xffff;
                const size_t o = (size_t)(by * 8 + y) * P.out_pitch + bx * 8;
                float r[3][8];
#pragma unroll
                for (int x = 0; x < 8; x++) {
                    const float *sp = tile + (y * 8 + x) * SMALL_PITCH + vbi * 3;
                    r[0][x] = sp[0]; r[1][x] = sp[1]; r[2][x] = sp[2];
                }
#pragma unroll
                for (int c = 0; c < 3; c++) {
                    float *op = (c == 0 ? P.out[0] : (c == 1 ? P.out[1] : P.out[2])) + o;
                    if (P.vec) {
                        reinterpret_cast<float4 *>(op)[0] = make_float4(r[c][0], r[c][1], r[c][2], r[c][3]);
                        reinterpret_cast<float4 *>(op)[1] = make_float4(r[c][4], r[c][5], r[c][6], r[c][7]);
                    } else {
#pragma unroll
                        for (int x = 0; x < 8; x++) op[x] = r[c][x];
                    }
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------------
// k1_medium: shapes with both sides in {8, 16, 32} except 8x8
// ------------------------------------------------------------------------------------------------------------
template <int N> __device__ __forceinline__ void line_idct(float *p, int stride) {
    float v[N];
#pragma unroll
    for (int i = 0; i < N; i++) v[i] = p[i * stride];
    RefIDCT<N>::run(v, CosLut());
#pragma unroll
    for (int i = 0; i < N; i++) p[i * stride] = v[i];
}

__host__ __device__ constexpr int cos_off(int l) { return l <= 1 ? 0 : cos_off(l - 1) + ((1 << (l - 1)) - 1) * (1 << (l - 1)); }

// HFCoefficients.finalizeLLF :218-226 for the whole DH x DW corner (DH, DW <= 4) of one varblock-channel, into d (pitch floats
// per row): forwardDCT2D = rows, then columns, each output * 1/N, in the reference's accumulation order; then * llfScale.  Every
// table index is a compile-time constant (constant-bank operands, no divergent indexing).
template <int DH, int DW> __device__ __forceinline__ void llf_corner(const float *lf, int wb, float *d, int pitch) {
    constexpr int LW = DW == 1 ? 0 : DW == 2 ? 1 : 2, LH = DH == 1 ? 0 : DH == 2 ? 1 : 2;
    const float invW = 1.0f / (float)DW, invH = 1.0f / (float)DH;
    float col[DH][DW];
#pragma unroll
    for (int y = 0; y < DH; y++) {
        float src[DW];
#pragma unroll
        for (int n = 0; n < DW; n++) src[n] = __ldg(lf + (size_t)y * wb + n);
#pragma unroll
        for (int kx = 0; kx < DW; kx++) {
            float d2;
            if (kx == 0) {
                d2 = src[0];
#pragma unroll
                for (int n = 1; n < DW; n++) d2 = __fadd_rn(d2, src[n]);
            } else {
                d2 = __fmul_rn(src[0], c_cos[cos_off(LW) + (kx - 1) * DW]);
#pragma unroll
                for (int n = 1; n < DW; n++) d2 = __fadd_rn(d2, __fmul_rn(src[n], c_cos[cos_off(LW) + (kx - 1) * DW + n]));
            }
            col[y][kx] = __fmul_rn(d2, invW);
        }
    }
#pragma unroll
    for (int ky = 0; ky < DH; ky++)
#pragma unroll
        for (int kx = 0; kx < DW; kx++) {
            float d2;
            if (ky == 0) {
                d2 = col[0][kx];
#pragma unroll
                for (int n = 1; n < DH; n++) d2 = __fadd_rn(d2, col[n][kx]);
            } else {
                d2 = __fmul_rn(col[0][kx], c_cos[cos_off(LH) + (ky - 1) * DH]);
#pragma unroll
                for (int n = 1; n < DH; n++) d2 = __fadd_rn(d2, __fmul_rn(col[n][kx], c_cos[cos_off(LH) + (ky - 1) * DH + n]));
            }
            d2 = __fmul_rn(d2, invH);
            // TransformType ctor :158-165: llfScale[y][x] = SCALE_F[y << (5 - yll)] * SCALE_F[x << (5 - xll)]
            const float sc = __fmul_rn(c_llf_scale[ky << (5 - LH)], c_llf_scale[kx << (5 - LW)]);
            d[ky * pitch + kx] = __fmul_rn(d2, sc);
        }
}

// Per-varblock constants of a k1_medium batch, formed once per varblock: make_vb's scale and the chroma-from-luma factors
// (HFCoefficients.chromaFromLuma :172-188) of the at most 2 x 2 tiles an 8-aligned varblock of side <= 32 touches, gate
// applied: a tile's factor is only "cached" once the varblock covering the tile's top-left pixel has been visited (raster
// order of origins); before that the Java reads 0.0f from its fresh arrays.
struct MedVB {
    int by, bx, origin;
    float sfc[3];
    float kx[4], kb[4];     // [2 * (tile row - first tile row) + tile column - first tile column]
};

template <int H, int W> __device__ void medium_batch(const K1Params &P, int type, const int *it, int nvb, float *tile, MedVB *s_vb) {
    constexpr int PITCH = W + 1, R = W / 4;       // a thread's unit: a run of four coefficients of a row
    constexpr int DH = H / 8, DW = W / 8;         // LLF corner
    const int tid = threadIdx.x, nt = blockDim.x;
    if (tid < 4 * nvb) {                          // four threads per varblock: tile s, and scale s < 3
        const int vbi = tid >> 2, s = tid & 3;
        const int item = it[vbi];
        const int by = item >> 16, bx = item & 0xffff, origin = by * P.wb + bx;
        MedVB &m = s_vb[vbi];
        if (s == 0) { m.by = by; m.bx = bx; m.origin = origin; }
        if (s < 3) m.sfc[s] = __fdiv_rn(P.sf[s], (float)P.hf_mul[origin]);
        const int ty = ((by * 8) >> 6) + (s >> 1), tx = ((bx * 8) >> 6) + (s & 1);
        float kX = 0.0f, kB = 0.0f;
        if (ty <= (by * 8 + H - 1) >> 6 && tx <= (bx * 8 + W - 1) >> 6) {
            const int t = ty * P.tw + tx;
            if (__ldg(P.cfl_gate + t) <= origin) {
                kX = __fadd_rn(P.base_x, __fdiv_rn((float)__ldg(P.xfy + t), P.color_factor));
                kB = __fadd_rn(P.base_b, __fdiv_rn((float)__ldg(P.bfy + t), P.color_factor));
            }
        }
        m.kx[s] = kX; m.kb[s] = kB;
    }
    __syncthreads();
    // load + dequant + CfL: one run of four per thread, runs fastest along x (coalesced rows), 128-bit loads of the
    // coefficients when P.vec holds and of the weights always (a run starts at a multiple of 4 of a weight table's row)
    const float *wt = P.wexp + c_tab.wexp_off[type];
    for (int i = tid; i < nvb * H * R; i += nt) {
        const int vbi = i / (H * R), r = i % (H * R);
        const int y = r / R, x0 = 4 * (r % R);
        const MedVB &m = s_vb[vbi];
        const int py = m.by * 8 + y, px = m.bx * 8 + x0;
        const size_t gi = (size_t)py * P.W + px;
        int q[3][4];
        float w[3][4];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const int32_t *qp = P.q[c] + gi;
            if (P.vec) {
                const int4 a = __ldg(reinterpret_cast<const int4 *>(qp));
                q[c][0] = a.x; q[c][1] = a.y; q[c][2] = a.z; q[c][3] = a.w;
            } else {
#pragma unroll
                for (int e = 0; e < 4; e++) q[c][e] = __ldg(qp + e);
            }
            const float4 b = __ldg(reinterpret_cast<const float4 *>(wt + c * H * W + y * W + x0));
            w[c][0] = b.x; w[c][1] = b.y; w[c][2] = b.z; w[c][3] = b.w;
        }
        const int s = 2 * ((py >> 6) - ((m.by * 8) >> 6)) + (px >> 6) - ((m.bx * 8) >> 6);
        const float kX = m.kx[s], kB = m.kb[s];
        float *d = tile + ((vbi * 3) * H + y) * PITCH + x0;
#pragma unroll
        for (int e = 0; e < 4; e++) {
            if (y < DH && x0 + e < DW) continue;   // the LLF corner, written below
            float X = dequant_one(q[0][e], P.qb[0], P.qbn, m.sfc[0], w[0][e]);
            const float Y = dequant_one(q[1][e], P.qb[1], P.qbn, m.sfc[1], w[1][e]);
            float B = dequant_one(q[2][e], P.qb[2], P.qbn, m.sfc[2], w[2][e]);
            X = __fadd_rn(X, __fmul_rn(kX, Y));
            B = __fadd_rn(B, __fmul_rn(kB, Y));
            d[e] = X; d[H * PITCH + e] = Y; d[2 * H * PITCH + e] = B;
        }
    }
    for (int j = tid; j < nvb * 3; j += nt) {
        const int vbi = j / 3, c = j % 3;
        const float *lf = c == 0 ? P.lf[0] : (c == 1 ? P.lf[1] : P.lf[2]);
        llf_corner<DH, DW>(lf + s_vb[vbi].origin, P.wb, tile + (j * H) * PITCH, PITCH);
    }
    __syncthreads();
    // columns (length H), then rows (length W): MathHelper.inverseDCT2D :110-120
    for (int l = tid; l < nvb * 3 * W; l += nt) line_idct<H>(tile + (l / W) * H * PITCH + (l % W), PITCH);
    __syncthreads();
    for (int l = tid; l < nvb * 3 * H; l += nt) line_idct<W>(tile + l * PITCH, 1);
    __syncthreads();
    for (int i = tid; i < nvb * H * R; i += nt) {
        const int vbi = i / (H * R), r = i % (H * R);
        const int y = r / R, x0 = 4 * (r % R);
        const MedVB &m = s_vb[vbi];
        const size_t o = (size_t)(m.by * 8 + y) * P.out_pitch + m.bx * 8 + x0;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const float *s = tile + ((vbi * 3 + c) * H + y) * PITCH + x0;
            float *op = P.out[c] + o;
            if (P.vec) {
                *reinterpret_cast<float4 *>(op) = make_float4(s[0], s[1], s[2], s[3]);
            } else {
#pragma unroll
                for (int e = 0; e < 4; e++) op[e] = s[e];
            }
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256) k1_medium(K1Params P, const Sched *__restrict__ S, const int *__restrict__ items) {
    __shared__ float tile[3 * MED_COEFFS * 9 / 8];
    __shared__ MedVB s_vb[MED_COEFFS / 128];
    const int total = S->med_cum[N_MED];
    for (int b = blockIdx.x; b < total; b += gridDim.x) {
        int ti = 0;
        while (b >= S->med_cum[ti + 1]) ti++;
        const int type = c_med_types[ti];
        const TTInfo tt = c_tt[type];
        const int per = MED_COEFFS / (tt.bh * tt.bw * 64);
        const int first = (b - S->med_cum[ti]) * per;
        const int nvb = min(per, S->cnt[type] - first);
        const int *it = items + S->start[type] + first;
        switch (type) {
        case 4: medium_batch<16, 16>(P, type, it, nvb, tile, s_vb); break;
        case 5: medium_batch<32, 32>(P, type, it, nvb, tile, s_vb); break;
        case 6: medium_batch<16, 8>(P, type, it, nvb, tile, s_vb); break;
        case 7: medium_batch<8, 16>(P, type, it, nvb, tile, s_vb); break;
        case 8: medium_batch<32, 8>(P, type, it, nvb, tile, s_vb); break;
        case 9: medium_batch<8, 32>(P, type, it, nvb, tile, s_vb); break;
        case 10: medium_batch<32, 16>(P, type, it, nvb, tile, s_vb); break;
        default: medium_batch<16, 32>(P, type, it, nvb, tile, s_vb); break;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// k1_big: varblocks with a side >= 64, two passes over 32-line strips, ONE CHANNEL per work item (a strip of one
// channel is 8..32 KB of shared memory, so several CTAs share an SM and the tail of the launch is short).
// PASS 0 = columns (reads coefficients, writes the plane), PASS 1 = rows (reads the plane, writes the plane).
// N = line length.  Both passes evaluate MathHelper.inverseDCTHorizontal's recurrence
//   out[k] = in[0] + sum_n fl(in[n] * lut[n-1][k])   in n order,
// forming each product once for out[k] and out[N-1-k] (the float table is exactly (anti)symmetric).
//   PASS 0  load phase: a lane takes four adjacent columns of a row, a warp four rows per 128-bit load (X and B items also
//           dequantise Y, which chroma-from-luma needs).  Walk: one column per warp, lanes = outputs k and their mirrors, over the column's
//           NON-ZERO coefficients only (ballot + ffs; adding a +-0 product changes no sum and ~95 % are zero): per live n
//           one shuffle for in[n] and one coalesced table-row read per 32 k.  Outputs replace the column in shared
//           memory and leave as 128-bit stores, four rows per warp.
//   PASS 1  the strip arrives by 128-bit loads.  lane = output index k (and its mirror).  A warp owns 32 k's of 16 rows: per n one coalesced table load
//           (issued four n ahead) and four 128-bit shared-memory broadcasts of in[row][n]; results go straight to the
//           plane, 128 bytes per row.
// Shared memory per CTA: PASS 0  A float[N][33] + llf scratch float[32][33];  PASS 1  A float[N][36].
// ------------------------------------------------------------------------------------------------------------
#define BIG_PITCH 33
#define BIG_PITCH1 36
template <int N, int PASS> struct BigCfg {
    // N = 32: one warp per CTA, which transforms its strip with RefIDCT<32> in registers; with more warps per CTA the others
    // waited at the barrier for it (42 % of those kernels' stall samples)
    static constexpr int kThreads = N == 32 ? 32 : (PASS == 0 ? 2 * N : N);
    static constexpr int kFloats = PASS == 0 ? N * BIG_PITCH + 32 * BIG_PITCH + N / 4 + 4 : (N == 32 ? N * BIG_PITCH : N * BIG_PITCH1);
    static constexpr int kBytes = kFloats * 4;
    // the column pass is latency-bound: resident warps matter more than registers per thread (48 warps per SM = 42 registers)
    static constexpr int kMinBlocks = N == 32 ? 24 : (PASS == 0 ? 1536 / kThreads : (N == 64 ? 14 : 1024 / kThreads));
};
__host__ __device__ constexpr int cos_big_off(int n) { return n == 64 ? 0 : n == 128 ? 63 * 64 : 63 * 64 + 127 * 128; }
#define COS_BIG_FLOATS (63 * 64 + 127 * 128 + 255 * 256)

__device__ __forceinline__ void ld_lut8(const float *p, float (&l)[8]) {
    const float4 *v = reinterpret_cast<const float4 *>(p);
    const float4 a = __ldg(v), b = __ldg(v + 1);
    l[0] = a.x; l[1] = a.y; l[2] = a.z; l[3] = a.w; l[4] = b.x; l[5] = b.y; l[6] = b.z; l[7] = b.w;
}

// One channel of a varblock: everything dequant_ch needs, fetched once per work item (c is a run-time value there)
struct ChanCtx {
    const int32_t *qc, *qy;      // this channel's and Y's coefficient planes
    const float *wc, *wy;        // weights in storage orientation
    const int32_t *fy;           // x_from_y or b_from_y
    float sfc_c, sfc_y, qb_c, qb_y, base;
    int c;
};
__device__ __forceinline__ ChanCtx make_chan(const K1Params &P, const VB &v, int c) {
    ChanCtx k;
    k.c = c;
    k.qc = c == 0 ? P.q[0] : (c == 1 ? P.q[1] : P.q[2]);
    k.qy = P.q[1];
    k.wc = c == 0 ? v.w[0] : (c == 1 ? v.w[1] : v.w[2]);
    k.wy = v.w[1];
    k.fy = c == 0 ? P.xfy : P.bfy;
    k.sfc_c = c == 0 ? v.sfc[0] : (c == 1 ? v.sfc[1] : v.sfc[2]);
    k.sfc_y = v.sfc[1];
    k.qb_c = c == 0 ? P.qb[0] : (c == 1 ? P.qb[1] : P.qb[2]);
    k.qb_y = P.qb[1];
    k.base = c == 0 ? P.base_x : P.base_b;
    return k;
}
// dequantise + CfL one channel of the coefficient at local (ly, lx) (outside the LLF corner)
__device__ __forceinline__ float dequant_ch(const K1Params &P, const VB &v, const ChanCtx &k, int ly, int lx) {
    const int py = v.by * 8 + ly, px = v.bx * 8 + lx;
    const size_t gi = (size_t)py * P.W + px;
    const int wi = ly * v.W + lx;
    const float Y = dequant_one(__ldg(k.qy + gi), k.qb_y, P.qbn, k.sfc_y, __ldg(k.wy + wi));
    if (k.c == 1) return Y;
    const float C = dequant_one(__ldg(k.qc + gi), k.qb_c, P.qbn, k.sfc_c, __ldg(k.wc + wi));
    const int tile = (py >> 6) * P.tw + (px >> 6);
    float f = 0.0f;   // chromaFromLuma :172-188, see MedVB
    if (__ldg(P.cfl_gate + tile) <= v.origin) f = __fadd_rn(k.base, __fdiv_rn((float)__ldg(k.fy + tile), P.color_factor));
    return __fadd_rn(C, __fmul_rn(f, Y));
}

template <int N, int PASS> __global__ void __launch_bounds__(BigCfg<N, PASS>::kThreads, BigCfg<N, PASS>::kMinBlocks)
k1_big(K1Params P, const Sched *__restrict__ S, const int *__restrict__ items, int cls, int *__restrict__ ticket) {
    extern __shared__ float smem[];
    __shared__ int s_wi;
    float *A = smem;
    float *scr = smem + N * BIG_PITCH;   // PASS 0 only
    const int tid = threadIdx.x, nt = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    // items are handed out through a counter (zeroed with the rest of Sched before K0): a strip with an LLF corner or a dense
    // column costs several times a sparse one, and a static round-robin left the last CTAs running alone
    const int total = S->big_cum[PASS][cls][3];
    for (;;) {
        if (tid == 0) s_wi = atomicAdd(ticket, 1);
        __syncthreads();
        const int wi = s_wi;     // every thread reads it before the barrier that ends the item, after which thread 0 rewrites it
        if (wi >= total) break;
        int j = 0;
        while (wi >= S->big_cum[PASS][cls][j + 1]) j++;
        const int type = c_big_types[PASS][cls][j];
        const TTInfo tt = c_tt[type];
        const int nstrips = (PASS == 0 ? tt.bw : tt.bh) / 4;
        const int local = wi - S->big_cum[PASS][cls][j];
        const int c = local % 3, strip = (local / 3) % nstrips;
        const VB v = make_vb(P, items[S->start[type] + local / (3 * nstrips)], type);
        const int Y0 = v.by * 8, X0 = v.bx * 8;
        float *plane = c == 0 ? P.out[0] : (c == 1 ? P.out[1] : P.out[2]);
        const float *lfc = c == 0 ? P.lf[0] : (c == 1 ? P.lf[1] : P.lf[2]);
        const ChanCtx kc = make_chan(P, v, c);

        if (PASS == 0) {
            // rows 0..N-1 of the strip's 32 columns.  lane = (row rs of a group of four rows, columns cx..cx+3): one 128-bit
            // streaming load per plane fetches four rows x 128 bytes per warp (X0 is a multiple of 8 and a strip offset a
            // multiple of 32, so the four columns are 16-byte aligned when P.vec holds and never straddle a 64x64 tile).  The
            // coefficient planes are read once (streaming: they must not evict the cosine table from L1); the weights are read
            // only for a run with a non-zero coefficient; the chroma-from-luma factor is formed once per 64-row band.  Staging is
            // conflict-free: bank = (rs + cx + e) mod 32.  The LLF corner is dequantised like any other run here and overwritten
            // below, behind a barrier, before anything reads it.
            {
                constexpr int NG = N / 4;                                // groups of four rows
                static_assert(NG % (BigCfg<N, PASS>::kThreads / 32) == 0, "row groups must tile the warps");
                const int rs = lane >> 3, cx = 4 * (lane & 7);
                const int lx = strip * 32 + cx, px = X0 + lx;
                const int32_t *qy0 = kc.qy + (size_t)(Y0 + rs) * P.W + px, *qc0 = kc.qc + (size_t)(Y0 + rs) * P.W + px;
                const float *wy0 = kc.wy + rs * v.W + lx, *wc0 = kc.wc + rs * v.W + lx;
                int last_band = -1;
                float f = 0.0f;
                // one group per lane and iteration: holding two groups' loads in flight spilled at the 42-register cap
                for (int g = warp; g < NG; g += nwarps) {
                    const int i = 4 * g + rs;
                    const size_t go = (size_t)(4 * g) * P.W;
                    int4 qy, qc = make_int4(0, 0, 0, 0);
                    if (P.vec) {
                        qy = __ldcs(reinterpret_cast<const int4 *>(qy0 + go));
                        if (c != 1) qc = __ldcs(reinterpret_cast<const int4 *>(qc0 + go));
                    } else {
                        qy = make_int4(__ldcs(qy0 + go), __ldcs(qy0 + go + 1), __ldcs(qy0 + go + 2), __ldcs(qy0 + go + 3));
                        if (c != 1) qc = make_int4(__ldcs(qc0 + go), __ldcs(qc0 + go + 1), __ldcs(qc0 + go + 2), __ldcs(qc0 + go + 3));
                    }
                    {
                        const int oy[4] = {qy.x, qy.y, qy.z, qy.w}, oc[4] = {qc.x, qc.y, qc.z, qc.w};
                        float val[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                        // both coefficients zero (most are): quant = 0, 0 * sfc * w = +0 and +0 + f * +0 = +0 whatever f's
                        // sign, so the weight is not needed.  Whole runs skip the arithmetic.
                        if ((oy[0] | oy[1] | oy[2] | oy[3] | oc[0] | oc[1] | oc[2] | oc[3]) != 0) {
                            const float4 wy4 = __ldg(reinterpret_cast<const float4 *>(wy0 + 4 * g * v.W));
                            const float wy[4] = {wy4.x, wy4.y, wy4.z, wy4.w};
                            float wc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                            if (c != 1) {
                                const float4 wc4 = __ldg(reinterpret_cast<const float4 *>(wc0 + 4 * g * v.W));
                                wc[0] = wc4.x; wc[1] = wc4.y; wc[2] = wc4.z; wc[3] = wc4.w;
                                const int band = (Y0 + i) >> 6;
                                if (band != last_band) {      // chromaFromLuma :172-188, see MedVB for the gate
                                    last_band = band;
                                    const int tile = band * P.tw + (px >> 6);
                                    f = 0.0f;
                                    if (__ldg(P.cfl_gate + tile) <= v.origin) f = __fadd_rn(kc.base, __fdiv_rn((float)__ldg(kc.fy + tile), P.color_factor));
                                }
                            }
#pragma unroll
                            for (int e = 0; e < 4; e++) {
                                if ((oy[e] | oc[e]) == 0) continue;
                                const float Y = dequant_one(oy[e], kc.qb_y, P.qbn, kc.sfc_y, wy[e]);
                                if (c == 1) {
                                    val[e] = Y;
                                } else {
                                    const float C = dequant_one(oc[e], kc.qb_c, P.qbn, kc.sfc_c, wc[e]);
                                    val[e] = __fadd_rn(C, __fmul_rn(f, Y));
                                }
                            }
                        }
                        float *a = A + i * BIG_PITCH + cx;
                        a[0] = val[0]; a[1] = val[1]; a[2] = val[2]; a[3] = val[3];
                    }
                }
            }
            if (strip == 0) {
                // finalizeLLF for a corner up to 32x32: row pass into scratch, column pass into A (overwrites)
                const int lw = ilog2_pow2(v.dsW), lh = ilog2_pow2(v.dsH);
                const float invW = 1.0f / (float)v.dsW, invH = 1.0f / (float)v.dsH;
                for (int i = tid; i < v.dsH * v.dsW; i += nt) {
                    const int y = i / v.dsW, kx = i % v.dsW;
                    const float *src = lfc + (size_t)(v.by + y) * P.wb + v.bx;
                    float d2;
                    if (kx == 0) {
                        d2 = src[0];
                        for (int n = 1; n < v.dsW; n++) d2 = __fadd_rn(d2, src[n]);
                    } else {
                        const float *lut = c_cos + c_cos_off[lw] + (kx - 1) * v.dsW;
                        d2 = __fmul_rn(src[0], lut[0]);
                        for (int n = 1; n < v.dsW; n++) d2 = __fadd_rn(d2, __fmul_rn(src[n], lut[n]));
                    }
                    scr[y * BIG_PITCH + kx] = __fmul_rn(d2, invW);
                }
                __syncthreads();
                for (int i = tid; i < v.dsH * v.dsW; i += nt) {
                    const int ky = i / v.dsW, kx = i % v.dsW;
                    const float *col = scr + kx;
                    float d2;
                    if (ky == 0) {
                        d2 = col[0];
                        for (int n = 1; n < v.dsH; n++) d2 = __fadd_rn(d2, col[n * BIG_PITCH]);
                    } else {
                        const float *lut = c_cos + c_cos_off[lh] + (ky - 1) * v.dsH;
                        d2 = __fmul_rn(col[0], lut[0]);
                        for (int n = 1; n < v.dsH; n++) d2 = __fadd_rn(d2, __fmul_rn(col[n * BIG_PITCH], lut[n]));
                    }
                    d2 = __fmul_rn(d2, invH);
                    const float sc = __fmul_rn(c_llf_scale[ky << (5 - lh)], c_llf_scale[kx << (5 - lw)]);
                    A[ky * BIG_PITCH + kx] = __fmul_rn(d2, sc);
                }
            }
        } else {
            // 32 rows x N columns of the intermediate plane into A[n][row]
            constexpr int PT = N == 32 ? BIG_PITCH : BIG_PITCH1;
            if (N == 64 && P.vec) {
                // 128-bit loads; a warp takes 16 rows x 8 columns, so that bank = (16 * (x / 4) + 4 * e + r) mod 32 (PT = 36)
                // differs across the warp for each of the four stores.  N = 128 and 256 keep the scalar loop: their row loops sit
                // at the 64-register cap, and with this loop beside them ptxas spilled a register (-Xptxas -v), while for N = 64
                // this loop is what removes the spill
                for (int w = warp; w < N / 4; w += nwarps) {
                    const int r = 16 * (w & 1) + (lane & 15), x = 8 * (w >> 1) + 4 * (lane >> 4);
                    const float4 t = *reinterpret_cast<const float4 *>(plane + (size_t)(Y0 + strip * 32 + r) * P.out_pitch + X0 + x);
                    A[x * PT + r] = t.x; A[(x + 1) * PT + r] = t.y; A[(x + 2) * PT + r] = t.z; A[(x + 3) * PT + r] = t.w;
                }
            } else {
                // N = 32 stays scalar: with pitch 33 a 128-bit mapping would put two lanes on each bank for every store
                for (int i = tid; i < 32 * N; i += nt) {
                    const int r = i / N, x = i % N;
                    A[x * PT + r] = plane[(size_t)(Y0 + strip * 32 + r) * P.out_pitch + X0 + x];
                }
            }
        }
        __syncthreads();

        if (N == 32) {
            if (warp == 0) {
                float vv[32];
#pragma unroll
                for (int m = 0; m < 32; m++) vv[m] = A[m * BIG_PITCH + lane];
                RefIDCT<32>::run(vv, CosLut());
                if (PASS == 0) {
#pragma unroll
                    for (int m = 0; m < 32; m++) plane[(size_t)(Y0 + m) * P.out_pitch + X0 + strip * 32 + lane] = vv[m];
                } else {
#pragma unroll
                    for (int m = 0; m < 32; m++) A[m * BIG_PITCH + lane] = vv[m];
                }
            }
            if (PASS == 1) {
                __syncthreads();
                for (int i = tid; i < 32 * N; i += nt) {
                    const int r = i / N, x = i % N;
                    plane[(size_t)(Y0 + strip * 32 + r) * P.out_pitch + X0 + x] = A[x * BIG_PITCH + r];
                }
            }
        } else if (PASS == 0) {
            // Sparse walk, one column of the strip per warp: lane l holds in[32 q + l] of chunk q, a ballot gives the column's
            // live n (most coefficients are zero and a +-0 product changes no sum), and for each live n -- in n order -- the
            // lanes own the outputs k = 32 m + lane and their mirrors: one coalesced table row read per 32 k, one shuffle for
            // in[n].  Work is proportional to the non-zeros of the column, not to the rows that are live anywhere in the strip.
            const float *__restrict__ lut = P.cos_big + cos_big_off(N);
            constexpr int KCH = N >= 64 ? N / 64 : 1, NCH = N / 32;
            for (int j = warp; j < 32; j += nwarps) {
                float vr[NCH];
                unsigned mk[NCH];
#pragma unroll
                for (int q = 0; q < NCH; q++) {
                    vr[q] = A[(32 * q + lane) * BIG_PITCH + j];
                    mk[q] = __ballot_sync(0xffffffffu, vr[q] != 0.0f);
                }
                mk[0] &= ~1u;                                   // n = 0 is the start value of every sum
                const float in0 = __shfl_sync(0xffffffffu, vr[0], 0);
                float lo[KCH], hi[KCH];
#pragma unroll
                for (int m = 0; m < KCH; m++) { lo[m] = in0; hi[m] = in0; }
#pragma unroll
                for (int q = 0; q < NCH; q++) {
                    unsigned m = mk[q];
                    while (m) {                                 // warp-uniform
                        const int b = __ffs(m) - 1;
                        m &= m - 1;
                        const float s2 = __shfl_sync(0xffffffffu, vr[q], b);
                        const float *row = lut + (32 * q + b - 1) * N + lane;
                        float l[KCH];
#pragma unroll
                        for (int u = 0; u < KCH; u++) l[u] = __ldg(row + 32 * u);
                        if (b & 1) {                            // n odd: the mirrored table entry is the negative
#pragma unroll
                            for (int u = 0; u < KCH; u++) {
                                const float pr = __fmul_rn(s2, l[u]);
                                lo[u] = __fadd_rn(lo[u], pr);
                                hi[u] = __fsub_rn(hi[u], pr);
                            }
                        } else {
#pragma unroll
                            for (int u = 0; u < KCH; u++) {
                                const float pr = __fmul_rn(s2, l[u]);
                                lo[u] = __fadd_rn(lo[u], pr);
                                hi[u] = __fadd_rn(hi[u], pr);
                            }
                        }
                    }
                }
                // column j of A belongs to this warp alone and has been read: it becomes the output column (other lanes read
                // the elements this lane overwrites: the ballots ordered that in practice, __syncwarp orders it formally)
                __syncwarp();
#pragma unroll
                for (int u = 0; u < KCH; u++) {
                    A[(32 * u + lane) * BIG_PITCH + j] = lo[u];
                    A[(N - 1 - 32 * u - lane) * BIG_PITCH + j] = hi[u];
                }
            }
            __syncthreads();
            if (P.vec) {                                       // four rows x 128 bytes per warp, lanes as in the load phase
                const int rs = lane >> 3, cx = 4 * (lane & 7);
                float *o = plane + (size_t)(Y0 + rs) * P.out_pitch + X0 + strip * 32 + cx;
                for (int g = warp; g < N / 4; g += nwarps) {
                    const float *a = A + (4 * g + rs) * BIG_PITCH + cx;
                    *reinterpret_cast<float4 *>(o + (size_t)(4 * g) * P.out_pitch) = make_float4(a[0], a[1], a[2], a[3]);
                }
            } else {
                for (int i = warp; i < N; i += nwarps)         // 128 bytes per row
                    plane[(size_t)(Y0 + i) * P.out_pitch + X0 + strip * 32 + lane] = A[i * BIG_PITCH + lane];
            }
        } else {
            const float *__restrict__ lut = P.cos_big + cos_big_off(N);
            constexpr int KCH = N / 64;                 // 32-lane chunks of k in [0, N/2)
            for (int w = warp; w < 2 * KCH; w += nwarps) {
                const int rg = w / KCH, k = (w % KCH) * 32 + lane;
                const float *src = A + 16 * rg;
                float lo[16], hi[16];
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const float4 t4 = *reinterpret_cast<const float4 *>(src + 4 * g);
                    lo[4 * g] = hi[4 * g] = t4.x; lo[4 * g + 1] = hi[4 * g + 1] = t4.y;
                    lo[4 * g + 2] = hi[4 * g + 2] = t4.z; lo[4 * g + 3] = hi[4 * g + 3] = t4.w;
                }
                // table entries four n ahead (L2 latency ~ 4 iterations of this loop)
                float lq[4];
#pragma unroll
                for (int u = 0; u < 4; u++) lq[u] = __ldg(lut + u * N + k);
#pragma unroll 1
                for (int n0 = 1; n0 < N; n0 += 4) {
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int n = n0 + u;
                        if (n >= N) break;
                        const float l = lq[u];
                        if (n + 4 < N) lq[u] = __ldg(lut + (n + 3) * N + k);
                        const float *sn = src + n * BIG_PITCH1;
#pragma unroll
                        for (int g = 0; g < 4; g++) {
                            const float4 t4 = *reinterpret_cast<const float4 *>(sn + 4 * g);
                            const float in4[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                            for (int e = 0; e < 4; e++) {
                                const float p = __fmul_rn(in4[e], l);
                                lo[4 * g + e] = __fadd_rn(lo[4 * g + e], p);
                                // n0 is odd, so n is odd exactly when u is even
                                hi[4 * g + e] = (u & 1) ? __fadd_rn(hi[4 * g + e], p) : __fsub_rn(hi[4 * g + e], p);
                            }
                        }
                    }
                }
#pragma unroll
                for (int r = 0; r < 16; r++) {
                    float *o = plane + (size_t)(Y0 + strip * 32 + 16 * rg + r) * P.out_pitch + X0;
                    o[k] = lo[r];
                    o[N - 1 - k] = hi[r];
                }
            }
        }
        __syncthreads();
    }
}
