// jxlb200.cu -- libjxlb200.so: context, buffers and the C ABI declared in include/jxlb200.h.
// Single translation unit (all kernels are included here) so __constant__ tables need no relocatable device code.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <algorithm>
#include <array>
#include <string>
#include <vector>

#include "common.cuh"
#include "k0_lists.cuh"
#include "k1_idct.cuh"
#include "k2_restore.cuh"
#include "k2_fused.cuh"
#include "k2_exact.cuh"
// measured-and-parked stage-2 variants: in the tree and tested (CPU emulator / opt-in builds), not in the default library
#include "k2_stream.cuh"     /* default stage 2: persistent CTAs streaming column strips through TMA-fed row rings, bit-exact */
#ifdef JXLB200_WITH_PAIR
#include "k2_pair.cuh"       /* packed FP32x2: bit-exact, measured slower (profiles/r1_k2_pair_ncu.md) */
#endif
#include "k3_modular.cuh"
#include "k6_subsample.cuh"
#include "k7_blend.cuh"
#include "k8_features.cuh"
#include "k9_device.cuh"
#include "k10_preview.cuh"
#include "k11_batch.cuh"
#include "splines_host.cuh"
#include "qm_tables.cuh"
#include "split_nccl.cuh"

// grow-only device allocation
#ifndef JXLB200_OVERLAP_ROWS
#define JXLB200_OVERLAP_ROWS 0   /* measured on B200, 8K frame: off 3.46 ms; 512 rows 4.29; 1024 3.79; 2048 3.62 -- per-slab launch tails cost more than the overlap wins */
#endif

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

struct jxlb200_ctx {
    int device = 0;
    int sms = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;   // copy engines of the pipelined host entry point
    // stage 1 fans out over six streams: its kernels touch disjoint varblocks and each is latency-bound on its own
    cudaStream_t k1_stream[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_p0[4] = {nullptr, nullptr, nullptr, nullptr}, ev_done[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    std::string err;
    int64_t launches = 0;
    bool have_weights = false;
    int opt_stage2 = 0;
    bool uniform_sigma = false;         // jxlb200_restore_uniform: one 1/sigma for every block instead of the hf_mul / sharpness maps
    float uniform_inv_sigma = 0.0f;
    int opt_pipe_rows = 0;              // host entry points: rows per pipelined slab (0 = the measured default for the output format)
    int opt_pipe_fanout = -1;           // stage 1 of a slab on six streams (1) or one (0); -1 = by slab height
    int opt_overlap_rows = JXLB200_OVERLAP_ROWS;   // device-resident whole path: slab height for overlapping stage 2 of slab j with stage 1 of slab j+2 (0 = off)
    std::vector<cudaEvent_t> ev_pool;

    DevBuf sched, items, gate, wraw, woff, wexp, cosbig, lut8, sigma, flags;
    bool flags_pending = false;         // a kernel that may raise an error flag was enqueued since check_flags last read them
    float lut8_host[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // what lut8 holds on the device, and the stream that put it there
    cudaStream_t lut8_stream = nullptr;
    bool lut8_valid = false;
    DevBuf mid;        // stage-1 output planes incl. halo rows (whole path on device)
    DevBuf pp[2];      // ping-pong planes of the staged stage 2
    DevBuf in_q, in_q16, in_lf, in_maps, out_planes, mod;   // staging for the host entry points
    // group-row split (split_nccl.cuh): communicator, its stream, the slab's stage-1 planes and block maps with room for the halos
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_world = 1;
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t ev_edge = nullptr, ev_halo = nullptr, ev_maps = nullptr;
    DevBuf split_xyb, split_maps;
    DevBuf pack_thr[4];     // threshold tables of the sample pipeline: (8 | 16 bits) x (as is | sRGB from linear)
    DevBuf packed;          // interleaved 8/16-bit samples of jxlb200_vardct_reconstruct_packed
    DevBuf blend;           // five compact rectangles of jxlb200_blend
    DevBuf sub, sub_maps;   // chroma-subsampled frames: per-channel planes + scratch, strided block maps
    DevBuf dtab;            // small host tables of the feature calls (upsampling weights, spline arcs, LF extraPrecision)
    DevBuf feat;            // scratch of the feature calls (noise samples)
    DevTables tab;

    int fail(int code, const char *what, cudaError_t e = cudaSuccess) {
        err = what;
        if (e != cudaSuccess) { err += ": "; err += cudaGetErrorString(e); }
        return code;
    }
};

namespace {

const float kAfvBasis[256] = {
#include "afv_basis.inc"
};
const float kScaleF[32] = {
    1.0000000000000000000f, 1.0003954307206444720f, 1.0015830492063566798f, 1.0035668445359847378f, 1.0063534990068075448f,
    1.0099524393750471170f, 1.0143759095929498827f, 1.0196390660646908181f, 1.0257600967811994622f, 1.0327603660498609462f,
    1.0406645869479269795f, 1.0495010240726261235f, 1.0593017296818027804f, 1.0701028169146909598f, 1.0819447744633102634f,
    1.0948728278735071820f, 1.1089373535928257701f, 1.1241943530045446156f, 1.1407059950032801390f, 1.1585412372562662921f,
    1.1777765381971696030f, 1.1984966740821024139f, 1.2207956782314713353f, 1.2447779229495839992f, 1.2705593687655135089f,
    1.2982690107340108228f, 1.3280505578212198723f, 1.3600643892400108061f, 1.3944898413648201160f, 1.4315278911623840964f,
    1.4714043176060183528f, 1.5143734423313919909f,
};

template <int N, int PASS> cudaError_t big_attr() {
    return cudaFuncSetAttribute(k1_big<N, PASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, BigCfg<N, PASS>::kBytes);
}

int upload_constants(jxlb200_ctx *ctx) {
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_tt, h_tt, sizeof(h_tt)));
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_small_types, h_small_types, sizeof(h_small_types)));
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_med_types, h_med_types, sizeof(h_med_types)));
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_big_types, h_big_types, sizeof(h_big_types)));
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_afv, kAfvBasis, sizeof(kAfvBasis)));
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_llf_scale, kScaleF, sizeof(kScaleF)));
    // MathHelper.cosineLut (J/util/MathHelper.java:19-30): (float)(sqrt2 * cos(pi (n+1) (k+0.5) / s)), double math
    float cosv[1302];
    int offs[6] = {0, 0, 0, 0, 0, 0}, o = 0;
    const double root2 = sqrt(2.0);
    for (int l = 1; l <= 5; l++) {
        const int s = 1 << l;
        offs[l] = o;
        for (int n = 0; n < s - 1; n++)
            for (int k = 0; k < s; k++) cosv[o++] = (float)(root2 * cos(M_PI * (n + 1) * (k + 0.5) / s));
    }
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_cos, cosv, sizeof(float) * o));
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_cos_off, offs, sizeof(offs)));
    // levels 6..8 (lengths 64, 128, 256) live in global memory; the kernels rely on the table's exact symmetry
    // lut[n-1][s-1-k] == (-1)^n lut[n-1][k] in float, so verify it here rather than assume it
    {
        float *big = (float *)malloc(sizeof(float) * COS_BIG_FLOATS);
        bool symmetric = true;
        for (int l = 1; l <= 8; l++) {
            const int s = 1 << l;
            float *dst = l >= 6 ? big + cos_big_off(s) : nullptr;
            for (int n = 0; n < s - 1; n++)
                for (int k = 0; k < s; k++) {
                    const float a = (float)(root2 * cos(M_PI * (n + 1) * (k + 0.5) / s));
                    const float b = (float)(root2 * cos(M_PI * (n + 1) * ((s - 1 - k) + 0.5) / s));
                    if (a != (((n + 1) & 1) ? -b : b)) symmetric = false;
                    if (dst) dst[n * s + k] = a;
                }
        }
        if (!symmetric) { free(big); return ctx->fail(JXLB200_E_CUDA, "cosine table is not exactly symmetric on this host libm"); }
        cudaError_t e = ctx->cosbig.ensure(sizeof(float) * COS_BIG_FLOATS);
        if (e == cudaSuccess) e = cudaMemcpy(ctx->cosbig.p, big, sizeof(float) * COS_BIG_FLOATS, cudaMemcpyHostToDevice);
        free(big);
        if (e != cudaSuccess) return ctx->fail(JXLB200_E_CUDA, "cosine table upload", e);
    }
    int wo = 0;
    for (int t = 0; t < 27; t++) { ctx->tab.wexp_off[t] = wo; wo += 3 * h_tt[t].bh * h_tt[t].bw * 64; }
    CUDA_TRY(ctx, cudaMemcpyToSymbol(c_tab, &ctx->tab, sizeof(DevTables)));
    CUDA_TRY(ctx, ctx->wexp.ensure(sizeof(float) * wo));
    CUDA_TRY(ctx, (big_attr<32, 0>()));  CUDA_TRY(ctx, (big_attr<64, 0>()));
    CUDA_TRY(ctx, (big_attr<128, 0>())); CUDA_TRY(ctx, (big_attr<256, 0>()));
    CUDA_TRY(ctx, (big_attr<32, 1>()));  CUDA_TRY(ctx, (big_attr<64, 1>()));
    CUDA_TRY(ctx, (big_attr<128, 1>())); CUDA_TRY(ctx, (big_attr<256, 1>()));
    CUDA_TRY(ctx, k2_fused_init_all());
    CUDA_TRY(ctx, k2_exact_init_all());
    CUDA_TRY(ctx, k2_stream_init_all());
#ifdef JXLB200_WITH_PAIR
    CUDA_TRY(ctx, k2_pair_init_all());
#endif
    return 0;
}

int check_params(jxlb200_ctx *ctx, const jxlb200_frame_params *p) {
    if (!ctx) return JXLB200_E_ARG;
    if (!p) return ctx->fail(JXLB200_E_ARG, "frame params are NULL");
    if (p->width <= 0 || p->height <= 0 || (p->width & 7) || (p->height & 7))
        return ctx->fail(JXLB200_E_ARG, "padded frame size must be positive multiples of 8");
    if (p->width > 65535 * 8 || p->height > 65535 * 8) return ctx->fail(JXLB200_E_ARG, "frame too large");
    for (int c = 0; c < 3; c++) {
        if (p->shift_x[c] < 0 || p->shift_x[c] > 1 || p->shift_y[c] < 0 || p->shift_y[c] > 1)
            return ctx->fail(JXLB200_E_ARG, "jpegUpsampling shift outside 0..1 (FrameHeader.java:98-117)");
        if ((p->shift_x[c] && (p->width & 15)) || (p->shift_y[c] && (p->height & 15)))
            return ctx->fail(JXLB200_E_ARG, "subsampled frame size must be padded to 16 (Frame.getPaddedFrameSize)");
    }
    if (p->epf_iters < 0 || p->epf_iters > 3) return ctx->fail(JXLB200_E_ARG, "epf_iters outside 0..3");
    if (p->global_scale == 0) return ctx->fail(JXLB200_E_ARG, "global_scale is 0");
    return 0;
}

template <int N, int PASS> void launch_big(jxlb200_ctx *ctx, const K1Params &P, int cls, cudaStream_t st) {
    using Cfg = BigCfg<N, PASS>;
    // persistent grid = exactly the CTAs that are resident at once (registers included: asked of the runtime, once)
    static int per_sm = 0;
    if (per_sm == 0) {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k1_big<N, PASS>, Cfg::kThreads, Cfg::kBytes) != cudaSuccess || n < 1) n = 1;
        per_sm = min(n, 16);
    }
    k1_big<N, PASS><<<ctx->sms * per_sm, Cfg::kThreads, Cfg::kBytes, st>>>(P, ctx->sched.as<Sched>(), ctx->items.as<int>(), cls,
                                                                                     &ctx->sched.as<Sched>()->ticket[PASS][cls]);
    ctx->launches++;
}

// the device error flags (check_flags), allocated and zeroed on first use
cudaError_t ensure_flags(jxlb200_ctx *ctx, cudaStream_t st) {
    if (ctx->flags.p) return cudaSuccess;
    cudaError_t e = ctx->flags.ensure(sizeof(int) * 4);
    return e == cudaSuccess ? cudaMemsetAsync(ctx->flags.p, 0, sizeof(int) * 4, st) : e;
}

bool is_subsampled(const jxlb200_frame_params *p) {
    for (int c = 0; c < 3; c++)
        if (p->shift_x[c] || p->shift_y[c]) return true;
    return false;
}

// stage 1 on device pointers
int invert_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const int32_t *const q[3], const float *const lf[3],
               const uint8_t *ds, const uint8_t *bo, const int32_t *hf_mul, const int32_t *xfy, const int32_t *bfy,
               float *const out[3], long long pitch, bool fanout = true, int frame_rows = 0) {
    if (is_subsampled(p)) return ctx->fail(JXLB200_E_UNSUPPORTED, "stage 1 alone does not take chroma-subsampled frames: use jxlb200_vardct_reconstruct[_dev]");
    if (!ctx->have_weights) return ctx->fail(JXLB200_E_ARG, "jxlb200_set_qm_weights has not been called");
    const int W = p->width, H = p->height, wb = W >> 3, hb = H >> 3, tw = (W + 63) >> 6, th = (H + 63) >> 6;
    CUDA_TRY(ctx, ctx->sched.ensure(sizeof(Sched)));
    CUDA_TRY(ctx, ctx->items.ensure(sizeof(int) * (size_t)wb * hb));
    CUDA_TRY(ctx, ctx->gate.ensure(sizeof(int) * (size_t)tw * th));
    CUDA_TRY(ctx, ensure_flags(ctx, ctx->stream));
    cudaStream_t st = ctx->stream;
    Sched *S = ctx->sched.as<Sched>();
    CUDA_TRY(ctx, cudaMemsetAsync(S, 0, sizeof(Sched), st));
    const int ncells = wb * hb;
    const int g0 = min(ctx->sms * 4, ceil_div(ncells, 256));
    const int fhb = frame_rows > 0 ? frame_rows >> 3 : hb;      // block rows of one frame (a batch is a vertical stack)
    k0_count<<<g0, 256, 0, st>>>(ds, bo, ncells, wb, fhb, S, ctx->flags.as<int>() + 2);
    ctx->flags_pending = true;
    k0_plan<<<1, 32, 0, st>>>(S);
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->gate.p, 0x7f, sizeof(int) * (size_t)tw * th, st));
    k0_scatter<<<g0, 256, 0, st>>>(ds, bo, hb, wb, fhb, S, ctx->items.as<int>(), ctx->gate.as<int>(), tw);
    ctx->launches += 3;

    K1Params P;
    for (int c = 0; c < 3; c++) { P.q[c] = q[c]; P.lf[c] = lf[c]; P.out[c] = out[c]; }
    P.out_pitch = pitch;
    P.dct_select = ds; P.hf_mul = hf_mul; P.xfy = xfy; P.bfy = bfy;
    P.cfl_gate = ctx->gate.as<int>();
    P.wexp = ctx->wexp.as<float>();
    P.cos_big = ctx->cosbig.as<float>();
    P.W = W; P.H = H; P.wb = wb; P.hb = hb; P.tw = tw;
    // HFCoefficients.dequantizeHFCoefficients :270-275
    const float gs = 65536.0f / p->global_scale;
    P.sf[0] = gs * (float)pow(0.8, p->xqm_scale - 2.0);
    P.sf[1] = gs;
    P.sf[2] = gs * (float)pow(0.8, p->bqm_scale - 2.0);
    for (int c = 0; c < 3; c++) P.qb[c] = p->quant_bias[c];
    P.qbn = p->quant_bias_numerator;
    P.base_x = p->base_corr_x; P.base_b = p->base_corr_b; P.color_factor = (float)p->color_factor;
    P.vec = (pitch & 3) == 0 && (W & 3) == 0;
    for (int c = 0; c < 3; c++)
        if (((uintptr_t)q[c] | (uintptr_t)out[c]) & 15) P.vec = 0;

    // fan out: small | medium | four line-length classes of the big kernels (pass 0, then pass 1 once every pass 0 is done:
    // a varblock's row pass runs in the class of its width, its column pass in the class of its height)
    if (!fanout) {
        // one stream: used by the slab-pipelined host entry point, where PCIe (not stage 1) is the bottleneck and the ~40
        // event calls per slab of the fan-out cost more host time than the overlap wins
        k1_small<<<min(ctx->sms * 8, ceil_div(ncells, SMALL_BATCH)), 128, 0, st>>>(P, S, ctx->items.as<int>());
        k1_medium<<<min(ctx->sms * 4, ceil_div(ncells, 2)), 256, 0, st>>>(P, S, ctx->items.as<int>());
        ctx->launches += 2;
        launch_big<256, 0>(ctx, P, 3, st); launch_big<128, 0>(ctx, P, 2, st); launch_big<64, 0>(ctx, P, 1, st); launch_big<32, 0>(ctx, P, 0, st);
        launch_big<128, 1>(ctx, P, 2, st); launch_big<256, 1>(ctx, P, 3, st); launch_big<64, 1>(ctx, P, 1, st); launch_big<32, 1>(ctx, P, 0, st);
        CUDA_TRY(ctx, cudaGetLastError());
        return 0;
    }
    cudaStream_t *ks = ctx->k1_stream;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, st));
    for (int i = 0; i < 6; i++) CUDA_TRY(ctx, cudaStreamWaitEvent(ks[i], ctx->ev_fork, 0));
    // the big column passes go first: every row pass waits for all of them, small / medium fill the SMs they leave (measured: 2.50 ->
    // 2.47 ms per 8K step; stream priorities change nothing)
    launch_big<256, 0>(ctx, P, 3, ks[5]); launch_big<128, 0>(ctx, P, 2, ks[4]); launch_big<64, 0>(ctx, P, 1, ks[3]); launch_big<32, 0>(ctx, P, 0, ks[2]);
    k1_small<<<min(ctx->sms * 8, ceil_div(ncells, SMALL_BATCH)), 128, 0, ks[0]>>>(P, S, ctx->items.as<int>());
    k1_medium<<<min(ctx->sms * 4, ceil_div(ncells, 2)), 256, 0, ks[1]>>>(P, S, ctx->items.as<int>());
    ctx->launches += 2;
    for (int k = 0; k < 4; k++) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_p0[k], ks[2 + k]));
    for (int k = 0; k < 4; k++)
        for (int j = 0; j < 4; j++)
            if (j != k) CUDA_TRY(ctx, cudaStreamWaitEvent(ks[2 + k], ctx->ev_p0[j], 0));
    launch_big<128, 1>(ctx, P, 2, ks[4]); launch_big<256, 1>(ctx, P, 3, ks[5]); launch_big<64, 1>(ctx, P, 1, ks[3]); launch_big<32, 1>(ctx, P, 0, ks[2]);
    for (int i = 0; i < 6; i++) {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_done[i], ks[i]));
        CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_done[i], 0));
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// Stage 1 of a chroma-subsampled frame (k6_subsample.cuh).  q[c], lf[c]: channel c's own (H >> sy) x (W >> sx) planes;
// out[c]: full-size planes.  Stage 1 runs once per channel on that channel's plane with strided block maps; the kernel's
// three channel slots all read the same plane and only slot c (which carries channel c's weights and scale) is kept.
// Chroma-from-luma is off for such frames (HFCoefficients.java:149-151): base correlations and factor maps are zero.
int invert_subsampled_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const int32_t *const q[3], const float *const lf[3],
                          const uint8_t *ds, const int32_t *hf_mul, float *const out[3]) {
    const int W = p->width, H = p->height, wb = W >> 3, hb = H >> 3;
    const size_t npx = (size_t)W * H, nb = (size_t)wb * hb, nt = (size_t)((W + 63) >> 6) * ((H + 63) >> 6);
    CUDA_TRY(ctx, ctx->sub.ensure(sizeof(float) * 4 * npx));
    const size_t nb4 = (nb + 3) & ~(size_t)3;
    CUDA_TRY(ctx, ctx->sub_maps.ensure(2 * nb4 + sizeof(int32_t) * (nb + 2 * nt)));
    CUDA_TRY(ctx, ensure_flags(ctx, ctx->stream));
    cudaStream_t st = ctx->stream;
    char *mb = (char *)ctx->sub_maps.p;
    uint8_t *ds_c = (uint8_t *)mb, *bo_c = (uint8_t *)(mb + nb4);
    int32_t *hf_c = (int32_t *)(mb + 2 * nb4), *zero_tiles = hf_c + nb;
    CUDA_TRY(ctx, cudaMemsetAsync(zero_tiles, 0, sizeof(int32_t) * 2 * nt, st));
    float *plane[4];
    for (int i = 0; i < 4; i++) plane[i] = ctx->sub.as<float>() + i * npx;
    for (int c = 0; c < 3; c++) {
        const int sy = p->shift_y[c], sx = p->shift_x[c];
        const int Hc = H >> sy, Wc = W >> sx, hbc = hb >> sy, wbc = wb >> sx;
        k6_submap<<<min(ctx->sms * 4, ceil_div(hbc * wbc, 256)), 256, 0, st>>>(ds, hf_mul, wb, hbc, wbc, sy, sx, ds_c, bo_c, hf_c, ctx->flags.as<int>() + 3);
        ctx->flags_pending = true;
        ctx->launches++;
        jxlb200_frame_params pc = *p;
        pc.width = Wc; pc.height = Hc;
        pc.base_corr_x = 0.0f; pc.base_corr_b = 0.0f;
        for (int k = 0; k < 3; k++) pc.shift_x[k] = pc.shift_y[k] = 0;
        const int32_t *q3[3] = {q[c], q[c], q[c]};
        const float *l3[3] = {lf[c], lf[c], lf[c]};
        float *keep = (sy | sx) ? plane[0] : out[c];          // slot c's plane; the other two slots are scratch
        float *o3[3];
        for (int k = 0, sc = 1; k < 3; k++) o3[k] = k == c ? keep : plane[sc++];
        int rc = invert_dev(ctx, &pc, q3, l3, ds_c, bo_c, hf_c, zero_tiles, zero_tiles + nt, o3, Wc);
        if (rc) return rc;
        // Frame.invertSubsampling: horizontal doublings first, then vertical
        const float *cur = keep;
        int h = Hc, w = Wc;
        if (sx) {
            float *dst = sy ? plane[3] : out[c];
            k6_upsample_h<<<min(ctx->sms * 8, ceil_div(h * w, 256)), 256, 0, st>>>(cur, h, w, dst);
            ctx->launches++;
            cur = dst; w *= 2;
        }
        if (sy) {
            k6_upsample_v<<<min(ctx->sms * 8, ceil_div(h * w, 256)), 256, 0, st>>>(cur, h, w, out[c]);
            ctx->launches++;
        }
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

void fill_k2(K2Params &K, const jxlb200_frame_params *p, const jxlb200_slab *slab) {
    memset(&K, 0, sizeof(K));
    K.W = p->width;
    K.rows = slab ? slab->rows : p->height;
    K.y0 = slab ? slab->y0 : 0;
    K.frame_h = slab ? slab->frame_height : p->height;
    K.has_top = slab ? slab->has_top : 0;
    K.has_bottom = slab ? slab->has_bottom : 0;
    K.wb = (p->width + 7) >> 3;          // Modular frames are not padded to 8 (Frame.getPaddedFrameSize :924-941)
    K.gab = p->gab; K.iters = p->epf_iters; K.color_mode = p->color_mode;
    for (int c = 0; c < 3; c++) {   // Frame.performGabConvolution :510-517
        const float w1 = p->gab_w1[c], w2 = p->gab_w2[c];
        const float mult = 1.0f / (1.0f + 4.0f * (w1 + w2));
        K.gab_base[c] = mult; K.gab_adj[c] = w1 * mult; K.gab_diag[c] = w2 * mult;
        K.ch_scale[c] = p->epf_channel_scale[c];
    }
    K.gscale = 65536.0f / p->global_scale;
    for (int i = 0; i < 8; i++) K.sharp_lut[i] = p->epf_sharp_lut[i];
    const float step = 1.65f * 4.0f * (1.0f - (float)sqrt(0.5));   // Frame.java:545
    K.sigma_scale[0] = step * p->epf_pass0_sigma_scale;
    K.sigma_scale[1] = step;
    K.sigma_scale[2] = step * p->epf_pass2_sigma_scale;
    K.border_mul = p->epf_border_sad_mul;
    const float it = 255.0f / p->intensity_target;                    // OpsinInverseMatrix.invertXYB :108-119
    for (int i = 0; i < 9; i++) K.m[i] = p->opsin_matrix[i] * it;
    for (int c = 0; c < 3; c++) { K.ob[c] = p->opsin_bias[c]; K.cob[c] = -(float)cbrt((double)p->opsin_bias[c]); }
}

// stage 2 on device pointers
int restore_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const jxlb200_slab *slab, const float *const xyb[3],
                long long pitch, const int32_t *hf_mul, const int32_t *sharp, float *const out[3], int n_frames = 1) {
    // n_frames > 1 (no slab, pitch == width, default stage 2 only): that many frames of p->height rows stacked vertically
    K2Params K;
    fill_k2(K, p, slab);
    const int W = K.W, rows = K.rows, wb = K.wb;
    if (slab && ((slab->y0 & 7) || (slab->rows & 7) || slab->rows <= 0 || slab->y0 + slab->rows > slab->frame_height))
        return ctx->fail(JXLB200_E_ARG, "slab must start on a block row and stay inside the frame");
    cudaStream_t st = ctx->stream;
    for (int c = 0; c < 3; c++) { K.in[c] = xyb[c]; K.out[c] = out[c]; }
    K.in_pitch = pitch; K.out_pitch = W;
    K.hf_mul = hf_mul; K.sharpness = sharp;

    // inverse sigma per block, with one extra block row towards each neighbour slab
    float *inv_sigma = nullptr;
    if (K.iters > 0) {
        CUDA_TRY(ctx, ctx->sigma.ensure(sizeof(float) * (size_t)wb * ((size_t)((rows + 7) / 8) * n_frames + 2)));
        CUDA_TRY(ctx, ctx->lut8.ensure(sizeof(float) * 8));
        CUDA_TRY(ctx, ensure_flags(ctx, st));
        // K.sharp_lut lives in pageable memory, and an asynchronous copy from pageable memory first waits for everything
        // enqueued on its stream: once per slab that stalled the host behind stage 1 and left the upload engine idle meanwhile.
        // The table rarely changes (RestorationFilter.java:18-44), so it goes up only when it differs from the device's copy.
        if (!ctx->lut8_valid || ctx->lut8_stream != st || memcmp(ctx->lut8_host, K.sharp_lut, sizeof(float) * 8) != 0) {
            CUDA_TRY(ctx, cudaMemcpyAsync(ctx->lut8.p, K.sharp_lut, sizeof(float) * 8, cudaMemcpyHostToDevice, st));
            memcpy(ctx->lut8_host, K.sharp_lut, sizeof(float) * 8);
            ctx->lut8_stream = st;
            ctx->lut8_valid = true;
        }
        inv_sigma = ctx->sigma.as<float>() + wb;
        const int br0 = K.has_top ? -1 : 0, br1 = ((rows + 7) / 8) * n_frames + (K.has_bottom ? 1 : 0);
        if (ctx->uniform_sigma)
            k2_sigma_fill<<<min(ctx->sms * 2, ceil_div((br1 - br0) * wb, 256)), 256, 0, st>>>(ctx->uniform_inv_sigma, (long long)br0 * wb, (long long)(br1 - br0) * wb, inv_sigma);
        else {
            k2_sigma<<<min(ctx->sms * 2, ceil_div((br1 - br0) * wb, 256)), 256, 0, st>>>(hf_mul, sharp, wb, br0, br1, K.gscale,
                                                                                         ctx->lut8.as<float>(), inv_sigma, ctx->flags.as<int>());
            ctx->flags_pending = true;
        }
        ctx->launches++;
    }
    // Two bit-exact fused kernels.  Default: the stream kernel where it is the faster one -- at least 0.6 MP, and Gaborish on or three EPF
    // passes (8K frame, gab + EPF 3: 1.36 ms against 1.66 ms; without Gaborish its first stage is a plain copy, which only three passes of
    // filtering outweigh, and a small frame does not fill 148 persistent CTAs: tools/stage2_matrix.py, profiles/r2_stage2_matrix.md) --
    // else the tile kernel.  5 forces the stream kernel wherever the planes can take TMA (16-byte aligned bases and pitches, sizes that are
    // multiples of 8, epf_iters >= 1), 6 forces the tile kernel.
    const bool stream_pays = (K.gab || K.iters == 3) && (long long)K.W * K.rows * n_frames >= 600000ll;
    if (((ctx->opt_stage2 == 0 && stream_pays) || ctx->opt_stage2 == 5) && k2_stream_supported(K, n_frames) &&
        k2_stream_launch(K, inv_sigma, st, n_frames, ctx->sms) == 0) {
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
        return 0;
    }
    if ((ctx->opt_stage2 == 0 || ctx->opt_stage2 == 3 || ctx->opt_stage2 == 5 || ctx->opt_stage2 == 6) && k2_exact_supported(K)) {
#ifdef JXLB200_WITH_PAIR
        if (ctx->opt_stage2 == 3) k2_pair_dispatch(K, inv_sigma, st, n_frames);      // two blocks per thread on packed FP32x2: same bits, measured slower
        else
#endif
        k2_exact_dispatch(K, inv_sigma, st, n_frames);                               // one 2x2 block per thread
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
        return 0;
    }
    if (n_frames > 1) return ctx->fail(JXLB200_E_ARG, "stacked frames go through the default stage 2 only");
    if (ctx->opt_stage2 == 2) {                                     // opt-in: fused with re-associated EPF sums
        if (!k2_fused_supported(K)) return ctx->fail(JXLB200_E_UNSUPPORTED, "fused stage 2 does not take this frame");
        k2_fused_dispatch(K, inv_sigma, st);
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
        return 0;
    }

    // ---- staged fallback-free path: one kernel per stage, planes ping-pong through ctx->pp ----
    const long long pp_pitch = W;
    const size_t plane = (size_t)(rows + 2 * JXLB200_HALO_ROWS) * W;
    int reach[4], n_epf = 0, pass_id[3];
    if (K.iters == 3) pass_id[n_epf++] = 0;
    if (K.iters >= 1) pass_id[n_epf++] = 1;
    if (K.iters >= 2) pass_id[n_epf++] = 2;
    static const int kReach[3] = {3, 2, 1};
    // reach[i] = rows of margin stage i's output still needs for the stages after it
    int acc = 0;
    for (int i = n_epf - 1; i >= 0; i--) { reach[i + 1] = acc; acc += kReach[pass_id[i]]; }
    reach[0] = acc;   // margin needed on the Gaborish output (or on the input if gab is off)
    const float *cur[3] = {xyb[0], xyb[1], xyb[2]};
    long long cur_pitch = pitch;
    int which = 0;
    const dim3 blk(32, 8);
    auto rows_range = [&](int margin, int &r0, int &r1) {
        r0 = K.has_top ? -margin : 0;
        r1 = rows + (K.has_bottom ? margin : 0);
    };
    if (K.gab || n_epf) {
        CUDA_TRY(ctx, ctx->pp[0].ensure(sizeof(float) * 3 * plane));
        CUDA_TRY(ctx, ctx->pp[1].ensure(sizeof(float) * 3 * plane));
    }
    auto pp_plane = [&](int w, int c) { return ctx->pp[w].as<float>() + (size_t)c * plane + (size_t)JXLB200_HALO_ROWS * W; };
    if (K.gab) {
        int r0, r1;
        rows_range(reach[0], r0, r1);
        const dim3 grid(ceil_div(W, 32), ceil_div(r1 - r0, 8));
        k2_gab<<<grid, blk, 0, st>>>(K, cur[0], cur[1], cur[2], pp_plane(which, 0), pp_plane(which, 1), pp_plane(which, 2),
                                     cur_pitch, pp_pitch, r0, r1);
        ctx->launches++;
        for (int c = 0; c < 3; c++) cur[c] = pp_plane(which, c);
        cur_pitch = pp_pitch;
        which ^= 1;
    }
    for (int i = 0; i < n_epf; i++) {
        int r0, r1;
        rows_range(reach[i + 1], r0, r1);
        const dim3 grid(ceil_div(W, 32), ceil_div(r1 - r0, 8));
        float *o0 = pp_plane(which, 0), *o1 = pp_plane(which, 1), *o2 = pp_plane(which, 2);
        if (cur_pitch != pp_pitch) {
            // EPF kernels use one pitch for input and output: bring the raw planes into a ping-pong set first
            int c0, c1;
            rows_range(reach[0], c0, c1);
            for (int c = 0; c < 3; c++)
                CUDA_TRY(ctx, cudaMemcpy2DAsync(pp_plane(which, c) + (long long)c0 * pp_pitch, sizeof(float) * pp_pitch,
                                                cur[c] + (long long)c0 * cur_pitch, sizeof(float) * cur_pitch,
                                                sizeof(float) * W, c1 - c0, cudaMemcpyDeviceToDevice, st));
            for (int c = 0; c < 3; c++) cur[c] = pp_plane(which, c);
            cur_pitch = pp_pitch;
            which ^= 1;
            o0 = pp_plane(which, 0); o1 = pp_plane(which, 1); o2 = pp_plane(which, 2);
        }
        switch (pass_id[i]) {
        case 0: k2_epf<0><<<grid, blk, 0, st>>>(K, cur[0], cur[1], cur[2], o0, o1, o2, pp_pitch, inv_sigma, r0, r1); break;
        case 1: k2_epf<1><<<grid, blk, 0, st>>>(K, cur[0], cur[1], cur[2], o0, o1, o2, pp_pitch, inv_sigma, r0, r1); break;
        default: k2_epf<2><<<grid, blk, 0, st>>>(K, cur[0], cur[1], cur[2], o0, o1, o2, pp_pitch, inv_sigma, r0, r1); break;
        }
        ctx->launches++;
        cur[0] = o0; cur[1] = o1; cur[2] = o2;
        which ^= 1;
    }
    {
        const dim3 grid(ceil_div(W, 32), ceil_div(rows, 8));
        k2_color<<<grid, blk, 0, st>>>(K, cur[0], cur[1], cur[2], cur_pitch, out[0], out[1], out[2], (long long)W);
        ctx->launches++;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// device error flags -> status: [0] sharpness outside 0..7, [1] palette scratch, [2] dct_select out of range, [3] subsampling with
// large varblocks.  Read (a synchronous round trip) only when a kernel that raises them ran since the last read.
int check_flags(jxlb200_ctx *ctx) {
    if (!ctx->flags_pending) return 0;
    ctx->flags_pending = false;
    int e[4] = {0, 0, 0, 0};
    CUDA_TRY(ctx, cudaMemcpy(e, ctx->flags.p, sizeof(e), cudaMemcpyDeviceToHost));
    if (!e[0] && !e[2] && !e[3]) return 0;
    cudaMemset(ctx->flags.p, 0, sizeof(e));
    if (e[3]) return ctx->fail(JXLB200_E_UNSUPPORTED, "chroma subsampling with varblocks larger than 8x8");
    if (e[2]) return ctx->fail(JXLB200_E_STREAM, "Invalid Transform Type in dct_select, or a varblock that leaves its group (HFMetadata.java:45-46, 93-119)");
    return ctx->fail(JXLB200_E_STREAM, "Invalid EPF Sharpness (Frame.java:565-566)");
}

struct HostMaps {   // device copies of the per-block maps, packed into one allocation
    uint8_t *ds, *bo;
    int32_t *hf, *sharp, *xfy, *bfy;
};

int upload_maps(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const uint8_t *ds, const uint8_t *bo, const int32_t *hf,
                const int32_t *xfy, const int32_t *bfy, const int32_t *sharp, HostMaps &M) {
    const size_t nb = (size_t)(p->width >> 3) * (p->height >> 3);
    const size_t nt = (size_t)((p->width + 63) >> 6) * ((p->height + 63) >> 6);
    const size_t nb4 = (nb + 3) & ~(size_t)3;
    CUDA_TRY(ctx, ctx->in_maps.ensure(2 * nb4 + sizeof(int32_t) * (2 * nb + 2 * nt)));
    char *base = (char *)ctx->in_maps.p;
    M.ds = (uint8_t *)base; M.bo = (uint8_t *)(base + nb4);
    M.hf = (int32_t *)(base + 2 * nb4); M.sharp = M.hf + nb; M.xfy = M.sharp + nb; M.bfy = M.xfy + nt;
    cudaStream_t st = ctx->stream;
    if (ds) CUDA_TRY(ctx, cudaMemcpyAsync(M.ds, ds, nb, cudaMemcpyHostToDevice, st));
    if (bo) CUDA_TRY(ctx, cudaMemcpyAsync(M.bo, bo, nb, cudaMemcpyHostToDevice, st));
    if (hf) CUDA_TRY(ctx, cudaMemcpyAsync(M.hf, hf, sizeof(int32_t) * nb, cudaMemcpyHostToDevice, st));
    if (sharp) CUDA_TRY(ctx, cudaMemcpyAsync(M.sharp, sharp, sizeof(int32_t) * nb, cudaMemcpyHostToDevice, st));
    if (xfy) CUDA_TRY(ctx, cudaMemcpyAsync(M.xfy, xfy, sizeof(int32_t) * nt, cudaMemcpyHostToDevice, st));
    if (bfy) CUDA_TRY(ctx, cudaMemcpyAsync(M.bfy, bfy, sizeof(int32_t) * nt, cudaMemcpyHostToDevice, st));
    return 0;
}

// One host array of a host entry point and the device region it is staged in: `in` is uploaded before the call's kernels,
// `out` downloaded after them (the same pointer for an array changed in place).  Every region is copied at least one way, so
// a region of non-zero size with neither pointer is a NULL argument.
struct Staged {
    DevBuf *buf;
    const void *in;
    void *out;
    size_t bytes;
    void *dev = nullptr;
};

size_t staged_bytes(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// Checks every host pointer and carves the regions out of their buffers on the context's device, then uploads the inputs.
// The regions of one buffer must be consecutive in r[]: they share one allocation (each region 256-byte aligned), and a later
// group of the same buffer would reallocate it under the earlier one.
int stage_in(jxlb200_ctx *ctx, Staged *r, int n) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    for (int i = 0; i < n;) {
        size_t total = 0;
        int end = i;
        for (; end < n && r[end].buf == r[i].buf; end++) {
            if (r[end].bytes && !r[end].in && !r[end].out) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
            total += staged_bytes(r[end].bytes);
        }
        CUDA_TRY(ctx, r[i].buf->ensure(total));
        for (char *at = (char *)r[i].buf->p; i < end; at += staged_bytes(r[i++].bytes)) r[i].dev = at;
    }
    for (int i = 0; i < n; i++)
        if (r[i].in && r[i].bytes) CUDA_TRY(ctx, cudaMemcpyAsync(r[i].dev, r[i].in, r[i].bytes, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

// Downloads the outputs, then synchronises and reports device errors as jxlb200_sync does.
int stage_out(jxlb200_ctx *ctx, const Staged *r, int n) {
    for (int i = 0; i < n; i++)
        if (r[i].out && r[i].bytes) CUDA_TRY(ctx, cudaMemcpyAsync(r[i].out, r[i].dev, r[i].bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return jxlb200_sync(ctx);
}

// r[0..2]: three input planes staged in `bin`, r[3..5]: three output planes staged in `bout`, `bytes` each
template <class I, class O> void stage_planes(Staged *r, DevBuf &bin, I *const in[3], DevBuf &bout, O *const out[3], size_t bytes) {
    for (int c = 0; c < 3; c++) {
        r[c] = {&bin, in[c], nullptr, bytes};
        r[3 + c] = {&bout, nullptr, out[c], bytes};
    }
}

// the device pointers of three staged planes (.data() is the `T *const [3]` argument of an enqueue routine)
template <class T> std::array<T *, 3> planes_of(const Staged *r) { return {(T *)r[0].dev, (T *)r[1].dev, (T *)r[2].dev}; }

}  // namespace

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
extern "C" {

int32_t jxlb200_create(int32_t device, jxlb200_ctx **out) {
    if (!out) return JXLB200_E_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return JXLB200_E_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return JXLB200_E_CUDA;
    jxlb200_ctx *ctx = new (std::nothrow) jxlb200_ctx();
    if (!ctx) return JXLB200_E_CUDA;
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return JXLB200_E_CUDA; }
    ctx->stream = ctx->own_stream;
    if (cudaStreamCreateWithFlags(&ctx->h2d_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking) != cudaSuccess) { jxlb200_destroy(ctx); return JXLB200_E_CUDA; }
    bool okst = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 6 && okst; i++)
        okst = cudaStreamCreateWithFlags(&ctx->k1_stream[i], cudaStreamNonBlocking) == cudaSuccess &&
               cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 4 && okst; i++) okst = cudaEventCreateWithFlags(&ctx->ev_p0[i], cudaEventDisableTiming) == cudaSuccess;
    if (!okst) { jxlb200_destroy(ctx); return JXLB200_E_CUDA; }
    int rc = upload_constants(ctx);
    if (rc) { fprintf(stderr, "jxlb200_create: %s\n", ctx->err.c_str()); jxlb200_destroy(ctx); return rc; }
    *out = ctx;
    return 0;
}

void jxlb200_destroy(jxlb200_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf *all[] = {&ctx->sched, &ctx->items, &ctx->gate, &ctx->wraw, &ctx->woff, &ctx->wexp, &ctx->cosbig, &ctx->lut8, &ctx->sigma, &ctx->flags,
                     &ctx->mid, &ctx->pp[0], &ctx->pp[1], &ctx->in_q, &ctx->in_q16, &ctx->in_lf, &ctx->in_maps, &ctx->out_planes, &ctx->mod, &ctx->sub, &ctx->sub_maps, &ctx->dtab, &ctx->feat, &ctx->blend, &ctx->packed, &ctx->split_xyb, &ctx->split_maps, &ctx->pack_thr[0], &ctx->pack_thr[1], &ctx->pack_thr[2], &ctx->pack_thr[3]};
    for (DevBuf *b : all) b->release();
    if (ctx->comm && nccl_api().ok) nccl_api().CommDestroy(ctx->comm);
    if (ctx->comm_stream) cudaStreamDestroy(ctx->comm_stream);
    for (cudaEvent_t e : {ctx->ev_edge, ctx->ev_halo, ctx->ev_maps}) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->h2d_stream) cudaStreamDestroy(ctx->h2d_stream);
    for (int i = 0; i < 6; i++) { if (ctx->k1_stream[i]) cudaStreamDestroy(ctx->k1_stream[i]); if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]); }
    for (int i = 0; i < 4; i++) if (ctx->ev_p0[i]) cudaEventDestroy(ctx->ev_p0[i]);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
    delete ctx;
}

const char *jxlb200_last_error(jxlb200_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }

int32_t jxlb200_set_stream(jxlb200_ctx *ctx, void *cuda_stream) {
    if (!ctx) return JXLB200_E_ARG;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return 0;
}

int32_t jxlb200_sync(jxlb200_ctx *ctx) {
    if (!ctx) return JXLB200_E_ARG;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return check_flags(ctx);
}

int64_t jxlb200_launch_count(jxlb200_ctx *ctx) { return ctx ? ctx->launches : 0; }

#ifdef K2S_PHASE_TIMING
// diagnostic builds only (tools/phase_timing.py): read and clear the per-stage cycle counters of k2_stream
extern "C" int32_t jxlb200_debug_phase_clocks(unsigned long long out[16]) {
    unsigned long long zero[16] = {0};
    if (cudaMemcpyFromSymbol(out, k2s_phase_clk, sizeof(zero)) != cudaSuccess) return -1;
    return cudaMemcpyToSymbol(k2s_phase_clk, zero, sizeof(zero)) == cudaSuccess ? 0 : -1;
}
#endif

int32_t jxlb200_set_option(jxlb200_ctx *ctx, int32_t option, int32_t value) {
    if (!ctx) return JXLB200_E_ARG;
    if (option == JXLB200_OPT_STAGE2 && value >= 0 && value <= 6) {
#ifndef JXLB200_WITH_PAIR
        if (value == 3) return ctx->fail(JXLB200_E_UNSUPPORTED, "this library was built without k2_pair (-DJXLB200_WITH_PAIR)");
#endif
        if (value == 4) return ctx->fail(JXLB200_E_ARG, "unknown option or value");
        ctx->opt_stage2 = value;
        return 0;
    }
    if (option == JXLB200_OPT_OVERLAP_ROWS && value >= 0 && (value & 255) == 0) { ctx->opt_overlap_rows = value; return 0; }
    if (option == JXLB200_OPT_PIPE_ROWS && value >= 0 && (value & 255) == 0) { ctx->opt_pipe_rows = value; return 0; }
    if (option == JXLB200_OPT_PIPE_FANOUT && value >= -1 && value <= 1) { ctx->opt_pipe_fanout = value; return 0; }
    return ctx->fail(JXLB200_E_ARG, "unknown option or value");
}

// Page-lock a caller's buffer once (a Panama Arena segment is pageable: the pipelined host entry points copy from and to it six
// times slower than from pinned memory).  The segment stays usable as ordinary memory; unregister before it is freed.
int32_t jxlb200_host_register(jxlb200_ctx *ctx, void *ptr, uint64_t bytes) {
    if (!ctx) return JXLB200_E_ARG;
    if (!ptr || bytes == 0) return ctx->fail(JXLB200_E_ARG, "NULL or empty buffer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable));
    return 0;
}
int32_t jxlb200_host_unregister(jxlb200_ctx *ctx, void *ptr) {
    if (!ctx) return JXLB200_E_ARG;
    if (!ptr) return ctx->fail(JXLB200_E_ARG, "NULL buffer");
    CUDA_TRY(ctx, cudaHostUnregister(ptr));
    return 0;
}

// diagnostic: the shared-reciprocal divide of k2_exact against __fdiv_rn on n operand pairs drawn like the kernel's (divisor 1..13,
// numerators image-like and arbitrary bit patterns); *mismatches must come back 0
int32_t jxlb200_selftest_divide(jxlb200_ctx *ctx, int64_t n, int32_t seed, int64_t *mismatches) {
    if (!ctx) return JXLB200_E_ARG;
    if (!mismatches || n < 1) return ctx->fail(JXLB200_E_ARG, "bad arguments");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    unsigned long long *d = nullptr, h = 0;
    CUDA_TRY(ctx, cudaMalloc(&d, sizeof(h)));
    cudaMemsetAsync(d, 0, sizeof(h), ctx->stream);
    kx_selftest_div<<<ctx->sms * 8, 256, 0, ctx->stream>>>((unsigned long long)n, (unsigned)seed, d);
    ctx->launches++;
    cudaError_t e = cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) return ctx->fail(JXLB200_E_CUDA, "selftest", e);
    *mismatches = (int64_t)h;
    return 0;
}

int32_t jxlb200_qm_default_params(jxlb200_qm_params out[17]) {
    if (!out) return JXLB200_E_ARG;
    qm::default_params(out);
    return 0;
}

int32_t jxlb200_qm_generate(const jxlb200_qm_params params[17], float *weights, int32_t offsets[51]) {
    if (!params || !weights || !offsets) return JXLB200_E_ARG;
    return qm::generate(params, weights, offsets);
}

int32_t jxlb200_set_qm_weights(jxlb200_ctx *ctx, const float *weights, const int32_t offsets[51]) {
    if (!ctx) return JXLB200_E_ARG;
    if (!weights || !offsets) return ctx->fail(JXLB200_E_ARG, "weights / offsets are NULL");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, ctx->wraw.ensure(sizeof(float) * JXLB200_QM_FLOATS));
    CUDA_TRY(ctx, ctx->woff.ensure(sizeof(int) * 51));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->wraw.p, weights, sizeof(float) * JXLB200_QM_FLOATS, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->woff.p, offsets, sizeof(int) * 51, cudaMemcpyHostToDevice, ctx->stream));
    k0_expand_weights<<<dim3(16, 27), 256, 0, ctx->stream>>>(ctx->wraw.as<float>(), ctx->woff.as<int>(), ctx->tab, ctx->wexp.as<float>());
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // host arrays may be freed by the caller after return
    ctx->have_weights = true;
    return 0;
}

int32_t jxlb200_vardct_invert_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p,
    const int32_t *const qcoeff[3], const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, float *const xyb[3], int64_t xyb_pitch) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!qcoeff || !lf || !dct_select || !block_origin || !hf_mul || !x_from_y || !b_from_y || !xyb || xyb_pitch < p->width)
        return ctx->fail(JXLB200_E_ARG, "NULL plane pointer or pitch < width");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return invert_dev(ctx, p, qcoeff, lf, dct_select, block_origin, hf_mul, x_from_y, b_from_y, xyb, xyb_pitch);
}

int32_t jxlb200_restore_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const jxlb200_slab *slab,
    const float *const xyb[3], int64_t xyb_pitch, const int32_t *hf_mul, const int32_t *sharpness, float *const out[3]) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!xyb || !out || xyb_pitch < p->width || (p->epf_iters > 0 && (!hf_mul || !sharpness)))
        return ctx->fail(JXLB200_E_ARG, "NULL plane pointer or pitch < width");
    for (int c = 0; c < 3; c++)
        if (xyb[c] == out[c]) return ctx->fail(JXLB200_E_ARG, "in-place restore is not allowed");
    if (slab && (slab->y0 & 255)) return ctx->fail(JXLB200_E_ARG, "slab must start on a group row and stay inside the frame");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return restore_dev(ctx, p, slab, xyb, xyb_pitch, hf_mul, sharpness, out);
}

int32_t jxlb200_vardct_reconstruct_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p,
    const int32_t *const qcoeff[3], const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, const int32_t *sharpness, float *const out[3]) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!qcoeff || !lf || !dct_select || !block_origin || !hf_mul || !x_from_y || !b_from_y || !out || (p->epf_iters > 0 && !sharpness))
        return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t plane = (size_t)p->width * p->height;
    CUDA_TRY(ctx, ctx->mid.ensure(sizeof(float) * 3 * plane));
    float *mid[3] = {ctx->mid.as<float>(), ctx->mid.as<float>() + plane, ctx->mid.as<float>() + 2 * plane};
    const int W = p->width, H = p->height, wb = W >> 3, tw = (W + 63) >> 6;
    const int SL = ctx->opt_overlap_rows;
    if (!is_subsampled(p) && SL >= 256 && H >= 2 * SL) {
        // Stage 1 is short of warps per SM, stage 2 short of issue slots it can fill on its own: run them side by side.
        // The frame is cut into slabs of group rows; stage 1 walks the slabs on the main stream, stage 2 of slab j follows on a
        // second stream as soon as stage 1 of slab j+1 (its lower halo rows) is done, so it overlaps stage 1 of slab j+2.
        const int nslab = ceil_div(H, SL);
        while ((int)ctx->ev_pool.size() < nslab + 1) {
            cudaEvent_t e;
            CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            ctx->ev_pool.push_back(e);
        }
        cudaStream_t main = ctx->stream, side = ctx->d2h_stream;
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[nslab], main));       // the side stream starts after whatever precedes this call
        CUDA_TRY(ctx, cudaStreamWaitEvent(side, ctx->ev_pool[nslab], 0));
        for (int i = 0; i <= nslab; i++) {
            if (i < nslab) {
                const int y0 = i * SL, rows = std::min(SL, H - y0);
                jxlb200_frame_params ps = *p;
                ps.height = rows;
                const int32_t *q3[3] = {qcoeff[0] + (size_t)y0 * W, qcoeff[1] + (size_t)y0 * W, qcoeff[2] + (size_t)y0 * W};
                const float *l3[3] = {lf[0] + (size_t)(y0 / 8) * wb, lf[1] + (size_t)(y0 / 8) * wb, lf[2] + (size_t)(y0 / 8) * wb};
                float *m3[3] = {mid[0] + (size_t)y0 * W, mid[1] + (size_t)y0 * W, mid[2] + (size_t)y0 * W};
                rc = invert_dev(ctx, &ps, q3, l3, dct_select + (size_t)(y0 / 8) * wb, block_origin + (size_t)(y0 / 8) * wb, hf_mul + (size_t)(y0 / 8) * wb,
                                x_from_y + (size_t)(y0 / 64) * tw, b_from_y + (size_t)(y0 / 64) * tw, m3, W);
                if (rc) return rc;
                CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[i], main));
            }
            if (i >= 1) {
                const int j = i - 1, y0 = j * SL, rows = std::min(SL, H - y0);
                CUDA_TRY(ctx, cudaStreamWaitEvent(side, ctx->ev_pool[std::min(i, nslab - 1)], 0));
                jxlb200_frame_params ps = *p;
                ps.height = rows;
                jxlb200_slab sl = {y0, rows, H, j > 0 ? 1 : 0, j < nslab - 1 ? 1 : 0};
                const float *m3[3] = {mid[0] + (size_t)y0 * W, mid[1] + (size_t)y0 * W, mid[2] + (size_t)y0 * W};
                float *o3[3] = {out[0] + (size_t)y0 * W, out[1] + (size_t)y0 * W, out[2] + (size_t)y0 * W};
                ctx->stream = side;
                rc = restore_dev(ctx, &ps, &sl, m3, W, hf_mul + (size_t)(y0 / 8) * wb, sharpness ? sharpness + (size_t)(y0 / 8) * wb : nullptr, o3);
                ctx->stream = main;
                if (rc) return rc;
            }
        }
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_pool[nslab], side));
        CUDA_TRY(ctx, cudaStreamWaitEvent(main, ctx->ev_pool[nslab], 0));
        return 0;
    }
    rc = is_subsampled(p) ? invert_subsampled_dev(ctx, p, qcoeff, lf, dct_select, hf_mul, mid)
                          : invert_dev(ctx, p, qcoeff, lf, dct_select, block_origin, hf_mul, x_from_y, b_from_y, mid, p->width);
    if (rc) return rc;
    return restore_dev(ctx, p, nullptr, mid, p->width, hf_mul, sharpness, out);
}

// A batch of equally sized frames stacked vertically in every array (frame f occupies rows [f * H, (f + 1) * H) of the planes
// and the matching rows of the block / tile maps; H a multiple of 64 so the 64x64 chroma-from-luma tiles of different frames do
// not mix).  Varblocks never leave their frame, so stage 1 runs ONCE over the stack -- one set of work lists and launches, which
// is what small frames need to fill the GPU -- and stage 2 runs per frame, each mirroring at its own edges.
int32_t jxlb200_vardct_reconstruct_batch_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, int32_t n_frames,
    const int32_t *const qcoeff[3], const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, const int32_t *sharpness, float *const out[3]) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (n_frames < 1) return ctx->fail(JXLB200_E_ARG, "n_frames < 1");
    if (is_subsampled(p)) return ctx->fail(JXLB200_E_UNSUPPORTED, "batched reconstruction of chroma-subsampled frames");
    if (p->height & 63) return ctx->fail(JXLB200_E_ARG, "batched frames need a padded height that is a multiple of 64");
    if ((long long)p->height * n_frames > 65535ll * 8) return ctx->fail(JXLB200_E_ARG, "batch too tall");
    if (!qcoeff || !lf || !dct_select || !block_origin || !hf_mul || !x_from_y || !b_from_y || !out || (p->epf_iters > 0 && !sharpness))
        return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int W = p->width, H = p->height, wb = W >> 3;
    const size_t plane = (size_t)W * H * n_frames;
    CUDA_TRY(ctx, ctx->mid.ensure(sizeof(float) * 3 * plane));
    float *mid[3] = {ctx->mid.as<float>(), ctx->mid.as<float>() + plane, ctx->mid.as<float>() + 2 * plane};
    jxlb200_frame_params ps = *p;
    ps.height = H * n_frames;
    rc = invert_dev(ctx, &ps, qcoeff, lf, dct_select, block_origin, hf_mul, x_from_y, b_from_y, mid, W, true, H);
    if (rc) return rc;
    K2Params K;
    fill_k2(K, p, nullptr);
    if ((ctx->opt_stage2 == 0 || ctx->opt_stage2 == 3 || ctx->opt_stage2 == 5 || ctx->opt_stage2 == 6) && k2_exact_supported(K)) {   // one launch over the whole stack
        const float *m3[3] = {mid[0], mid[1], mid[2]};
        return restore_dev(ctx, p, nullptr, m3, W, hf_mul, sharpness, out, n_frames);
    }
    for (int f = 0; f < n_frames; f++) {
        const size_t po = (size_t)f * H * W, bo_ = (size_t)f * (H >> 3) * wb;
        const float *m3[3] = {mid[0] + po, mid[1] + po, mid[2] + po};
        float *o3[3] = {out[0] + po, out[1] + po, out[2] + po};
        rc = restore_dev(ctx, p, nullptr, m3, W, hf_mul + bo_, sharpness ? sharpness + bo_ : nullptr, o3);
        if (rc) return rc;
    }
    return 0;
}

// ---- one frame split by group rows over several GPUs (split_nccl.cuh) ----
#define NCCL_TRY(ctx, expr)                                                                          \
    do {                                                                                             \
        ncclResult_t r__ = (expr);                                                                   \
        if (r__ != ncclSuccess) {                                                                    \
            (ctx)->err = std::string(#expr ": ") + nccl_api().GetErrorString(r__);                   \
            return JXLB200_E_CUDA;                                                                   \
        }                                                                                            \
    } while (0)

int32_t jxlb200_comm_unique_id(uint8_t id[JXLB200_COMM_ID_BYTES]) {
    if (!id) return JXLB200_E_ARG;
    if (!nccl_api().ok) return JXLB200_E_UNSUPPORTED;
    static_assert(sizeof(ncclUniqueId) == JXLB200_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    ncclUniqueId u;
    if (nccl_api().GetUniqueId(&u) != ncclSuccess) return JXLB200_E_CUDA;
    memcpy(id, &u, sizeof(u));
    return 0;
}

int32_t jxlb200_comm_init(jxlb200_ctx *ctx, const uint8_t id[JXLB200_COMM_ID_BYTES], int32_t rank, int32_t world) {
    if (!ctx) return JXLB200_E_ARG;
    if (!id || world < 1 || rank < 0 || rank >= world) return ctx->fail(JXLB200_E_ARG, "bad communicator arguments");
    if (!nccl_api().ok) return ctx->fail(JXLB200_E_UNSUPPORTED, "libnccl.so.2 could not be loaded");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (ctx->comm) { nccl_api().CommDestroy(ctx->comm); ctx->comm = nullptr; }
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    NCCL_TRY(ctx, nccl_api().CommInitRank(&ctx->comm, world, u, rank));
    ctx->comm_rank = rank; ctx->comm_world = world;
    if (!ctx->comm_stream) {
        CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->comm_stream, cudaStreamNonBlocking));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_edge, cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_halo, cudaEventDisableTiming));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_maps, cudaEventDisableTiming));
    }
    return 0;
}

int32_t jxlb200_comm_destroy(jxlb200_ctx *ctx) {
    if (!ctx) return JXLB200_E_ARG;
    if (ctx->comm && nccl_api().ok) nccl_api().CommDestroy(ctx->comm);
    ctx->comm = nullptr; ctx->comm_world = 1; ctx->comm_rank = 0;
    return 0;
}

int32_t jxlb200_vardct_reconstruct_split_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const jxlb200_slab *slab,
    const int32_t *const qcoeff[3], const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, const int32_t *sharpness, float *const out[3]) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!slab || !qcoeff || !lf || !dct_select || !block_origin || !hf_mul || !x_from_y || !b_from_y || !sharpness || !out)
        return ctx->fail(JXLB200_E_ARG, "NULL pointer");
    if (is_subsampled(p)) return ctx->fail(JXLB200_E_UNSUPPORTED, "group-row split of chroma-subsampled frames");
    const int W = p->width, R = p->height, wb = W >> 3, tw = (W + 63) >> 6;
    if (slab->rows != R || (slab->y0 & 255) || slab->y0 + R > slab->frame_height || (R & 7))
        return ctx->fail(JXLB200_E_ARG, "slab must start on a group row, match p->height and stay inside the frame");
    const bool up = slab->has_top != 0, down = slab->has_bottom != 0;
    if ((up || down) && !ctx->comm) return ctx->fail(JXLB200_E_ARG, "jxlb200_comm_init has not been called");
    if ((up && ctx->comm_rank == 0) || (down && ctx->comm_rank == ctx->comm_world - 1))
        return ctx->fail(JXLB200_E_ARG, "slab has a neighbour where the communicator has no rank");
    if ((up || down) && R < 2 * JXLB200_HALO_ROWS) return ctx->fail(JXLB200_E_ARG, "slab shorter than its two halos");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int HR = JXLB200_HALO_ROWS;
    const size_t plane = (size_t)(R + 2 * HR) * W, mrows = (size_t)(R / 8 + 2) * wb;
    CUDA_TRY(ctx, ctx->split_xyb.ensure(sizeof(float) * 3 * plane));
    CUDA_TRY(ctx, ctx->split_maps.ensure(sizeof(int32_t) * 2 * mrows));
    float *xyb[3];
    for (int c = 0; c < 3; c++) xyb[c] = ctx->split_xyb.as<float>() + c * plane + (size_t)HR * W;     // row 0 of the slab
    int32_t *hm = ctx->split_maps.as<int32_t>() + wb, *sh = hm + mrows;                                 // block row 0 of the slab
    cudaStream_t main = ctx->stream, cs = ctx->comm_stream;
    NcclApi &N = nccl_api();

    // block maps with one neighbour block row each side (a frame edge keeps benign values there: nothing reads them)
    CUDA_TRY(ctx, cudaMemcpyAsync(hm, hf_mul, sizeof(int32_t) * (size_t)(R / 8) * wb, cudaMemcpyDeviceToDevice, main));
    CUDA_TRY(ctx, cudaMemcpyAsync(sh, sharpness, sizeof(int32_t) * (size_t)(R / 8) * wb, cudaMemcpyDeviceToDevice, main));
    if (!up) { CUDA_TRY(ctx, cudaMemsetAsync(hm - wb, 0, sizeof(int32_t) * wb, main)); CUDA_TRY(ctx, cudaMemsetAsync(sh - wb, 0, sizeof(int32_t) * wb, main)); }
    if (!down) { CUDA_TRY(ctx, cudaMemsetAsync(hm + (size_t)(R / 8) * wb, 0, sizeof(int32_t) * wb, main)); CUDA_TRY(ctx, cudaMemsetAsync(sh + (size_t)(R / 8) * wb, 0, sizeof(int32_t) * wb, main)); }

    auto stage1 = [&](int y0, int rows) -> int {           // group rows [y0, y0 + rows) of the slab
        if (rows <= 0) return 0;
        jxlb200_frame_params ps = *p;
        ps.height = rows;
        const size_t off = (size_t)y0 * W, bo_ = (size_t)(y0 / 8) * wb, to = (size_t)(y0 / 64) * tw;
        const int32_t *q3[3] = {qcoeff[0] + off, qcoeff[1] + off, qcoeff[2] + off};
        const float *l3[3] = {lf[0] + bo_, lf[1] + bo_, lf[2] + bo_};
        float *m3[3] = {xyb[0] + off, xyb[1] + off, xyb[2] + off};
        return invert_dev(ctx, &ps, q3, l3, dct_select + bo_, block_origin + bo_, hf_mul + bo_, x_from_y + to, b_from_y + to, m3, W);
    };
    auto stage2 = [&](int a, int b, bool top_nb, bool bottom_nb) -> int {      // rows [a, b) of the slab
        if (b <= a) return 0;
        jxlb200_frame_params ps = *p;
        ps.height = b - a;
        jxlb200_slab sl = {slab->y0 + a, b - a, slab->frame_height, top_nb ? 1 : 0, bottom_nb ? 1 : 0};
        const float *m3[3] = {xyb[0] + (size_t)a * W, xyb[1] + (size_t)a * W, xyb[2] + (size_t)a * W};
        float *o3[3] = {out[0] + (size_t)a * W, out[1] + (size_t)a * W, out[2] + (size_t)a * W};
        return restore_dev(ctx, &ps, &sl, m3, W, hm + (size_t)(a / 8) * wb, sh + (size_t)(a / 8) * wb, o3);
    };

    if (!up && !down) {                                     // a "split" over one rank
        if ((rc = stage1(0, R))) return rc;
        return stage2(0, R, false, false);
    }
    // 1. stage 1 of the whole slab in one go.  (Running the two boundary group rows first, so that the exchange could start earlier,
    // was measured and dropped: every extra stage-1 call costs ~0.3 ms of launch latency -- a dozen persistent launches --, more than
    // the 0.1 ms exchange it would hide; the exchange hides behind stage 2 of the interior rows anyway.  8 B200s, 16384^2: 3.23 -> see
    // profiles/r2_multigpu.md.)
    if ((rc = stage1(0, R))) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_edge, main));
    // 2. halo rows and the neighbours' block rows, one NCCL group on the comm stream
    CUDA_TRY(ctx, cudaStreamWaitEvent(cs, ctx->ev_edge, 0));
    NCCL_TRY(ctx, N.GroupStart());
    const size_t hn = (size_t)HR * W;
    for (int c = 0; c < 3; c++) {
        if (up) {
            NCCL_TRY(ctx, N.Send(xyb[c], hn, ncclFloat, ctx->comm_rank - 1, ctx->comm, cs));                          // my first rows
            NCCL_TRY(ctx, N.Recv(xyb[c] - hn, hn, ncclFloat, ctx->comm_rank - 1, ctx->comm, cs));                     // its last rows
        }
        if (down) {
            NCCL_TRY(ctx, N.Send(xyb[c] + (size_t)(R - HR) * W, hn, ncclFloat, ctx->comm_rank + 1, ctx->comm, cs));    // my last rows
            NCCL_TRY(ctx, N.Recv(xyb[c] + (size_t)R * W, hn, ncclFloat, ctx->comm_rank + 1, ctx->comm, cs));           // its first rows
        }
    }
    for (int32_t *m : {hm, sh}) {
        if (up) {
            NCCL_TRY(ctx, N.Send(m, wb, ncclInt32, ctx->comm_rank - 1, ctx->comm, cs));
            NCCL_TRY(ctx, N.Recv(m - wb, wb, ncclInt32, ctx->comm_rank - 1, ctx->comm, cs));
        }
        if (down) {
            NCCL_TRY(ctx, N.Send(m + (size_t)(R / 8 - 1) * wb, wb, ncclInt32, ctx->comm_rank + 1, ctx->comm, cs));
            NCCL_TRY(ctx, N.Recv(m + (size_t)(R / 8) * wb, wb, ncclInt32, ctx->comm_rank + 1, ctx->comm, cs));
        }
    }
    NCCL_TRY(ctx, N.GroupEnd());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_halo, cs));
    // 3. stage 2 of the rows that need no halo, beside the exchange
    const int a = up ? HR : 0, b = down ? R - HR : R;
    if ((rc = stage2(a, b, up, down))) return rc;
    // 4. the rows next to the neighbours
    CUDA_TRY(ctx, cudaStreamWaitEvent(main, ctx->ev_halo, 0));
    if (up && (rc = stage2(0, HR, true, true))) return rc;
    if (down && (rc = stage2(R - HR, R, true, true))) return rc;
    // the next call's stage 1 overwrites rows the comm stream may still be sending from only after this event
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_maps, main));
    CUDA_TRY(ctx, cudaStreamWaitEvent(cs, ctx->ev_maps, 0));
    return 0;
}

// host-buffer entry points ------------------------------------------------------------------------------------
// Whole path on host buffers.  Frames taller than one slab are pipelined by group rows over three streams: while slab i
// is uploaded (copy engine 1), stage 1 and stage 2 of slab i-1 run, and slab i-2's pixels go back (copy engine 2) -- PCIe
// is full duplex, so the call costs about max(upload, download, compute) instead of their sum.  Stage 2 needs HALO rows
// of stage-1 output below the rows it produces, so the stage-2 / download ranges are the upload slabs SHIFTED UP by
// JXLB200_HALO_ROWS: after stage 1 of slab i = rows [s_i, s_i+1), stage 2 runs on rows [s_i - 8, s_i+1 - 8) (from 0 for the
// first slab, to the frame's end for the last) -- everything it reads exists already, and no slab waits for the next
// one's upload.  The planes are contiguous on the device, so "halo rows" are simply the neighbouring rows (jxlb200_slab
// with has_top / has_bottom; the kernels only need a range to start on a block row).
// Slab schedule of the pipelined host entry point: the first two and the last two slabs are one group row (256) each so
// that the pipeline fills and drains quickly, the ones in between are JXLB200_PIPE_ROWS.
static void host_slab_schedule(int H, std::vector<int> &slab_start, int pipe_rows = 0);
#ifndef JXLB200_HOST_TWO_COMPUTE_STREAMS
#define JXLB200_HOST_TWO_COMPUTE_STREAMS 1   /* measured on B200, 8K frame, int32 / int16 coefficients: one compute stream 10.40 / 9.29 ms, two 10.31 / 9.21 ms (256-row slabs: 11.07 / 11.49 -> 10.53 / 10.39) */
#endif
#ifndef JXLB200_PIPE_ROWS_PACKED
#define JXLB200_PIPE_ROWS_PACKED 768   /* packed samples out: measured on B200, profiles/r2_host_entry_packed.md (512 / 768 / 1024 rows with the stage-1 fan-out: 5.70 / 5.53 / 5.64 ms) */
#endif
#ifndef JXLB200_PIPE_ROWS
#define JXLB200_PIPE_ROWS 512   /* measured on B200, 8K frame: 256 rows 12.0 ms, 512 rows 11.2 ms, 1024 rows 12.7 ms; again with the 2.9 ms kernels: 256 / 512 / 768 rows 11.4 / 11.2 / 11.7 ms; PCIe floor (398 MB each way, duplex) 8.4 ms */
#endif
static void host_slab_schedule(int H, std::vector<int> &slab_start, int pipe_rows) {
    const int G = (H + 255) / 256, per = (pipe_rows > 0 ? pipe_rows : JXLB200_PIPE_ROWS) / 256;     // group rows in the frame / per middle slab
    const int edge = G >= 4 + per ? 2 : (G >= 2 + per ? 1 : 0);        // single-group-row slabs at each end
    int g = 0;
    slab_start.clear();
    while (g < G) {
        slab_start.push_back(g * 256);
        const int left = G - g;
        int take = (g < edge || left <= edge) ? 1 : min(per, left - edge);
        if (take < 1) take = 1;
        g += take;
    }
}
// rows [a, b) that stage 2 produces (and the download returns) once stage 1 of slab i has run: the slab shifted up by the halo
static inline void host_stage2_range(const std::vector<int> &slab_start, int H, int i, int &a, int &b) {
    const int n = (int)slab_start.size();
    a = i > 0 ? slab_start[i] - JXLB200_HALO_ROWS : 0;
    b = i + 1 < n ? slab_start[i + 1] - JXLB200_HALO_ROWS : H;
}
int32_t jxlb200_host_stage2_ranges(int32_t height, int32_t *first_rows, int32_t *end_rows, int32_t capacity) {
    if (height <= 0 || (height & 7)) return JXLB200_E_ARG;
    std::vector<int> v;
    host_slab_schedule(height, v);
    for (int i = 0; i < (int)v.size() && first_rows && end_rows && i < capacity; i++) {
        int a, b;
        host_stage2_range(v, height, i, a, b);
        first_rows[i] = a; end_rows[i] = b;
    }
    return (int32_t)v.size();
}
// the schedule, for callers that want to overlap their own work with the slabs and for the CPU tests (no device needed)
int32_t jxlb200_host_slab_schedule(int32_t height, int32_t *starts, int32_t capacity) {
    if (height <= 0 || (height & 7)) return JXLB200_E_ARG;
    std::vector<int> v;
    host_slab_schedule(height, v);
    for (int i = 0; i < (int)v.size() && starts && i < capacity; i++) starts[i] = v[i];
    return (int32_t)v.size();
}
// int16 coefficients (jxlb200_vardct_reconstruct_i16) are widened on the device: 8 per thread, one 128-bit load, two
// 128-bit stores; the few elements of a plane that is not a multiple of 8 long go through the scalar tail.
__global__ void k9_widen_i16(const int16_t *__restrict__ in, int32_t *__restrict__ out, size_t n) {
    const size_t n8 = n >> 3, stride = (size_t)gridDim.x * blockDim.x, t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t i = t; i < n8; i += stride) {
        const int4 v = __ldg(reinterpret_cast<const int4 *>(in) + i);
        int4 lo, hi;
        lo.x = (int)(short)(v.x & 0xffff); lo.y = v.x >> 16; lo.z = (int)(short)(v.y & 0xffff); lo.w = v.y >> 16;
        hi.x = (int)(short)(v.z & 0xffff); hi.y = v.z >> 16; hi.z = (int)(short)(v.w & 0xffff); hi.w = v.w >> 16;
        reinterpret_cast<int4 *>(out)[2 * i] = lo;
        reinterpret_cast<int4 *>(out)[2 * i + 1] = hi;
    }
    for (size_t i = (n8 << 3) + t; i < n; i += stride) out[i] = in[i];
}
static void widen_i16(jxlb200_ctx *ctx, const int16_t *in, int32_t *out, size_t n, cudaStream_t st) {
    const size_t want = ((n >> 3) + 255) / 256 + 1;
    const int grid = (int)(want < (size_t)ctx->sms * 8 ? want : (size_t)ctx->sms * 8);
    k9_widen_i16<<<grid, 256, 0, st>>>(in, out, n);
    ctx->launches++;
}

// qbytes = 4: qcoeff planes are int32 (HFCoefficients.quantizedCoeffs as the reference holds them); 2: int16
// Packed output (jxlb200_vardct_reconstruct_packed): the colour planes leave the device as interleaved 8- or 16-bit samples
struct PackedOut {
    uint8_t *dst = nullptr;     // crop_h x crop_w x 3 samples
    int bits = 0, linear = 0, crop_w = 0, crop_h = 0;
};

static int reconstruct_host(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const void *const qcoeff[3], int qbytes,
    const float *const lf[3], const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, const int32_t *sharpness, float *const out[3], const PackedOut *pk = nullptr) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!qcoeff || !lf || !dct_select || !block_origin || !hf_mul || !x_from_y || !b_from_y || !sharpness || (!out && !pk))
        return ctx->fail(JXLB200_E_ARG, "NULL pointer");
    for (int c = 0; c < 3; c++)
        if (!qcoeff[c] || !lf[c] || (!pk && !out[c])) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    const size_t pk_row = pk ? (size_t)pk->crop_w * 3 * (pk->bits > 8 ? 2 : 1) : 0;
    const float *pk_thr = nullptr;
    if (pk) {
        CUDA_TRY(ctx, ctx->packed.ensure(pk_row * pk->crop_h + 64));
        // the sample pipeline as a threshold table (k8_features.cuh), one per (bits, linear), built on first use
        const int slot = (pk->bits > 8 ? 2 : 0) + (pk->linear ? 1 : 0);
        if (!ctx->pack_thr[slot].p) {
            std::vector<float> thr;
            pack_thresholds(pk->bits, pk->linear, thr);
            thr.resize((size_t)1 << pk->bits, INFINITY);        // the 16-bit search reads whole 256-entry segments
            CUDA_TRY(ctx, ctx->pack_thr[slot].ensure(sizeof(float) * thr.size()));
            CUDA_TRY(ctx, cudaMemcpy(ctx->pack_thr[slot].p, thr.data(), sizeof(float) * thr.size(), cudaMemcpyHostToDevice));
        }
        pk_thr = ctx->pack_thr[slot].as<float>();
    }
    // rows [a, b) of the device planes -> packed samples -> host, on stream st (enqueued after stage 2 of those rows)
    auto send_packed = [&](float *const dplanes[3], int a, int b, cudaStream_t kst, cudaStream_t cst, cudaEvent_t ev) -> int {
        b = b < pk->crop_h ? b : pk->crop_h;
        if (a >= b) return 0;
        const long long quads = (long long)(b - a) * ((pk->crop_w + 3) >> 2);
        const int grid = (int)(quads / 256 + 1 < (long long)ctx->sms * 8 ? quads / 256 + 1 : (long long)ctx->sms * 8);
        if (pk->bits == 8) k8_pack_rgb<8><<<grid, 256, 0, kst>>>(dplanes[0], dplanes[1], dplanes[2], p->width, a, b, pk->crop_w, pk_thr, ctx->packed.as<unsigned char>());
        else k8_pack_rgb<16><<<grid, 256, 0, kst>>>(dplanes[0], dplanes[1], dplanes[2], p->width, a, b, pk->crop_w, pk_thr, ctx->packed.as<unsigned char>());
        ctx->launches++;
        if (kst != cst) { cudaEventRecord(ev, kst); cudaStreamWaitEvent(cst, ev, 0); }
        cudaError_t e = cudaMemcpyAsync(pk->dst + pk_row * a, ctx->packed.as<unsigned char>() + pk_row * a, pk_row * (b - a), cudaMemcpyDeviceToHost, cst);
        return e == cudaSuccess ? 0 : ctx->fail(JXLB200_E_CUDA, "cudaMemcpyAsync (packed download)", e);
    };
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int W = p->width, H = p->height, wb = W >> 3, tw = (W + 63) >> 6;
    const size_t npx = (size_t)W * H, nb = npx / 64;
    const bool narrow = qbytes == 2;
    CUDA_TRY(ctx, ctx->in_q.ensure(3 * sizeof(int32_t) * npx));
    if (narrow) CUDA_TRY(ctx, ctx->in_q16.ensure(3 * sizeof(int16_t) * npx));
    CUDA_TRY(ctx, ctx->in_lf.ensure(3 * sizeof(float) * nb));
    CUDA_TRY(ctx, ctx->mid.ensure(3 * sizeof(float) * npx));
    CUDA_TRY(ctx, ctx->out_planes.ensure(3 * sizeof(float) * npx));
    int32_t *dq[3]; int16_t *dq16[3]; float *dlf[3], *mid[3], *dout[3];
    for (int c = 0; c < 3; c++) {
        dq[c] = ctx->in_q.as<int32_t>() + c * npx;
        dq16[c] = narrow ? ctx->in_q16.as<int16_t>() + c * npx : nullptr;
        dlf[c] = ctx->in_lf.as<float>() + c * nb;
        mid[c] = ctx->mid.as<float>() + c * npx;
        dout[c] = ctx->out_planes.as<float>() + c * npx;
    }
    if (is_subsampled(p)) {
        // chroma-subsampled frame: plain upload -> stage 1 per channel + upsampling -> stage 2 -> download
        const int32_t *q3[3]; const float *l3[3];
        for (int c = 0; c < 3; c++) {
            const size_t nc = (size_t)(W >> p->shift_x[c]) * (H >> p->shift_y[c]);
            if (narrow) {
                CUDA_TRY(ctx, cudaMemcpyAsync(dq16[c], qcoeff[c], sizeof(int16_t) * nc, cudaMemcpyHostToDevice, ctx->stream));
                widen_i16(ctx, dq16[c], dq[c], nc, ctx->stream);
            } else {
                CUDA_TRY(ctx, cudaMemcpyAsync(dq[c], qcoeff[c], sizeof(int32_t) * nc, cudaMemcpyHostToDevice, ctx->stream));
            }
            CUDA_TRY(ctx, cudaMemcpyAsync(dlf[c], lf[c], sizeof(float) * (nc / 64), cudaMemcpyHostToDevice, ctx->stream));
            q3[c] = dq[c]; l3[c] = dlf[c];
        }
        HostMaps M;
        if ((rc = upload_maps(ctx, p, dct_select, block_origin, hf_mul, x_from_y, b_from_y, sharpness, M))) return rc;
        if ((rc = invert_subsampled_dev(ctx, p, q3, l3, M.ds, M.hf, mid))) return rc;
        if ((rc = restore_dev(ctx, p, nullptr, mid, W, M.hf, M.sharp, dout))) return rc;
        if (pk) {
            if ((rc = send_packed(dout, 0, H, ctx->stream, ctx->stream, nullptr))) return rc;
            CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            return check_flags(ctx);
        }
        Staged r[3];
        for (int c = 0; c < 3; c++) r[c] = {&ctx->out_planes, nullptr, out[c], sizeof(float) * npx, dout[c]};
        return stage_out(ctx, r, 3);
    }
    // stage 2 of one slab and stage 1 of the next touch disjoint rows and disjoint context buffers, so they run on two
    // streams: on slab-sized pieces stage 1 is a chain of short latency-bound launches, which hide under the issue-bound k2
    cudaStream_t comp = ctx->stream, up = ctx->h2d_stream, down = ctx->d2h_stream;
    cudaStream_t comp2 = JXLB200_HOST_TWO_COMPUTE_STREAMS ? ctx->k1_stream[0] : comp;
    HostMaps M;
    {   // the small per-block maps go first, on the upload stream
        cudaStream_t keep = ctx->stream;
        ctx->stream = up;
        rc = upload_maps(ctx, p, dct_select, block_origin, hf_mul, x_from_y, b_from_y, sharpness, M);
        ctx->stream = keep;
        if (rc) return rc;
        for (int c = 0; c < 3; c++)      // the LF planes are 1/64 of the coefficients: whole, up front
            CUDA_TRY(ctx, cudaMemcpyAsync(dlf[c], lf[c], sizeof(float) * nb, cudaMemcpyHostToDevice, up));
    }
    // Slab height.  Every slab costs stage 1 about 0.6 ms of launch latency whatever its size (a dozen persistent launches in a row:
    // JXLB200_TIMELINE shows it), so 11 slabs of 512 rows make stage 1, not the bus, the limit of an 8K call as soon as the download is
    // small.  With float32 planes going back (12 B/px down) the bus is the limit and short slabs keep it busy; with packed samples
    // (3 or 6 B/px down) taller slabs win.
    const int pipe_rows = ctx->opt_pipe_rows > 0 ? ctx->opt_pipe_rows : (pk ? JXLB200_PIPE_ROWS_PACKED : JXLB200_PIPE_ROWS);
    std::vector<int> slab_start;
    host_slab_schedule(H, slab_start, pipe_rows);
    const int nslab = (int)slab_start.size();
    // stage 1 of a slab on six streams: a win whenever the bus is not the limit (int16 coefficients in or packed samples out: 9.19 ->
    // 8.75 ms and 7.58 -> 5.70 ms per 8K frame), a small loss when it is (int32 in, float32 out: 10.28 -> 10.69 ms)
    const bool s1_fanout = ctx->opt_pipe_fanout >= 0 ? ctx->opt_pipe_fanout != 0 : (narrow || pk != nullptr);
    // JXLB200_TIMELINE=1: per-slab event times of this call on stderr (upload done | stage 1 done | stage 2 done | download done)
    static const bool timeline = getenv("JXLB200_TIMELINE") != nullptr;
    const unsigned evflag = timeline ? cudaEventDefault : cudaEventDisableTiming;
    std::vector<cudaEvent_t> ev_up(nslab), ev_k2(nslab), ev_k1(nslab), ev_dn(timeline ? nslab : 0);
    cudaEvent_t ev_t0 = nullptr;
    for (int i = 0; i < nslab; i++) {
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev_up[i], evflag));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev_k2[i], evflag));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev_k1[i], evflag));
        if (timeline) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev_dn[i], evflag));
    }
    if (timeline) { CUDA_TRY(ctx, cudaEventCreate(&ev_t0)); cudaEventRecord(ev_t0, up); }
    rc = 0;
    for (int i = 0; i < nslab && !rc; i++) {
        const int y0 = slab_start[i], y1 = i + 1 < nslab ? slab_start[i + 1] : H, rows = y1 - y0;
        const size_t off = (size_t)y0 * W, cnt = (size_t)rows * W;
        for (int c = 0; c < 3 && !rc; c++) {
            cudaError_t e = narrow
                ? cudaMemcpyAsync(dq16[c] + off, (const int16_t *)qcoeff[c] + off, sizeof(int16_t) * cnt, cudaMemcpyHostToDevice, up)
                : cudaMemcpyAsync(dq[c] + off, (const int32_t *)qcoeff[c] + off, sizeof(int32_t) * cnt, cudaMemcpyHostToDevice, up);
            if (e != cudaSuccess) rc = ctx->fail(JXLB200_E_CUDA, "cudaMemcpyAsync (upload)", e);
        }
        if (rc) break;
        cudaEventRecord(ev_up[i], up);
        cudaStreamWaitEvent(comp, ev_up[i], 0);
        if (narrow)
            for (int c = 0; c < 3; c++) widen_i16(ctx, dq16[c] + off, dq[c] + off, cnt, comp);
        {   // stage 1 of slab i: a frame of `rows` rows whose planes start at row y0
            jxlb200_frame_params ps = *p;
            ps.height = rows;
            const int32_t *q3[3] = {dq[0] + off, dq[1] + off, dq[2] + off};
            const float *l3[3] = {dlf[0] + (size_t)(y0 / 8) * wb, dlf[1] + (size_t)(y0 / 8) * wb, dlf[2] + (size_t)(y0 / 8) * wb};
            float *m3[3] = {mid[0] + off, mid[1] + off, mid[2] + off};
            rc = invert_dev(ctx, &ps, q3, l3, M.ds + (size_t)(y0 / 8) * wb, M.bo + (size_t)(y0 / 8) * wb, M.hf + (size_t)(y0 / 8) * wb,
                            M.xfy + (size_t)(y0 / 64) * tw, M.bfy + (size_t)(y0 / 64) * tw, m3, W, s1_fanout);
            if (rc) break;
        }
        {   // stage 2 of the rows whose lower halo now exists: the slab shifted up by HALO rows
            int a, b;
            host_stage2_range(slab_start, H, i, a, b);
            const int r2 = b - a;
            const size_t o2 = (size_t)a * W;
            jxlb200_frame_params ps = *p;
            ps.height = r2;
            jxlb200_slab sl = {a, r2, H, a > 0 ? 1 : 0, b < H ? 1 : 0};
            const float *m3[3] = {mid[0] + o2, mid[1] + o2, mid[2] + o2};
            float *o3[3] = {dout[0] + o2, dout[1] + o2, dout[2] + o2};
            if (comp2 != comp || timeline) {
                cudaEventRecord(ev_k1[i], comp);
                if (comp2 != comp) cudaStreamWaitEvent(comp2, ev_k1[i], 0);
            }
            ctx->stream = comp2;
            rc = restore_dev(ctx, &ps, nslab > 1 ? &sl : nullptr, m3, W, M.hf + (size_t)(a / 8) * wb, M.sharp + (size_t)(a / 8) * wb, o3);
            ctx->stream = comp;
            if (rc) break;
            if (pk) {       // sRGB + quantise + interleave on the compute stream, then a quarter (or half) of the bytes go back
                rc = send_packed(dout, a, b, comp2, down, ev_k2[i]);
                if (rc) break;
                if (timeline) cudaEventRecord(ev_dn[i], down);
                continue;
            }
            cudaEventRecord(ev_k2[i], comp2);
            cudaStreamWaitEvent(down, ev_k2[i], 0);
            for (int c = 0; c < 3 && !rc; c++) {
                cudaError_t e = cudaMemcpyAsync(out[c] + o2, o3[c], sizeof(float) * (size_t)r2 * W, cudaMemcpyDeviceToHost, down);
                if (e != cudaSuccess) rc = ctx->fail(JXLB200_E_CUDA, "cudaMemcpyAsync (download)", e);
            }
            if (timeline) cudaEventRecord(ev_dn[i], down);
        }
    }
    cudaError_t e1 = cudaStreamSynchronize(up), e2 = cudaStreamSynchronize(comp), e3 = cudaStreamSynchronize(down);
    if (comp2 != comp && e2 == cudaSuccess) e2 = cudaStreamSynchronize(comp2);
    if (timeline && !rc && e1 == cudaSuccess && e2 == cudaSuccess && e3 == cudaSuccess) {
        fprintf(stderr, "[jxlb200 timeline] %d slabs, %s coefficients, %s out (ms since the call's first upload)\n", nslab, narrow ? "int16" : "int32", pk ? "packed" : "float32");
        for (int i = 0; i < nslab; i++) {
            float a = 0, b = 0, c = 0, d = 0;
            cudaEventElapsedTime(&a, ev_t0, ev_up[i]); cudaEventElapsedTime(&b, ev_t0, ev_k1[i]);
            cudaEventElapsedTime(&c, ev_t0, ev_k2[i]); cudaEventElapsedTime(&d, ev_t0, ev_dn[i]);
            fprintf(stderr, "[jxlb200 timeline] slab %2d rows %4d..%4d: uploaded %.3f  stage1 %.3f  stage2 %.3f  downloaded %.3f\n", i, slab_start[i],
                    i + 1 < nslab ? slab_start[i + 1] : H, a, b, c, d);
        }
    }
    if (timeline) { for (cudaEvent_t e : ev_dn) cudaEventDestroy(e); if (ev_t0) cudaEventDestroy(ev_t0); }
    for (int i = 0; i < nslab; i++) { cudaEventDestroy(ev_up[i]); cudaEventDestroy(ev_k2[i]); cudaEventDestroy(ev_k1[i]); }
    if (rc) return rc;
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)
        return ctx->fail(JXLB200_E_CUDA, "stream synchronize", e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3));
    return check_flags(ctx);
}

int32_t jxlb200_vardct_reconstruct(jxlb200_ctx *ctx, const jxlb200_frame_params *p,
    const int32_t *const qcoeff[3], const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, const int32_t *sharpness, float *const out[3]) {
    return reconstruct_host(ctx, p, (const void *const *)qcoeff, 4, lf, dct_select, block_origin, hf_mul, x_from_y, b_from_y, sharpness, out);
}

int32_t jxlb200_vardct_reconstruct_i16(jxlb200_ctx *ctx, const jxlb200_frame_params *p,
    const int16_t *const qcoeff[3], const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, const int32_t *sharpness, float *const out[3]) {
    return reconstruct_host(ctx, p, (const void *const *)qcoeff, 2, lf, dct_select, block_origin, hf_mul, x_from_y, b_from_y, sharpness, out);
}

int32_t jxlb200_vardct_reconstruct_packed(jxlb200_ctx *ctx, const jxlb200_frame_params *p,
    const void *const qcoeff[3], int32_t coeff_bytes, const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, const int32_t *sharpness,
    int32_t bits, int32_t linear, int32_t crop_width, int32_t crop_height, uint8_t *out) {
    if (!ctx) return JXLB200_E_ARG;
    if (coeff_bytes != 2 && coeff_bytes != 4) return ctx->fail(JXLB200_E_ARG, "coeff_bytes must be 4 (int32) or 2 (int16)");
    if (bits != 8 && bits != 16) return ctx->fail(JXLB200_E_ARG, "PNG only supports 8 and 16 (PNGWriter.java:57-58)");
    if (!p || !out || crop_width < 1 || crop_height < 1 || crop_width > p->width || crop_height > p->height)
        return ctx->fail(JXLB200_E_ARG, "crop size must lie inside the padded frame");
    PackedOut pk;
    pk.dst = out; pk.bits = bits; pk.linear = linear ? 1 : 0; pk.crop_w = crop_width; pk.crop_h = crop_height;
    return reconstruct_host(ctx, p, qcoeff, coeff_bytes, lf, dct_select, block_origin, hf_mul, x_from_y, b_from_y, sharpness, nullptr, &pk);
}

int32_t jxlb200_vardct_invert(jxlb200_ctx *ctx, const jxlb200_frame_params *p,
    const int32_t *const qcoeff[3], const float *const lf[3],
    const uint8_t *dct_select, const uint8_t *block_origin, const int32_t *hf_mul,
    const int32_t *x_from_y, const int32_t *b_from_y, float *const xyb[3]) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!qcoeff || !lf || !dct_select || !block_origin || !hf_mul || !x_from_y || !b_from_y || !xyb)
        return ctx->fail(JXLB200_E_ARG, "NULL pointer");
    const size_t npx = (size_t)p->width * p->height, nb = npx / 64;
    Staged r[9];
    stage_planes(r, ctx->in_q, qcoeff, ctx->out_planes, xyb, sizeof(float) * npx);
    for (int c = 0; c < 3; c++) r[6 + c] = {&ctx->in_lf, lf[c], nullptr, sizeof(float) * nb};
    if ((rc = stage_in(ctx, r, 9))) return rc;
    HostMaps M;
    if ((rc = upload_maps(ctx, p, dct_select, block_origin, hf_mul, x_from_y, b_from_y, nullptr, M))) return rc;
    if ((rc = invert_dev(ctx, p, planes_of<const int32_t>(r).data(), planes_of<const float>(r + 6).data(), M.ds, M.bo, M.hf, M.xfy, M.bfy,
                         planes_of<float>(r + 3).data(), p->width)))
        return rc;
    return stage_out(ctx, r, 9);
}

// one restoration stage on device planes: mode 0 Gaborish only, 1 EPF only, 2 colour only (what the host form and the _dev form share)
static int stage_enqueue(jxlb200_ctx *ctx, const jxlb200_frame_params *p, int mode, const float *const din[3],
                         const int32_t *hf_mul, const int32_t *sharp, float *const dout[3]) {
    jxlb200_frame_params q = *p;
    q.gab = mode == 0 ? 1 : 0;
    q.epf_iters = mode == 1 ? p->epf_iters : 0;
    q.color_mode = mode == 2 ? p->color_mode : 0;
    return restore_dev(ctx, &q, nullptr, din, p->width, hf_mul, sharp, dout);
}

// frame params and three input and three output planes (the restoration stages)
static int check_planes(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float *const in[3], float *const out[3]) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!in || !out) return ctx->fail(JXLB200_E_ARG, "NULL pointer");
    for (int c = 0; c < 3; c++)
        if (!in[c] || !out[c]) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    return 0;
}

// one restoration stage on host planes: stage in, stage_enqueue, stage out
static int host_stage(jxlb200_ctx *ctx, const jxlb200_frame_params *p, int mode, const float *const in[3],
                      const int32_t *hf_mul, const int32_t *sharp, float *const out[3]) {
    int rc = check_planes(ctx, p, in, out);
    if (rc) return rc;
    if (mode == 1 && (!hf_mul || !sharp)) return ctx->fail(JXLB200_E_ARG, "EPF needs hf_mul and sharpness");
    Staged r[6];
    stage_planes(r, ctx->in_q, in, ctx->out_planes, out, sizeof(float) * p->width * p->height);
    if ((rc = stage_in(ctx, r, 6))) return rc;
    HostMaps M{};
    if (mode == 1 && (rc = upload_maps(ctx, p, nullptr, nullptr, hf_mul, nullptr, nullptr, sharp, M))) return rc;
    if ((rc = stage_enqueue(ctx, p, mode, planes_of<const float>(r).data(), M.hf, M.sharp, planes_of<float>(r + 3).data()))) return rc;
    return stage_out(ctx, r, 6);
}

// Gaborish + EPF of a Modular-encoded frame (Frame.decodeFrame :457-461 with header.encoding == MODULAR): one sigma for the frame
static int check_uniform(jxlb200_ctx *ctx, const jxlb200_frame_params *p, float epf_sigma_for_modular, const float *const in[3],
                         float *const out[3]) {
    if (!ctx) return JXLB200_E_ARG;
    if (!p || !in || !out) return ctx->fail(JXLB200_E_ARG, "NULL pointer");
    for (int c = 0; c < 3; c++)
        if (!in[c] || !out[c]) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    // a Modular frame has its own size, not a multiple of 8; sizes the tile kernel does not take go through the staged kernels
    if (p->width <= 0 || p->height <= 0 || p->width > 65535 * 8 || p->height > 65535 * 8) return ctx->fail(JXLB200_E_ARG, "bad frame size");
    if ((p->gab || p->epf_iters) && (p->width < 4 || p->height < 4))
        return ctx->fail(JXLB200_E_UNSUPPORTED, "filters on a frame narrower than 4 pixels (mirrorCoordinate reflects more than once)");
    if (p->epf_iters < 0 || p->epf_iters > 3) return ctx->fail(JXLB200_E_ARG, "epf_iters outside 0..3");
    if (!(epf_sigma_for_modular == epf_sigma_for_modular)) return ctx->fail(JXLB200_E_ARG, "sigma is NaN");
    return 0;
}

static int restore_uniform_enqueue(jxlb200_ctx *ctx, const jxlb200_frame_params *p, float epf_sigma_for_modular,
                                   const float *const din[3], float *const dout[3]) {
    const size_t npx = (size_t)p->width * p->height;
    if (!p->gab && p->epf_iters == 0 && p->color_mode == 0) {
        for (int c = 0; c < 3; c++) CUDA_TRY(ctx, cudaMemcpyAsync(dout[c], din[c], sizeof(float) * npx, cudaMemcpyDeviceToDevice, ctx->stream));
        return 0;
    }
    ctx->uniform_sigma = true;
    ctx->uniform_inv_sigma = 1.0f / epf_sigma_for_modular;        // Frame.java:574
    // hf_mul / sharpness are not read in this mode; any non-NULL pointers satisfy the argument checks below
    const int rc = restore_dev(ctx, p, nullptr, din, p->width, (const int32_t *)din[0], (const int32_t *)din[0], dout);
    ctx->uniform_sigma = false;
    return rc;
}

int32_t jxlb200_restore_uniform(jxlb200_ctx *ctx, const jxlb200_frame_params *p, float epf_sigma_for_modular,
    const float *const in[3], float *const out[3]) {
    int rc = check_uniform(ctx, p, epf_sigma_for_modular, in, out);
    if (rc) return rc;
    Staged r[6];
    stage_planes(r, ctx->in_q, in, ctx->out_planes, out, sizeof(float) * p->width * p->height);
    if ((rc = stage_in(ctx, r, 6))) return rc;
    if ((rc = restore_uniform_enqueue(ctx, p, epf_sigma_for_modular, planes_of<const float>(r).data(), planes_of<float>(r + 3).data()))) return rc;
    return stage_out(ctx, r, 6);
}

int32_t jxlb200_restore_uniform_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, float epf_sigma_for_modular,
    const float *const in[3], float *const out[3]) {
    int rc = check_uniform(ctx, p, epf_sigma_for_modular, in, out);
    if (rc) return rc;
    for (int c = 0; c < 3; c++)
        for (int d = 0; d < 3; d++)
            if (in[c] == out[d]) return ctx->fail(JXLB200_E_ARG, "in-place restore is not allowed");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return restore_uniform_enqueue(ctx, p, epf_sigma_for_modular, in, out);
}

int32_t jxlb200_gaborish(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float *const in[3], float *const out[3]) {
    return host_stage(ctx, p, 0, in, nullptr, nullptr, out);
}
int32_t jxlb200_epf(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float *const in[3], const int32_t *hf_mul,
                    const int32_t *sharpness, float *const out[3]) {
    return host_stage(ctx, p, 1, in, hf_mul, sharpness, out);
}
int32_t jxlb200_color_transform(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float *const in[3], float *const out[3]) {
    return host_stage(ctx, p, 2, in, nullptr, nullptr, out);
}
int32_t jxlb200_color_transform_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float *const in[3], float *const out[3]) {
    int rc = check_planes(ctx, p, in, out);
    if (rc) return rc;
    for (int c = 0; c < 3; c++)
        for (int d = 0; d < 3; d++)
            if (in[c] == out[d]) return ctx->fail(JXLB200_E_ARG, "in-place colour transform is not allowed");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return stage_enqueue(ctx, p, 2, in, nullptr, nullptr, out);
}

// ---- Modular: each host form stages its arrays around the _dev form ----
static int rct_check(jxlb200_ctx *ctx, int32_t *const ch[3], int32_t h, int32_t w, int32_t rct_type) {
    if (!ctx) return JXLB200_E_ARG;
    if (!ch || !ch[0] || !ch[1] || !ch[2] || h < 0 || w < 0) return ctx->fail(JXLB200_E_ARG, "bad RCT arguments");
    if (rct_type < 0 || rct_type >= 42) return ctx->fail(JXLB200_E_ARG, "rct_type outside 0..41");
    return 0;
}

static int squeeze_check(jxlb200_ctx *ctx, const int32_t *avg, const int32_t *res, int32_t h_avg, int32_t w_avg, int32_t h_res,
                         int32_t w_res, int32_t horizontal, const int32_t *out) {
    if (!ctx) return JXLB200_E_ARG;
    if (!avg || !out || h_avg < 0 || w_avg < 0 || h_res < 0 || w_res < 0) return ctx->fail(JXLB200_E_ARG, "bad squeeze arguments");
    if (horizontal) {
        if ((w_avg != w_res && w_avg != 1 + w_res) || h_res != h_avg) return ctx->fail(JXLB200_E_ARG, "Corrupted squeeze transform");
    } else {
        if ((h_avg != h_res && h_avg != 1 + h_res) || w_res != w_avg) return ctx->fail(JXLB200_E_ARG, "Corrupted squeeze transform");
    }
    if (!res && h_res > 0 && w_res > 0) return ctx->fail(JXLB200_E_ARG, "bad squeeze arguments");
    return 0;
}

static int palette_check(jxlb200_ctx *ctx, const int32_t *idx, const int32_t *palette, int32_t h, int32_t w, int32_t num_c,
                         int32_t nb_colors, int32_t d_pred, int32_t *const out[]) {
    if (!ctx) return JXLB200_E_ARG;
    if (!idx || !out || h < 0 || w < 0 || num_c < 1 || nb_colors < 0 || (nb_colors > 0 && !palette))
        return ctx->fail(JXLB200_E_ARG, "bad palette arguments");
    if (d_pred < 0 || d_pred > 13) return ctx->fail(JXLB200_E_ARG, "d_pred outside 0..13");
    if (d_pred == 6) return ctx->fail(JXLB200_E_UNSUPPORTED, "palette delta with the weighted predictor (reference dereferences null pred[][])");
    for (int c = 0; c < num_c; c++)
        if (!out[c]) return ctx->fail(JXLB200_E_ARG, "NULL palette output channel");
    return 0;
}

int32_t jxlb200_modular_rct_dev(jxlb200_ctx *ctx, int32_t *const ch[3], int32_t h, int32_t w, int32_t rct_type) {
    int rc = rct_check(ctx, ch, h, w, rct_type);
    if (rc || h == 0 || w == 0) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const long long n = (long long)h * w;
    const int grid = (int)min((long long)ctx->sms * 8, (n + 255) / 256);
    k3_rct<<<grid, 256, 0, ctx->stream>>>(ch[0], ch[1], ch[2], n, rct_type % 7, rct_type / 7);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int32_t jxlb200_modular_squeeze_dev(jxlb200_ctx *ctx, const int32_t *avg, const int32_t *res, int32_t h_avg, int32_t w_avg,
    int32_t h_res, int32_t w_res, int32_t horizontal, int32_t *out) {
    int rc = squeeze_check(ctx, avg, res, h_avg, w_avg, h_res, w_res, horizontal, out);
    if (rc || h_avg == 0 || w_avg == 0) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (horizontal) k5_squeeze_h<<<ceil_div(h_avg, 32), 32, 0, ctx->stream>>>(avg, res, h_avg, w_avg, w_res, out);
    else k5_squeeze_v<<<ceil_div(w_avg, 128), 128, 0, ctx->stream>>>(avg, res, h_avg, h_res, w_avg, out);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int32_t jxlb200_modular_palette_dev(jxlb200_ctx *ctx, const int32_t *idx, const int32_t *palette, int32_t h, int32_t w,
    int32_t num_c, int32_t nb_colors, int32_t nb_deltas, int32_t d_pred, int32_t bit_depth, int32_t *const out[]) {
    int rc = palette_check(ctx, idx, palette, h, w, num_c, nb_colors, d_pred, out);
    if (rc || h == 0 || w == 0) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, ensure_flags(ctx, ctx->stream));
    int *any = ctx->flags.as<int>() + 1;
    PalArgs A{idx, palette, h, w, num_c, nb_colors, nb_deltas, d_pred, bit_depth};
    const long long n = (long long)h * w;
    const int grid = (int)min((long long)ctx->sms * 8, (n + 255) / 256);
    CUDA_TRY(ctx, cudaMemsetAsync(any, 0, sizeof(int), ctx->stream));
    for (int c = 0; c < num_c; c++) {
        k4_palette_gather<<<grid, 256, 0, ctx->stream>>>(A, c, out[c], any);
        ctx->launches++;
    }
    if (d_pred != 0)   // predictor 0 adds 0 to every delta pixel
        for (int c = 0; c < num_c; c++) {
            k4_palette_delta<<<1, 1024, 0, ctx->stream>>>(A, out[c], any);
            ctx->launches++;
        }
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int32_t jxlb200_modular_rct(jxlb200_ctx *ctx, int32_t *const ch[3], int32_t h, int32_t w, int32_t rct_type) {
    int rc = rct_check(ctx, ch, h, w, rct_type);
    if (rc || h == 0 || w == 0) return rc;
    Staged r[3];
    for (int c = 0; c < 3; c++) r[c] = {&ctx->mod, ch[c], ch[c], sizeof(int32_t) * h * w};
    if ((rc = stage_in(ctx, r, 3))) return rc;
    if ((rc = jxlb200_modular_rct_dev(ctx, planes_of<int32_t>(r).data(), h, w, rct_type))) return rc;
    return stage_out(ctx, r, 3);
}

int32_t jxlb200_modular_squeeze(jxlb200_ctx *ctx, const int32_t *avg, const int32_t *res, int32_t h_avg, int32_t w_avg,
    int32_t h_res, int32_t w_res, int32_t horizontal, int32_t *out) {
    int rc = squeeze_check(ctx, avg, res, h_avg, w_avg, h_res, w_res, horizontal, out);
    if (rc || h_avg == 0 || w_avg == 0) return rc;
    const size_t na = (size_t)h_avg * w_avg, nr = (size_t)h_res * w_res;
    Staged r[3] = {{&ctx->mod, avg, nullptr, sizeof(int32_t) * na}, {&ctx->mod, res, nullptr, sizeof(int32_t) * nr},
                   {&ctx->mod, nullptr, out, sizeof(int32_t) * (na + nr)}};
    if ((rc = stage_in(ctx, r, 3))) return rc;
    if ((rc = jxlb200_modular_squeeze_dev(ctx, (const int32_t *)r[0].dev, (const int32_t *)r[1].dev, h_avg, w_avg, h_res, w_res,
                                          horizontal, (int32_t *)r[2].dev)))
        return rc;
    return stage_out(ctx, r, 3);
}

int32_t jxlb200_modular_palette(jxlb200_ctx *ctx, const int32_t *idx, const int32_t *palette, int32_t h, int32_t w,
    int32_t num_c, int32_t nb_colors, int32_t nb_deltas, int32_t d_pred, int32_t bit_depth, int32_t *const out[]) {
    if (ctx && num_c > 4096) return ctx->fail(JXLB200_E_ARG, "bad palette arguments");   // before palette_check reads out[0 .. num_c)
    int rc = palette_check(ctx, idx, palette, h, w, num_c, nb_colors, d_pred, out);
    if (rc || h == 0 || w == 0) return rc;
    const size_t n = (size_t)h * w;
    std::vector<Staged> r(2 + num_c);
    r[0] = {&ctx->mod, idx, nullptr, sizeof(int32_t) * n};
    r[1] = {&ctx->mod, palette, nullptr, sizeof(int32_t) * num_c * nb_colors};
    for (int c = 0; c < num_c; c++) r[2 + c] = {&ctx->mod, nullptr, out[c], sizeof(int32_t) * n};
    if ((rc = stage_in(ctx, r.data(), 2 + num_c))) return rc;
    std::vector<int32_t *> dout(num_c);
    for (int c = 0; c < num_c; c++) dout[c] = (int32_t *)r[2 + c].dev;
    if ((rc = jxlb200_modular_palette_dev(ctx, (const int32_t *)r[0].dev, (const int32_t *)r[1].dev, h, w, num_c, nb_colors, nb_deltas,
                                          d_pred, bit_depth, dout.data())))
        return rc;
    return stage_out(ctx, r.data(), 2 + num_c);
}


// ---- frame / patch blending on host rectangles (k7_blend.cuh) ----
int32_t jxlb200_blend(jxlb200_ctx *ctx, const jxlb200_blend_op *op, int32_t h, int32_t w,
    void *canvas, int64_t canvas_pitch, const void *frame, int64_t frame_pitch, const void *ref, int64_t ref_pitch,
    const float *frame_alpha, int64_t frame_alpha_pitch, const float *ref_alpha, int64_t ref_alpha_pitch) {
    if (!ctx) return JXLB200_E_ARG;
    if (!op || !canvas || !frame || !ref || h < 0 || w < 0) return ctx->fail(JXLB200_E_ARG, "NULL pointer or negative size");
    if (op->mode < 1 || op->mode > 4) return ctx->fail(JXLB200_E_STREAM, "Illegal blend mode");
    if (h == 0 || w == 0) return 0;
    int mode = op->mode;
    if ((mode == 2 || mode == 3) && !op->has_extra) mode = 1;
    if (op->is_int && mode != 1) return ctx->fail(JXLB200_E_ARG, "integer samples only blend with ADD (the reference casts to float first)");
    const bool need_fa = (mode == 2 && !op->is_alpha) || mode == 3, need_ra = mode == 2 && !op->is_alpha;
    if ((need_fa && !frame_alpha) || (need_ra && !ref_alpha)) return ctx->fail(JXLB200_E_ARG, "alpha plane missing");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)h * w, row = sizeof(float) * (size_t)w;
    CUDA_TRY(ctx, ctx->blend.ensure(5 * sizeof(float) * n));
    char *base = (char *)ctx->blend.p;
    cudaStream_t st = ctx->stream;
    BlendArgs A;
    A.mode = op->mode; A.is_int = op->is_int; A.is_alpha = op->is_alpha; A.has_extra = op->has_extra; A.clamp = op->clamp; A.premult = op->premult;
    A.h = h; A.w = w;
    A.pa = A.pb = A.pfa = A.pra = A.pout = 0;
    A.a = base; A.b = base + sizeof(float) * n; A.fa = (const float *)(base + 2 * sizeof(float) * n);
    A.ra = (const float *)(base + 3 * sizeof(float) * n); A.out = base + 4 * sizeof(float) * n;
    CUDA_TRY(ctx, cudaMemcpy2DAsync((void *)A.a, row, frame, sizeof(float) * frame_pitch, row, h, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpy2DAsync((void *)A.b, row, ref, sizeof(float) * ref_pitch, row, h, cudaMemcpyHostToDevice, st));
    if (need_fa) CUDA_TRY(ctx, cudaMemcpy2DAsync((void *)A.fa, row, frame_alpha, sizeof(float) * frame_alpha_pitch, row, h, cudaMemcpyHostToDevice, st));
    if (need_ra) CUDA_TRY(ctx, cudaMemcpy2DAsync((void *)A.ra, row, ref_alpha, sizeof(float) * ref_alpha_pitch, row, h, cudaMemcpyHostToDevice, st));
    k7_blend<<<min(ctx->sms * 8, ceil_div((int)std::min<size_t>(n, 1u << 30), 256)), 256, 0, st>>>(A);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpy2DAsync(canvas, sizeof(float) * canvas_pitch, A.out, row, row, h, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    return 0;
}


// ---- a frame's whole compositing in one call (SURVEY.md 8f-3): the planes involved go to the device ONCE (only the rows any
// rectangle touches), every rectangle of every channel is blended there in the order given -- later items see what earlier ones
// wrote, as blendFrame / computePatches do (J/JXLCodestreamDecoder.java:212-254, 415-537) -- and the written planes come back once.
// patches-lossless.jxl: ~2000 rectangles, two PCIe round trips instead of ~8000. ----
// Checks the items against the planes and records the rows [lo, hi) of each plane that some rectangle touches.
static int blend_items_check(jxlb200_ctx *ctx, int32_t n_planes, void *const planes[], const int32_t plane_h[], const int32_t plane_w[],
    const int32_t writable[], int32_t n_items, const jxlb200_blend_item *items, std::vector<int> &lo, std::vector<int> &hi) {
    lo.assign(n_planes, 1 << 30);
    hi.assign(n_planes, -1);
    for (int k = 0; k < n_items; k++) {
        const jxlb200_blend_item &it = items[k];
        if (it.op.mode < 1 || it.op.mode > 4) return ctx->fail(JXLB200_E_STREAM, "Illegal blend mode");
        if (it.h < 1 || it.w < 1) return ctx->fail(JXLB200_E_ARG, "empty blend rectangle");
        int mode = it.op.mode;
        if ((mode == 2 || mode == 3) && !it.op.has_extra) mode = 1;
        if (it.op.is_int && mode != 1) return ctx->fail(JXLB200_E_ARG, "integer samples only blend with ADD (the reference casts to float first)");
        const bool need_fa = (mode == 2 && !it.op.is_alpha) || mode == 3, need_ra = mode == 2 && !it.op.is_alpha;
        for (int r = 0; r < 5; r++) {
            const bool needed = r < 3 || (r == 3 && need_fa) || (r == 4 && need_ra);
            const int pl = it.plane[r];
            if (!needed) continue;
            if (pl < 0 || pl >= n_planes || !planes[pl]) return ctx->fail(JXLB200_E_ARG, "blend item names a plane that was not given");
            if (it.y[r] < 0 || it.x[r] < 0 || it.y[r] + it.h > plane_h[pl] || it.x[r] + it.w > plane_w[pl])
                return ctx->fail(JXLB200_E_STREAM, "blend rectangle outside its buffer");
            lo[pl] = std::min(lo[pl], it.y[r]); hi[pl] = std::max(hi[pl], it.y[r] + it.h);
        }
        if (writable && !writable[it.plane[0]]) return ctx->fail(JXLB200_E_ARG, "blend item writes a plane not marked writable");
    }
    return 0;
}

// One k7_blend launch per item, in order.  row0[pl] is the device address of row 0 of plane pl (plane_w[pl] samples per row); only
// rows hi[pl] > lo[pl] of a plane are dereferenced.
static int blend_items_enqueue(jxlb200_ctx *ctx, int32_t n_planes, const std::vector<uintptr_t> &row0, const std::vector<int> &hi,
    const int32_t plane_w[], int32_t n_items, const jxlb200_blend_item *items) {
    cudaStream_t st = ctx->stream;
    for (int k = 0; k < n_items; k++) {
        const jxlb200_blend_item &it = items[k];
        BlendArgs A;
        A.mode = it.op.mode; A.is_int = it.op.is_int; A.is_alpha = it.op.is_alpha; A.has_extra = it.op.has_extra; A.clamp = it.op.clamp; A.premult = it.op.premult;
        A.h = it.h; A.w = it.w;
        auto at = [&](int r) -> char * {
            const int pl = it.plane[r];
            if (pl < 0 || pl >= n_planes || hi[pl] < 0) return nullptr;
            return (char *)(row0[pl] + ((size_t)it.y[r] * plane_w[pl] + it.x[r]) * 4);
        };
        auto pitch = [&](int r) -> long long { const int pl = it.plane[r]; return (pl < 0 || pl >= n_planes) ? 1 : plane_w[pl]; };
        A.out = at(0); A.a = at(1); A.b = at(2); A.fa = (const float *)at(3); A.ra = (const float *)at(4);
        A.pout = pitch(0); A.pa = pitch(1); A.pb = pitch(2); A.pfa = pitch(3); A.pra = pitch(4);
        const long long n = (long long)it.h * it.w;
        k7_blend<<<(int)std::min<long long>(ctx->sms * 8, (n + 255) / 256), 256, 0, st>>>(A);
        ctx->launches++;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int32_t jxlb200_blend_batch(jxlb200_ctx *ctx, int32_t n_planes, void *const planes[], const int32_t plane_h[], const int32_t plane_w[],
    const int32_t writable[], int32_t n_items, const jxlb200_blend_item *items) {
    if (!ctx) return JXLB200_E_ARG;
    if (n_planes < 1 || n_planes > 64 || !planes || !plane_h || !plane_w || !writable || n_items < 0 || (n_items > 0 && !items))
        return ctx->fail(JXLB200_E_ARG, "bad arguments");
    if (n_items == 0) return 0;
    std::vector<int> lo, hi;
    int rc = blend_items_check(ctx, n_planes, planes, plane_h, plane_w, writable, n_items, items, lo, hi);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<size_t> off(n_planes, 0);
    size_t total = 0;
    for (int pl = 0; pl < n_planes; pl++) {
        if (hi[pl] < 0) continue;
        off[pl] = total;
        total += ((size_t)(hi[pl] - lo[pl]) * plane_w[pl] * 4 + 255) & ~(size_t)255;
    }
    CUDA_TRY(ctx, ctx->blend.ensure(total));
    cudaStream_t st = ctx->stream;
    char *base = (char *)ctx->blend.p;
    std::vector<uintptr_t> row0(n_planes, 0);
    for (int pl = 0; pl < n_planes; pl++)
        if (hi[pl] >= 0) {
            row0[pl] = (uintptr_t)(base + off[pl]) - (uintptr_t)lo[pl] * plane_w[pl] * 4;   // the staged rows start at row lo[pl]
            CUDA_TRY(ctx, cudaMemcpyAsync(base + off[pl], (const char *)planes[pl] + (size_t)lo[pl] * plane_w[pl] * 4,
                                          (size_t)(hi[pl] - lo[pl]) * plane_w[pl] * 4, cudaMemcpyHostToDevice, st));
        }
    if ((rc = blend_items_enqueue(ctx, n_planes, row0, hi, plane_w, n_items, items))) return rc;
    for (int pl = 0; pl < n_planes; pl++)
        if (hi[pl] >= 0 && writable[pl])
            CUDA_TRY(ctx, cudaMemcpyAsync((char *)planes[pl] + (size_t)lo[pl] * plane_w[pl] * 4, base + off[pl],
                                          (size_t)(hi[pl] - lo[pl]) * plane_w[pl] * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    return 0;
}

int32_t jxlb200_blend_batch_dev(jxlb200_ctx *ctx, int32_t n_planes, void *const planes[], const int32_t plane_h[], const int32_t plane_w[],
    int32_t n_items, const jxlb200_blend_item *items) {
    if (!ctx) return JXLB200_E_ARG;
    if (n_planes < 1 || n_planes > 64 || !planes || !plane_h || !plane_w || n_items < 0 || (n_items > 0 && !items))
        return ctx->fail(JXLB200_E_ARG, "bad arguments");
    if (n_items == 0) return 0;
    std::vector<int> lo, hi;
    int rc = blend_items_check(ctx, n_planes, planes, plane_h, plane_w, nullptr, n_items, items, lo, hi);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<uintptr_t> row0(n_planes, 0);
    for (int pl = 0; pl < n_planes; pl++) row0[pl] = (uintptr_t)planes[pl];
    return blend_items_enqueue(ctx, n_planes, row0, hi, plane_w, n_items, items);
}


// ---- k x k upsampling of one float channel (k8_features.cuh) ----
static int upsample_check(jxlb200_ctx *ctx, const void *in, int32_t h, int32_t w, int32_t k, const float *weights, const void *out) {
    if (!ctx) return JXLB200_E_ARG;
    if (!in || !weights || !out || h <= 0 || w <= 0) return ctx->fail(JXLB200_E_ARG, "NULL pointer or empty channel");
    if (k != 2 && k != 4 && k != 8) return ctx->fail(JXLB200_E_ARG, "upsampling factor must be 2, 4 or 8 (FrameHeader.java:121-123)");
    return 0;
}
static int upsample_enqueue(jxlb200_ctx *ctx, const float *d_in, int32_t h, int32_t w, int32_t k, const float *weights, float *d_out) {
    const size_t n = (size_t)h * w, nw = (size_t)k * k * 25;
    CUDA_TRY(ctx, ctx->dtab.ensure(sizeof(float) * nw));
    float *d_w = ctx->dtab.as<float>();
    cudaStream_t st = ctx->stream;
    CUDA_TRY(ctx, cudaMemcpyAsync(d_w, weights, sizeof(float) * nw, cudaMemcpyHostToDevice, st));
    k8_upsample<<<min(ctx->sms * 8, ceil_div((int)std::min<size_t>(n, 1u << 30), 128)), 128, sizeof(float) * nw, st>>>(d_in, h, w, k, d_w, d_out);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
int32_t jxlb200_upsample(jxlb200_ctx *ctx, const float *in, int32_t h, int32_t w, int32_t k, const float *weights, float *out) {
    int rc = upsample_check(ctx, in, h, w, k, weights, out);
    if (rc) return rc;
    const size_t n = (size_t)h * w;
    Staged r[2] = {{&ctx->blend, in, nullptr, sizeof(float) * n}, {&ctx->blend, nullptr, out, sizeof(float) * n * k * k}};
    if ((rc = stage_in(ctx, r, 2))) return rc;
    if ((rc = upsample_enqueue(ctx, (const float *)r[0].dev, h, w, k, weights, (float *)r[1].dev))) return rc;
    return stage_out(ctx, r, 2);
}
int32_t jxlb200_upsample_dev(jxlb200_ctx *ctx, const float *in, int32_t h, int32_t w, int32_t k, const float *weights, float *out) {
    int rc = upsample_check(ctx, in, h, w, k, weights, out);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return upsample_enqueue(ctx, in, h, w, k, weights, out);
}


// ---- noise synthesis (k8_features.cuh): Frame.initializeNoise + synthesizeNoise, in place on device planes ----
static int noise_check(jxlb200_ctx *ctx, float *const planes[3], int32_t h, int32_t w, int32_t group_dim, const float *lut) {
    if (!ctx) return JXLB200_E_ARG;
    if (!planes || !planes[0] || !planes[1] || !planes[2] || !lut || h <= 0 || w <= 0) return ctx->fail(JXLB200_E_ARG, "NULL pointer or empty frame");
    if (group_dim != 128 && group_dim != 256 && group_dim != 512 && group_dim != 1024) return ctx->fail(JXLB200_E_ARG, "group_dim must be 128 << 0..3");
    return 0;
}
static int noise_enqueue(jxlb200_ctx *ctx, float *const d_planes[3], int32_t h, int32_t w, int32_t group_dim, int64_t seed0,
    const float lut[8], float base_corr_x, float base_corr_b) {
    const size_t n = (size_t)h * w;
    CUDA_TRY(ctx, ctx->feat.ensure(sizeof(float) * 3 * n));
    NoiseArgs A;
    for (int c = 0; c < 3; c++) { A.local[c] = ctx->feat.as<float>() + c * n; A.plane[c] = d_planes[c]; }
    A.h = h; A.w = w; A.group_dim = group_dim;
    A.log_dim = group_dim == 128 ? 7 : group_dim == 256 ? 8 : group_dim == 512 ? 9 : 10;
    A.group_cols = ceil_div(w, group_dim);
    A.num_groups = A.group_cols * ceil_div(h, group_dim);
    A.seed0 = (unsigned long long)seed0;
    for (int i = 0; i < 8; i++) A.lut[i] = lut[i];
    A.base_x = base_corr_x; A.base_b = base_corr_b;
    cudaStream_t st = ctx->stream;
    k8_noise_rng<<<ceil_div(A.num_groups * 8, 64), 64, 0, st>>>(A);
    k8_noise_apply<<<min(ctx->sms * 8, ceil_div((int)std::min<size_t>(n, 1u << 30), 256)), 256, 0, st>>>(A);
    ctx->launches += 2;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
int32_t jxlb200_noise(jxlb200_ctx *ctx, float *const planes[3], int32_t h, int32_t w, int32_t group_dim, int64_t seed0,
    const float lut[8], float base_corr_x, float base_corr_b) {
    int rc = noise_check(ctx, planes, h, w, group_dim, lut);
    if (rc) return rc;
    Staged r[3];
    for (int c = 0; c < 3; c++) r[c] = {&ctx->blend, planes[c], planes[c], sizeof(float) * h * w};
    if ((rc = stage_in(ctx, r, 3))) return rc;
    if ((rc = noise_enqueue(ctx, planes_of<float>(r).data(), h, w, group_dim, seed0, lut, base_corr_x, base_corr_b))) return rc;
    return stage_out(ctx, r, 3);
}
int32_t jxlb200_noise_dev(jxlb200_ctx *ctx, float *const planes[3], int32_t h, int32_t w, int32_t group_dim, int64_t seed0,
    const float lut[8], float base_corr_x, float base_corr_b) {
    int rc = noise_check(ctx, planes, h, w, group_dim, lut);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return noise_enqueue(ctx, planes, h, w, group_dim, seed0, lut, base_corr_x, base_corr_b);
}


// ---- splines (splines_host.cuh + k8_splines): Frame.renderSplines, in place ----
// Spline.computeCoeffs and the arcs of every spline, on the host (both forms)
static int splines_arcs(jxlb200_ctx *ctx, float *const planes[3], int32_t h, int32_t w, int32_t num_splines, const int32_t *npoints,
    const int32_t *points, const int32_t *coeff, int32_t quant_adjust, float base_corr_x, float base_corr_b, std::vector<SplineArcDev> &arcs) {
    if (!ctx) return JXLB200_E_ARG;
    if (!planes || !planes[0] || !planes[1] || !planes[2] || !npoints || !points || !coeff || h <= 0 || w <= 0 || num_splines < 0)
        return ctx->fail(JXLB200_E_ARG, "NULL pointer or empty frame");
    if (num_splines == 0) return 0;
    // Spline.computeCoeffs with splineID 0 (see splines_host.cuh)
    splines_host::Track trk[4];
    {
        const float qa = quant_adjust / 8.0f;
        const float inv_qa = qa >= 0 ? 1.0f / (1.0f + qa) : 1.0f - qa;
        const float ya = 0.106066017f * inv_qa, xa = 0.005939697f * inv_qa, ba = 0.098994949f * inv_qa, sa = 0.47135738f * inv_qa;
        for (int i = 0; i < 32; i++) {
            trk[1].c[i] = coeff[32 + i] * ya;
            trk[0].c[i] = coeff[i] * xa + base_corr_x * trk[1].c[i];
            trk[2].c[i] = coeff[64 + i] * ba + base_corr_b * trk[1].c[i];
            trk[3].c[i] = coeff[96 + i] * sa;
        }
    }
    const int32_t *pts = points;
    for (int s = 0; s < num_splines; s++) {
        if (npoints[s] < 1) return ctx->fail(JXLB200_E_ARG, "a spline needs at least one control point");
        splines_host::build(pts, npoints[s], trk, h, w, arcs);
        pts += 2 * npoints[s];
    }
    return 0;
}
static int splines_enqueue(jxlb200_ctx *ctx, float *const d[3], int32_t h, int32_t w, const std::vector<SplineArcDev> &arcs) {
    const size_t abytes = sizeof(SplineArcDev) * arcs.size();
    CUDA_TRY(ctx, ctx->dtab.ensure(abytes));
    SplineArcDev *d_arcs = ctx->dtab.as<SplineArcDev>();
    cudaStream_t st = ctx->stream;
    CUDA_TRY(ctx, cudaMemcpyAsync(d_arcs, arcs.data(), abytes, cudaMemcpyHostToDevice, st));
    k8_splines<<<dim3(ceil_div(w, 32), ceil_div(h, 8)), 256, 0, st>>>(d[0], d[1], d[2], h, w, d_arcs, (int)arcs.size(), (float)sqrt(0.125));
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
int32_t jxlb200_splines(jxlb200_ctx *ctx, float *const planes[3], int32_t h, int32_t w, int32_t num_splines, const int32_t *npoints,
    const int32_t *points, const int32_t *coeff, int32_t quant_adjust, float base_corr_x, float base_corr_b) {
    std::vector<SplineArcDev> arcs;
    int rc = splines_arcs(ctx, planes, h, w, num_splines, npoints, points, coeff, quant_adjust, base_corr_x, base_corr_b, arcs);
    if (rc || arcs.empty()) return rc;
    Staged r[3];
    for (int c = 0; c < 3; c++) r[c] = {&ctx->blend, planes[c], planes[c], sizeof(float) * h * w};
    if ((rc = stage_in(ctx, r, 3))) return rc;
    if ((rc = splines_enqueue(ctx, planes_of<float>(r).data(), h, w, arcs))) return rc;
    return stage_out(ctx, r, 3);
}
int32_t jxlb200_splines_dev(jxlb200_ctx *ctx, float *const planes[3], int32_t h, int32_t w, int32_t num_splines, const int32_t *npoints,
    const int32_t *points, const int32_t *coeff, int32_t quant_adjust, float base_corr_x, float base_corr_b) {
    std::vector<SplineArcDev> arcs;
    int rc = splines_arcs(ctx, planes, h, w, num_splines, npoints, points, coeff, quant_adjust, base_corr_x, base_corr_b, arcs);
    if (rc || arcs.empty()) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return splines_enqueue(ctx, planes, h, w, arcs);
}


// ---- LF coefficients (k8_lf_dequant): LFCoefficients' dequantisation + LF chroma-from-luma + adaptive smoothing ----
static int lf_check(jxlb200_ctx *ctx, int32_t hb, int32_t wb, const float scaled_dequant[3], const int32_t *const lf_quant[3],
    const uint8_t *extra_precision, float *const out[3]) {
    if (!ctx) return JXLB200_E_ARG;
    if (hb < 1 || wb < 1 || !scaled_dequant || !lf_quant || !extra_precision || !out) return ctx->fail(JXLB200_E_ARG, "bad arguments");
    for (int c = 0; c < 3; c++)
        if (!lf_quant[c] || !out[c]) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    const int ng = ((wb + 255) >> 8) * ((hb + 255) >> 8);
    for (int g = 0; g < ng; g++)
        if (extra_precision[g] > 3) return ctx->fail(JXLB200_E_STREAM, "extraPrecision is a 2-bit field");
    return 0;
}
static int lf_enqueue(jxlb200_ctx *ctx, int32_t hb, int32_t wb, const float scaled_dequant[3], float k_x, float k_b,
    int32_t cfl, int32_t adaptive_smoothing, const int32_t *const d_q[3], const uint8_t *extra_precision, float *const d_out[3]) {
    const size_t n = (size_t)hb * wb;
    const int gcols = (wb + 255) >> 8, ng = gcols * ((hb + 255) >> 8);
    CUDA_TRY(ctx, ctx->dtab.ensure(ng));
    uint8_t *dep = ctx->dtab.as<uint8_t>();
    cudaStream_t st = ctx->stream;
    CUDA_TRY(ctx, cudaMemcpyAsync(dep, extra_precision, ng, cudaMemcpyHostToDevice, st));
    LfArgs A;
    for (int c = 0; c < 3; c++) { A.q[c] = d_q[c]; A.out[c] = d_out[c]; A.sd[c] = scaled_dequant[c]; }
    A.ep = dep; A.hb = hb; A.wb = wb; A.gcols = gcols; A.cfl = cfl ? 1 : 0; A.smooth = adaptive_smoothing ? 1 : 0; A.kx = k_x; A.kb = k_b;
    k8_lf_dequant<<<(int)std::min<size_t>((size_t)ctx->sms * 8, (n + 255) / 256), 256, 0, st>>>(A);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
int32_t jxlb200_lf_dequant(jxlb200_ctx *ctx, int32_t hb, int32_t wb, const float scaled_dequant[3], float k_x, float k_b,
    int32_t cfl, int32_t adaptive_smoothing, const int32_t *const lf_quant[3], const uint8_t *extra_precision, float *const out[3]) {
    int rc = lf_check(ctx, hb, wb, scaled_dequant, lf_quant, extra_precision, out);
    if (rc) return rc;
    Staged r[6];
    stage_planes(r, ctx->blend, lf_quant, ctx->blend, out, sizeof(float) * hb * wb);
    if ((rc = stage_in(ctx, r, 6))) return rc;
    if ((rc = lf_enqueue(ctx, hb, wb, scaled_dequant, k_x, k_b, cfl, adaptive_smoothing, planes_of<const int32_t>(r).data(), extra_precision,
                         planes_of<float>(r + 3).data())))
        return rc;
    return stage_out(ctx, r, 6);
}
int32_t jxlb200_lf_dequant_dev(jxlb200_ctx *ctx, int32_t hb, int32_t wb, const float scaled_dequant[3], float k_x, float k_b,
    int32_t cfl, int32_t adaptive_smoothing, const int32_t *const lf_quant[3], const uint8_t *extra_precision, float *const out[3]) {
    int rc = lf_check(ctx, hb, wb, scaled_dequant, lf_quant, extra_precision, out);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return lf_enqueue(ctx, hb, wb, scaled_dequant, k_x, k_b, cfl, adaptive_smoothing, lf_quant, extra_precision, out);
}


// ---- 1:8 previews (k10_preview.cuh) ----
static int preview_check(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float scaled_dequant[3], int32_t adaptive_smoothing,
    const int32_t *const lf_quant[3], const uint8_t *extra_precision, int32_t n_extra_precision, int32_t out_h, int32_t out_w,
    float *const out[3]) {
    int rc = check_params(ctx, p);
    if (rc) return rc;
    if (!scaled_dequant || !lf_quant || !extra_precision || !out) return ctx->fail(JXLB200_E_ARG, "NULL pointer");
    for (int c = 0; c < 3; c++)
        if (!lf_quant[c] || !out[c]) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    const int hb = p->height >> 3, wb = p->width >> 3;
    if (out_h < 1 || out_w < 1 || out_h > hb || out_w > wb) return ctx->fail(JXLB200_E_ARG, "preview size outside the frame's LF grid");
    const int ng = ((wb + 255) >> 8) * ((hb + 255) >> 8);
    if (n_extra_precision != ng) return ctx->fail(JXLB200_E_ARG, "extra_precision must hold one byte per LF group");
    for (int g = 0; g < ng; g++)
        if (extra_precision[g] > 3) return ctx->fail(JXLB200_E_STREAM, "extraPrecision is a 2-bit field");
    const bool subsampled = p->shift_x[0] | p->shift_x[1] | p->shift_x[2] | p->shift_y[0] | p->shift_y[1] | p->shift_y[2];
    if (subsampled && adaptive_smoothing) return ctx->fail(JXLB200_E_STREAM, "adaptive LF smoothing with chroma subsampling");
    return 0;
}
static int preview_enqueue(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float scaled_dequant[3], float k_x, float k_b,
    int32_t adaptive_smoothing, const int32_t *const d_q[3], const uint8_t *extra_precision, int32_t out_h, int32_t out_w,
    float *const d_out[3]) {
    PreviewArgs A;
    LfArgs &L = A.lf;
    L.hb = p->height >> 3; L.wb = p->width >> 3;
    L.gcols = (L.wb + 255) >> 8;
    const int ng = L.gcols * ((L.hb + 255) >> 8);
    cudaStream_t st = ctx->stream;
    CUDA_TRY(ctx, ctx->dtab.ensure(ng));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->dtab.p, extra_precision, ng, cudaMemcpyHostToDevice, st));
    L.ep = ctx->dtab.as<uint8_t>();
    A.subsampled = 0;
    for (int c = 0; c < 3; c++) {
        L.q[c] = d_q[c]; L.out[c] = nullptr; L.sd[c] = scaled_dequant[c];
        A.sy[c] = p->shift_y[c]; A.sx[c] = p->shift_x[c];
        A.subsampled |= A.sy[c] | A.sx[c];
        A.out[c] = d_out[c];
    }
    L.cfl = !A.subsampled; L.smooth = adaptive_smoothing ? 1 : 0; L.kx = k_x; L.kb = k_b;
    A.out_h = out_h; A.out_w = out_w;
    fill_k2(A.P, p, nullptr);
    const long long n = (long long)out_h * out_w;
    k10_lf_preview<<<(int)std::min<long long>((long long)ctx->sms * 8, (n + 255) / 256), 256, 0, st>>>(A);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
int32_t jxlb200_lf_preview(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float scaled_dequant[3], float k_x, float k_b,
    int32_t adaptive_smoothing, const int32_t *const lf_quant[3], const uint8_t *extra_precision, int32_t n_extra_precision,
    int32_t out_h, int32_t out_w, float *const out[3]) {
    int rc = preview_check(ctx, p, scaled_dequant, adaptive_smoothing, lf_quant, extra_precision, n_extra_precision, out_h, out_w, out);
    if (rc) return rc;
    Staged r[6];
    for (int c = 0; c < 3; c++) {
        r[c] = {&ctx->blend, lf_quant[c], nullptr, sizeof(int32_t) * (size_t)((p->height >> 3) >> p->shift_y[c]) * ((p->width >> 3) >> p->shift_x[c])};
        r[3 + c] = {&ctx->blend, nullptr, out[c], sizeof(float) * (size_t)out_h * out_w};
    }
    if ((rc = stage_in(ctx, r, 6))) return rc;
    if ((rc = preview_enqueue(ctx, p, scaled_dequant, k_x, k_b, adaptive_smoothing, planes_of<const int32_t>(r).data(), extra_precision,
                              out_h, out_w, planes_of<float>(r + 3).data())))
        return rc;
    return stage_out(ctx, r, 6);
}
int32_t jxlb200_lf_preview_dev(jxlb200_ctx *ctx, const jxlb200_frame_params *p, const float scaled_dequant[3], float k_x, float k_b,
    int32_t adaptive_smoothing, const int32_t *const lf_quant[3], const uint8_t *extra_precision, int32_t n_extra_precision,
    int32_t out_h, int32_t out_w, float *const out[3]) {
    int rc = preview_check(ctx, p, scaled_dequant, adaptive_smoothing, lf_quant, extra_precision, n_extra_precision, out_h, out_w, out);
    if (rc) return rc;
    for (int c = 0; c < 3; c++)
        for (int d = 0; d < 3; d++)
            if ((const void *)lf_quant[c] == (const void *)out[d]) return ctx->fail(JXLB200_E_ARG, "an output plane aliases an input plane");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return preview_enqueue(ctx, p, scaled_dequant, k_x, k_b, adaptive_smoothing, lf_quant, extra_precision, out_h, out_w, out);
}

static int area_check(jxlb200_ctx *ctx, int32_t n_channels, const void *const planes[], const int32_t is_int[], const int32_t depth[],
    int32_t h, int32_t w, float *const out[]) {
    if (!ctx) return JXLB200_E_ARG;
    if (!planes || !is_int || !depth || !out || n_channels < 1 || h <= 0 || w <= 0) return ctx->fail(JXLB200_E_ARG, "bad arguments");
    for (int c = 0; c < n_channels; c++) {
        if (!planes[c] || !out[c]) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
        if (is_int[c] && (depth[c] < 1 || depth[c] > 31)) return ctx->fail(JXLB200_E_ARG, "bit depth outside 1..31");
    }
    return 0;
}
static int area_enqueue(jxlb200_ctx *ctx, int32_t n_channels, const void *const d_planes[], const int32_t is_int[], const int32_t depth[],
    int32_t h, int32_t w, float *const d_out[]) {
    AreaArgs A;
    A.h = h; A.w = w; A.oh = (h + 7) >> 3; A.ow = (w + 7) >> 3;
    const long long n = (long long)A.oh * A.ow;
    for (int c0 = 0; c0 < n_channels; c0 += kAreaChannels) {
        const int nc = std::min(kAreaChannels, n_channels - c0);
        for (int k = 0; k < nc; k++) {
            const int c = c0 + k;
            A.plane[k] = d_planes[c]; A.out[k] = d_out[c]; A.is_int[k] = is_int[c] ? 1 : 0;
            A.scale[k] = is_int[c] ? 1.0f / (float)((1u << depth[c]) - 1u) : 1.0f;      // ImageBuffer.castToFloat
        }
        const dim3 grid((unsigned)std::min<long long>((long long)ctx->sms * 8, (n + 255) / 256), (unsigned)nc);
        k10_area_mean8<<<grid, 256, 0, ctx->stream>>>(A);
        ctx->launches++;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
int32_t jxlb200_area_mean8(jxlb200_ctx *ctx, int32_t n_channels, const void *const planes[], const int32_t is_int[], const int32_t depth[],
    int32_t h, int32_t w, float *const out[]) {
    int rc = area_check(ctx, n_channels, planes, is_int, depth, h, w, out);
    if (rc) return rc;
    const size_t in_bytes = 4 * (size_t)h * w, out_bytes = sizeof(float) * (size_t)((h + 7) >> 3) * ((w + 7) >> 3);
    std::vector<Staged> r(2 * (size_t)n_channels);
    for (int c = 0; c < n_channels; c++) {
        r[c] = {&ctx->blend, planes[c], nullptr, in_bytes};
        r[n_channels + c] = {&ctx->blend, nullptr, out[c], out_bytes};
    }
    if ((rc = stage_in(ctx, r.data(), 2 * n_channels))) return rc;
    std::vector<const void *> d(n_channels);
    std::vector<float *> o(n_channels);
    for (int c = 0; c < n_channels; c++) { d[c] = r[c].dev; o[c] = (float *)r[n_channels + c].dev; }
    if ((rc = area_enqueue(ctx, n_channels, d.data(), is_int, depth, h, w, o.data()))) return rc;
    return stage_out(ctx, r.data(), 2 * n_channels);
}
int32_t jxlb200_area_mean8_dev(jxlb200_ctx *ctx, int32_t n_channels, const void *const planes[], const int32_t is_int[], const int32_t depth[],
    int32_t h, int32_t w, float *const out[]) {
    int rc = area_check(ctx, n_channels, planes, is_int, depth, h, w, out);
    if (rc) return rc;
    for (int c = 0; c < n_channels; c++)
        for (int d = 0; d < n_channels; d++)
            if (planes[c] == (const void *)out[d]) return ctx->fail(JXLB200_E_ARG, "an output plane aliases an input plane");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return area_enqueue(ctx, n_channels, planes, is_int, depth, h, w, out);
}


// ---- PNG-ready samples (k8_pack_samples) ----
static int pack_check(jxlb200_ctx *ctx, const void *const planes[], const int32_t is_int[], const int32_t depth[],
    int32_t n_channels, int32_t h, int32_t w, int32_t bits, const void *out) {
    if (!ctx) return JXLB200_E_ARG;
    if (!planes || !is_int || !depth || !out || n_channels < 1 || n_channels > 8 || h <= 0 || w <= 0) return ctx->fail(JXLB200_E_ARG, "bad arguments");
    if (bits != 8 && bits != 16) return ctx->fail(JXLB200_E_ARG, "PNG only supports 8 and 16 (PNGWriter.java:57-58)");
    for (int c = 0; c < n_channels; c++)
        if (!planes[c] || depth[c] < 1 || depth[c] > 31) return ctx->fail(JXLB200_E_ARG, "NULL plane or bad depth");
    return 0;
}
static int pack_enqueue(jxlb200_ctx *ctx, const void *const d_planes[], const int32_t is_int[], const int32_t depth[],
    int32_t n_channels, int32_t n_color, int32_t linear, int32_t h, int32_t w, int32_t bits, int32_t layout, uint8_t *d_out) {
    const size_t n = (size_t)h * w;
    PackArgs A;
    for (int c = 0; c < n_channels; c++) { A.plane[c] = d_planes[c]; A.is_int[c] = is_int[c]; A.depth[c] = depth[c]; }
    A.n_channels = n_channels; A.n_color = n_color; A.linear = linear; A.h = h; A.w = w; A.bits = bits; A.layout = layout;
    A.out = d_out;
    k8_pack_samples<<<min(ctx->sms * 8, ceil_div((int)std::min<size_t>(n, 1u << 30), 256)), 256, 0, ctx->stream>>>(A);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
int32_t jxlb200_pack_samples(jxlb200_ctx *ctx, const void *const planes[], const int32_t is_int[], const int32_t depth[],
    int32_t n_channels, int32_t n_color, int32_t linear, int32_t h, int32_t w, int32_t bits, uint8_t *out) {
    int rc = pack_check(ctx, planes, is_int, depth, n_channels, h, w, bits, out);
    if (rc) return rc;
    const size_t n = (size_t)h * w;
    Staged r[9];
    for (int c = 0; c < n_channels; c++) r[c] = {&ctx->blend, planes[c], nullptr, 4 * n};
    r[n_channels] = {&ctx->blend, nullptr, out, n * n_channels * (bits > 8 ? 2 : 1)};
    if ((rc = stage_in(ctx, r, n_channels + 1))) return rc;
    const void *d[8];
    for (int c = 0; c < n_channels; c++) d[c] = r[c].dev;
    if ((rc = pack_enqueue(ctx, d, is_int, depth, n_channels, n_color, linear, h, w, bits, 0, (uint8_t *)r[n_channels].dev))) return rc;
    return stage_out(ctx, r, n_channels + 1);
}
int32_t jxlb200_pack_samples_dev(jxlb200_ctx *ctx, const void *const planes[], const int32_t is_int[], const int32_t depth[],
    int32_t n_channels, int32_t n_color, int32_t linear, int32_t h, int32_t w, int32_t bits, int32_t layout, uint8_t *out) {
    int rc = pack_check(ctx, planes, is_int, depth, n_channels, h, w, bits, out);
    if (rc) return rc;
    if (layout != 0 && layout != 1) return ctx->fail(JXLB200_E_ARG, "layout must be 0 (PNG bytes) or 1 (planar samples)");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return pack_enqueue(ctx, planes, is_int, depth, n_channels, n_color, linear, h, w, bits, layout, out);
}

// ---- batch output (k11_pack_batch) ----
int32_t jxlb200_pack_batch_dev(jxlb200_ctx *ctx, const jxlb200_batch_item *items, int32_t n, int32_t c, int32_t bits, int32_t out_h,
    int32_t out_w, void *out) {
    if (!ctx) return JXLB200_E_ARG;
    if (!items || !out || n < 1) return ctx->fail(JXLB200_E_ARG, "NULL pointer or an empty batch");
    if (c != 1 && c != 3 && c != 4) return ctx->fail(JXLB200_E_ARG, "c must be 1, 3 or 4");
    if (bits != 8 && bits != 16) return ctx->fail(JXLB200_E_ARG, "bits must be 8 or 16");
    if (out_h < 1 || out_w < 1) return ctx->fail(JXLB200_E_ARG, "slot smaller than 1 x 1");
    const size_t bytes = bits > 8 ? 2 : 1;
    const uintptr_t o0 = (uintptr_t)out, o1 = o0 + (size_t)n * c * out_h * out_w * bytes;
    for (int i = 0; i < n; i++) {
        const jxlb200_batch_item &I = items[i];
        if (I.orientation < 1 || I.orientation > 8) return ctx->fail(JXLB200_E_ARG, "orientation outside 1..8");
        if (I.h < 1 || I.w < 1) return ctx->fail(JXLB200_E_ARG, "image smaller than 1 x 1");
        const int oh = I.orientation >= 5 ? I.w : I.h, ow = I.orientation >= 5 ? I.h : I.w;
        if (oh > out_h || ow > out_w) return ctx->fail(JXLB200_E_ARG, "oriented image larger than its slot");
        for (int k = 0; k < c; k++) {
            if (!I.plane[k]) continue;
            if (I.pitch[k] < I.w) return ctx->fail(JXLB200_E_ARG, "plane pitch below the image width");
            if (I.is_int[k] && (I.depth[k] < 1 || I.depth[k] > 31)) return ctx->fail(JXLB200_E_ARG, "bit depth outside 1..31");
            const uintptr_t p0 = (uintptr_t)I.plane[k], p1 = p0 + 4 * ((size_t)(I.h - 1) * I.pitch[k] + I.w);
            if (p0 < o1 && o0 < p1) return ctx->fail(JXLB200_E_ARG, "the output overlaps an input plane");
        }
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t tab = sizeof(jxlb200_batch_item) * (size_t)n;
    CUDA_TRY(ctx, ctx->dtab.ensure(tab));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->dtab.p, items, tab, cudaMemcpyHostToDevice, ctx->stream));
    const int px = 16 / (int)bytes;                                     // samples per thread: one 16-byte store per channel
    const int vec = (o0 % 16) == 0 && ((size_t)out_w * bytes) % 16 == 0;
    const dim3 block(32, 8), grid((unsigned)ceil_div(out_w, 32 * px), (unsigned)ceil_div(out_h, 8), (unsigned)std::min(n, 65535));
    if (bits == 8) k11_pack_batch<8><<<grid, block, 0, ctx->stream>>>(ctx->dtab.as<jxlb200_batch_item>(), n, c, out_h, out_w, vec, out);
    else k11_pack_batch<16><<<grid, block, 0, ctx->stream>>>(ctx->dtab.as<jxlb200_batch_item>(), n, c, out_h, out_w, vec, out);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}


// ---- glue of the frame loop on device buffers (k9_device.cuh) ----
int32_t jxlb200_cast_to_float_dev(jxlb200_ctx *ctx, const int32_t *in, int64_t n, float scale, float *out) {
    if (!ctx) return JXLB200_E_ARG;
    if (!in || !out || n < 0) return ctx->fail(JXLB200_E_ARG, "NULL pointer or negative size");
    if (n == 0) return 0;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    k9_cast_to_float<<<(int)std::min<long long>((long long)ctx->sms * 8, (n + 255) / 256), 256, 0, ctx->stream>>>(in, n, scale, out);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int32_t jxlb200_modular_xyb_dev(jxlb200_ctx *ctx, const int32_t *const in[3], int64_t n, const float lf_dequant[3], float *const out[3]) {
    if (!ctx) return JXLB200_E_ARG;
    if (!in || !out || !lf_dequant || n < 0) return ctx->fail(JXLB200_E_ARG, "NULL pointer or negative size");
    for (int c = 0; c < 3; c++)
        if (!in[c] || !out[c]) return ctx->fail(JXLB200_E_ARG, "NULL plane pointer");
    if (n == 0) return 0;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    XybArgs A;
    A.y = in[0]; A.x = in[1]; A.b = in[2];
    for (int c = 0; c < 3; c++) { A.out[c] = out[c]; A.dq[c] = lf_dequant[c]; }
    A.n = n;
    k9_modular_xyb<<<(int)std::min<long long>((long long)ctx->sms * 8, (n + 255) / 256), 256, 0, ctx->stream>>>(A);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

}  // extern "C"
