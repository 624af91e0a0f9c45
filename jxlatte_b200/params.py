"""Frame-level scalars handed across the C ABI (include/jxlb200.h: jxlb200_frame_params).

Defaults follow the reference's own defaults; J/ = /root/reference/java/com/traneptora/jxlatte/:
  - OpsinInverseMatrix defaults        J/color/OpsinInverseMatrix.java:11-27
  - RestorationFilter defaults         J/frame/features/RestorationFilter.java:14-44
  - LFChannelCorrelation defaults      J/frame/vardct/LFChannelCorrelation.java:23-29
"""
import ctypes as C

import numpy as np

# TransformType table: (type) -> (parameterIndex, transformMethod, pixelHeight, pixelWidth)
# J/frame/vardct/TransformType.java:10-36
TRANSFORM_TYPES = [
    (0, 0, 8, 8), (1, 3, 8, 8), (2, 1, 8, 8), (3, 2, 8, 8), (4, 0, 16, 16), (5, 0, 32, 32),
    (6, 0, 16, 8), (6, 0, 8, 16), (7, 0, 32, 8), (7, 0, 8, 32), (8, 0, 32, 16), (8, 0, 16, 32),
    (9, 5, 8, 8), (9, 4, 8, 8), (10, 6, 8, 8), (10, 6, 8, 8), (10, 6, 8, 8), (10, 6, 8, 8),
    (11, 0, 64, 64), (12, 0, 64, 32), (12, 0, 32, 64), (13, 0, 128, 128), (14, 0, 128, 64), (14, 0, 64, 128),
    (15, 0, 256, 256), (16, 0, 256, 128), (16, 0, 128, 256),
]
TRANSFORM_NAMES = [
    "DCT8", "HORNUSS", "DCT2", "DCT4", "DCT16", "DCT32", "DCT16_8", "DCT8_16", "DCT32_8", "DCT8_32",
    "DCT32_16", "DCT16_32", "DCT4_8", "DCT8_4", "AFV0", "AFV1", "AFV2", "AFV3", "DCT64", "DCT64_32",
    "DCT32_64", "DCT128", "DCT128_64", "DCT64_128", "DCT256", "DCT256_128", "DCT128_256",
]

COLOR_NONE, COLOR_XYB, COLOR_YCBCR = 0, 1, 2


class FrameParams(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("global_scale", C.c_int32),
        ("xqm_scale", C.c_int32), ("bqm_scale", C.c_int32),
        ("quant_bias", C.c_float * 3), ("quant_bias_numerator", C.c_float),
        ("color_factor", C.c_int32), ("base_corr_x", C.c_float), ("base_corr_b", C.c_float),
        ("shift_x", C.c_int32 * 3), ("shift_y", C.c_int32 * 3),
        ("gab", C.c_int32), ("gab_w1", C.c_float * 3), ("gab_w2", C.c_float * 3),
        ("epf_iters", C.c_int32), ("epf_sharp_lut", C.c_float * 8), ("epf_channel_scale", C.c_float * 3),
        ("epf_pass0_sigma_scale", C.c_float), ("epf_pass2_sigma_scale", C.c_float), ("epf_border_sad_mul", C.c_float),
        ("color_mode", C.c_int32),
        ("opsin_matrix", C.c_float * 9), ("opsin_bias", C.c_float * 3), ("intensity_target", C.c_float),
    ]

    def copy(self):
        return FrameParams.from_buffer_copy(bytes(self))


def default_frame_params(width, height, *, epf_iters=3, gab=True, color_mode=COLOR_XYB, global_scale=4096,
                         xqm_scale=3, bqm_scale=2, intensity_target=255.0):
    """Scalars of a frame with all-default metadata (the synthetic configs of SURVEY.md 8(d))."""
    if width % 8 or height % 8 or width <= 0 or height <= 0:
        raise ValueError("padded frame size must be positive multiples of 8 (Frame.getPaddedFrameSize)")
    p = FrameParams()
    p.width, p.height = width, height
    p.global_scale = global_scale
    p.xqm_scale, p.bqm_scale = xqm_scale, bqm_scale
    p.quant_bias[:] = [0.945349926692846, 0.9299455010825141, 0.9500648966626564]
    p.quant_bias_numerator = 0.145
    p.color_factor = 84
    p.base_corr_x, p.base_corr_b = 0.0, 1.0
    p.shift_x[:] = [0, 0, 0]
    p.shift_y[:] = [0, 0, 0]
    p.gab = 1 if gab else 0
    p.gab_w1[:] = [0.115169525] * 3
    p.gab_w2[:] = [0.061248592] * 3
    p.epf_iters = epf_iters
    quant_mul = np.float32(0.46)
    for i in range(8):  # epfSharpLut = {0, 1f/7f, ..., 1f} * epfQuantMul, in float32
        base = np.float32(1.0) if i == 7 else np.float32(i) / np.float32(7)
        p.epf_sharp_lut[i] = float(np.float32(base * quant_mul))
    p.epf_channel_scale[:] = [40.0, 5.0, 3.5]
    p.epf_pass0_sigma_scale = 0.9
    p.epf_pass2_sigma_scale = 6.5
    p.epf_border_sad_mul = float(np.float32(2.0) / np.float32(3.0))
    p.color_mode = color_mode
    p.opsin_matrix[:] = [11.031566901960783, -9.866943921568629, -0.16462299647058826,
                         -3.254147380392157, 4.418770392156863, -0.16462299647058826,
                         -3.6588512862745097, 2.7129230470588235, 1.9459282392156863]
    p.opsin_bias[:] = [-0.0037930732552754493] * 3
    p.intensity_target = intensity_target
    return p


# the per-block / per-tile maps of the VarDCT state, in the C ABI's argument order, and their dtypes
STATE_MAPS = (("dct_select", np.uint8), ("block_origin", np.uint8), ("hf_mul", np.int32), ("x_from_y", np.int32), ("b_from_y", np.int32),
              ("sharpness", np.int32))


def state_shapes(p, subsampled=True):
    """Expected shape of each VarDCT state array of a frame with params p: "qcoeff" and "lf" hold one shape per channel (a
    chroma-subsampled channel is smaller by its shifts unless subsampled=False), the STATE_MAPS one shape each."""
    H, W = p.height, p.width
    hb, wb, th, tw = H // 8, W // 8, (H + 63) // 64, (W + 63) // 64
    shifts = [(p.shift_y[c], p.shift_x[c]) if subsampled else (0, 0) for c in range(3)]
    return dict(qcoeff=[(H >> sy, W >> sx) for sy, sx in shifts], lf=[(hb >> sy, wb >> sx) for sy, sx in shifts],
                dct_select=(hb, wb), block_origin=(hb, wb), hf_mul=(hb, wb), x_from_y=(th, tw), b_from_y=(th, tw), sharpness=(hb, wb))


def check_state_shapes(p, arrays, subsampled=True):
    """ValueError unless every array of `arrays` (numpy or torch, keyed as in the state dict) has its state_shapes(p) shape."""
    want = state_shapes(p, subsampled)
    for c in range(3):
        q, lf = tuple(arrays["qcoeff"][c].shape), tuple(arrays["lf"][c].shape)
        if q != want["qcoeff"][c] or lf != want["lf"][c]:
            raise ValueError("qcoeff[%d] / lf[%d] have shapes %s / %s, expected %s / %s" % (c, c, q, lf, want["qcoeff"][c], want["lf"][c]))
    for k, a in arrays.items():
        if k not in ("qcoeff", "lf") and tuple(a.shape) != want[k]:
            raise ValueError("%s has shape %s, expected %s" % (k, tuple(a.shape), want[k]))


def check_lf_planes(p, planes):
    """The three quantised LF planes of a frame (numpy or torch), each of its state_shapes(p)["lf"] shape; ValueError otherwise."""
    want = state_shapes(p)["lf"]
    for c in range(3):
        if tuple(planes[c].shape) != want[c]:
            raise ValueError("lf_quant[%d] has shape %s, expected %s" % (c, tuple(planes[c].shape), want[c]))
    return planes


def check_channels(channels):
    """Equally sized 2-D channels (numpy or torch) -> their (h, w); ValueError otherwise."""
    shapes = {tuple(a.shape) for a in channels}
    if not channels or len(shapes) != 1 or len(next(iter(shapes))) != 2:
        raise ValueError("channels must be 2-D and of one size, got %s" % sorted(shapes))
    return next(iter(shapes))


def check_planes(p, planes):
    """The three colour planes of a frame, each p.height x p.width (numpy or torch); ValueError otherwise."""
    for a in planes:
        if tuple(a.shape) != (p.height, p.width):
            raise ValueError("planes have shape %s, expected %s" % (tuple(a.shape), (p.height, p.width)))
    return planes
