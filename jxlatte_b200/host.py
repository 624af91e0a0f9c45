"""Host side of the drop-in boundary, above the C ABI (include/jxlb200.h).

jxlatte is Java and this image has no JDK, so the Panama shim of INTEGRATION.md cannot be compiled here; this module
makes the same downcalls through ctypes and mirrors the reference's method seams by name and argument meaning, so the
parity tests read like tests of the reference itself (J/ = java/com/traneptora/jxlatte/ in the reference tree):

    Reconstructor.generateWeights              HFGlobal.generateWeights             J/frame/vardct/HFGlobal.java:347-432
    Reconstructor.invertVarDCT                 Frame.decodePassGroups tail          J/frame/Frame.java:361-374
    Reconstructor.performGabConvolution        Frame.performGabConvolution          J/frame/Frame.java:505-542
    Reconstructor.performEdgePreservingFilter  Frame.performEdgePreservingFilter    J/frame/Frame.java:544-636
    Reconstructor.performColorTransforms       JXLCodestreamDecoder.performColorTransforms  J/JXLCodestreamDecoder.java:256-283
    ModularTransforms.applyTransforms          ModularStream.applyTransforms        J/frame/modular/ModularStream.java:224-380

Errors keep the reference's types: IllegalArgumentException -> ValueError, InvalidBitstreamException (an IOException)
-> InvalidBitstreamError(IOError), UnsupportedOperationException -> NotImplementedError, CUDA failure -> IOError.
Everything computes on the GPU; nothing here falls back to the CPU.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import QmParams, Slab  # noqa: F401
from .params import STATE_MAPS, FrameParams, check_channels, check_lf_planes, check_planes, check_state_shapes


class InvalidBitstreamError(IOError):
    """J/io/InvalidBitstreamException.java"""


def _raise(rc, msg):
    if rc == _lib.E_ARG:
        raise ValueError(msg)
    if rc == _lib.E_STREAM:
        raise InvalidBitstreamError(msg)
    if rc == _lib.E_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise IOError(msg)


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _ptr(a):
    return a.ctypes.data


def narrow_coefficients(qcoeff):
    """The three coefficient planes as contiguous int16 arrays for jxlb200_vardct_reconstruct_i16.  Planes that already are
    int16 pass through untouched (no copy: pinned buffers stay pinned); wider ones are range-checked first -- a coefficient
    beyond int16 is legal JPEG XL, it just has to take the int32 call."""
    out = []
    for c in range(3):
        a = np.asarray(qcoeff[c])
        if a.dtype != np.int16:
            if a.dtype.kind not in "iu":
                raise ValueError("qcoeff[%d] is not an integer array" % c)
            if a.size and (int(a.max()) > 32767 or int(a.min()) < -32768):
                raise ValueError("qcoeff[%d] does not fit int16: use narrow=False" % c)
            a = a.astype(np.int16)
        out.append(np.ascontiguousarray(a))
    return out


def _spline_arrays(splines):
    npts = np.array([len(s["points"]) // 2 for s in splines], np.int32)
    pts = np.array([v for s in splines for v in s["points"]], np.int32)
    cf = np.array([v for s in splines for v in s["coeff"]], np.int32)
    return npts, pts, cf


def _extra_precision(extra_precision, hb, wb):
    ep = _c(np.asarray(extra_precision).reshape(-1), np.uint8)
    if ep.size != ((hb + 255) // 256) * ((wb + 255) // 256):
        raise ValueError("extra_precision must hold one byte per LF group")
    return ep


def _preview_args(scaled_dequant, extra_precision):
    """The scaledDequant array and the flat extraPrecision bytes of jxlb200_lf_preview[_dev] (the library checks their count)."""
    return (C.c_float * 3)(*[float(v) for v in scaled_dequant]), _c(np.asarray(extra_precision).reshape(-1), np.uint8)


def _area_args(is_int, depths):
    """The is_int and depth arrays of jxlb200_area_mean8[_dev]."""
    return np.array([1 if v else 0 for v in is_int], np.int32), np.array(depths, np.int32)


def _upsampling_weights(weights, k):
    wt = _c(weights, np.float32)
    if wt.shape != (k, k, 5, 5):
        raise ValueError("weights must be [k][k][5][5]")
    return wt


def _pack_args(ptrs, is_int, depths):
    """The plane pointer, is_int and depth arrays of jxlb200_pack_samples[_dev]."""
    return (C.c_void_p * len(ptrs))(*ptrs), np.array([1 if v else 0 for v in is_int], np.int32), np.array(depths, np.int32)


def qm_default_params():
    """HFGlobal.getDefaultParams (J/frame/vardct/HFGlobal.java:79-188)."""
    prm = (QmParams * 17)()
    rc = _lib.lib().jxlb200_qm_default_params(prm)
    if rc:
        _raise(rc, "jxlb200_qm_default_params failed")
    return prm


def qm_generate(prm=None):
    """HFGlobal.generateWeights for the 17 parameter sets -> (weights f32[3*131584], offsets i32[51]).  Host-side
    table build, no GPU needed (the reference builds it once per frame in the HFGlobal constructor)."""
    if prm is None:
        prm = qm_default_params()
    w = np.zeros(_lib.QM_FLOATS, np.float32)
    off = np.zeros(51, np.int32)
    rc = _lib.lib().jxlb200_qm_generate(prm, _ptr(w), _ptr(off))
    if rc == _lib.E_STREAM:
        raise InvalidBitstreamError("Negative or infinite weight")
    if rc:
        _raise(rc, "jxlb200_qm_generate failed")
    return w, off


def _blend_items(items):
    """(op dict, (h, w), [(plane index, y, x) or None] * 5) tuples -> jxlb200_blend_item array."""
    arr = (_lib.BlendItem * len(items))()
    for k, (op, (h, w), refs) in enumerate(items):
        it = arr[k]
        it.op = _lib.BlendOp(int(op["mode"]), int(op["is_int"]), int(op["is_alpha"]), int(op["has_extra"]), int(op["clamp"]), int(op["premult"]))
        it.h, it.w = int(h), int(w)
        for r in range(5):
            if refs[r] is None:
                it.plane[r], it.y[r], it.x[r] = -1, 0, 0
            else:
                it.plane[r], it.y[r], it.x[r] = int(refs[r][0]), int(refs[r][1]), int(refs[r][2])
    return arr


class Reconstructor:
    """One per decoder instance (JXLDecoder ctor / close(), J/JXLDecoder.java:17-46).  Not thread-safe, like the reference."""

    def __init__(self, device=0):
        self._L = _lib.lib()
        h = C.c_void_p()
        rc = self._L.jxlb200_create(int(device), C.byref(h))
        if rc:
            raise IOError("jxlb200_create(device=%d) failed with %d: no usable CUDA device (there is no CPU fallback)" % (device, rc))
        self._h = h
        self.device = device
        self._weights = None

    def close(self):
        if self._h:
            self._L.jxlb200_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing --
    @property
    def handle(self):
        return self._h

    def _check(self, rc):
        if rc:
            _raise(rc, self._L.jxlb200_last_error(self._h).decode())

    def set_stream(self, cuda_stream_ptr):
        self._check(self._L.jxlb200_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def sync(self):
        self._check(self._L.jxlb200_sync(self._h))

    def launch_count(self):
        return int(self._L.jxlb200_launch_count(self._h))

    def host_register(self, array):
        """Page-lock a numpy array in place (jxlb200_host_register); pair with host_unregister before the array is freed."""
        self._check(self._L.jxlb200_host_register(self._h, C.c_void_p(array.ctypes.data), int(array.nbytes)))

    def host_unregister(self, array):
        self._check(self._L.jxlb200_host_unregister(self._h, C.c_void_p(array.ctypes.data)))

    def selftest_divide(self, n, seed=1):
        """Mismatches between stage 2's shared-reciprocal divide and __fdiv_rn on n operand pairs (must be 0)."""
        bad = C.c_int64(-1)
        self._check(self._L.jxlb200_selftest_divide(self._h, int(n), int(seed), C.byref(bad)))
        return int(bad.value)

    def set_option(self, option, value):
        self._check(self._L.jxlb200_set_option(self._h, int(option), int(value)))

    # -- HFGlobal --
    def generateWeights(self, prm=None):
        w, off = qm_generate(prm)
        self.setWeights(w, off)
        return w, off

    def setWeights(self, weights, offsets):
        w, off = _c(weights, np.float32), _c(offsets, np.int32)
        if w.size != _lib.QM_FLOATS or off.size != 51:
            raise ValueError("weights must hold 3*131584 floats and offsets 51 ints")
        self._check(self._L.jxlb200_set_qm_weights(self._h, _ptr(w), _ptr(off)))
        self._weights = (w, off)

    # -- VarDCT --
    def _state_args(self, st, p, with_sharp, narrow=False, subsampled=True):
        """qcoeff (int16 through narrow_coefficients when narrow), lf, then the STATE_MAPS (sharpness when with_sharp) as contiguous
        arrays of their shapes."""
        q = narrow_coefficients(st["qcoeff"]) if narrow else [_c(st["qcoeff"][c], np.int32) for c in range(3)]
        a = dict(qcoeff=q, lf=[_c(st["lf"][c], np.float32) for c in range(3)])
        a.update((k, _c(st[k], dt)) for k, dt in STATE_MAPS if with_sharp or k != "sharpness")
        check_state_shapes(p, a, subsampled)
        return tuple(a.values())

    def invertVarDCT(self, p, st):
        """bakeDequantizedCoeffs + invertVarDCT for every pass group of the frame -> XYB planes f32[3,H,W]."""
        # full-size planes only: stage 1 alone refuses chroma-subsampled frames (NotImplementedError from the library)
        q, lf, ds, bo, hm, xf, bf = self._state_args(st, p, False, subsampled=False)
        out = np.empty((3, p.height, p.width), np.float32)
        self._check(self._L.jxlb200_vardct_invert(
            self._h, C.byref(p), _lib.planes([_ptr(a) for a in q]), _lib.planes([_ptr(a) for a in lf]),
            _ptr(ds), _ptr(bo), _ptr(hm), _ptr(xf), _ptr(bf), _lib.planes([_ptr(out[c]) for c in range(3)])))
        return out

    def _stage(self, fn, p, planes_in, *extra):
        inp = check_planes(p, [_c(planes_in[c], np.float32) for c in range(3)])
        out = np.empty((3, p.height, p.width), np.float32)
        self._check(fn(self._h, C.byref(p), _lib.planes([_ptr(a) for a in inp]), *extra,
                       _lib.planes([_ptr(out[c]) for c in range(3)])))
        return out

    def performGabConvolution(self, p, planes_in):
        return self._stage(self._L.jxlb200_gaborish, p, planes_in)

    def performEdgePreservingFilter(self, p, planes_in, hf_mul, sharpness):
        hm, sh = _c(hf_mul, np.int32), _c(sharpness, np.int32)
        shp = (p.height // 8, p.width // 8)
        if hm.shape != shp or sh.shape != shp:
            raise ValueError("hf_mul / sharpness must have shape %s" % (shp,))
        return self._stage(self._L.jxlb200_epf, p, planes_in, _ptr(hm), _ptr(sh))

    def restoreModularFrame(self, p, planes_in, epf_sigma_for_modular):
        """Gaborish + EPF (+ p.color_mode) of a Modular-encoded frame: one sigma for the frame (jxlb200_restore_uniform)."""
        sigma = C.c_float(float(epf_sigma_for_modular))
        return self._stage(lambda h, pp, inp, out: self._L.jxlb200_restore_uniform(h, pp, sigma, inp, out), p, planes_in)

    def performColorTransforms(self, p, planes_in):
        return self._stage(self._L.jxlb200_color_transform, p, planes_in)

    def reconstruct(self, p, st, out=None, narrow=False):
        """The whole path on host buffers: invertVarDCT -> Gaborish -> EPF -> colour transform.

        narrow=True sends the coefficients as int16 (jxlb200_vardct_reconstruct_i16: half the upload, same result);
        planes that already are int16 go as they are, int32 planes are range-checked and narrowed here."""
        q, lf, ds, bo, hm, xf, bf, sh = self._state_args(st, p, True, narrow)
        if out is None:
            out = np.empty((3, p.height, p.width), np.float32)
        fn = self._L.jxlb200_vardct_reconstruct_i16 if narrow else self._L.jxlb200_vardct_reconstruct
        self._check(fn(
            self._h, C.byref(p), _lib.planes([_ptr(a) for a in q]), _lib.planes([_ptr(a) for a in lf]),
            _ptr(ds), _ptr(bo), _ptr(hm), _ptr(xf), _ptr(bf), _ptr(sh), _lib.planes([_ptr(out[c]) for c in range(3)])))
        return out

    def reconstruct_packed(self, p, st, bits=8, linear=True, crop=None, out=None, narrow=False):
        """The whole path ending in PNG-ready samples (jxlb200_vardct_reconstruct_packed): sRGB transfer (when `linear`),
        8/16-bit quantisation and R,G,B interleave on the device; returns uint8 [crop_h, crop_w, 3 * bits/8] (16-bit samples big
        endian, as PNGWriter writes them).  crop = (width, height) of the image inside the padded frame."""
        cw, ch = crop if crop is not None else (p.width, p.height)
        q, lf, ds, bo, hm, xf, bf, sh = self._state_args(st, p, True, narrow)
        nb = 3 * (2 if bits > 8 else 1)
        if out is None:
            out = np.empty((ch, cw, nb), np.uint8)
        self._check(self._L.jxlb200_vardct_reconstruct_packed(
            self._h, C.byref(p), _lib.planes([_ptr(a) for a in q]), 2 if narrow else 4, _lib.planes([_ptr(a) for a in lf]),
            _ptr(ds), _ptr(bo), _ptr(hm), _ptr(xf), _ptr(bf), _ptr(sh), int(bits), 1 if linear else 0, int(cw), int(ch), _ptr(out)))
        return out

    # -- device-pointer calls (bench, multi-GPU): integers are CUdeviceptr values --
    def reconstruct_dev(self, p, q, lf, ds, bo, hm, xf, bf, sh, out):
        self._check(self._L.jxlb200_vardct_reconstruct_dev(self._h, C.byref(p), _lib.planes(q), _lib.planes(lf), ds, bo, hm, xf, bf, sh,
                                                           _lib.planes(out)))

    def reconstruct_batch_dev(self, p, n_frames, q, lf, ds, bo, hm, xf, bf, sh, out):
        """n_frames equally sized frames stacked vertically in every array (p describes ONE frame, height % 64 == 0):
        stage 1 runs once over the stack, stage 2 once per frame."""
        self._check(self._L.jxlb200_vardct_reconstruct_batch_dev(self._h, C.byref(p), int(n_frames), _lib.planes(q), _lib.planes(lf),
                                                                 ds, bo, hm, xf, bf, sh, _lib.planes(out)))

    # -- one frame split by group rows over the GPUs of a box (jxlb200_comm_* / ..._split_dev) --
    @staticmethod
    def comm_unique_id():
        """128 bytes made by rank 0 (ncclGetUniqueId) and handed to every rank's comm_init."""
        buf = (C.c_uint8 * 128)()
        rc = _lib.lib().jxlb200_comm_unique_id(buf)
        if rc:
            raise (NotImplementedError if rc == _lib.E_UNSUPPORTED else RuntimeError)("jxlb200_comm_unique_id: status %d" % rc)
        return bytes(buf)

    def comm_init(self, unique_id, rank, world):
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        self._check(self._L.jxlb200_comm_init(self._h, buf, int(rank), int(world)))

    def comm_destroy(self):
        self._check(self._L.jxlb200_comm_destroy(self._h))

    def reconstruct_split_dev(self, p, slab, q, lf, ds, bo, hm, xf, bf, sh, out):
        """This rank's slab of a frame split by group rows: stage 1, NCCL halo rows (overlapped), stage 2.  Device pointers of
        the slab's own rows only."""
        self._check(self._L.jxlb200_vardct_reconstruct_split_dev(self._h, C.byref(p), C.byref(slab), _lib.planes(q), _lib.planes(lf),
                                                                 ds, bo, hm, xf, bf, sh, _lib.planes(out)))

    def invert_dev(self, p, q, lf, ds, bo, hm, xf, bf, xyb, pitch):
        self._check(self._L.jxlb200_vardct_invert_dev(self._h, C.byref(p), _lib.planes(q), _lib.planes(lf), ds, bo, hm, xf, bf,
                                                      _lib.planes(xyb), int(pitch)))

    def restore_dev(self, p, slab, xyb, pitch, hm, sh, out):
        self._check(self._L.jxlb200_restore_dev(self._h, C.byref(p), C.byref(slab) if slab is not None else None,
                                                _lib.planes(xyb), int(pitch), hm, sh, _lib.planes(out)))

    # -- upsampling (Frame.performUpsampling) --
    def performUpsampling(self, plane, k, weights):
        """One float32 channel h x w -> (h*k) x (w*k); weights float32 [k][k][5][5] (jxlatte_b200.upsampling.up_weights)."""
        a = _c(plane, np.float32)
        if a.ndim != 2:
            raise ValueError("plane must be 2-D")
        wt = _upsampling_weights(weights, k)
        out = np.empty((a.shape[0] * k, a.shape[1] * k), np.float32)
        self._check(self._L.jxlb200_upsample(self._h, _ptr(a), a.shape[0], a.shape[1], int(k), _ptr(wt), _ptr(out)))
        return out

    # -- noise (Frame.initializeNoise + synthesizeNoise) --
    def synthesizeNoise(self, planes, group_dim, seed0, lut, base_corr_x, base_corr_b):
        """X, Y, B planes [3, h, w] -> planes with the frame's noise added."""
        buf = [np.array(planes[c], dtype=np.float32, order="C", copy=True) for c in range(3)]
        lt = _c(lut, np.float32)
        h, w = buf[0].shape
        self._check(self._L.jxlb200_noise(self._h, _lib.planes([_ptr(a) for a in buf]), h, w, int(group_dim), int(seed0),
                                          _ptr(lt), float(base_corr_x), float(base_corr_b)))
        return np.stack(buf)

    # -- splines (Frame.renderSplines) --
    def renderSplines(self, planes, splines, quant_adjust, base_corr_x, base_corr_b):
        """X, Y, B planes [3, h, w] -> planes with the splines drawn.  splines: [{"points": [x0, y0, ...], "coeff": 128 ints}]."""
        buf = [np.array(planes[c], dtype=np.float32, order="C", copy=True) for c in range(3)]
        h, w = buf[0].shape
        npts, pts, cf = _spline_arrays(splines)
        self._check(self._L.jxlb200_splines(self._h, _lib.planes([_ptr(a) for a in buf]), h, w, len(splines), _ptr(npts), _ptr(pts),
                                            _ptr(cf), int(quant_adjust), float(base_corr_x), float(base_corr_b)))
        return np.stack(buf)

    # -- PNG samples (JXLImage.transfer + ImageBuffer.castToInt + PNGWriter interleave) --
    def packSamples(self, channels, depths, n_color, linear, bits):
        """channels: 2-D float32 / int32 arrays of one size -> uint8 [h, w, C * bits/8], big-endian for 16 bit."""
        ch = [np.ascontiguousarray(c if c.dtype == np.float32 else c.astype(np.int32)) for c in channels]
        h, w = ch[0].shape
        n = len(ch)
        ptrs, is_int, dep = _pack_args([c.ctypes.data for c in ch], [c.dtype != np.float32 for c in ch], depths)
        out = np.empty((h, w, n * (2 if bits > 8 else 1)), np.uint8)
        self._check(self._L.jxlb200_pack_samples(self._h, ptrs, _ptr(is_int), _ptr(dep), n, int(n_color), int(bool(linear)), h, w, int(bits), _ptr(out)))
        return out

    # -- blending (JXLCodestreamDecoder.blendAdd / blendMult / blendBlend / blendMulAdd) --
    def blend(self, op, canvas, a, b, fa=None, ra=None):
        """One rectangle of one channel; op = dict(mode, is_int, is_alpha, has_extra, clamp, premult); canvas, a (the Java's
        `frame` argument), b (`ref`), fa / ra (frame / reference alpha) are equally sized 2-D numpy views with contiguous
        rows; canvas is written in place and may alias a or b."""
        def rect(v):
            if v is None:
                return None, 0
            if v.ndim != 2 or v.shape != canvas.shape or (v.shape[1] > 1 and v.strides[1] != v.itemsize) or v.itemsize != 4:
                raise ValueError("blend operands must be equally sized 2-D views of 4-byte samples with contiguous rows")
            return C.c_void_p(v.ctypes.data), v.strides[0] // v.itemsize
        o = _lib.BlendOp(int(op["mode"]), int(op["is_int"]), int(op["is_alpha"]), int(op["has_extra"]), int(op["clamp"]), int(op["premult"]))
        h, w = canvas.shape
        (cp, cpi), (ap, api), (bp, bpi), (fp, fpi), (rp, rpi) = rect(canvas), rect(a), rect(b), rect(fa), rect(ra)
        self._check(self._L.jxlb200_blend(self._h, C.byref(o), h, w, cp, cpi, ap, api, bp, bpi, fp, fpi, rp, rpi))

    def dequantLF(self, lf_quant, extra_precision, scaled_dequant, kx, kb, cfl=True, smooth=True):
        """LFCoefficients (J/frame/vardct/LFCoefficients.java:61-103, 113-179) on the device: quantised LF planes [3, hb, wb] in X, Y, B
        order + extraPrecision per LF group -> the dequantised, smoothed `lf` planes of the reconstruction call."""
        q = [_c(lf_quant[c], np.int32) for c in range(3)]
        hb, wb = q[0].shape
        if any(a.shape != (hb, wb) for a in q):
            raise ValueError("lf_quant planes must share a shape")
        ep = _extra_precision(extra_precision, hb, wb)
        sd = (C.c_float * 3)(*[float(v) for v in scaled_dequant])
        out = np.empty((3, hb, wb), np.float32)
        self._check(self._L.jxlb200_lf_dequant(self._h, hb, wb, sd, C.c_float(float(kx)), C.c_float(float(kb)), 1 if cfl else 0, 1 if smooth else 0,
                                               _lib.planes([_ptr(a) for a in q]), _ptr(ep), _lib.planes([_ptr(out[c]) for c in range(3)])))
        return out

    # -- 1:8 previews (k10_preview.cuh) --
    def lfPreview(self, p, lf_quant, extra_precision, scaled_dequant, kx, kb, smooth, out_h, out_w):
        """A VarDCT frame rendered from its LF image alone (jxlb200_lf_preview): the quantised LF planes X, Y, B (each of its
        state_shapes(p)["lf"] shape) + extraPrecision per LF group -> the frame at 1:8 after p's colour transform, f32[3, out_h, out_w]."""
        q = check_lf_planes(p, [_c(lf_quant[c], np.int32) for c in range(3)])
        sd, ep = _preview_args(scaled_dequant, extra_precision)
        out = np.empty((3, out_h, out_w), np.float32)
        self._check(self._L.jxlb200_lf_preview(self._h, C.byref(p), sd, C.c_float(float(kx)), C.c_float(float(kb)), 1 if smooth else 0,
                                               _lib.planes([_ptr(a) for a in q]), _ptr(ep), ep.size, int(out_h), int(out_w),
                                               _lib.planes([_ptr(out[c]) for c in range(3)])))
        return out

    def areaMean8(self, channels, depths):
        """The 8x8 area mean of equally sized float32 / int32 channels (jxlb200_area_mean8; int32 ones cast by castToFloat(depth) first)
        -> one float32 plane of ceil(h / 8) x ceil(w / 8) per channel."""
        ch = [np.ascontiguousarray(c if c.dtype == np.float32 else c.astype(np.int32)) for c in channels]
        h, w = check_channels(ch)
        ii, dep = _area_args([c.dtype != np.float32 for c in ch], depths)
        out = [np.empty(((h + 7) // 8, (w + 7) // 8), np.float32) for _ in ch]
        self._check(self._L.jxlb200_area_mean8(self._h, len(ch), _lib.planes([_ptr(a) for a in ch]), _ptr(ii), _ptr(dep), h, w,
                                               _lib.planes([_ptr(a) for a in out])))
        return out

    def blend_batch(self, planes, writable, items):
        """A frame's whole compositing in one call (jxlb200_blend_batch).  planes: 2-D C-contiguous 4-byte numpy arrays (written in
        place when writable[i]); items: (op dict, (h, w), [(plane index, y, x) or None] * 5) in the order canvas, `frame`, `ref`,
        frame alpha, reference alpha -- blended on the device in that order, each seeing what the earlier ones wrote."""
        n = len(planes)
        for a in planes:
            if a.ndim != 2 or a.itemsize != 4 or not a.flags["C_CONTIGUOUS"]:
                raise ValueError("blend planes must be 2-D C-contiguous arrays of 4-byte samples")
        ptrs = (C.c_void_p * n)(*[a.ctypes.data for a in planes])
        ph = np.array([a.shape[0] for a in planes], np.int32)
        pw = np.array([a.shape[1] for a in planes], np.int32)
        wr = np.array([1 if w else 0 for w in writable], np.int32)
        arr = _blend_items(items)
        self._check(self._L.jxlb200_blend_batch(self._h, n, ptrs, _ptr(ph), _ptr(pw), _ptr(wr), len(items), C.byref(arr) if len(items) else None))

    # -- device-resident frame loop (jxlatte_b200.decoder.DeviceEngine): integers are CUdeviceptr values; enqueued, not synchronised --
    def lf_dequant_dev(self, hb, wb, scaled_dequant, kx, kb, cfl, smooth, lf_quant, extra_precision, out):
        """jxlb200_lf_dequant_dev: lf_quant / out are three device pointers each; extra_precision a host array (one byte per LF group)."""
        ep = _extra_precision(extra_precision, hb, wb)
        sd = (C.c_float * 3)(*[float(v) for v in scaled_dequant])
        self._check(self._L.jxlb200_lf_dequant_dev(self._h, int(hb), int(wb), sd, C.c_float(float(kx)), C.c_float(float(kb)), 1 if cfl else 0,
                                                   1 if smooth else 0, _lib.planes(lf_quant), _ptr(ep), _lib.planes(out)))

    def lf_preview_dev(self, p, scaled_dequant, kx, kb, smooth, lf_quant, extra_precision, out_h, out_w, out):
        """jxlb200_lf_preview_dev: lf_quant / out are three device pointers each; extra_precision a host array."""
        sd, ep = _preview_args(scaled_dequant, extra_precision)
        self._check(self._L.jxlb200_lf_preview_dev(self._h, C.byref(p), sd, C.c_float(float(kx)), C.c_float(float(kb)), 1 if smooth else 0,
                                                   _lib.planes(lf_quant), _ptr(ep), ep.size, int(out_h), int(out_w), _lib.planes(out)))

    def area_mean8_dev(self, planes, is_int, depths, h, w, out):
        ii, dep = _area_args(is_int, depths)
        self._check(self._L.jxlb200_area_mean8_dev(self._h, len(planes), _lib.planes(planes), _ptr(ii), _ptr(dep), int(h), int(w), _lib.planes(out)))

    def restore_uniform_dev(self, p, epf_sigma_for_modular, planes_in, out):
        self._check(self._L.jxlb200_restore_uniform_dev(self._h, C.byref(p), C.c_float(float(epf_sigma_for_modular)), _lib.planes(planes_in),
                                                        _lib.planes(out)))

    def color_transform_dev(self, p, planes_in, out):
        self._check(self._L.jxlb200_color_transform_dev(self._h, C.byref(p), _lib.planes(planes_in), _lib.planes(out)))

    def upsample_dev(self, plane, h, w, k, weights, out):
        wt = _upsampling_weights(weights, k)
        self._check(self._L.jxlb200_upsample_dev(self._h, plane, int(h), int(w), int(k), _ptr(wt), out))

    def noise_dev(self, planes, h, w, group_dim, seed0, lut, base_corr_x, base_corr_b):
        lt = _c(lut, np.float32)
        self._check(self._L.jxlb200_noise_dev(self._h, _lib.planes(planes), int(h), int(w), int(group_dim), int(seed0), _ptr(lt),
                                              float(base_corr_x), float(base_corr_b)))

    def splines_dev(self, planes, h, w, splines, quant_adjust, base_corr_x, base_corr_b):
        npts, pts, cf = _spline_arrays(splines)
        self._check(self._L.jxlb200_splines_dev(self._h, _lib.planes(planes), int(h), int(w), len(splines), _ptr(npts), _ptr(pts), _ptr(cf),
                                                int(quant_adjust), float(base_corr_x), float(base_corr_b)))

    def blend_batch_dev(self, planes, items):
        """planes: [(device pointer, h, w)] of 4-byte samples, pitch == w; items as for blend_batch.  Blended in place, in order."""
        n = len(planes)
        ptrs = (C.c_void_p * n)(*[int(p) for p, _, _ in planes])
        ph = np.array([h for _, h, _ in planes], np.int32)
        pw = np.array([w for _, _, w in planes], np.int32)
        arr = _blend_items(items)
        self._check(self._L.jxlb200_blend_batch_dev(self._h, n, ptrs, _ptr(ph), _ptr(pw), len(items), C.byref(arr) if len(items) else None))

    def pack_samples_dev(self, planes, is_int, depths, n_color, linear, h, w, bits, layout, out):
        n = len(planes)
        ptrs, ii, dep = _pack_args([int(p) for p in planes], is_int, depths)
        self._check(self._L.jxlb200_pack_samples_dev(self._h, ptrs, _ptr(ii), _ptr(dep), n, int(n_color), int(bool(linear)), int(h), int(w),
                                                     int(bits), int(layout), out))

    def pack_batch_dev(self, items, c, bits, out_h, out_w, out):
        """jxlb200_pack_batch_dev.  items: one (planes, is_int, depths, h, w, pitches, orientation, linear) per image, planes as
        device pointers (0: filled with the maximum sample value), one entry per output channel; out: the device pointer of
        [len(items)][c][out_h][out_w] samples."""
        arr = (_lib.BatchItem * len(items))()
        for it, (planes, is_int, depths, h, w, pitches, orientation, linear) in zip(arr, items):
            for k in range(len(planes)):
                it.plane[k], it.is_int[k], it.depth[k], it.pitch[k] = int(planes[k]) or None, int(bool(is_int[k])), int(depths[k]), int(pitches[k])
            it.h, it.w, it.orientation, it.linear = int(h), int(w), int(orientation), int(bool(linear))
        self._check(self._L.jxlb200_pack_batch_dev(self._h, arr, len(items), int(c), int(bits), int(out_h), int(out_w), out))

    def cast_to_float_dev(self, src, n, scale, out):
        self._check(self._L.jxlb200_cast_to_float_dev(self._h, src, int(n), C.c_float(float(scale)), out))

    def modular_xyb_dev(self, channels, n, lf_dequant, out):
        dq = np.array([np.float32(v) for v in lf_dequant], np.float32)
        self._check(self._L.jxlb200_modular_xyb_dev(self._h, _lib.planes(channels), int(n), _ptr(dq), _lib.planes(out)))

    def modular_rct_dev(self, channels, h, w, rct_type):
        self._check(self._L.jxlb200_modular_rct_dev(self._h, _lib.planes(channels), int(h), int(w), int(rct_type)))

    def modular_palette_dev(self, idx, palette, h, w, num_c, nb_colors, nb_deltas, d_pred, bit_depth, out):
        self._check(self._L.jxlb200_modular_palette_dev(self._h, idx, palette or None, int(h), int(w), int(num_c), int(nb_colors), int(nb_deltas),
                                                        int(d_pred), int(bit_depth), _lib.planes(out)))

    def modular_squeeze_dev(self, avg, res, h_avg, w_avg, h_res, w_res, horizontal, out):
        self._check(self._L.jxlb200_modular_squeeze_dev(self._h, avg, res or None, int(h_avg), int(w_avg), int(h_res), int(w_res),
                                                        1 if horizontal else 0, out))

    # -- Modular --
    def inverseRCT(self, channels, rct_type):
        """ModularStream.applyTransforms RCT branch: three equal-size channels, returns them as the reference leaves
        channels[beginC .. beginC+2] (permutation applied)."""
        v = [np.array(channels[c], dtype=np.int32, order="C", copy=True) for c in range(3)]
        if not (v[0].shape == v[1].shape == v[2].shape):
            raise InvalidBitstreamError("RCT must be performed on three equal size channels")
        h, w = v[0].shape
        self._check(self._L.jxlb200_modular_rct(self._h, _lib.planes([_ptr(a) for a in v]), h, w, int(rct_type)))
        return v

    def inversePalette(self, index_channel, palette, nb_deltas, d_pred, bit_depth):
        """Palette branch: index channel [h,w] + palette [num_c, nb_colors] -> num_c channels."""
        idx = _c(index_channel, np.int32)
        pal = _c(palette, np.int32)
        if pal.ndim != 2:
            raise ValueError("palette must be [num_c, nb_colors]")
        num_c, nb_colors = pal.shape
        h, w = idx.shape
        out = [np.zeros((h, w), np.int32) for _ in range(num_c)]
        self._check(self._L.jxlb200_modular_palette(self._h, _ptr(idx), _ptr(pal) if pal.size else None, h, w, num_c, nb_colors,
                                                    int(nb_deltas), int(d_pred), int(bit_depth),
                                                    _lib.planes([_ptr(a) for a in out])))
        return out

    def inverseHorizontalSqueeze(self, orig, res):
        return self._squeeze(orig, res, 1)

    def inverseVerticalSqueeze(self, orig, res):
        return self._squeeze(orig, res, 0)

    def _squeeze(self, orig, res, horizontal):
        a, r = _c(orig, np.int32), _c(res, np.int32)
        ha, wa = a.shape
        hr, wr = r.shape
        out = np.zeros((ha, wa + wr) if horizontal else (ha + hr, wa), np.int32)
        self._check(self._L.jxlb200_modular_squeeze(self._h, _ptr(a), _ptr(r) if r.size else None, ha, wa, hr, wr, horizontal, _ptr(out)))
        return out


# ---------------------------------------------------------------------------------------------------------------
# ModularStream channel-list bookkeeping (host logic, J/frame/modular/ModularStream.java:66-185 and :224-380)
# ---------------------------------------------------------------------------------------------------------------
RCT, PALETTE, SQUEEZE = 0, 1, 2


def default_squeeze_params(sizes, nb_meta):
    """Default SqueezeParam list when the bitstream gives none (ModularStream.java:110-131).
    sizes: [(h, w)] of the channel list at that point.  Returns [(horizontal, in_place, begin_c, num_c)]."""
    first = nb_meta
    count = len(sizes) - first
    h, w = sizes[0]
    out = []
    if count > 2 and (h, w) == tuple(sizes[first + 1]):
        out.append((True, False, first + 1, 2))
        out.append((False, False, first + 1, 2))
    if h >= w and h > 8:
        out.append((False, True, first, count))
        h = (h + 1) // 2
    while w > 8 or h > 8:
        if w > 8:
            out.append((True, True, first, count))
            w = (w + 1) // 2
        if h > 8:
            out.append((False, True, first, count))
            h = (h + 1) // 2
    return out


def forward_channel_layout(sizes, squeeze_params):
    """Replay of the constructor's squeeze bookkeeping (ModularStream.java:135-168): channel sizes after the forward
    squeeze steps.  sizes: [(h, w)]; returns the new size list."""
    ch = [tuple(s) for s in sizes]
    for (horizontal, in_place, begin, num_c) in squeeze_params:
        end = begin + num_c - 1
        offset = end + 1 if in_place else len(ch)
        for k in range(begin, end + 1):
            h, w = ch[k]
            if horizontal:
                ch[k] = (h, (w + 1) // 2)
                residu = (h, w // 2)
            else:
                ch[k] = ((h + 1) // 2, w)
                residu = (h // 2, w)
            ch.insert(offset + k - begin, residu)
    return ch


class ModularTransforms:
    """ModularStream.applyTransforms over a decoded channel list, every transform running on the GPU.

    transforms: list of dicts in bitstream order (they are undone in reverse, :228):
        {"tr": RCT, "begin_c": b, "rct_type": t}
        {"tr": PALETTE, "begin_c": b, "num_c": n, "nb_colors": k, "nb_deltas": d, "d_pred": p}
        {"tr": SQUEEZE, "sp": [(horizontal, in_place, begin_c, num_c), ...]}   # explicit or default list
    """

    def __init__(self, reconstructor, bit_depth=8):
        self.r = reconstructor
        self.bit_depth = bit_depth

    @staticmethod
    def own(c):
        """The channel list is edited in place: each channel becomes an int32 C-contiguous array of the transforms' own."""
        return np.array(c, dtype=np.int32, order="C")

    def applyTransforms(self, channels, transforms):
        ch = [self.own(c) for c in channels]
        for tr in reversed(transforms):
            if tr["tr"] == SQUEEZE:
                for (horizontal, in_place, begin, num_c) in reversed(tr["sp"]):
                    end = begin + num_c - 1
                    offset = end + 1 if in_place else len(ch) + begin - end - 1
                    for c in range(begin, end + 1):
                        r = offset + c - begin
                        ch[c] = (self.r.inverseHorizontalSqueeze if horizontal else self.r.inverseVerticalSqueeze)(ch[c], ch[r])
                    del ch[offset:offset + end - begin + 1]
            elif tr["tr"] == RCT:
                b = tr["begin_c"]
                ch[b:b + 3] = self.r.inverseRCT(ch[b:b + 3], tr["rct_type"])
            elif tr["tr"] == PALETTE:
                first = tr["begin_c"] + 1
                outs = self.r.inversePalette(ch[first], ch[0][:tr["num_c"], :tr["nb_colors"]], tr["nb_deltas"], tr["d_pred"], self.bit_depth)
                ch[first:first + 1] = outs
                del ch[0]
            else:
                raise InvalidBitstreamError("Illegal Transform %r" % (tr["tr"],))
        return ch
