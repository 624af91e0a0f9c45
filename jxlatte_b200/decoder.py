"""JXLDecoder / JXLImage / PNGWriter mirrors: .jxl bytes -> C++ front end (entropy decoding, headers; libjxlfront.so)
-> CUDA reconstruction (libjxlb200.so) -> image planes.

Mirrors the reference's only public API (J/JXLDecoder.java:17-46, J/JXLImage.java, J/io/PNGWriter.java:61-65,191-212,
J/io/PFMWriter.java:22-49) for the part of the format this build covers:
  * VarDCT frames, 4:4:4, XYB or YCbCr, any TransformType mix, custom or default quant tables, Gaborish, EPF;
  * Modular frames / extra channels: channels decoded on the host, RCT / Palette / Squeeze undone on the GPU;
  * frame blending mode REPLACE onto the canvas (crop offsets honoured).
Everything the frame loop of JXLCodestreamDecoder.decode (:588-626) does beyond that -- upsampling, noise, splines,
patches, the other blend modes, LF frames, chroma subsampling -- raises NotImplementedError (SURVEY.md 8f-2..4).

`engine` is the reconstruction back end.  The default is the CUDA library (jxlatte_b200.host.Reconstructor) on host buffers;
DeviceEngine keeps every buffer of the frame loop on the device and returns the image as CUDA tensors.  There is no CPU fallback
in this module -- the CPU tests inject the oracle explicitly (tests/test_frontend.py).

The frame loop is written once.  Where it creates, copies or casts a buffer it goes through the engine's `arrays` (NumpyArrays
for engines that work on host arrays, the DeviceEngine itself for CUDA tensors), so the same loop runs on either.
"""
import ctypes as C
import os
import struct
import zlib

import numpy as np

from . import frontend, host
from .params import STATE_MAPS, FrameParams, check_channels, check_lf_planes, check_planes, check_state_shapes
from .upsampling import up_weights

ENC_VARDCT, ENC_MODULAR = 0, 1
FLAG_NOISE, FLAG_PATCHES, FLAG_SPLINES, FLAG_USE_LF_FRAME = 1, 2, 16, 32
TF_SRGB, TF_LINEAR = (1 << 24) + 13, (1 << 24) + 8


def locate_view(v):
    """A rectangle view of a channel buffer -> (a 2-D C-contiguous plane it is a window of, y, x), or None when it is not such a
    window (the rectangle then takes the immediate blend call).  numpy collapses view chains onto the owning array, so the plane is
    the owner seen as rows of the view's own row pitch: a [C, H, W] owner becomes one plane of C * H rows."""
    if not isinstance(v, np.ndarray) or v.ndim != 2 or v.itemsize != 4:
        return None
    base = v
    while isinstance(base.base, np.ndarray):
        base = base.base
    if base.itemsize != 4 or not base.flags["C_CONTIGUOUS"] or base.ndim < 1:
        return None
    if v.shape[1] > 1 and v.strides[1] != 4:
        return None
    if v.shape[0] > 1:
        if v.strides[0] <= 0 or v.strides[0] % 4:
            return None
        W = v.strides[0] // 4
    else:
        W = base.shape[-1]
    off = v.ctypes.data - base.ctypes.data
    if off < 0 or off % 4 or W < 1 or base.size % W:
        return None
    y, x = divmod(off // 4, W)
    plane = base.reshape(-1, W)
    if y + v.shape[0] > plane.shape[0] or x + v.shape[1] > W:
        return None
    return plane, y, x


def locate_tensor_view(v):
    """locate_view for torch tensors: a 2-D view with unit column stride -> (the rows of its storage at the view's row pitch, as a
    2-D tensor from storage offset 0; y; x), or None when the view is not such a window.  Slicing keeps the parent's row stride, so
    the pitch is stride(0) and the origin follows from the storage offset."""
    if v.dim() != 2 or v.element_size() != 4:
        return None
    if v.shape[1] > 1 and v.stride(1) != 1:
        return None
    W = v.stride(0)
    if W < 1 or W < v.shape[1]:
        return None
    total = v.untyped_storage().nbytes() // 4
    y, x = divmod(v.storage_offset(), W)
    rows = total // W
    if y + v.shape[0] > rows or x + v.shape[1] > W:
        return None
    return v.as_strided((rows, W), (W, 1), 0), y, x


class NumpyArrays:
    """The buffer operations of the frame loop on host numpy arrays (CudaEngine, the oracle engine)."""

    @staticmethod
    def is_float(a):
        return a.dtype == np.float32

    @staticmethod
    def zeros(shape, like=None):
        return np.zeros(shape, np.float32 if like is None else like.dtype)

    @staticmethod
    def copy(a):
        return a.copy()

    @staticmethod
    def contiguous(a):
        return np.ascontiguousarray(a)

    @staticmethod
    def stack(planes):
        return np.stack(planes)

    @staticmethod
    def upload(a):
        return a

    @staticmethod
    def cast_to_float(a, depth):
        """ImageBuffer.castToFloat: (float)v * (1f / ((1 << depth) - 1))."""
        return a.astype(np.float32) * (np.float32(1.0) / np.float32((1 << depth) - 1))

    @staticmethod
    def modular_xyb(y, x, b, dq):
        """Frame.decodeFrame :429-447 on the Modular channels Y, X, B - Y -> float X, Y, B."""
        dq = [np.float32(v) for v in dq]
        return [dq[0] * x.astype(np.float32), dq[1] * y.astype(np.float32), dq[2] * (y + b).astype(np.float32)]

    @staticmethod
    def orient(a, o):
        """JXLCodestreamDecoder.transposeBuffer (:43-112) for orientation o != 1."""
        if o == 2:
            a = a[:, ::-1]
        elif o == 3:
            a = a[::-1, ::-1]
        elif o == 4:
            a = a[::-1, :]
        elif o == 5:
            a = a.T
        elif o == 6:
            a = a.T[:, ::-1]
        elif o == 7:
            a = a[::-1, ::-1].T
        else:
            a = a.T[::-1, :]
        return np.ascontiguousarray(a)


_NUMPY = NumpyArrays()


def _arrays(engine):
    return getattr(engine, "arrays", None) or _NUMPY


def preview_route(info):
    """How JXLOptions(preview=True) renders a stream, from its headers (a parse with frontend.FLAG_LF_ONLY has them all): "lf" when
    every frame's 1:8 image is its LF image -- VarDCT, type 0 or 3, no LF frame used or present, no patches, splines or noise, no
    upsampling, no extra channels in the image, blend mode REPLACE and an origin on the 8 x 8 grid -- else "full"."""
    if info["extra_channels"]:
        return "full"
    for f in info["frames"]:
        if (f["encoding"] != ENC_VARDCT or f["type"] not in (0, 3) or f["flags"] & (FLAG_USE_LF_FRAME | FLAG_PATCHES | FLAG_SPLINES | FLAG_NOISE)
                or f["upsampling"] != 1 or f["blend_mode"] != 0 or f["x0"] % 8 or f["y0"] % 8):
            return "full"
    return "lf"


def parse_stream(data, preview, threads=None):
    """The front end of a decode: .jxl bytes -> (ParsedImage, preview route or None).  A preview parses up to the LF images
    (frontend.FLAG_LF_ONLY) and, when preview_route() sends the stream to "full", parses it again in full.  threads: OpenMP threads
    of the calling thread's parses (frontend.parse)."""
    def parse(flags):
        return frontend.parse(data, flags, threads=threads) if threads else frontend.parse(data, flags)
    if not preview:
        return parse(0), None
    parsed = parse(frontend.FLAG_LF_ONLY)
    route = preview_route(parsed.info)
    if route == "full":
        parsed.close()
        parsed = parse(0)
    return parsed, route


class JXLOptions:
    """The reference's JXLOptions (J/JXLOptions.java:7-50), the fields that reach the reconstruction path."""
    OUTPUT_DEFAULT, OUTPUT_PNG, OUTPUT_PFM = -1, 0, 1

    def __init__(self, outputFormat=-1, outputDepth=-1, preview=False):
        self.outputFormat = outputFormat    # OUTPUT_PNG: the caller will quantise with PNGWriter; OUTPUT_PFM / default: float samples
        self.outputDepth = outputDepth      # -1: PNGWriter picks 8 for images of up to 8 bits per sample, else 16
        # preview: every displayed image at 1:8, ceil(H / 8) x ceil(W / 8) before orientation, as float32 channels (linear when
        # xyb_encoded).  Streams preview_route() accepts are rendered from the frames' LF images without decoding any HF data; the
        # others are decoded in full and each channel is averaged over 8 x 8 areas.
        self.preview = preview

    def quantises_to_8_bits(self, bits_per_sample):
        """True when the only consumer of the planes is PNGWriter at 8 bits: the tolerance "<= 1e-4 and <= 1 LSB" of the north
        star is then met by the re-associated filter sums too, and the engine may use them (JXLB200_OPT_STAGE2 = 2).  16-bit PNG
        and PFM output keep the bit-exact kernels (profiles/r2_exact_vs_fast.md has the price of each)."""
        if self.outputFormat != self.OUTPUT_PNG:
            return False
        depth = self.outputDepth if self.outputDepth > 0 else (8 if bits_per_sample <= 8 else 16)
        return depth <= 8


class CudaEngine:
    """The product back end: every data-parallel stage on the GPU through the C ABI."""

    def __init__(self, device=0, allow_tolerance_mode=False):
        """allow_tolerance_mode: let JXLOptions(OUTPUT_PNG, 8) select the re-associated stage 2 (JXLB200_OPT_STAGE2 = 2).  OFF by
        default: measured on B200 that kernel (k2_fused) is inside the tolerance but SLOWER than the bit-exact kernels (2.40 ms per
        8K frame with three EPF passes against 1.31 ms for k2_stream and 1.65 ms for k2_exact; 0.58 against 0.55 ms with one pass:
        profiles/r2_exact_vs_fast.md), so there is nothing to buy with the error."""
        from . import host
        self._host = host
        self.rec = host.Reconstructor(device)
        self._qm_default = None
        self._uploaded = None
        self.allow_tolerance_mode = allow_tolerance_mode
        self.tolerance_mode = False         # set per image by JXLDecoder from JXLOptions
        self.batch_blends = True
        self._batch_planes, self._batch_writable, self._batch_items, self._batch_index = [], [], [], {}

    def qm_default(self):
        if self._qm_default is None:        # HFGlobal.defaultParams tables: built once, shared by every frame that uses them
            self._qm_default = self._host.qm_generate()
        return self._qm_default

    def qm_generate(self, prm):
        return self._host.qm_generate(prm)

    def qm_params(self):
        return self._host.qm_default_params()

    def reconstruct(self, p, st):
        if st["qm_weights"] is not self._uploaded:      # same table object as the previous frame: already on the device
            self.rec.setWeights(st["qm_weights"], st["qm_offsets"])
            self._uploaded = st["qm_weights"]
        # the tolerance kernel is faster only with fewer than three EPF passes (profiles/r2_exact_vs_fast.md)
        if not (self.tolerance_mode and self.allow_tolerance_mode and p.epf_iters < 3 and (p.gab or p.epf_iters)):
            return self._reconstruct(p, st)
        from . import _lib
        self.rec.set_option(_lib.OPT_STAGE2, _lib.STAGE2_FUSED)
        try:
            return self._reconstruct(p, st)
        finally:
            self.rec.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)

    def _reconstruct(self, p, st):
        return self.rec.reconstruct(p, st)

    def modular(self, channels, transforms, bit_depth):
        return self._host.ModularTransforms(self.rec, bit_depth).applyTransforms(channels, transforms)

    def color(self, p, planes):
        return self.rec.performColorTransforms(p, planes)

    def restore_modular(self, p, planes, sigma):
        return self.rec.restoreModularFrame(p, planes, sigma)

    def lf_dequant(self, q, ep, scaled_dequant, kx, kb, smooth):
        return self.rec.dequantLF(q, ep, scaled_dequant, kx, kb, cfl=True, smooth=smooth)

    def lf_preview(self, p, q, ep, scaled_dequant, kx, kb, smooth, out_h, out_w):
        return self.rec.lfPreview(p, q, ep, scaled_dequant, kx, kb, smooth, out_h, out_w)

    def area_mean8(self, channels, depths):
        return self.rec.areaMean8(channels, depths)

    # ---- compositing: the blends of a frame are queued and run in ONE device call (jxlb200_blend_batch) ----
    def _locate(self, v):
        loc = locate_view(v)
        if loc is None:
            return None
        plane, y, x = loc
        key = plane.ctypes.data
        if key not in self._batch_index:
            self._batch_index[key] = len(self._batch_planes)
            self._batch_planes.append(plane)
            self._batch_writable.append(False)
        return self._batch_index[key], y, x

    def blend(self, op, canvas, a, b, fa, ra):
        if self.batch_blends:
            refs = [self._locate(v) if v is not None else None for v in (canvas, a, b, fa, ra)]
            if refs[0] is not None and refs[1] is not None and refs[2] is not None and (fa is None or refs[3] is not None) and (ra is None or refs[4] is not None):
                self._batch_writable[refs[0][0]] = True
                self._batch_items.append((dict(op), canvas.shape, refs))
                return
            self.flush_blends()
        self._blend_now(op, canvas, a, b, fa, ra)

    def flush_blends(self):
        """Run the queued rectangles (in order) and bring the written planes back.  Called before anything else touches the
        buffers: a cast, a plain copy, the end of a frame's patches or of its blend."""
        if self._batch_items:
            planes, wr, items = self._batch_planes, self._batch_writable, self._batch_items
            self._batch_planes, self._batch_writable, self._batch_items, self._batch_index = [], [], [], {}
            self.rec.blend_batch(planes, wr, items)
        else:
            self._batch_planes, self._batch_writable, self._batch_index = [], [], {}

    def _blend_now(self, op, canvas, a, b, fa, ra):
        self.rec.blend(op, canvas, a, b, fa, ra)

    def upsample(self, plane, k, weights):
        return self.rec.performUpsampling(plane, k, weights)

    def pack(self, channels, depths, n_color, linear, bits):
        return self.rec.packSamples(channels, depths, n_color, linear, bits)

    def pack_batch(self, items, c, bits, out_h, out_w):
        """DeviceEngine.pack_batch's contract on host arrays -> numpy [len(items), c, out_h, out_w] uint8 / uint16.  The samples of
        each image come from the pack kernel's host form (jxlb200_pack_samples), so both engines agree byte for byte; orientation,
        channel expansion and placement are numpy (NumpyArrays.orient)."""
        maxv = (1 << bits) - 1
        out = np.zeros((len(items), c, out_h, out_w), np.uint16 if bits > 8 else np.uint8)
        for i, (planes, depths, o, linear) in enumerate(items):
            k = sum(p is not None for p in planes)        # the planes present come first: only a missing alpha is filled
            raw = self.pack(planes[:k], depths[:k], min(c, 3), linear, bits)
            samples = raw.view(">u2") if bits > 8 else raw
            for ch in range(c):
                a = samples[:, :, ch] if ch < k else np.full(planes[0].shape, maxv, out.dtype)
                a = NumpyArrays.orient(a, o) if o != 1 else a
                out[i, ch, :a.shape[0], :a.shape[1]] = a
        return out

    def noise(self, planes, group_dim, seed0, lut, base_x, base_b):
        return self.rec.synthesizeNoise(planes, group_dim, seed0, lut, base_x, base_b)

    def splines(self, planes, splines, quant_adjust, base_x, base_b):
        return self.rec.renderSplines(planes, splines, quant_adjust, base_x, base_b)

    def close(self):
        self.rec.close()


class DeviceEngine(CudaEngine):
    """CudaEngine on CUDA tensors: every buffer of the frame loop stays on the device.  The front end's arrays of a frame are
    uploaded once, each stage runs through the library's _dev entry points on torch's current stream of `device`, and nothing
    comes back to the host until the image is: JXLImage.channels / planes are CUDA tensors, to_int / packed run the pack kernel on
    the device.  The decoder synchronises once per displayed image (sync), which is where stream errors of the kernels surface."""

    def __init__(self, device=0, allow_tolerance_mode=False):
        import torch
        self._torch = torch
        super().__init__(device, allow_tolerance_mode)
        self.device = torch.device("cuda", device)
        # the legacy default stream is 0 to torch but "the context's own stream" to jxlb200_set_stream: pass cudaStreamLegacy (1)
        self.stream = torch.cuda.current_stream(self.device)
        self.rec.set_stream(self.stream.cuda_stream or 1)
        self.arrays = self
        self._dtypes = {np.dtype(np.int32): torch.int32, np.dtype(np.float32): torch.float32, np.dtype(np.uint8): torch.uint8}

    def _on_stream(self):
        """The library's kernels and the frame loop's torch work must share one stream; the library is bound to the stream that was
        current when the engine was made.  Decoding under another stream would race with it, so that is an error."""
        if self._torch.cuda.current_stream(self.device) != self.stream:
            raise RuntimeError("DeviceEngine is bound to %r; decode on that stream (torch.cuda.stream(engine.stream))" % (self.stream,))

    def sync(self):
        """jxlb200_sync: wait for the decode's work and raise the first stream error it met (the host path's exception classes)."""
        self._on_stream()
        self.rec.sync()

    # ---- buffer operations of the frame loop (NumpyArrays on tensors) ----
    def is_float(self, a):
        return a.dtype == self._torch.float32

    def zeros(self, shape, like=None):
        self._on_stream()
        return self._torch.zeros(tuple(shape), dtype=self._torch.float32 if like is None else like.dtype, device=self.device)

    def empty(self, shape, dtype=None):
        self._on_stream()
        return self._torch.empty(tuple(shape), dtype=dtype or self._torch.float32, device=self.device)

    def copy(self, a):
        self._on_stream()
        return a.clone(memory_format=self._torch.contiguous_format)

    def contiguous(self, a):
        return a.contiguous()

    def stack(self, planes):
        self._on_stream()
        return self._torch.stack(list(planes))

    def upload(self, a, dtype=None):
        """A front-end (numpy) array -> a contiguous tensor on the device; tensors pass through (made contiguous).  Host arrays are
        copied into pinned memory from torch's caching host allocator (the front end may free its arrays as soon as this returns)
        and sent with a non-blocking copy, so the host runs ahead of the device instead of waiting for each upload."""
        torch = self._torch
        self._on_stream()
        if isinstance(a, torch.Tensor):
            t = a.to(self.device)
        else:
            a = np.ascontiguousarray(a, dtype)
            t = torch.from_numpy(a).pin_memory().to(self.device, non_blocking=True)
        if dtype is not None and t.dtype != self._dtypes[np.dtype(dtype)]:
            raise ValueError("device array has dtype %s, expected %s" % (t.dtype, np.dtype(dtype)))
        return t.contiguous()

    def cast_to_float(self, a, depth):
        a = a.contiguous()
        out = self.empty(a.shape)
        self.rec.cast_to_float_dev(a.data_ptr(), a.numel(), np.float32(1.0) / np.float32((1 << depth) - 1), out.data_ptr())
        return out

    def modular_xyb(self, y, x, b, dq):
        y, x, b = y.contiguous(), x.contiguous(), b.contiguous()
        out = self.empty((3,) + tuple(y.shape))
        self.rec.modular_xyb_dev([y.data_ptr(), x.data_ptr(), b.data_ptr()], y.numel(), dq, [out[c].data_ptr() for c in range(3)])
        return [out[0], out[1], out[2]]

    def orient(self, a, o):
        torch = self._torch
        if o == 2:
            a = torch.flip(a, (1,))
        elif o == 3:
            a = torch.flip(a, (0, 1))
        elif o == 4:
            a = torch.flip(a, (0,))
        elif o == 5:
            a = a.t()
        elif o == 6:
            a = torch.flip(a.t(), (1,))
        elif o == 7:
            a = torch.flip(a, (0, 1)).t()
        else:
            a = torch.flip(a.t(), (0,))
        return a.contiguous()

    # ---- stages ----
    def _reconstruct(self, p, st):
        a = dict(qcoeff=[self.upload(st["qcoeff"][c], np.int32) for c in range(3)], lf=[self.upload(st["lf"][c], np.float32) for c in range(3)])
        a.update((k, self.upload(st[k], dt)) for k, dt in STATE_MAPS)
        check_state_shapes(p, a)
        out = self.empty((3, p.height, p.width))
        self.rec.reconstruct_dev(p, [t.data_ptr() for t in a["qcoeff"]], [t.data_ptr() for t in a["lf"]], *[a[k].data_ptr() for k, _ in STATE_MAPS],
                                 [out[c].data_ptr() for c in range(3)])
        return out

    def lf_dequant(self, q, ep, scaled_dequant, kx, kb, smooth):
        qd = [self.upload(q[c], np.int32) for c in range(3)]
        hb, wb = qd[0].shape
        if any(tuple(a.shape) != (hb, wb) for a in qd):
            raise ValueError("lf_quant planes must share a shape")
        out = self.empty((3, hb, wb))
        self.rec.lf_dequant_dev(hb, wb, scaled_dequant, kx, kb, True, smooth, [a.data_ptr() for a in qd], ep, [out[c].data_ptr() for c in range(3)])
        return out

    def lf_preview(self, p, q, ep, scaled_dequant, kx, kb, smooth, out_h, out_w):
        qd = check_lf_planes(p, [self.upload(q[c], np.int32) for c in range(3)])
        out = self.empty((3, out_h, out_w))
        self.rec.lf_preview_dev(p, scaled_dequant, kx, kb, smooth, [a.data_ptr() for a in qd], ep, out_h, out_w, [out[c].data_ptr() for c in range(3)])
        return out

    def area_mean8(self, channels, depths):
        ch = [c.contiguous() for c in channels]
        h, w = check_channels(ch)
        out = self.empty((len(ch), (h + 7) // 8, (w + 7) // 8))
        self.rec.area_mean8_dev([c.data_ptr() for c in ch], [not self.is_float(c) for c in ch], depths, h, w, [o.data_ptr() for o in out])
        return list(out)

    def modular(self, channels, transforms, bit_depth):
        return _DeviceModularTransforms(_DeviceModularOps(self), bit_depth).applyTransforms([self.upload(c, np.int32) for c in channels], transforms)

    def _planes3(self, p, planes):
        return check_planes(p, [self.upload(planes[c], np.float32) for c in range(3)])

    def color(self, p, planes):
        inp = self._planes3(p, planes)
        out = self.empty((3, p.height, p.width))
        self.rec.color_transform_dev(p, [a.data_ptr() for a in inp], [out[c].data_ptr() for c in range(3)])
        return out

    def restore_modular(self, p, planes, sigma):
        inp = self._planes3(p, planes)
        out = self.empty((3, p.height, p.width))
        self.rec.restore_uniform_dev(p, sigma, [a.data_ptr() for a in inp], [out[c].data_ptr() for c in range(3)])
        return out

    def upsample(self, plane, k, weights):
        a = self.upload(plane, np.float32)
        if a.dim() != 2:
            raise ValueError("plane must be 2-D")
        h, w = a.shape
        out = self.empty((h * k, w * k))
        self.rec.upsample_dev(a.data_ptr(), h, w, k, weights, out.data_ptr())
        return out

    def noise(self, planes, group_dim, seed0, lut, base_x, base_b):
        buf = self.upload(planes, np.float32).clone()       # the argument is left as it is, as CudaEngine.noise does
        h, w = buf.shape[1:]
        self.rec.noise_dev([buf[c].data_ptr() for c in range(3)], h, w, group_dim, seed0, lut, base_x, base_b)
        return buf

    def splines(self, planes, splines, quant_adjust, base_x, base_b):
        buf = self.upload(planes, np.float32).clone()       # the argument is left as it is, as CudaEngine.splines does
        h, w = buf.shape[1:]
        self.rec.splines_dev([buf[c].data_ptr() for c in range(3)], h, w, splines, quant_adjust, base_x, base_b)
        return buf

    def pack(self, channels, depths, n_color, linear, bits, layout=0):
        """layout 0: uint8 [h, w, C * bits/8] PNG bytes (big-endian 16 bit); 1: [C, h, w] uint8 / uint16 samples."""
        torch = self._torch
        self._on_stream()
        ch = [c.contiguous() for c in channels]
        h, w = ch[0].shape
        n = len(ch)
        if layout == 1:
            out = torch.empty((n, h, w), dtype=torch.uint16 if bits > 8 else torch.uint8, device=self.device)
        else:
            out = torch.empty((h, w, n * (2 if bits > 8 else 1)), dtype=torch.uint8, device=self.device)
        self.rec.pack_samples_dev([c.data_ptr() for c in ch], [not self.is_float(c) for c in ch], depths, n_color, linear, h, w, bits, layout,
                                  out.data_ptr())
        return out

    def pack_batch(self, items, c, bits, out_h, out_w):
        """Every image of a batch into one CUDA [len(items), c, out_h, out_w] uint8 / uint16 tensor, in one launch (k11_pack_batch):
        oriented, each sample through to_int's pipeline, at the top-left of its slot, the rest of the slot 0.  items: (planes, depths,
        orientation, linear) per image; planes: c stored-orientation 2-D tensors (repeats allowed), None for a channel filled with the
        maximum sample value; depths: the bit depth of each."""
        torch = self._torch
        self._on_stream()
        out = torch.empty((len(items), c, out_h, out_w), dtype=torch.uint16 if bits > 8 else torch.uint8, device=self.device)
        keep, args = [], []
        for planes, depths, o, linear in items:
            planes = [p if p is None or p.stride(1) == 1 else p.contiguous() for p in planes]
            keep.append(planes)
            h, w = next(p for p in planes if p is not None).shape
            args.append(([0 if p is None else p.data_ptr() for p in planes], [p is not None and not self.is_float(p) for p in planes],
                         [d if p is not None else 0 for p, d in zip(planes, depths)], h, w, [w if p is None else p.stride(0) for p in planes],
                         o, linear))
        self.rec.pack_batch_dev(args, c, bits, out_h, out_w, out.data_ptr())
        return out

    # ---- compositing: the rectangles of a frame are queued and blended in one call on the device planes ----
    def _locate(self, v):
        loc = locate_tensor_view(v)
        if loc is None:
            return None
        plane, y, x = loc
        key = (plane.data_ptr(), plane.shape[1])
        if key not in self._batch_index:
            self._batch_index[key] = len(self._batch_planes)
            self._batch_planes.append(plane)
        return self._batch_index[key], y, x

    def blend(self, op, canvas, a, b, fa, ra):
        refs = [self._locate(v) if v is not None else None for v in (canvas, a, b, fa, ra)]
        if any(r is None and v is not None for r, v in zip(refs, (canvas, a, b, fa, ra))):
            raise ValueError("blend operands must be 2-D windows of device planes with contiguous rows")
        self._batch_items.append((dict(op), tuple(canvas.shape), refs))

    def flush_blends(self):
        planes, items = self._batch_planes, self._batch_items
        self._batch_planes, self._batch_writable, self._batch_items, self._batch_index = [], [], [], {}
        if items:
            self._on_stream()
            self.rec.blend_batch_dev([(pl.data_ptr(), pl.shape[0], pl.shape[1]) for pl in planes], items)


class _DeviceModularOps:
    """ModularStream's inverse transforms on device channels (int32 CUDA tensors) through the _dev entry points."""

    def __init__(self, engine):
        self.e = engine

    def inverseRCT(self, channels, rct_type):
        v = [c.clone(memory_format=self.e._torch.contiguous_format) for c in channels[:3]]
        if not (v[0].shape == v[1].shape == v[2].shape):
            raise host.InvalidBitstreamError("RCT must be performed on three equal size channels")
        h, w = v[0].shape
        self.e.rec.modular_rct_dev([a.data_ptr() for a in v], h, w, rct_type)
        return v

    def inversePalette(self, index_channel, palette, nb_deltas, d_pred, bit_depth):
        idx, pal = index_channel.contiguous(), palette.contiguous()
        num_c, nb_colors = pal.shape
        h, w = idx.shape
        out = [self.e.zeros((h, w), idx) for _ in range(num_c)]       # zero-initialised, as the host form's outputs
        self.e.rec.modular_palette_dev(idx.data_ptr(), pal.data_ptr() if pal.numel() else 0, h, w, num_c, nb_colors, nb_deltas, d_pred,
                                       bit_depth, [a.data_ptr() for a in out])
        return out

    def inverseHorizontalSqueeze(self, orig, res):
        return self._squeeze(orig, res, True)

    def inverseVerticalSqueeze(self, orig, res):
        return self._squeeze(orig, res, False)

    def _squeeze(self, orig, res, horizontal):
        a, r = orig.contiguous(), res.contiguous()
        ha, wa = a.shape
        hr, wr = r.shape
        out = self.e.zeros((ha, wa + wr) if horizontal else (ha + hr, wa), a)
        self.e.rec.modular_squeeze_dev(a.data_ptr(), r.data_ptr() if r.numel() else 0, ha, wa, hr, wr, horizontal, out.data_ptr())
        return out


class _DeviceModularTransforms(host.ModularTransforms):
    """ModularStream.applyTransforms, unchanged, over channels DeviceEngine.modular has already uploaded as int32 tensors."""

    @staticmethod
    def own(c):
        return c            # fresh uploads of the front end's channels: nobody else holds them


def _f32(x):
    return np.float32(x)


def _conversion_matrix(color):
    """ColorManagement.getConversionMatrix(target = the image's tagged primaries / white point, current = sRGB / D65)
    (J/color/ColorManagement.java:150-161).  Identity for sRGB/D65-tagged images, which is every lossy sample here."""
    srgb = [0.639998686, 0.330010138, 0.300003784, 0.600003357, 0.150002046, 0.059997204]
    same_prim = all(abs(a - b) < 1e-6 for a, b in zip(color["prim_xy"], srgb))
    same_wp = abs(color["white_xy"][0] - 0.3127) < 1e-6 and abs(color["white_xy"][1] - 0.3290) < 1e-6
    if same_prim and same_wp:
        return np.eye(3, dtype=np.float32)

    def xyz(xy):
        inv = _f32(1.0) / _f32(xy[1])
        return np.array([_f32(xy[0]) * inv, _f32(1.0), (_f32(1.0) - _f32(xy[0]) - _f32(xy[1])) * inv], np.float32)

    def prim_to_xyz(prim, wp):
        m = np.stack([xyz(prim[0:2]), xyz(prim[2:4]), xyz(prim[4:6])]).T.astype(np.float32)
        s = np.linalg.inv(m.astype(np.float64)).astype(np.float32) @ xyz(wp)
        return (m @ np.diag(s)).astype(np.float32)

    bradford = np.array([[0.8951, 0.2664, -0.1614], [-0.7502, 1.7135, 0.0367], [0.0389, -0.0685, 1.0296]], np.float32)
    wp_t, wp_c = color["white_xy"], [0.3127, 0.3290]
    adapt = np.eye(3, dtype=np.float32)
    if not same_wp:
        lc, lt = bradford @ xyz(wp_c), bradford @ xyz(wp_t)
        adapt = (np.linalg.inv(bradford.astype(np.float64)).astype(np.float32) @ np.diag(lt / lc) @ bradford).astype(np.float32)
    forward = prim_to_xyz(srgb, wp_c)
    reverse = np.linalg.inv(prim_to_xyz(color["prim_xy"], wp_t).astype(np.float64)).astype(np.float32)
    return (reverse @ adapt @ forward).astype(np.float32)


class _Buf:
    """ImageBuffer (J/util/ImageBuffer.java): one channel, int32 or float32, type changed in place by castToFloat so that
    every alias (canvas, reference slots) sees it.  `xp`: the array operations of the engine that owns the buffer."""

    def __init__(self, a, xp=_NUMPY):
        self.a = a
        self.xp = xp

    @property
    def is_int(self):
        return not self.xp.is_float(self.a)

    before_mutation = staticmethod(lambda: None)     # set by the decoder: queued device blends must land before a buffer changes

    def cast_to_float(self, depth):
        if self.is_int:
            _Buf.before_mutation()
            self.a = self.xp.cast_to_float(self.a, depth)


class JXLImage:
    """Decoded image.  `channels`: one 2-D array per channel (colour first, then extra channels): float32 linear light in
    the tagged primaries for XYB images (what PFMWriter writes), float32 in [0, 1] for other lossy images, int32 samples for
    lossless Modular images.  `planes` stacks them (cast to float when the types are mixed).

    With `engine` (a DeviceEngine) the channels are CUDA tensors of the same dtypes and shapes; `planes`, `to_int` and `packed`
    then stay on the device, and write_png / write_pfm copy to the host once."""

    def __init__(self, channels, info, linear, engine=None):
        self.channels = list(channels)
        self.info = info
        self.linear = linear
        self.engine = engine
        self._xp = _arrays(engine)

    @property
    def planes(self):
        if len({c.dtype for c in self.channels}) == 1:
            return self._xp.stack(self.channels)
        return self._xp.stack([self._as_float(i) for i in range(len(self.channels))])

    def _depths(self):
        return [self._depth(i) for i in range(len(self.channels))]

    def _depth(self, i):
        ncol = self.info["color_channels"]
        return self.info["bits_per_sample"] if i < ncol else self.info["extra_channels"][i - ncol]["bits_per_sample"]

    def _as_float(self, i):
        c = self.channels[i]
        if self._xp.is_float(c):
            return c
        return self._xp.cast_to_float(c, self._depth(i))

    @property
    def width(self):
        return self.channels[0].shape[1]

    @property
    def height(self):
        return self.channels[0].shape[0]

    def to_int(self, bits=8):
        """PNGWriter's sample pipeline: TF_SRGB.fromLinearF for linear images, then (int)(v * max + 0.5f) clamped
        (J/color/TransferFunction.java:39-43, J/util/ImageBuffer.java:129-145).  Integer channels whose depth already is
        `bits` are only clamped.  Device images: a CUDA [C, H, W] uint8 / uint16 tensor from the pack kernel."""
        if self.engine is not None:
            return self.engine.pack(self.channels, self._depths(), self.info["color_channels"], self.linear, bits, layout=1)
        if all(c.dtype != np.float32 and self._depth(i) == bits for i, c in enumerate(self.channels)):
            return np.clip(np.stack(self.channels), 0, (1 << bits) - 1).astype(np.uint16 if bits > 8 else np.uint8)
        v = np.stack([self._as_float(i) for i in range(len(self.channels))])
        ncol = self.info["color_channels"]
        if self.linear:
            c = v[:ncol]
            with np.errstate(invalid="ignore"):
                hi = np.float32(1.055) * np.power(c.astype(np.float64), 0.4166666666666667).astype(np.float32) + np.float32(-0.055)
            v = v.copy()
            v[:ncol] = np.where(c < np.float32(0.00313066844250063), c * np.float32(12.92), hi)
        maxv = (1 << bits) - 1
        q = (v * np.float32(maxv) + np.float32(0.5))
        q = np.where(np.isnan(q), 0, q)
        return np.clip(q.astype(np.int64), 0, maxv).astype(np.uint16 if bits > 8 else np.uint8)

    def packed(self, bits=8, engine=None):
        """uint8 [h, w, C * bits/8] in PNG sample order (big-endian for 16 bit).  With an engine the transfer function,
        quantisation and interleave run on the GPU (jxlb200_pack_samples); without one, in numpy (the PNGWriter mirror).  Device
        images: the same bytes as a CUDA uint8 tensor, from the pack kernel on the device planes."""
        if self.engine is not None:
            return self.engine.pack(self.channels, self._depths(), self.info["color_channels"], self.linear, bits)
        if engine is not None:
            return engine.pack(self.channels, self._depths(), self.info["color_channels"], self.linear, bits)
        rows = np.moveaxis(self.to_int(bits), 0, 2)
        if bits > 8:
            rows = rows.astype(">u2")
        return np.ascontiguousarray(rows).view(np.uint8).reshape(rows.shape[0], rows.shape[1], -1)

    def write_png(self, path, bits=8, engine=None):
        rows = self.packed(bits, engine)
        if self.engine is not None:
            rows = rows.cpu().numpy()
        c = len(self.channels)
        ctype = {1: 0, 2: 4, 3: 2, 4: 6}[c]
        raw = b"".join(b"\x00" + rows[y].tobytes() for y in range(rows.shape[0]))

        def chunk(tag, data):
            return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xffffffff)
        with open(path, "wb") as f:
            f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", self.width, self.height, 16 if bits > 8 else 8, ctype, 0, 0, 0)) +
                    chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))

    def write_pfm(self, path):
        v = [self._as_float(i) for i in range(len(self.channels))]
        p = self._xp.stack(v[:3] if len(v) >= 3 else v[:1])
        if self.engine is not None:
            p = p.cpu().numpy()
        with open(path, "wb") as f:
            f.write(("PF\n" if p.shape[0] == 3 else "Pf\n").encode() + ("%d %d\n1.0\n" % (self.width, self.height)).encode())
            f.write(np.moveaxis(p, 0, 2)[::-1].astype(">f4").tobytes())


class JXLDecoder:
    def __init__(self, source, engine=None, options=None):
        self.options = options if options is not None else JXLOptions()
        if isinstance(source, (bytes, bytearray, memoryview)):
            self.data = bytes(source)
        elif isinstance(source, str):
            with open(source, "rb") as f:
                self.data = f.read()
        else:
            self.data = source.read()
        self._own = engine is None
        self.engine = engine
        self.timings = {}
        self.preview_route = None           # JXLOptions(preview=True): "lf" or "full" (preview_route()) once the stream is parsed
        self._images = None
        self._next = None
        self._buffered = False
        self._parsed = None                 # _from_parsed: the stream, already through the front end
        self._batch = False

    @classmethod
    def _from_parsed(cls, parsed, route, engine, options):
        """decode_batch's decoder: `parsed` (and, with JXLOptions(preview=True), its preview `route`) came from parse_stream.  Its
        images are left in stored orientation (info["orientation"] still to apply) and are not synchronised: the batch's pack
        kernel orients them, and the batch synchronises once at its end."""
        d = cls(b"", engine, options)
        d._parsed, d.preview_route, d._batch = parsed, route, True
        return d

    def close(self):
        if self._own and self.engine is not None:
            self.engine.close()
            self.engine = None

    @property
    def _xp(self):
        return _arrays(self.engine)

    def _buf(self, a):
        return _Buf(a, self._xp)

    # ---- frame-level pieces ----
    def frame_params(self, info, f):
        p = FrameParams()
        p.width, p.height = f["padded_width"], f["padded_height"]
        p.global_scale = f["global_scale"]
        p.xqm_scale, p.bqm_scale = f["xqm_scale"], f["bqm_scale"]
        p.quant_bias[:] = info["quant_bias"]
        p.quant_bias_numerator = info["quant_bias_numerator"]
        p.color_factor = f["color_factor"]
        p.base_corr_x, p.base_corr_b = f["base_corr_x"], f["base_corr_b"]
        p.shift_x[:] = f["shift_x"]
        p.shift_y[:] = f["shift_y"]
        p.gab = 1 if f["gab"] else 0
        p.gab_w1[:] = f["gab_w1"]
        p.gab_w2[:] = f["gab_w2"]
        p.epf_iters = f["epf_iters"]
        p.epf_sharp_lut[:] = f["epf_sharp_lut"]
        p.epf_channel_scale[:] = f["epf_channel_scale"]
        p.epf_pass0_sigma_scale = f["epf_pass0_sigma_scale"]
        p.epf_pass2_sigma_scale = f["epf_pass2_sigma_scale"]
        p.epf_border_sad_mul = f["epf_border_sad_mul"]
        p.color_mode = 1 if info["xyb_encoded"] else (2 if f["do_ycbcr"] else 0)
        m = (_conversion_matrix(info["color"]) @ np.array(info["opsin_inverse"], np.float32).reshape(3, 3)).astype(np.float32)
        p.opsin_matrix[:] = [float(x) for x in m.reshape(-1)]
        p.opsin_bias[:] = info["opsin_bias"]
        p.intensity_target = info["intensity_target"]
        return p

    def quant_tables(self, parsed, k, f):
        if f["quant_all_default"]:
            return self.engine.qm_default()
        prm = self.engine.qm_params()          # library defaults, overwritten where the stream codes its own
        keep = []
        for i, q in enumerate(f["quant_params"]):
            if q["mode"] == 0:
                continue
            prm[i].mode, prm[i].n_dct, prm[i].n_param, prm[i].n_4x4 = q["mode"], q["n_dct"], q["n_param"], q["n_4x4"]
            prm[i].denominator = q["denominator"]
            for c in range(3):
                prm[i].dct_param[c][:] = q["dct_param"][17 * c:17 * c + 17]
                prm[i].param[c][:] = q["param"][9 * c:9 * c + 9]
                prm[i].params4x4[c][:] = q["params4x4"][17 * c:17 * c + 17]
                if q["mode"] == 7:
                    raw = np.ascontiguousarray(parsed.array(k, "qraw", 3 * i + c), np.float32)
                    keep.append(raw)
                    prm[i].raw[c] = raw.ctypes.data_as(C.POINTER(C.c_float))
        out = self.engine.qm_generate(prm)
        del keep
        return out

    # ---- one frame: Frame.decodeFrame (+ the colour transform when nothing has to happen in between) ----
    def decode_frame(self, parsed, k, lf_store=None):
        """-> (list of _Buf of frame size: colour channels then extra channels, colour transform still pending?, params)."""
        info, f = parsed.info, parsed.frames[k]
        xp, buf = self._xp, self._buf
        h, w = f["height"], f["width"]
        bits = info["bits_per_sample"]
        mod = None
        if f["modular"]["channels"]:
            tr = [dict(tr=t["tr"], begin_c=t["begin_c"], rct_type=t["rct_type"], num_c=t["num_c"], nb_colors=t["nb_colors"],
                       nb_deltas=t["nb_deltas"], d_pred=t["d_pred"], sp=[(bool(s[0]), bool(s[1]), s[2], s[3]) for s in t["sp"]])
                  for t in f["modular"]["transforms"]]
            mod = self.engine.modular(parsed.modular_channels(k), tr, bits)
        pending, p = False, None
        if f["encoding"] == ENC_VARDCT:
            st = parsed.vardct_state(k, copy=False)
            st["qm_weights"], st["qm_offsets"] = self.quant_tables(parsed, k, f)
            p = self.frame_params(info, f)
            if f["flags"] & FLAG_USE_LF_FRAME:
                # LFCoefficients.java:39-52: dequantLFCoeff is cut out of the LF frame stored for this level
                src = lf_store[f["lf_level"]] if lf_store else None
                if src is None:
                    raise frontend.InvalidBitstreamError("LF Level too large")
                bh, bw = f["padded_height"] // 8, f["padded_width"] // 8
                lf = xp.zeros((3, bh, bw))
                for c in range(3):
                    src[c].cast_to_float(info["bits_per_sample"])
                    a = src[c].a[:bh, :bw]
                    if a.shape != (bh, bw):
                        raise frontend.InvalidBitstreamError("LF frame smaller than the frame that uses it")
                    lf[c] = a
                st["lf"] = lf
            else:
                # LFCoefficients' dequantisation + LF chroma-from-luma + adaptive smoothing on the device (jxlb200_lf_dequant) from the
                # quantised LF the front end decoded; the front end's own host result (the same arithmetic in C++) is what the oracle
                # engine keeps using, so the whole-file parity tests hold the two to each other bit for bit
                lfq = parsed.lf_quantised(k) if hasattr(self.engine, "lf_dequant") and hasattr(parsed, "lf_quantised") else None
                if lfq is not None:
                    st["lf"] = self.engine.lf_dequant(*lfq)
            if f["type"] == 1:
                p.color_mode = 0                      # LF frames are kept as they leave Frame.decodeFrame (no colour transform)
            # patches and saveBeforeCT act on the planes BEFORE the colour transform (JXLCodestreamDecoder.java:611-616)
            upsampled = f["upsampling"] != 1 or any(u != 1 for u in f["ec_upsampling"])
            pending = p.color_mode != 0 and (bool(f["flags"] & (FLAG_PATCHES | FLAG_SPLINES | FLAG_NOISE)) or f["save_before_ct"] or upsampled)
            if pending:
                q = p.copy()
                q.color_mode = 0
                rec = self.engine.reconstruct(q, st)
            else:
                rec = self.engine.reconstruct(p, st)
            bufs = [buf(xp.contiguous(rec[c][:h, :w])) for c in range(3)]
            first = 0
        else:
            if f["do_ycbcr"]:
                raise NotImplementedError("YCbCr Modular frames")
            if info["xyb_encoded"]:
                # lossy Modular: channels are Y, X, B - Y in integers; Frame.decodeFrame :429-447 scales them by LFGlobal.lfDequant
                # (X, Y, B order) into float XYB planes, which then take the same colour transform as VarDCT frames
                y, x, b = (xp.contiguous(mod[c][:h, :w]) for c in range(3))
                bufs = [buf(xp.contiguous(pl)) for pl in xp.modular_xyb(y, x, b, f["lf_dequant"])]
                p = self.frame_params(info, dict(f, padded_width=-(-w // 8) * 8, padded_height=-(-h // 8) * 8, global_scale=1))
                pending = True
                first = 3
            else:
                ncol = info["color_channels"]
                bufs = [buf(xp.contiguous(mod[c][:h, :w])) for c in range(ncol)]          # int32 samples (Frame.java:452-455)
                first = ncol
            if f["gab"] or f["epf_iters"] > 0:
                bufs = self._restore_modular(info, f, bufs, first, h, w)
        for e in range(len(info["extra_channels"])):
            bufs.append(buf(xp.contiguous(mod[first + e][:h, :w])))
        return bufs, pending, p

    def _restore_modular(self, info, f, bufs, ncol, h, w):
        """Frame.decodeFrame :457-461 on a Modular-encoded frame: Gaborish and the edge-preserving filter cast the colour buffers
        to float (castToFloat(bitsPerSample)) and run at the frame's own size with ONE sigma, 1f / epfSigmaForModular
        (Frame.java:573-575, 604-607).  A one-colour frame filters channel 0 with the three distance terms all taken on that
        channel (`colors == 1 ? 0 : c`, :642, 661): three copies of the plane through the same kernels, channel 0 kept."""
        for c in range(ncol):
            bufs[c].cast_to_float(info["bits_per_sample"])
        p = self.frame_params(info, dict(f, padded_width=w, padded_height=h, global_scale=1))
        p.color_mode = 0
        if ncol == 1:
            for c in (1, 2):
                p.gab_w1[c], p.gab_w2[c] = p.gab_w1[0], p.gab_w2[0]
            planes = [bufs[0].a, bufs[0].a, bufs[0].a]
        else:
            planes = [bufs[c].a for c in range(3)]
        out = self.engine.restore_modular(p, planes, f["epf_sigma_for_modular"])
        for c in range(ncol):
            bufs[c] = self._buf(self._xp.contiguous(out[c]))
        return bufs

    # ---- JXLCodestreamDecoder.blendBuffers (:415-497) ----
    def _blend_buffers(self, info, canvas, frame_bufs, ref_bufs, patch_start, frame_offset, ref_offset, size, idx, frame_colors, binfo, patch):
        colors = info["color_channels"]
        extras = info["extra_channels"]
        frame_buf = frame_bufs[(1 if idx == 0 else idx + 2) if colors != frame_colors else idx]
        ex = idx - colors
        is_extra, has_extra = ex >= 0, len(extras) > 0
        is_alpha = is_extra and extras[ex]["type"] == 0
        mode, alpha_ch, clamp = binfo
        alpha_info = extras[alpha_ch] if has_extra else None
        depth = extras[ex]["bits_per_sample"] if is_extra else info["bits_per_sample"]
        premult = bool(has_extra and alpha_info["alpha_associated"])
        h, w = size

        def rect(buf, off):
            v = buf.a[off[0]:off[0] + h, off[1]:off[1] + w]
            if off[0] < 0 or off[1] < 0 or v.shape != (h, w):
                raise frontend.InvalidBitstreamError("blend rectangle outside its buffer")
            return v
        if canvas.is_int != frame_buf.is_int:
            frame_buf.cast_to_float(depth)
            canvas.cast_to_float(depth)
        if mode == 0 or (ref_bufs is None and mode == 1):
            self._flush_blends()
            rect(canvas, patch_start)[...] = rect(frame_buf, frame_offset)
            return
        if ref_bufs is None:
            raise frontend.InvalidBitstreamError("blending against a reference frame that was never stored")
        if ref_bufs[idx] is None:
            ref_bufs[idx] = self._buf(self._xp.zeros(canvas.a.shape, canvas.a))
        ref_buf = ref_bufs[idx]
        ref_alpha = ref_bufs[colors + alpha_ch] if has_extra else None
        frame_alpha = frame_bufs[frame_colors + alpha_ch] if has_extra else None
        if has_extra and mode in (2, 3):
            adepth = alpha_info["bits_per_sample"]
            if mode == 2:
                if ref_alpha is None:
                    ref_alpha = self._buf(self._xp.zeros(canvas.a.shape))
                    ref_bufs[colors + alpha_ch] = ref_alpha
                ref_alpha.cast_to_float(adepth)
            frame_alpha.cast_to_float(adepth)
        should_cast = mode == 4 or (mode == 2 and has_extra) or (mode == 3 and has_extra and not is_alpha)
        if should_cast or ref_buf.is_int != frame_buf.is_int:
            frame_buf.cast_to_float(depth)
            canvas.cast_to_float(depth)
            ref_buf.cast_to_float(depth)
        below = False
        if patch:
            if mode == 5:
                mode, below = 2, True
            elif mode == 6:
                mode = 3
            elif mode == 7:
                mode, below = 3, True
            else:
                mode -= 1
        old_buf, new_buf = (ref_buf, frame_buf) if below else (frame_buf, ref_buf)     # passed as the Java's `frame`, `ref`
        if mode == 3 and has_extra and is_alpha:
            self._flush_blends()
            rect(canvas, patch_start)[...] = rect(new_buf, frame_offset)                # copyToCanvas(..., ref), :389-391
            return
        if mode < 1 or mode > 4:
            raise frontend.InvalidBitstreamError("Illegal blend mode")
        eff = 1 if (mode in (2, 3) and not has_extra) else mode
        need_fa = (eff == 2 and not is_alpha) or eff == 3
        need_ra = eff == 2 and not is_alpha
        op = dict(mode=mode, is_int=int(canvas.is_int), is_alpha=int(is_alpha), has_extra=int(has_extra), clamp=int(clamp), premult=int(premult))
        if eff == 1 and not (canvas.is_int == old_buf.is_int == new_buf.is_int):
            raise frontend.InvalidBitstreamError("blendAdd over buffers of different types")
        self.engine.blend(op, rect(canvas, patch_start), rect(old_buf, frame_offset), rect(new_buf, ref_offset),
                          rect(frame_alpha, frame_offset) if need_fa else None, rect(ref_alpha, ref_offset) if need_ra else None)

    def _flush_blends(self):
        fl = getattr(self.engine, "flush_blends", None)
        if fl is not None:
            fl()

    # ---- JXLCodestreamDecoder.computePatches (:212-254) ----
    def _compute_patches(self, info, f, frame_bufs, frame_colors, reference):
        try:
            self._compute_patches_queued(info, f, frame_bufs, frame_colors, reference)
        finally:
            self._flush_blends()

    def _compute_patches_queued(self, info, f, frame_bufs, frame_colors, reference):
        colors, nextra = info["color_channels"], len(info["extra_channels"])
        for patch in f["patches"]:
            if patch["ref"] > 3:
                raise frontend.InvalidBitstreamError("Patch out of range")
            ref = reference[patch["ref"]]
            if ref is None:
                continue
            if patch["y0"] + patch["h"] > ref[0].a.shape[0] or patch["x0"] + patch["w"] > ref[0].a.shape[1]:
                raise frontend.InvalidBitstreamError("Patch too large")
            npos = len(patch["pos"]) // 2
            for j in range(npos):
                x0, y0 = patch["pos"][2 * j], patch["pos"][2 * j + 1]
                if y0 < 0 or x0 < 0 or patch["h"] + y0 > f["height"] or patch["w"] + x0 > f["width"]:
                    raise frontend.InvalidBitstreamError("Patch size out of bounds")
                for d in range(colors + nextra):
                    c = 0 if d < colors else d - colors + 1
                    b = patch["blend"][3 * (j * (nextra + 1) + c):3 * (j * (nextra + 1) + c) + 3]
                    if b[0] == 0:
                        continue
                    self._blend_buffers(info, frame_bufs[d], frame_bufs, ref, (y0, x0), (y0, x0), (patch["y0"], patch["x0"]),
                                        (patch["h"], patch["w"]), d, frame_colors, (b[0], b[1], bool(b[2])), True)

    def decode(self):
        """JXLDecoder.decode(): the next displayed image -- frames are composed until one has a duration or is the last
        (JXLCodestreamDecoder.java:588-626: `while (!header.isLast && header.duration == 0)`); None once the stream is
        exhausted (atEnd()).  A still image yields one JXLImage; an animation one per displayed frame."""
        self._advance()
        self._buffered = False
        return self._next

    def atEnd(self):
        """JXLDecoder.atEnd(): no further image in the stream."""
        self._advance()
        return self._next is None

    def _advance(self):
        if self._images is None:
            self._images = self._compose()
        if not self._buffered:
            self._next = next(self._images, None)
            self._buffered = True

    def _compose(self):
        """Generator over the displayed images: JXLCodestreamDecoder.decode's frame loop for the features this build renders."""
        import time
        if self._parsed is None:
            t0 = time.perf_counter()
            parsed, self.preview_route = parse_stream(self.data, self.options.preview)
            self.timings["front_end_s"] = time.perf_counter() - t0
        else:
            parsed, self._parsed = self._parsed, None
        if self.engine is None:
            self.engine = CudaEngine()
        if self.preview_route == "lf":
            yield from self._compose_lf(parsed)
            return
        info = parsed.info
        xp, buf = self._xp, self._buf
        sync = None if self._batch else getattr(self.engine, "sync", None)
        _Buf.before_mutation = staticmethod(self._flush_blends)
        if hasattr(self.engine, "tolerance_mode"):
            self.engine.tolerance_mode = self.options.quantises_to_8_bits(info["bits_per_sample"])
        colors, nextra = info["color_channels"], len(info["extra_channels"])
        canvas = None                      # list of _Buf
        reference = [None, None, None, None]
        linear = bool(info["xyb_encoded"])
        t1 = time.perf_counter()
        visible_frames = invisible_frames = 0
        lf_store = [None] * 5                       # JXLCodestreamDecoder.lfBuffer
        for k, f in enumerate(parsed.frames):
            bufs, pending, p = self.decode_frame(parsed, k, lf_store)
            if f["lf_level"] > 0:
                lf_store[f["lf_level"] - 1] = bufs
            if f["type"] == 1:
                continue
            frame_colors = 3 if (info["xyb_encoded"] or f["encoding"] == ENC_VARDCT) else colors
            save = (f["save_as_reference"] != 0 or f["duration"] == 0) and not f["is_last"] and f["type"] != 1
            if f["type"] in (0, 3) and (f["duration"] != 0 or f["is_last"]):          # Frame.isVisible
                visible_frames, invisible_frames = visible_frames + 1, 0
            else:
                invisible_frames += 1
            # Frame.upsample (:725-737): every channel by its own factor, the frame rectangle by the colour factor
            fh, fw, fy0, fx0 = f["height"], f["width"], f["y0"], f["x0"]
            ups = f["upsampling"]
            for c, b in enumerate(bufs):
                kk = ups if c < frame_colors else f["ec_upsampling"][c - frame_colors]
                if kk > 1:
                    b.cast_to_float(info["bits_per_sample"] if c < frame_colors else info["extra_channels"][c - frame_colors]["bits_per_sample"])
                    b.a = self.engine.upsample(b.a, kk, up_weights(kk, info["up%d" % kk]))
            fh, fw, fy0, fx0 = fh * ups, fw * ups, fy0 * ups, fx0 * ups
            fr = dict(f, height=fh, width=fw, y0=fy0, x0=fx0)
            has_noise = bool(f["flags"] & FLAG_NOISE)
            if save and f["save_before_ct"]:
                reference[f["save_as_reference"]] = [buf(xp.copy(b.a)) for b in bufs]
            self._compute_patches(info, fr, bufs, frame_colors, reference)
            if f["flags"] & FLAG_SPLINES and f["splines"]:
                for c in range(3):
                    bufs[c].cast_to_float(info["bits_per_sample"])
                xyb = self.engine.splines(xp.stack([bufs[c].a for c in range(3)]), f["splines"], f["spline_quant_adjust"], f["base_corr_x"], f["base_corr_b"])
                for c in range(3):
                    bufs[c].a = xp.contiguous(xyb[c])
            if has_noise:
                for c in range(3):
                    bufs[c].cast_to_float(info["bits_per_sample"])
                seed0 = (visible_frames << 32) | invisible_frames
                xyb = self.engine.noise(xp.stack([bufs[c].a for c in range(3)]), f["group_dim"], seed0, f["noise"], f["base_corr_x"], f["base_corr_b"])
                for c in range(3):
                    bufs[c].a = xp.contiguous(xyb[c])
            if pending:
                hh, ww = bufs[0].a.shape
                ph, pw = -(-hh // 8) * 8, -(-ww // 8) * 8          # the ABI takes padded planes; the transform is per pixel
                q = p.copy()
                q.width, q.height = pw, ph
                xyb = xp.zeros((3, ph, pw))
                for c in range(3):
                    xyb[c, :hh, :ww] = bufs[c].a
                rgb = self.engine.color(q, xyb)
                for c in range(3):
                    bufs[c] = buf(xp.contiguous(rgb[c, :hh, :ww]))
            adopt = False
            if canvas is None:
                # The usual still image: ONE VarDCT frame that covers the image and REPLACEs.  copyToCanvas would copy every
                # sample of it into a zeroed canvas (page faults included: 2 ms per megapixel and channel); the planes are
                # freshly made numpy arrays nobody else holds, so they become the canvas.
                adopt = (f["type"] in (0, 3) and f["encoding"] == ENC_VARDCT and nextra == 0 and colors == frame_colors == len(bufs)
                         and (fy0, fx0) == (0, 0) and all(b.a.shape == (info["height"], info["width"]) and not b.is_int for b in bufs)
                         and (f["blend_mode"] == 0 or (f["blend_mode"] == 1 and reference[f["blend_source"]] is None)))
                if adopt:
                    canvas = list(bufs)
                else:
                    canvas = [buf(xp.zeros((info["height"], info["width"]), bufs[0].a)) for _ in range(colors + nextra)]
            if f["type"] in (0, 3) and not adopt:
                aliased = any(reference[i] is canvas and i != f["save_as_reference"] for i in range(4))
                if aliased:
                    canvas = [buf(xp.copy(b.a)) for b in canvas]
                # blendFrame (:499-523)
                ih, iw = info["height"], info["width"]
                ps = (min(max(fy0, 0), ih), min(max(fx0, 0), iw))
                fo = (ps[0] - fy0, ps[1] - fx0)
                size = (min(fy0 + fh, ih) - ps[0], min(fx0 + fw, iw) - ps[1])
                if size[0] > 0 and size[1] > 0:
                    for c in range(len(canvas)):
                        if c >= colors:
                            m, a, cl, src = f["ec_blending"][c - colors]
                        else:
                            m, a, cl, src = f["blend_mode"], f["blend_alpha"], f["blend_clamp"], f["blend_source"]
                        self._blend_buffers(info, canvas[c], bufs, reference[src], ps, fo, ps, size, c, frame_colors, (m, a, bool(cl)), False)
                    self._flush_blends()
            if save and not f["save_before_ct"]:
                reference[f["save_as_reference"]] = canvas
            if f["is_last"] or f["duration"] != 0:
                if sync is None:
                    self.timings["reconstruct_s"] = time.perf_counter() - t1
                shown, copy = canvas, not f["is_last"]
                if self.options.preview:
                    shown, copy = self._area_mean8(canvas, info), False
                img = self._finish(shown, info, linear, copy=copy, xp=xp, engine=self.engine if xp is not _NUMPY else None, orient=not self._batch)
                if sync is not None:
                    sync()                  # device engines: the image is complete, and stream errors surface here
                    self.timings["reconstruct_s"] = time.perf_counter() - t1
                yield img
                t1 = time.perf_counter()
        parsed.close()

    def _area_mean8(self, canvas, info):
        """The preview of a composed canvas: each channel's 8 x 8 area means (float32; int32 channels cast by their bit depth first)."""
        depths = [info["bits_per_sample"]] * info["color_channels"] + [e["bits_per_sample"] for e in info["extra_channels"]]
        return [self._buf(a) for a in self.engine.area_mean8([b.a for b in canvas], depths[:len(canvas)])]

    def _compose_lf(self, parsed):
        """The displayed images of a stream preview_route() sends to "lf", at 1:8: each frame rendered from its LF image by the engine's
        lf_preview (one kernel), REPLACEd into a ceil(H / 8) x ceil(W / 8) canvas at (y0 / 8, x0 / 8) with blendFrame's crop clipping,
        and shown when it is the last or has a duration, as _compose shows frames."""
        import time
        info, xp, buf = parsed.info, self._xp, self._buf
        sync = None if self._batch else getattr(self.engine, "sync", None)
        colors = info["color_channels"]
        ih, iw = -(-info["height"] // 8), -(-info["width"] // 8)
        canvas = None
        t1 = time.perf_counter()
        for k, f in enumerate(parsed.frames):
            fh, fw, fy0, fx0 = -(-f["height"] // 8), -(-f["width"] // 8), f["y0"] // 8, f["x0"] // 8
            q, ep, sd, kx, kb, smooth = parsed.lf_state(k)
            planes = self.engine.lf_preview(self.frame_params(info, f), q, ep, sd, kx, kb, smooth, fh, fw)
            chans = [planes[1]] if colors == 1 else [planes[c] for c in range(3)]      # a grey image shows Y, as blendBuffers picks it
            if canvas is None and (fy0, fx0, fh, fw) == (0, 0, ih, iw):
                canvas = chans                          # fresh planes nobody else holds
            else:
                if canvas is None:
                    canvas = [xp.zeros((ih, iw)) for _ in range(colors)]
                ps = (min(max(fy0, 0), ih), min(max(fx0, 0), iw))
                fo = (ps[0] - fy0, ps[1] - fx0)
                size = (min(fy0 + fh, ih) - ps[0], min(fx0 + fw, iw) - ps[1])
                if size[0] > 0 and size[1] > 0:
                    for c in range(colors):
                        canvas[c][ps[0]:ps[0] + size[0], ps[1]:ps[1] + size[1]] = chans[c][fo[0]:fo[0] + size[0], fo[1]:fo[1] + size[1]]
            if f["is_last"] or f["duration"] != 0:
                if sync is None:
                    self.timings["reconstruct_s"] = time.perf_counter() - t1
                img = self._finish([buf(a) for a in canvas], info, bool(info["xyb_encoded"]), copy=not f["is_last"], xp=xp,
                                   engine=self.engine if xp is not _NUMPY else None, orient=not self._batch)
                if sync is not None:
                    sync()
                    self.timings["reconstruct_s"] = time.perf_counter() - t1
                yield img
                t1 = time.perf_counter()
        parsed.close()

    @staticmethod
    def _finish(canvas, info, linear, copy, xp=_NUMPY, engine=None, orient=True):
        o = info["orientation"] if orient else 1
        out = []
        for b in canvas:
            a = xp.copy(b.a) if copy else b.a
            if o != 1:                    # JXLCodestreamDecoder.transposeBuffer (:43-112)
                a = xp.orient(a, o)
            out.append(a)
        return JXLImage(out, info, linear, engine=engine)


# ---- batch decode ----
BATCH_MODES = {"rgb": 3, "rgba": 4, "grey": 1}


class BatchResult:
    """decode_batch's result.  images: [N, C, H, W] uint8 / uint16 (a CUDA tensor from DeviceEngine, numpy from CudaEngine);
    sizes: [N, 2] int64 (h, w) of each image as displayed, after orientation (a CPU tensor, or numpy); routes: each file's preview
    route ("lf" / "full") with JXLOptions(preview=True), else None for each; timings: parse_s (front-end time summed over files),
    parse_wall_s (first parse start to last parse end), device_wall_s (first composition start to the end of the batch's
    synchronise), total_s (the whole call)."""

    def __init__(self, images, sizes, routes, timings):
        self.images, self.sizes, self.routes, self.timings = images, sizes, routes, timings


def _source_name(src):
    if isinstance(src, (str, os.PathLike)):
        return os.fspath(src)
    if isinstance(src, (bytes, bytearray, memoryview)):
        return "<%d bytes>" % len(src)
    return str(getattr(src, "name", type(src).__name__))


def _read_source(src):
    if isinstance(src, (str, os.PathLike)):
        with open(src, "rb") as f:
            return f.read()
    return bytes(src)


def _attributed(e, i, name):
    """e, re-raised as its own type with the source it came from in front of its message."""
    try:
        return type(e)("source %d (%s): %s" % (i, name, e))
    except Exception:
        return e


def _slot_channels(info, mode):
    """The image channel each output channel shows, None for one filled with the maximum sample value.  A grey image is
    replicated into R, G and B; "rgba" takes the first alpha channel (a missing one is filled); other extra channels are dropped."""
    ncol = info["color_channels"]
    if mode == "grey":
        if ncol != 1:
            raise ValueError("mode 'grey' needs a grey image; this one has %d colour channels" % ncol)
        return [0]
    slots = [0, 0, 0] if ncol == 1 else [0, 1, 2]
    if mode == "rgba":
        slots.append(next((ncol + k for k, e in enumerate(info["extra_channels"]) if e["type"] == 0), None))
    return slots


def _compose_first(parsed, route, engine, options):
    """The first displayed image of a parsed stream, composed on `engine`, in stored orientation and not synchronised."""
    d = JXLDecoder._from_parsed(parsed, route, engine, options)
    img = d.decode()
    d._images.close()                   # later frames of an animation are not decoded
    if img is None:
        raise frontend.InvalidBitstreamError("the stream has no displayed image")
    return img


def decode_batch(sources, engine, *, bits=8, mode="rgb", size=None, workers=None, options=None):
    """Decode many JPEG XL files into one [N, C, H, W] batch.

    sources: paths, bytes or binary file objects (file objects are read on the calling thread, paths by the parsing threads).
    engine: a DeviceEngine (images: a CUDA tensor) or a CudaEngine (numpy, the same bytes).  bits: 8 or 16 -> uint8 / uint16
    samples, each through JXLImage.to_int's pipeline.  mode: "rgb", "rgba" or "grey" -> C = 3, 4 or 1 (see _slot_channels; a
    colour image in "grey" is a ValueError: no luma formula is applied).  A missing alpha is the maximum sample value.
    size: (H, W) of every slot; by default the largest displayed size in the batch.  Each image sits at the top-left of its slot
    after orientation, and the rest of the slot is 0.  Nothing is resampled or cropped: an image larger than `size` is a
    ValueError naming it.  options: a JXLOptions; preview=True gives the 1:8 previews (BatchResult.routes says which route each
    took), and outputFormat / outputDepth keep their meaning.

    Only the first displayed image of each file is decoded: a still image, or an animation's first frame.  Frames are not
    batched across files (their quantisation tables and filters differ) and nothing is colour managed beyond to_int.

    Pipelining: `workers` threads (default min(len(sources), os.cpu_count() // 2)) run the front end, each parse with
    os.cpu_count() // workers OpenMP threads for the sections of a frame, so parsing threads times OpenMP threads stays within the
    cores.  The calling thread composes the files in order on the engine's stream while later files parse; at most 2 * workers
    parsed files are alive at once, and each is closed as soon as its image is composed.  All device work, one pack launch and
    one synchronise for the batch, runs on the calling thread: composition must stay single-threaded, because _Buf.before_mutation
    is a class-level hook that points at the composing decoder's blend queue.

    A failure names the index and source it came from and fails the whole call; stream errors found at the batch's synchronise
    name the batch.  Returns a BatchResult."""
    import time
    from concurrent.futures import ThreadPoolExecutor
    t_start = time.perf_counter()
    sources = list(sources)
    n = len(sources)
    if n == 0:
        raise ValueError("decode_batch needs at least one source")
    if bits not in (8, 16):
        raise ValueError("bits must be 8 or 16, not %r" % (bits,))
    if mode not in BATCH_MODES:
        raise ValueError("mode must be one of %s, not %r" % (", ".join(BATCH_MODES), mode))
    if size is not None and (len(size) != 2 or any(int(v) < 1 for v in size)):
        raise ValueError("size must be (H, W) with H, W >= 1, not %r" % (size,))
    if engine is None or not hasattr(engine, "pack_batch"):
        raise ValueError("decode_batch needs a DeviceEngine or a CudaEngine")
    options = options if options is not None else JXLOptions()
    cores = os.cpu_count() or 1
    workers = max(1, min(n, cores // 2)) if workers is None else int(workers)
    if workers < 1:
        raise ValueError("workers must be >= 1")
    threads = max(1, cores // workers)
    c = BATCH_MODES[mode]
    names = [_source_name(s) for s in sources]
    datas = [s if isinstance(s, (str, os.PathLike, bytes, bytearray, memoryview)) else s.read() for s in sources]
    frontend.lib()                      # loaded (and built if need be) here, not by the parsing threads at once

    def parse(i):
        t = time.perf_counter()
        parsed, route = parse_stream(_read_source(datas[i]), options.preview, threads)
        return parsed, route, t, time.perf_counter()

    futures = {}
    items, sizes, routes, spans = [], [], [], []
    t_dev = None
    pool = ThreadPoolExecutor(workers)
    try:
        submitted = 0
        for i in range(n):
            while submitted < min(n, i + 2 * workers):
                futures[submitted] = pool.submit(parse, submitted)
                submitted += 1
            try:
                parsed, route, t0, t1 = futures.pop(i).result()
            except Exception as e:
                raise _attributed(e, i, names[i]) from e
            spans.append((t0, t1))
            try:
                t_dev = t_dev or time.perf_counter()
                img = _compose_first(parsed, route, engine, options)
                slots = _slot_channels(img.info, mode)
                o = img.info["orientation"]
                h, w = img.height, img.width
                shown = (w, h) if o >= 5 else (h, w)
                if size is not None and (shown[0] > size[0] or shown[1] > size[1]):
                    raise ValueError("image is %d x %d, larger than the batch size %d x %d" % (shown[0], shown[1], size[0], size[1]))
            except Exception as e:
                raise _attributed(e, i, names[i]) from e
            finally:
                parsed.close()
            items.append(([None if k is None else img.channels[k] for k in slots], [None if k is None else img._depth(k) for k in slots],
                          o, img.linear))
            sizes.append(shown)
            routes.append(route)
        out_h, out_w = (int(size[0]), int(size[1])) if size is not None else tuple(max(v) for v in zip(*sizes))
        images = engine.pack_batch(items, c, bits, out_h, out_w)
        del items
        sync = getattr(engine, "sync", None)
        if sync is not None:
            try:
                sync()
            except Exception as e:
                raise _attributed(e, -1, "the batch of %d sources" % n) from e
    except BaseException:
        pool.shutdown(wait=True, cancel_futures=True)
        for f in futures.values():              # parses that finished before the failure
            if not f.cancelled() and f.exception() is None:
                f.result()[0].close()
        sync = getattr(engine, "sync", None)
        if sync is not None:
            try:
                sync()                          # drain the batch's device work; the failure being raised is the one to report
            except Exception:
                pass
        raise
    pool.shutdown(wait=True)
    t_end = time.perf_counter()
    timings = dict(parse_s=sum(b - a for a, b in spans), parse_wall_s=max(b for _, b in spans) - min(a for a, _ in spans),
                   device_wall_s=t_end - t_dev, total_s=t_end - t_start)
    if isinstance(images, np.ndarray):
        sizes = np.array(sizes, np.int64)
    else:
        import torch
        sizes = torch.tensor(sizes, dtype=torch.int64)
    return BatchResult(images, sizes, routes, timings)
