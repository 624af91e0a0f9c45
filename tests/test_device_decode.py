"""Device-resident decoding (decoder.DeviceEngine): the frame loop on CUDA tensors must compute what the host-buffer engine
(CudaEngine) computes, bit for bit -- both run the same kernels -- and must not copy image data back to the host before the image
is returned."""
import copy
import os

import numpy as np
import pytest

from jxlatte_b200 import frontend, synth, default_frame_params
from jxlatte_b200.decoder import JXLDecoder, locate_tensor_view

S = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "samples")
SAMPLES = ["ants", "art", "bbb", "bench", "blendmodes_5", "george-tiled", "lenna", "patches-lossless", "quilt", "sollevante-hdr",
           "wb-rainbow", "white"]


# ---- the tensor view locator (CPU) ----
def test_locate_tensor_view_windows():
    torch = pytest.importorskip("torch")
    a = torch.zeros((10, 12), dtype=torch.float32)
    plane, y, x = locate_tensor_view(a[3:7, 2:9])
    assert (y, x) == (3, 2) and tuple(plane.shape) == (10, 12) and plane.data_ptr() == a.data_ptr()
    plane, y, x = locate_tensor_view(a[5:6, 0:12])                 # one row keeps the parent's pitch
    assert (y, x) == (5, 0) and tuple(plane.shape) == (10, 12)
    plane, y, x = locate_tensor_view(a[:, 11:12])                  # one column
    assert (y, x) == (0, 11)
    plane, y, x = locate_tensor_view(a)
    assert (y, x) == (0, 0) and tuple(plane.shape) == (10, 12)
    # a [C, H, W] owner is one plane of C * H rows
    b = torch.zeros((3, 8, 16), dtype=torch.int32)
    plane, y, x = locate_tensor_view(b[2, 1:5, 4:10])
    assert (y, x) == (2 * 8 + 1, 4) and tuple(plane.shape) == (24, 16) and plane.data_ptr() == b.data_ptr()
    plane[y, x] = 7
    assert int(b[2, 1, 4]) == 7


def test_locate_tensor_view_rejects_non_windows():
    torch = pytest.importorskip("torch")
    a = torch.zeros((10, 12), dtype=torch.float32)
    assert locate_tensor_view(a.t()[2:5, 1:4]) is None             # columns not contiguous
    assert locate_tensor_view(a[:, ::2]) is None
    assert locate_tensor_view(a[0]) is None                        # not 2-D
    assert locate_tensor_view(torch.zeros((4, 4), dtype=torch.float64)) is None


# ---- GPU ----
def _engines():
    from jxlatte_b200.decoder import CudaEngine, DeviceEngine
    return CudaEngine(), DeviceEngine()


def _assert_same_image(dev, ref, host_engine):
    torch = pytest.importorskip("torch")
    assert len(dev.channels) == len(ref.channels)
    for d, r in zip(dev.channels, ref.channels):
        assert isinstance(d, torch.Tensor) and d.is_cuda
        dn = d.cpu().numpy()
        assert dn.dtype == r.dtype and dn.shape == r.shape
        assert np.array_equal(dn, r, equal_nan=dn.dtype == np.float32)
    pd, pr = dev.planes.cpu().numpy(), ref.planes
    assert pd.dtype == pr.dtype and pd.shape == pr.shape
    assert np.array_equal(pd, pr, equal_nan=True)
    for bits in (8, 16):
        want_packed = ref.packed(bits, engine=host_engine)
        got_packed = dev.packed(bits)
        assert got_packed.is_cuda and got_packed.dtype == torch.uint8
        assert np.array_equal(got_packed.cpu().numpy(), want_packed)
        got = dev.to_int(bits)
        assert got.is_cuda and got.dtype == (torch.uint16 if bits > 8 else torch.uint8)
        got = got.cpu().numpy()
        # the host image's samples from the same kernel, in planar layout
        want = want_packed.view(">u2").astype(np.uint16) if bits > 8 else want_packed
        want = np.moveaxis(want, 2, 0)
        assert got.shape == want.shape and np.array_equal(got, want)
        # and the numpy mirror: the device pow and host libm may differ in the last bit of a double, once in ~1e8 samples
        d = np.abs(got.astype(np.int64) - ref.to_int(bits).astype(np.int64))
        assert int(d.max()) <= 1 and float((d != 0).mean()) < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("name", SAMPLES)
def test_device_decode_equals_host_decode(name):
    host, dev = _engines()
    path = os.path.join(S, name + ".jxl")
    hd, dd = JXLDecoder(path, engine=host), JXLDecoder(path, engine=dev)
    n = 0
    while True:
        ref, got = hd.decode(), dd.decode()
        assert (ref is None) == (got is None)
        if ref is None:
            break
        _assert_same_image(got, ref, host)
        n += 1
    assert n >= 1 and dd.timings["reconstruct_s"] > 0
    host.close()
    dev.close()


@pytest.mark.gpu
def test_device_decode_lf_frame_and_lossy_modular(monkeypatch):
    """The LF frame + lossy-Modular pair of test_frontend, built the same way, on both engines."""
    from jxlatte_b200 import decoder as dec_mod
    real = frontend.parse_file(os.path.join(S, "lenna.jxl"))
    st = real.vardct_state(0)
    lf = st["lf"]
    step = np.float32(1.0 / 65536.0)
    yq = np.rint(lf[1] / step).astype(np.int32)
    xq = np.rint(lf[0] / step).astype(np.int32)
    bq = np.rint(lf[2] / step).astype(np.int32) - yq
    info = copy.deepcopy(real.info)
    f1 = copy.deepcopy(info["frames"][0])
    f0 = copy.deepcopy(f1)
    f0.update(type=1, lf_level=1, encoding=1, width=64, height=64, padded_width=64, padded_height=64, gab=False, epf_iters=0,
              lf_dequant=[float(step)] * 3, flags=0, is_last=False, save_as_reference=0, num_groups=1,
              modular=dict(nb_meta=0, transformed=False, channels=[dict(h=64, w=64, hshift=0, vshift=0)] * 3, transforms=[]))
    f1.update(flags=f1["flags"] | 32, modular=dict(nb_meta=0, transformed=False, channels=[], transforms=[]))
    info["frames"] = [f0, f1]
    st1 = dict(st)
    st1["lf"] = np.zeros_like(lf)
    fake = _FakeParsed(info, {1: st1}, {0: [yq, xq, bq], 1: []})
    monkeypatch.setattr(dec_mod.frontend, "parse", lambda data, flags=0, strict=True: fake)
    host, dev = _engines()
    ref = JXLDecoder(b"unused", engine=host).decode()
    got = JXLDecoder(b"unused", engine=dev).decode()
    _assert_same_image(got, ref, host)
    host.close()
    dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [dict(w=67, h=45, gab=True, iters=2, ncolor=3), dict(w=40, h=33, gab=True, iters=3, ncolor=1),
                                 dict(w=64, h=48, gab=False, iters=1, ncolor=3)])
def test_device_decode_modular_gaborish_epf(monkeypatch, cfg):
    """Gaborish / EPF on a Modular frame, fabricated as test_frontend does, on both engines."""
    from jxlatte_b200 import decoder as dec_mod
    real = frontend.parse_file(os.path.join(S, "lenna.jxl"))
    rng = np.random.default_rng(cfg["w"])
    w, h, nc = cfg["w"], cfg["h"], cfg["ncolor"]
    base = rng.integers(90, 160, size=(nc, h, w)) + (rng.random((nc, h, w)) < 0.02) * 60
    chans = [np.ascontiguousarray(base[c], np.int32) for c in range(nc)]
    info = copy.deepcopy(real.info)
    f = copy.deepcopy(info["frames"][0])
    f.update(type=0, lf_level=0, encoding=1, width=w, height=h, padded_width=w, padded_height=h, gab=cfg["gab"], epf_iters=cfg["iters"],
             epf_sigma_for_modular=1.75, lf_dequant=[1.0 / 4096] * 3, flags=0, is_last=True, save_as_reference=0, num_groups=1,
             upsampling=1, do_ycbcr=False,
             modular=dict(nb_meta=0, transformed=False, channels=[dict(h=h, w=w, hshift=0, vshift=0)] * nc, transforms=[]))
    info["frames"] = [f]
    info.update(width=w, height=h, xyb_encoded=False, color_channels=nc, bits_per_sample=8, orientation=1)
    fake = _FakeParsed(info, {}, {0: chans})
    monkeypatch.setattr(dec_mod.frontend, "parse", lambda data, flags=0, strict=True: fake)
    host, dev = _engines()
    ref = JXLDecoder(b"unused", engine=host).decode()
    got = JXLDecoder(b"unused", engine=dev).decode()
    _assert_same_image(got, ref, host)
    host.close()
    dev.close()


class _FakeParsed:
    def __init__(self, info, states, modulars):
        self.info, self._states, self._mod = info, states, modulars

    @property
    def frames(self):
        return self.info["frames"]

    def vardct_state(self, k, copy=True):
        return dict(self._states[k])

    def modular_channels(self, k):
        return self._mod[k]

    def array(self, *a, **kw):
        raise KeyError(a)

    def close(self):
        pass


@pytest.mark.gpu
def test_cast_to_float_and_modular_xyb_kernels():
    """The two new kernels against the numpy lines they replace, on random int32 including values near +-2^31 and Y + B wrapping."""
    import torch
    from jxlatte_b200.decoder import DeviceEngine, NumpyArrays
    eng = DeviceEngine()
    rng = np.random.default_rng(3)
    n = 1 << 16
    edge = np.array([2**31 - 1, 2**31 - 2, -2**31, -2**31 + 1, 0, 1, -1, 16777217, -16777217, 2**30], np.int64)
    a = np.concatenate([rng.integers(-2**31, 2**31, n, dtype=np.int64), edge]).astype(np.int32).reshape(-1, 1)
    for depth in (1, 8, 12, 16, 24, 31):
        got = eng.cast_to_float(eng.upload(a, np.int32), depth).cpu().numpy()
        assert np.array_equal(got, NumpyArrays.cast_to_float(a, depth))
    y = np.concatenate([rng.integers(-2**31, 2**31, n, dtype=np.int64), edge]).astype(np.int32).reshape(-1, 1)
    b = np.concatenate([rng.integers(-2**31, 2**31, n, dtype=np.int64), edge[::-1]]).astype(np.int32).reshape(-1, 1)
    b[0, 0], y[0, 0] = 2**31 - 1, 5                       # y + b wraps
    x = a[::-1].copy()
    with np.errstate(over="ignore"):
        assert int(y[0, 0]) + int(b[0, 0]) > 2**31 - 1 and int((y + b)[0, 0]) < 0
        want = NumpyArrays.modular_xyb(y, x, b, [1.0 / 4096, 0.00123, 3.5])
    got = eng.modular_xyb(*(eng.upload(v, np.int32) for v in (y, x, b)), [1.0 / 4096, 0.00123, 3.5])
    for g, w_ in zip(got, want):
        assert g.dtype == torch.float32 and np.array_equal(g.cpu().numpy(), w_)
    eng.close()


def _state(W, H, p, seed=1, **kw):
    from jxlatte_b200.host import qm_generate
    qw, qo = qm_generate()
    return synth.make_state(W, H, seed=seed, params=p, qm_weights=qw, qm_offsets=qo, **kw), qw, qo


@pytest.mark.gpu
def test_device_stream_errors_surface_at_sync():
    """Errors the kernels find on the device come back with the host path's exception classes, at the synchronise."""
    from jxlatte_b200.decoder import DeviceEngine
    from jxlatte_b200.host import InvalidBitstreamError
    eng = DeviceEngine()
    p = default_frame_params(64, 64)
    st, qw, qo = _state(64, 64, p, mix="dct8")
    st = dict(st, qm_weights=qw, qm_offsets=qo)
    st["dct_select"] = st["dct_select"].copy()
    st["dct_select"][3, 3] = 31
    eng.reconstruct(p, st)
    with pytest.raises(InvalidBitstreamError):
        eng.sync()
    W, H = 256, 256
    p = default_frame_params(W, H, epf_iters=0, gab=False, color_mode=2)
    p.shift_y[:] = (1, 0, 1)
    p.shift_x[:] = (1, 0, 1)
    st, qw, qo = _state(W, H, p, seed=5)
    st = dict(st, qm_weights=qw, qm_offsets=qo)
    st["qcoeff"] = [np.ascontiguousarray(st["qcoeff"][c][:H >> p.shift_y[c], :W >> p.shift_x[c]]) for c in range(3)]
    st["lf"] = [np.ascontiguousarray(st["lf"][c][:(H // 8) >> p.shift_y[c], :(W // 8) >> p.shift_x[c]]) for c in range(3)]
    eng.reconstruct(p, st)
    with pytest.raises(NotImplementedError):
        eng.sync()
    eng.sync()                                  # the error is reported once; the context stays usable
    eng.close()


def _dtoh_copies(fn, tmp_path):
    """-> the byte counts of the device-to-host memcpys the CUDA activity trace records while fn runs."""
    import json
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    trace = str(tmp_path / "trace.json")
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    return [int(e.get("args", {}).get("bytes", -1)) for e in events
            if e.get("cat") == "gpu_memcpy" and ("DtoH" in e.get("name", "") or "Device -> Host" in e.get("name", ""))]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["george-tiled", "wb-rainbow"])
def test_device_decode_copies_nothing_back(name, tmp_path):
    """Under torch.profiler: the device path's only device-to-host copies are jxlb200_sync's flag reads (16 bytes), at most one per
    displayed image; the host path, profiled the same way, shows its own copies of image data back (so the profiler does see the
    library's copies)."""
    from jxlatte_b200.decoder import CudaEngine, DeviceEngine
    path = os.path.join(S, name + ".jxl")
    dev = DeviceEngine()
    JXLDecoder(path, engine=dev).decode()              # warm-up: allocations, lazy module loads
    images = []

    def run_dev():
        d = JXLDecoder(path, engine=dev)
        while True:
            img = d.decode()
            if img is None:
                break
            images.append(img)
    copies = _dtoh_copies(run_dev, tmp_path)
    assert len(images) >= 1
    assert len(copies) <= len(images) and all(b == 16 for b in copies), copies[:8]
    dev.close()
    host = CudaEngine()
    JXLDecoder(path, engine=host).decode()
    host_copies = _dtoh_copies(lambda: JXLDecoder(path, engine=host).decode(), tmp_path)
    assert sum(1 for b in host_copies if b > 16) >= 1, host_copies[:8]
    host.close()


@pytest.mark.gpu
def test_device_engine_refuses_another_stream():
    """The library is bound to the stream current at the engine's creation; decoding under another one would race, so it raises."""
    import torch
    from jxlatte_b200.decoder import DeviceEngine
    path = os.path.join(S, "lenna.jxl")
    eng = DeviceEngine()
    other = torch.cuda.Stream()
    with torch.cuda.stream(other):
        with pytest.raises(RuntimeError):
            JXLDecoder(path, engine=eng).decode()
    eng.sync()
    with torch.cuda.stream(eng.stream):
        assert JXLDecoder(path, engine=eng).decode().to_int(8).is_cuda
    eng.close()


@pytest.mark.gpu
def test_device_decode_on_a_second_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from jxlatte_b200.decoder import DeviceEngine
    path = os.path.join(S, "bbb.jxl")
    e0, e1 = DeviceEngine(0), DeviceEngine(1)
    a = JXLDecoder(path, engine=e0).decode()
    b = JXLDecoder(path, engine=e1).decode()
    assert b.planes.device == torch.device("cuda", 1)
    assert np.array_equal(a.planes.cpu().numpy(), b.planes.cpu().numpy(), equal_nan=True)
    assert np.array_equal(a.to_int(8).cpu().numpy(), b.to_int(8).cpu().numpy())
    e0.close()
    e1.close()
