"""Batch decode (decoder.decode_batch): many files into one [N, C, H, W] tensor, the front end on worker threads overlapping the
composition of earlier files, and every image oriented and packed into its slot by one k11_pack_batch launch."""
import copy
import json
import os
import random
import tempfile
import threading
import time

import numpy as np
import pytest

from jxlatte_b200 import decoder, frontend
from jxlatte_b200.decoder import JXLDecoder, JXLImage, JXLOptions, NumpyArrays, decode_batch

S = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "samples")
SAMPLES = ["ants", "art", "bbb", "bench", "blendmodes_5", "george-tiled", "lenna", "patches-lossless", "quilt", "sollevante-hdr",
           "wb-rainbow", "white"]
PATHS = [os.path.join(S, n + ".jxl") for n in SAMPLES]


# ---- fakes for the host-side pipeline (CPU) ----
class _Recorder:
    def __init__(self):
        self.lock = threading.Lock()
        self.events = []
        self.alive = self.max_alive = 0
        self.parse_started = {}

    def log(self, *e):
        with self.lock:
            self.events.append(e)


class _FakeParsed:
    def __init__(self, rec, i):
        self.rec, self.i, self.open = rec, i, True
        with rec.lock:
            rec.alive += 1
            rec.max_alive = max(rec.max_alive, rec.alive)

    def close(self):
        if self.open:
            self.open = False
            with self.rec.lock:
                self.rec.alive -= 1


class _FakeEngine:
    def __init__(self):
        self.calls = []

    def pack_batch(self, items, c, bits, out_h, out_w):
        self.calls.append((len(items), c, bits, out_h, out_w))
        return np.zeros((len(items), c, out_h, out_w), np.uint16 if bits > 8 else np.uint8)


def _fake_image(h, w, ncol=3, orientation=1, alpha=False):
    info = dict(color_channels=ncol, bits_per_sample=8, orientation=orientation,
                extra_channels=[dict(type=0, bits_per_sample=8)] if alpha else [])
    return JXLImage([np.zeros((h, w), np.float32) for _ in range(ncol + alpha)], info, False)


def _install_fakes(monkeypatch, rec, shapes, parse_s=0.0, compose=None):
    """decode_batch with fake front end and composition: source i is the int i; its image has shape shapes[i] ((h, w[, ncol])."""
    def parse_stream(data, preview, threads=None):
        i = int(data.decode())
        rec.log("parse_start", i)
        with rec.lock:
            ev = rec.parse_started.setdefault(i, threading.Event())
        ev.set()
        time.sleep(parse_s)
        rec.log("parse_end", i)
        return _FakeParsed(rec, i), None

    def compose_first(parsed, route, engine, options):
        rec.log("compose_start", parsed.i)
        if compose:
            compose(parsed.i)
        rec.log("compose_end", parsed.i)
        return _fake_image(*shapes[parsed.i])
    monkeypatch.setattr(decoder, "parse_stream", parse_stream)
    monkeypatch.setattr(decoder, "_compose_first", compose_first)


def _sources(n):
    return [str(i).encode() for i in range(n)]


# ---- CPU ----
def test_batch_argument_checks(monkeypatch):
    rec = _Recorder()
    _install_fakes(monkeypatch, rec, {0: (8, 8), 1: (20, 9), 2: (8, 8, 1)})
    eng = _FakeEngine()
    with pytest.raises(ValueError):
        decode_batch([], eng)
    for bad in (dict(bits=12), dict(bits=0), dict(mode="bgr"), dict(mode="RGB"), dict(size=(0, 8)), dict(workers=0)):
        with pytest.raises(ValueError):
            decode_batch(_sources(1), eng, **bad)
    assert not eng.calls
    # a colour image in "grey" is refused, naming the source; a grey image is fine in every mode
    with pytest.raises(ValueError, match=r"source 1 \(<1 bytes>\).*grey"):
        decode_batch([b"2", b"0"], eng, mode="grey")
    r = decode_batch([b"2"], eng, mode="grey", workers=1)
    assert r.images.shape == (1, 1, 8, 8)
    for mode, c in (("rgb", 3), ("rgba", 4)):
        assert decode_batch([b"2", b"0"], eng, mode=mode).images.shape == (2, c, 8, 8)
    # an image larger than `size` is an error that names the file
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "wide.jxl")
        with open(path, "wb") as f:
            f.write(b"1")
        with pytest.raises(ValueError, match=r"source 1 \(.*wide\.jxl\).*20 x 9"):
            decode_batch([b"0", path], eng, size=(16, 16))
    # the default size is the largest displayed size; bits picks the dtype
    r = decode_batch(_sources(2), eng, bits=16)
    assert r.images.shape == (2, 3, 20, 9) and r.images.dtype == np.uint16
    assert r.sizes.tolist() == [[8, 8], [20, 9]] and r.routes == [None, None]
    assert set(r.timings) == {"parse_s", "parse_wall_s", "device_wall_s", "total_s"}


def test_batch_sizes_follow_orientation(monkeypatch):
    rec = _Recorder()
    _install_fakes(monkeypatch, rec, {0: (10, 30, 3, 6), 1: (12, 5, 3, 1), 2: (4, 7, 3, 8)})
    eng = _FakeEngine()
    r = decode_batch(_sources(3), eng)
    assert r.sizes.tolist() == [[30, 10], [12, 5], [7, 4]] and r.images.shape == (3, 3, 30, 10)
    with pytest.raises(ValueError, match="source 0"):
        decode_batch(_sources(3), eng, size=(29, 30))


@pytest.mark.parametrize("workers", [1, 2, 3])
def test_batch_pipeline_overlaps_and_bounds_parsed_files(monkeypatch, workers):
    """Composition of file i waits until the parse of file i + 1 has started: a serial pipeline would time out here.  No more than
    2 * workers parsed files are alive at any time, every one is closed, and results follow the order of `sources`."""
    n = 12
    rec = _Recorder()

    def compose(i):
        if i + 1 < n:
            with rec.lock:
                ev = rec.parse_started.setdefault(i + 1, threading.Event())
            assert ev.wait(10.0), "parse of file %d had not started while file %d was composed" % (i + 1, i)
        time.sleep(0.01)
    shapes = {i: (4 + i, 5) for i in range(n)}
    _install_fakes(monkeypatch, rec, shapes, parse_s=0.002, compose=compose)
    r = decode_batch(_sources(n), _FakeEngine(), workers=workers)
    assert r.sizes.tolist() == [[4 + i, 5] for i in range(n)]
    assert 1 <= rec.max_alive <= 2 * workers and rec.alive == 0
    composed = [e[1] for e in rec.events if e[0] == "compose_start"]
    assert composed == list(range(n))
    for i in range(n - 1):                      # the start of parse i + 1 comes before the end of composition i
        assert rec.events.index(("parse_start", i + 1)) < rec.events.index(("compose_end", i))


def test_batch_failure_names_the_source_and_closes_everything(monkeypatch):
    rec = _Recorder()
    _install_fakes(monkeypatch, rec, {i: (4, 4) for i in range(6)})
    real = decoder.parse_stream

    def parse_stream(data, preview, threads=None):
        if data == b"3":
            raise frontend.InvalidBitstreamError("broken")
        return real(data, preview, threads)
    monkeypatch.setattr(decoder, "parse_stream", parse_stream)
    with pytest.raises(frontend.InvalidBitstreamError, match=r"source 3 .*broken"):
        decode_batch(_sources(6), _FakeEngine(), workers=2)
    assert rec.alive == 0


def _kernel_orient(a, o):
    """k11_pack_batch's index map (orient_source in csrc/k11_batch.cuh), restated: output (y, x) shows stored (sy, sx)."""
    h, w = a.shape
    oh, ow = (w, h) if o >= 5 else (h, w)
    y, x = np.meshgrid(np.arange(oh), np.arange(ow), indexing="ij")
    sy, sx = {1: (y, x), 2: (y, w - 1 - x), 3: (h - 1 - y, w - 1 - x), 4: (h - 1 - y, x), 5: (x, y), 6: (h - 1 - x, y),
              7: (h - 1 - x, w - 1 - y), 8: (x, w - 1 - y)}[o]
    return a[sy, sx]


@pytest.mark.parametrize("shape", [(5, 9), (9, 5), (1, 7), (6, 1)])
def test_kernel_orientation_map_matches_numpy_orient(shape):
    a = np.arange(shape[0] * shape[1], dtype=np.int32).reshape(shape)
    assert np.array_equal(_kernel_orient(a, 1), a)
    for o in range(2, 9):
        assert np.array_equal(_kernel_orient(a, o), NumpyArrays.orient(a, o)), o


# ---- GPU ----
def _expand(samples, info, mode, bits):
    """A single-file to_int result [C_img, h, w] expanded by decode_batch's channel rule."""
    ncol = info["color_channels"]
    rgb = [samples[0]] * 3 if ncol == 1 else [samples[0], samples[1], samples[2]]
    if mode == "grey":
        return samples[:1]
    if mode == "rgb":
        return np.stack(rgb)
    alpha = [ncol + k for k, e in enumerate(info["extra_channels"]) if e["type"] == 0]
    a = samples[alpha[0]] if alpha else np.full(samples[0].shape, (1 << bits) - 1, samples.dtype)
    return np.stack(rgb + [a])


def _single(path, engine, bits, options=None):
    img = JXLDecoder(path, engine=engine, options=options).decode()
    return img.to_int(bits).cpu().numpy(), img.info


def _check_slots(images, sizes, refs, mode, bits):
    assert images.shape[0] == len(refs)
    for i, (samples, info) in enumerate(refs):
        want = _expand(samples, info, mode, bits)
        h, w = want.shape[1:]
        assert tuple(sizes[i]) == (h, w)
        assert np.array_equal(images[i, :, :h, :w], want), i
        assert not images[i, :, h:, :].any() and not images[i, :, :, w:].any(), "padding of slot %d is not zero" % i


@pytest.fixture(scope="module")
def engines():
    from jxlatte_b200.decoder import CudaEngine, DeviceEngine
    e = dict(device=DeviceEngine(), host=CudaEngine())
    yield e
    for v in e.values():
        v.close()


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [8, 16])
def test_batch_of_all_samples_equals_single_decodes(engines, bits):
    import torch
    dev, host = engines["device"], engines["host"]
    refs = [_single(p, dev, bits) for p in PATHS]
    assert refs[SAMPLES.index("bench")][1]["orientation"] == 5
    assert refs[SAMPLES.index("patches-lossless")][1]["extra_channels"][0]["type"] == 0
    for mode in ("rgb", "rgba"):
        r = decode_batch(PATHS, dev, bits=bits, mode=mode)
        assert r.images.is_cuda and r.images.dtype == (torch.uint16 if bits > 8 else torch.uint8)
        assert r.images.shape[:2] == (len(PATHS), len(mode))
        got = r.images.cpu().numpy()
        _check_slots(got, r.sizes.tolist(), refs, mode, bits)
        if mode == "rgba":
            hr = decode_batch(PATHS, host, bits=bits, mode=mode)
            assert isinstance(hr.images, np.ndarray) and hr.images.dtype == got.dtype
            assert np.array_equal(hr.images, got) and hr.sizes.tolist() == r.sizes.tolist()
    with pytest.raises(ValueError, match="grey"):
        decode_batch(PATHS[:2], dev, mode="grey")


@pytest.mark.gpu
def test_batch_preview(engines):
    dev = engines["device"]
    opts = JXLOptions(preview=True)
    refs, routes = [], []
    for p in PATHS:
        d = JXLDecoder(p, engine=dev, options=opts)
        img = d.decode()
        refs.append((img.to_int(8).cpu().numpy(), img.info))
        routes.append(d.preview_route)
    r = decode_batch(PATHS, dev, options=opts, mode="rgba")
    assert r.routes == routes and "lf" in routes and "full" in routes
    _check_slots(r.images.cpu().numpy(), r.sizes.tolist(), refs, "rgba", 8)


@pytest.mark.gpu
def test_batch_order_follows_sources(engines):
    dev = engines["device"]
    base = decode_batch(PATHS, dev, bits=8)
    order = list(range(len(PATHS))) * 2
    random.Random(5).shuffle(order)
    src = [PATHS[i] for i in order]
    src[1] = open(src[1], "rb").read()                  # bytes and file objects are sources too
    with open(src[2], "rb") as f:
        src[2] = f
        one = decode_batch(src, dev, bits=8, workers=1, size=tuple(base.images.shape[2:]))
    src[2] = PATHS[order[2]]
    eight = decode_batch(src, dev, bits=8, workers=8, size=tuple(base.images.shape[2:]))
    a, b, ref = one.images.cpu().numpy(), eight.images.cpu().numpy(), base.images.cpu().numpy()
    assert np.array_equal(a, b)
    assert np.array_equal(a, ref[order]) and one.sizes.tolist() == base.sizes[order].tolist()


@pytest.mark.gpu
def test_batch_grey_images(monkeypatch, engines):
    """A grey Modular image (fabricated as test_device_decode does) with orientation 6: "grey" keeps its one channel, "rgb"
    replicates it, "rgba" adds an opaque alpha; each slot equals the single-file decode."""
    real = frontend.parse_file(os.path.join(S, "lenna.jxl"))
    rng = np.random.default_rng(7)
    h, w = 37, 58
    chan = np.ascontiguousarray(rng.integers(0, 256, size=(h, w)), np.int32)
    info = copy.deepcopy(real.info)
    real.close()
    f = copy.deepcopy(info["frames"][0])
    f.update(type=0, lf_level=0, encoding=1, width=w, height=h, padded_width=w, padded_height=h, gab=False, epf_iters=0, flags=0,
             is_last=True, save_as_reference=0, num_groups=1, upsampling=1, do_ycbcr=False,
             modular=dict(nb_meta=0, transformed=False, channels=[dict(h=h, w=w, hshift=0, vshift=0)], transforms=[]))
    info["frames"] = [f]
    info.update(width=w, height=h, xyb_encoded=False, color_channels=1, bits_per_sample=8, orientation=6, extra_channels=[])

    class Fake:
        def __init__(self):
            self.info = info

        @property
        def frames(self):
            return self.info["frames"]

        def modular_channels(self, k):
            return [chan]

        def close(self):
            pass
    monkeypatch.setattr(decoder.frontend, "parse", lambda data, flags=0, strict=True, threads=None: Fake())
    dev = engines["device"]
    ref = _single(b"unused", dev, 8)
    for mode in ("grey", "rgb", "rgba"):
        r = decode_batch([b"a", b"b"], dev, mode=mode, size=(64, 64))
        assert r.sizes.tolist() == [[w, h]] * 2
        _check_slots(r.images.cpu().numpy(), r.sizes.tolist(), [ref, ref], mode, 8)


# Run in a child process: its torch.profiler session records decode_batch's parsing threads, and such a session left the test
# process in a state where later kernel traces there (tests/kernel_trace.py) came back without the stage-2 kernels they ran.
_PROFILE_CHILD = r"""
import json, os, sys, tempfile
import torch
from torch.profiler import ProfilerActivity, profile
from jxlatte_b200.decoder import DeviceEngine, decode_batch
src = sys.argv[1:]
dev = DeviceEngine()
decode_batch(src, dev, mode="rgba")                     # warm-up
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    r = decode_batch(src, dev, mode="rgba")
    torch.cuda.synchronize()
fd, path = tempfile.mkstemp(suffix=".json")
os.close(fd)
try:
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
finally:
    os.unlink(path)
kernels = [e.get("name", "") for e in events if e.get("cat") == "kernel"]
dtoh = [int(e.get("args", {}).get("bytes", -1)) for e in events
        if e.get("cat") == "gpu_memcpy" and ("DtoH" in e.get("name", "") or "Device -> Host" in e.get("name", ""))]
dev.close()
print(json.dumps(dict(n=int(r.images.shape[0]), kernels=kernels, dtoh=dtoh)))
"""


@pytest.mark.gpu
def test_batch_launches_one_pack_and_copies_only_the_flags():
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = [os.path.join(S, n + ".jxl") for n in ("bench", "patches-lossless", "lenna", "art", "white")]
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([root] + [v for v in [os.environ.get("PYTHONPATH")] if v]))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _PROFILE_CHILD] + src
    p = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-4000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    kernels, dtoh = res["kernels"], res["dtoh"]
    assert res["n"] == len(src)
    assert sum("k11_pack_batch" in k for k in kernels) == 1, [k for k in kernels if "pack" in k]
    assert not any("k8_pack_samples" in k for k in kernels)
    assert len(dtoh) <= 1 and all(b == 16 for b in dtoh), dtoh


@pytest.mark.gpu
def test_batch_corrupt_file_fails_the_batch_and_the_engine_recovers(engines):
    dev = engines["device"]
    data = open(PATHS[SAMPLES.index("lenna")], "rb").read()
    bad = data[:len(data) // 2]
    src = [PATHS[1], PATHS[3], bad, PATHS[6]]
    with pytest.raises(frontend.InvalidBitstreamError, match=r"source 2 "):
        decode_batch(src, dev)
    r = decode_batch([PATHS[1], PATHS[3], PATHS[6]], dev, bits=16)
    refs = [_single(p, dev, 16) for p in (PATHS[1], PATHS[3], PATHS[6])]
    _check_slots(r.images.cpu().numpy(), r.sizes.tolist(), refs, "rgb", 16)


@pytest.mark.gpu
def test_pack_batch_dev_refuses_bad_arguments():
    import ctypes as C
    import torch
    from jxlatte_b200 import _lib
    from jxlatte_b200.host import Reconstructor
    rec = Reconstructor(0)
    plane = torch.zeros((6, 10), dtype=torch.float32, device="cuda")
    iplane = torch.zeros((6, 10), dtype=torch.int32, device="cuda")
    out = torch.zeros((2, 4, 16, 16), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()                            # the context runs on its own stream

    def items(n=1, **kw):
        arr = (_lib.BatchItem * n)()
        for it in arr:
            for k in range(4):
                it.plane[k], it.is_int[k], it.depth[k], it.pitch[k] = plane.data_ptr(), 0, 8, 10
            it.h, it.w, it.orientation, it.linear = 6, 10, 1, 0
        for key, v in kw.items():
            if key == "int_depth":
                arr[n - 1].plane[1], arr[n - 1].is_int[1], arr[n - 1].depth[1] = iplane.data_ptr(), 1, v
            elif key == "plane0":
                arr[n - 1].plane[0] = v
            else:
                setattr(arr[n - 1], key, v)
        return arr

    def call(arr, n, c=4, bits=8, oh=16, ow=16, dst=None):
        return rec._L.jxlb200_pack_batch_dev(rec._h, arr, n, c, bits, oh, ow, dst if dst is not None else out.data_ptr())
    assert call(items(2), 2) == _lib.OK                  # the arguments below differ from this one in one thing each
    rec.sync()
    before = rec.launch_count()
    bad = [(items(), 0, {}), (items(), 1, dict(c=2)), (items(), 1, dict(c=5)), (items(), 1, dict(bits=12)),
           (items(2, orientation=0), 2, {}), (items(2, orientation=9), 2, {}),
           (items(2, h=17), 2, {}), (items(2, orientation=5, h=12, w=17), 2, {}), (items(), 1, dict(oh=5)),
           (items(2, int_depth=0), 2, {}), (items(2, int_depth=32), 2, {}),
           (items(2, plane0=out.data_ptr() + 64), 2, {}), (items(), 1, dict(dst=plane.data_ptr() + 8))]
    for arr, n, kw in bad:
        assert call(arr, n, **kw) == _lib.E_ARG, (n, kw)
    assert rec.launch_count() == before
    rec.close()
