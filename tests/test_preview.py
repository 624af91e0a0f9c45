"""1:8 previews (JXLOptions(preview=True)): the front end's LF-only parse, the route each stream takes, the two preview kernels
(k10_lf_preview, k10_area_mean8) against numpy / oracle references, and the two engines against each other."""
import copy
import os

import numpy as np
import pytest

from jxlatte_b200 import default_frame_params, frontend
from jxlatte_b200.decoder import JXLDecoder, JXLOptions, NumpyArrays, preview_route

S = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "samples")
ROUTES = {"ants": "lf", "art": "full", "bbb": "lf", "bench": "lf", "blendmodes_5": "full", "george-tiled": "lf", "lenna": "lf",
          "patches-lossless": "full", "quilt": "full", "sollevante-hdr": "lf", "wb-rainbow": "full", "white": "lf"}
SAMPLES = sorted(ROUTES)
LF_SAMPLES = [n for n in SAMPLES if ROUTES[n] == "lf"]
HF_ARRAYS = ("qcoeff", "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y")


def _data(name):
    with open(os.path.join(S, name + ".jxl"), "rb") as f:
        return f.read()


def _headers(info):
    """The header JSON an LF-only parse shares with the full parse: without "lf_only", without the parse's coverage counters (it opens
    fewer entropy streams) and without the HfGlobal fields it does not read."""
    info = copy.deepcopy(info)
    info.pop("lf_only", None)
    info.pop("coverage")
    for f in info["frames"]:
        f.pop("quant_all_default", None)
        f.pop("quant_params", None)
    return info


# ---- the LF-only parse (CPU) ----
@pytest.mark.parametrize("name", SAMPLES)
def test_lf_only_parse_equals_full_parse(name):
    full, lf = frontend.parse(_data(name)), frontend.parse(_data(name), frontend.FLAG_LF_ONLY)
    assert lf.info["lf_only"] is True and "lf_only" not in full.info
    assert _headers(lf.info) == _headers(full.info)
    for k, f in enumerate(full.frames):
        if f["encoding"] != 0:
            continue
        for c in range(3):
            assert np.array_equal(lf.array(k, "lf", c), full.array(k, "lf", c))
            assert np.array_equal(lf.array(k, "lf_quant", c), full.array(k, "lf_quant", c))
        assert np.array_equal(lf.array(k, "lf_extra_precision"), full.array(k, "lf_extra_precision"))
        for a in HF_ARRAYS:
            full.array(k, a)
            with pytest.raises(KeyError):
                lf.array(k, a)


def test_lf_state_of_a_subsampled_frame():
    """ants is chroma-subsampled (X and B at half width): lf_state gives each channel its own grid, lf_quantised keeps refusing."""
    p = frontend.parse(_data("ants"), frontend.FLAG_LF_ONLY)
    f = p.frames[0]
    assert f["shift_x"] == [1, 0, 1] and f["shift_y"] == [0, 0, 0]
    hb, wb = f["padded_height"] // 8, f["padded_width"] // 8
    q, ep, sd, kx, kb, smooth = p.lf_state(0)
    assert [a.shape for a in q] == [(hb, wb // 2), (hb, wb), (hb, wb // 2)] and all(a.dtype == np.int32 for a in q)
    assert ep.size == ((hb + 255) // 256) * ((wb + 255) // 256) and not smooth
    assert p.lf_quantised(0) is None


def test_lf_only_refuses_host_transforms():
    """The host-side Modular transforms need the channels an LF-only parse leaves empty: the combination is an argument error."""
    with pytest.raises(RuntimeError):
        frontend.parse(_data("quilt"), frontend.FLAG_LF_ONLY | frontend.FLAG_HOST_TRANSFORMS)


def test_hf_sections_are_never_read():
    """lenna with garbage in place of its HfGlobal and pass-group sections: the LF-only parse still gives the clean file's LF image;
    the full parse of the same bytes does not (the positive control)."""
    data = _data("lenna")
    clean = frontend.parse(data)
    f = clean.frames[0]
    lengths, first = f["toc_lengths"], f["toc_first_section"]
    assert len(lengths) == 2 + f["num_lf_groups"] + f["num_groups"] and not clean.info["coverage"]["permuted_toc"]
    start = first + sum(lengths[:1 + f["num_lf_groups"]])        # HfGlobal, then the pass groups, to the end of the frame
    end = first + sum(lengths)
    garbage = np.random.default_rng(7).integers(0, 256, end - start, dtype=np.uint8).tobytes()
    crafted = data[:start] + garbage + data[end:]
    assert len(crafted) == len(data) and crafted != data
    lf = frontend.parse(crafted, frontend.FLAG_LF_ONLY)
    for c in range(3):
        assert np.array_equal(lf.array(0, "lf", c), clean.array(0, "lf", c))
        assert np.array_equal(lf.array(0, "lf_quant", c), clean.array(0, "lf_quant", c))
    assert np.array_equal(lf.array(0, "lf_extra_precision"), clean.array(0, "lf_extra_precision"))
    try:
        full = frontend.parse(crafted)
    except (frontend.InvalidBitstreamError, NotImplementedError, RuntimeError):
        return
    assert not np.array_equal(full.array(0, "qcoeff", 1), clean.array(0, "qcoeff", 1))


# ---- route selection, on headers (CPU) ----
@pytest.mark.parametrize("name", SAMPLES)
def test_route_pinned_per_sample(name):
    assert preview_route(frontend.parse(_data(name), frontend.FLAG_LF_ONLY).info) == ROUTES[name]


@pytest.fixture(scope="module")
def lenna_info():
    info = frontend.parse(_data("lenna"), frontend.FLAG_LF_ONLY).info
    assert preview_route(info) == "lf"
    return info


def _with_frame(info, **fields):
    info = copy.deepcopy(info)
    info["frames"][0].update(fields)
    return info


def test_route_needs_vardct(lenna_info):
    assert preview_route(_with_frame(lenna_info, encoding=1)) == "full"


@pytest.mark.parametrize("ftype,route", [(0, "lf"), (3, "lf"), (1, "full"), (2, "full")])
def test_route_frame_types(lenna_info, ftype, route):
    """Types 0 and 3 are rendered; an LF frame (1) or a reference-only frame (2) anywhere in the stream sends it to the full route."""
    info = copy.deepcopy(lenna_info)
    extra = copy.deepcopy(info["frames"][0])
    extra.update(type=ftype, is_last=False)
    info["frames"].insert(0, extra)
    assert preview_route(info) == route


def test_route_refuses_a_frame_using_an_lf_frame(lenna_info):
    assert preview_route(_with_frame(lenna_info, flags=lenna_info["frames"][0]["flags"] | 32)) == "full"


@pytest.mark.parametrize("flag", [1, 2, 16])        # noise, patches, splines
def test_route_refuses_features(lenna_info, flag):
    assert preview_route(_with_frame(lenna_info, flags=lenna_info["frames"][0]["flags"] | flag)) == "full"


def test_route_refuses_upsampling(lenna_info):
    assert preview_route(_with_frame(lenna_info, upsampling=2)) == "full"


def test_route_refuses_extra_channels(lenna_info):
    info = copy.deepcopy(lenna_info)
    info["extra_channels"] = [dict(type=0, bits_per_sample=8, exp_bits=0, dim_shift=0, name="", alpha_associated=False)]
    assert preview_route(info) == "full"


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_route_needs_replace(lenna_info, mode):
    assert preview_route(_with_frame(lenna_info, blend_mode=mode)) == "full"


@pytest.mark.parametrize("x0,y0,route", [(8, 16, "lf"), (-8, -24, "lf"), (4, 0, "full"), (0, 12, "full"), (-3, 0, "full")])
def test_route_needs_an_origin_on_the_block_grid(lenna_info, x0, y0, route):
    assert preview_route(_with_frame(lenna_info, x0=x0, y0=y0)) == route


# ---- numpy references ----
F32 = np.float32


def _double_h(a):
    """k6_upsample_h in numpy: out[y][2x] = .75 a[y][x] + .25 a[y][max(x-1, 0)], out[y][2x+1] = .75 a[y][x] + .25 a[y][min(x+1, w-1)]."""
    w = a.shape[1]
    b75 = F32(0.75) * a
    out = np.empty((a.shape[0], 2 * w), np.float32)
    out[:, 0::2] = b75 + F32(0.25) * a[:, np.r_[0, 0:w - 1]]
    out[:, 1::2] = b75 + F32(0.25) * a[:, np.r_[1:w, w - 1]]
    return out


def _double_v(a):
    return np.ascontiguousarray(_double_h(np.ascontiguousarray(a.T)).T)


def _mean8(a, depth):
    """k10_area_mean8 in numpy: castToFloat for int32, a float32 sum from 0 in row-major order over each 8 x 8 area, one divide by the
    area's pixel count.  Zeros fill the partial areas: adding +0 never changes a sum that starts at +0."""
    if a.dtype != np.float32:
        a = NumpyArrays.cast_to_float(a, depth)
    h, w = a.shape
    oh, ow = -(-h // 8), -(-w // 8)
    pad = np.zeros((oh * 8, ow * 8), np.float32)
    pad[:h, :w] = a
    blocks = pad.reshape(oh, 8, ow, 8).transpose(0, 2, 1, 3).reshape(oh, ow, 64)
    s = np.zeros((oh, ow), np.float32)
    for k in range(64):
        s = s + blocks[:, :, k]
    rows = np.minimum(8, h - 8 * np.arange(oh))[:, None]
    cols = np.minimum(8, w - 8 * np.arange(ow))[None, :]
    return s / (rows * cols).astype(np.float32)


def _lf_reference(orc, dec, parsed, k):
    """One frame's 1:8 image from the front end's own LF planes: the 0.75 / 0.25 doubling of subsampled channels, the crop, then
    the oracle's colour transform."""
    info, f = parsed.info, parsed.frames[k]
    hb, wb = f["padded_height"] // 8, f["padded_width"] // 8
    oh, ow = -(-f["height"] // 8), -(-f["width"] // 8)
    planes = []
    for c in range(3):
        a = parsed.array(k, "lf", c, (hb >> f["shift_y"][c], wb >> f["shift_x"][c]))
        if f["shift_x"][c]:
            a = _double_h(a)
        if f["shift_y"][c]:
            a = _double_v(a)
        planes.append(np.ascontiguousarray(a[:oh, :ow]))
    p = dec.frame_params(info, f).copy()
    p.width, p.height = ow, oh
    return orc.color(p, planes)


def _unorient(a, o):
    """The inverse of JXLCodestreamDecoder.transposeBuffer for orientation o."""
    return a if o == 1 else NumpyArrays.orient(a, {6: 8, 8: 6}.get(o, o))


def _depths(info, n):
    return ([info["bits_per_sample"]] * info["color_channels"] + [e["bits_per_sample"] for e in info["extra_channels"]])[:n]


def _decode_all(name, engine, preview=True):
    d = JXLDecoder(os.path.join(S, name + ".jxl"), engine=engine, options=JXLOptions(preview=preview))
    images = []
    while True:
        img = d.decode()
        if img is None:
            break
        images.append(img)
    return d, images


# ---- GPU ----
@pytest.fixture(scope="module")
def engines():
    from jxlatte_b200.decoder import CudaEngine, DeviceEngine
    host, dev = CudaEngine(), DeviceEngine()
    yield host, dev
    host.close()
    dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", LF_SAMPLES)
def test_lf_route_bit_exact(engines, orc, name):
    """Every frame's DeviceEngine preview equals the reference from the front end's LF planes; 4:4:4 frames also equal
    lf_dequant_dev + color_transform_dev on the same inputs; the decoded image is those frames composed at 1:8."""
    host, dev = engines
    parsed = frontend.parse(_data(name), frontend.FLAG_LF_ONLY)
    info = parsed.info
    dec = JXLDecoder(b"", engine=dev)
    ih, iw = -(-info["height"] // 8), -(-info["width"] // 8)
    canvas = np.zeros((3, ih, iw), np.float32)
    for k, f in enumerate(parsed.frames):
        p = dec.frame_params(info, f)
        oh, ow = -(-f["height"] // 8), -(-f["width"] // 8)
        q, ep, sd, kx, kb, smooth = parsed.lf_state(k)
        got = dev.lf_preview(p, q, ep, sd, kx, kb, smooth, oh, ow).cpu().numpy()
        want = _lf_reference(orc, dec, parsed, k)
        assert np.array_equal(got, want, equal_nan=True), (name, k)
        if not any(f["shift_x"]) and not any(f["shift_y"]):
            lf = dev.lf_dequant(np.stack(q), ep, sd, kx, kb, smooth)
            hb, wb = lf.shape[1:]
            pad = dev.zeros((3, -(-hb // 8) * 8, -(-wb // 8) * 8))
            pad[:, :hb, :wb] = lf
            pc = p.copy()
            pc.height, pc.width = pad.shape[1:]
            two_step = dev.color(pc, pad)[:, :oh, :ow].cpu().numpy()
            assert np.array_equal(got, two_step, equal_nan=True), (name, k)
        y0, x0 = f["y0"] // 8, f["x0"] // 8
        ys, xs = max(y0, 0), max(x0, 0)
        ye, xe = min(y0 + oh, ih), min(x0 + ow, iw)
        if ye > ys and xe > xs:
            canvas[:, ys:ye, xs:xe] = want[:, ys - y0:ye - y0, xs - x0:xe - x0]
    _, images = _decode_all(name, dev)
    assert len(images) == 1
    img = images[0]
    o = info["orientation"]
    assert np.array_equal(np.stack([c.cpu().numpy() for c in img.channels]), np.stack([NumpyArrays.orient(c, o) if o != 1 else c for c in canvas]),
                          equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SAMPLES)
def test_preview_host_equals_device(engines, name):
    """CudaEngine and DeviceEngine previews are bit-identical in planes, to_int(8 / 16) and packed, on either route."""
    from test_device_decode import _assert_same_image
    host, dev = engines
    dh, ref = _decode_all(name, host)
    dd, got = _decode_all(name, dev)
    assert dh.preview_route == dd.preview_route == ROUTES[name]
    assert len(ref) == len(got) >= 1
    info = frontend.parse(_data(name), frontend.FLAG_HEADERS_ONLY).info
    for r, g in zip(ref, got):
        w8, h8 = -(-info["width"] // 8), -(-info["height"] // 8)
        shape = (w8, h8) if info["orientation"] > 4 else (h8, w8)
        assert all(c.shape == shape and c.dtype == np.float32 for c in r.channels)
        _assert_same_image(g, r, host)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SAMPLES)
def test_area_mean8_bit_exact(engines, name):
    """k10_area_mean8 on each sample's full decode (before orientation) equals the numpy loop, on both engines: float canvases, int32
    canvases (lossless Modular: art, quilt), 500 x 606 (bench), orientation 5 (bench).  Full-route previews are exactly those means, oriented."""
    import torch
    host, dev = engines
    d, full = _decode_all(name, host, preview=False)
    _, prev = _decode_all(name, host)
    info = frontend.parse(_data(name), frontend.FLAG_HEADERS_ONLY).info
    o = info["orientation"]
    assert len(full) == len(prev)
    for img, pimg in zip(full, prev):
        canvas = [_unorient(c, o) for c in img.channels]
        depths = _depths(info, len(canvas))
        want = [_mean8(c, dp) for c, dp in zip(canvas, depths)]
        got_h = host.area_mean8(canvas, depths)
        got_d = dev.area_mean8([torch.from_numpy(np.ascontiguousarray(c)).cuda() for c in canvas], depths)
        for w_, gh, gd in zip(want, got_h, got_d):
            assert np.array_equal(gh, w_, equal_nan=True) and np.array_equal(gd.cpu().numpy(), w_, equal_nan=True)
        if ROUTES[name] == "full":
            for w_, c in zip(want, pimg.channels):
                assert np.array_equal(c, NumpyArrays.orient(w_, o) if o != 1 else w_, equal_nan=True)
    if name == "bench":
        assert (info["width"], info["height"], o) == (500, 606, 5)
    if name in ("art", "quilt"):
        assert full[0].channels[0].dtype == np.int32


def _psnr8(a, b):
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return float("inf") if mse == 0 else 10.0 * np.log10(255.0 ** 2 / mse)


@pytest.mark.gpu
@pytest.mark.parametrize("name", LF_SAMPLES)
def test_routes_agree(engines, monkeypatch, name):
    """The LF route (colour of the block mean, no restoration filters) against the full route (mean of the colour) in 8-bit sRGB:
    different definitions, so a PSNR floor rather than equality."""
    from jxlatte_b200 import decoder as dec_mod
    host, _ = engines
    _, lf = _decode_all(name, host)
    monkeypatch.setattr(dec_mod, "preview_route", lambda info: "full")
    d, full = _decode_all(name, host)
    assert d.preview_route == "full"
    for a, b in zip(lf, full):
        ta, tb = a.to_int(8), b.to_int(8)
        assert ta.shape == tb.shape
        psnr = _psnr8(ta, tb)
        print("%s: LF route vs full route, 8-bit sRGB PSNR %.2f dB" % (name, psnr))
        assert psnr >= 30.0, (name, psnr)


@pytest.mark.gpu
def test_lf_route_kernels_and_copies(engines, tmp_path):
    """An LF-route preview on the device launches k10_lf_preview once per frame (george-tiled: 135 cropped frames) and no stage-1 /
    stage-2 kernel, and copies nothing back but the sync's 16-byte flag reads."""
    from kernel_trace import launched_kernels
    from test_device_decode import _dtoh_copies
    _, dev = engines
    name = "george-tiled"
    nframes = len(frontend.parse(_data(name), frontend.FLAG_LF_ONLY).frames)
    _decode_all(name, dev)                                    # warm-up
    (d, images), names = launched_kernels(lambda: _decode_all(name, dev))
    assert d.preview_route == "lf" and len(images) == 1
    assert sum(1 for n in names if "k10_lf_preview" in n) == nframes
    stage = [n for n in names if any(k in n for k in ("k0_", "k1_", "k2_", "k6_", "k8_lf_dequant"))]
    assert not stage, stage[:4]
    copies = _dtoh_copies(lambda: _decode_all(name, dev), tmp_path)
    assert len(copies) <= len(images) and all(b == 16 for b in copies), copies[:8]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [dict(sy=(1, 0, 1), sx=(1, 0, 1), color=2), dict(sy=(0, 0, 0), sx=(1, 0, 1), color=2),
                                 dict(sy=(1, 0, 1), sx=(0, 0, 0), color=0), dict(sy=(0, 1, 0), sx=(1, 0, 0), color=1)])
def test_lf_preview_kernel_subsampled(recon, orc, cfg):
    """Subsampled channels over several LF groups with different extraPrecision, odd crops: dequantisation, doubling, colour."""
    W, H = 16 * 136, 16 * 264                     # LF grid 272 x 528: 2 x 3 LF groups
    p = default_frame_params(W, H, color_mode=cfg["color"])
    p.shift_y[:], p.shift_x[:] = cfg["sy"], cfg["sx"]
    hb, wb = H // 8, W // 8
    rng = np.random.default_rng(sum(cfg["sy"]) * 4 + sum(cfg["sx"]) + cfg["color"])
    q = [rng.integers(-400, 400, (hb >> cfg["sy"][c], wb >> cfg["sx"][c])).astype(np.int32) for c in range(3)]
    ep = rng.integers(0, 4, 6).astype(np.uint8)
    sd = [F32(1 / 4096.0), F32(1 / 512.0), F32(1 / 256.0)]
    oh, ow = hb - 3, wb - 5
    got = recon.lfPreview(p, q, ep, sd, 0.0, 1.0, False, oh, ow)
    planes = []
    for c in range(3):
        sy, sx = cfg["sy"][c], cfg["sx"][c]
        gy = (np.arange(hb >> sy) << sy) >> 8
        gx = (np.arange(wb >> sx) << sx) >> 8
        div = (F32(1) * (1 << ep[gy[:, None] * 2 + gx[None, :]].astype(np.int64))).astype(np.float32)
        a = q[c].astype(np.float32) * (F32(sd[c]) / div)
        if sx:
            a = _double_h(a)
        if sy:
            a = _double_v(a)
        planes.append(np.ascontiguousarray(a[:oh, :ow]))
    pc = p.copy()
    pc.width, pc.height = ow, oh
    assert np.array_equal(got, orc.color(pc, planes), equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("smooth", [True, False])
def test_lf_preview_kernel_444(recon, orc, smooth):
    """4:4:4 over several LF groups: the oracle's LFCoefficients (dequantisation, chroma-from-luma, smoothing), cropped, coloured."""
    W, H = 8 * 300, 8 * 520
    p = default_frame_params(W, H, color_mode=1)
    rng = np.random.default_rng(11 + smooth)
    q = rng.integers(-300, 300, (3, H // 8, W // 8)).astype(np.int32)
    ep = rng.integers(0, 4, 6).astype(np.uint8)
    sd = [F32(1 / 4096.0), F32(1 / 512.0), F32(1 / 256.0)]
    kx, kb = F32(0.03125), F32(0.9375)
    oh, ow = H // 8 - 7, W // 8 - 1
    got = recon.lfPreview(p, q, ep, sd, kx, kb, smooth, oh, ow)
    lf = orc.lf_dequant(q, ep, sd, kx, kb, cfl=True, smooth=smooth)
    pc = p.copy()
    pc.width, pc.height = ow, oh
    assert np.array_equal(got, orc.color(pc, [np.ascontiguousarray(lf[c, :oh, :ow]) for c in range(3)]), equal_nan=True)


@pytest.mark.gpu
def test_preview_argument_errors(recon):
    import torch
    from jxlatte_b200.host import InvalidBitstreamError
    W, H = 512, 256
    hb, wb = H // 8, W // 8
    q = [np.zeros((hb, wb), np.int32) for _ in range(3)]
    ep = np.zeros(1, np.uint8)
    sd = [1.0, 1.0, 1.0]
    p = default_frame_params(W, H)
    assert recon.lfPreview(p, q, ep, sd, 0.0, 1.0, True, hb, wb).shape == (3, hb, wb)
    with pytest.raises(ValueError):                                 # preview larger than the LF grid
        recon.lfPreview(p, q, ep, sd, 0.0, 1.0, True, hb + 1, wb)
    with pytest.raises(ValueError):
        recon.lfPreview(p, q, ep, sd, 0.0, 1.0, True, hb, wb + 1)
    with pytest.raises(ValueError):                                 # one extraPrecision byte per LF group
        recon.lfPreview(p, q, np.zeros(2, np.uint8), sd, 0.0, 1.0, True, hb, wb)
    with pytest.raises(InvalidBitstreamError):                      # a 2-bit field
        recon.lfPreview(p, q, np.full(1, 4, np.uint8), sd, 0.0, 1.0, True, hb, wb)
    with pytest.raises(ValueError):                                 # planes of the wrong shape
        recon.lfPreview(p, [a[:-1] for a in q], ep, sd, 0.0, 1.0, True, hb, wb)
    ps = default_frame_params(W, H)
    ps.shift_x[:] = (1, 0, 1)
    qs = [np.zeros((hb, wb >> s), np.int32) for s in (1, 0, 1)]
    assert recon.lfPreview(ps, qs, ep, sd, 0.0, 1.0, False, hb, wb).shape == (3, hb, wb)
    with pytest.raises(InvalidBitstreamError):                      # adaptive smoothing with subsampling
        recon.lfPreview(ps, qs, ep, sd, 0.0, 1.0, True, hb, wb)
    ps.shift_x[:] = (2, 0, 2)
    with pytest.raises(ValueError):                                 # shifts outside {0, 1}
        recon.lfPreview(ps, [np.zeros((hb, wb >> s), np.int32) for s in (2, 0, 2)], ep, sd, 0.0, 1.0, False, hb, wb)
    qd = [torch.zeros((hb, wb), dtype=torch.int32, device="cuda") for _ in range(3)]
    out = [torch.empty((hb, wb), dtype=torch.float32, device="cuda") for _ in range(3)]
    with pytest.raises(ValueError):                                 # an output plane aliases an input plane
        recon.lf_preview_dev(p, sd, 0.0, 1.0, True, [a.data_ptr() for a in qd], ep, hb, wb, [qd[0].data_ptr()] + [o.data_ptr() for o in out[1:]])
    ch = [np.zeros((20, 30), np.int32), np.zeros((20, 30), np.float32)]
    assert [a.shape for a in recon.areaMean8(ch, [8, 8])] == [(3, 4), (3, 4)]
    with pytest.raises(ValueError):                                 # int32 channel without a usable depth
        recon.areaMean8(ch, [0, 8])
    with pytest.raises(ValueError):                                 # channels of different sizes
        recon.areaMean8([ch[0], np.zeros((20, 31), np.float32)], [8, 8])
    a = torch.zeros((16, 16), dtype=torch.float32, device="cuda")
    with pytest.raises(ValueError):
        recon.area_mean8_dev([a.data_ptr()], [False], [8], 16, 16, [a.data_ptr()])
    torch.cuda.synchronize()
