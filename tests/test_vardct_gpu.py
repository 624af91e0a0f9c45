"""Parity of the CUDA VarDCT path (through the C ABI) against the CPU oracle on identical synthetic frame state.

Tolerances (BASELINE.json north_star): max abs error <= 1e-4 on linear float planes; <= 1 LSB after sRGB 8/16-bit
quantisation.  Stage 1 (dequant/CfL/LLF/IDCT) and the staged stage 2 evaluate the reference's float operations in the
reference's order, so they are held to BIT-EXACT equality with the oracle; the fused stage-2 kernel reassociates the EPF
sums and is held to the stated tolerances.
"""
import numpy as np
import pytest

from jxlatte_b200 import synth, default_frame_params
from jxlatte_b200 import _lib
from jxlatte_b200.host import InvalidBitstreamError, qm_generate
from jxlatte_b200.params import TRANSFORM_TYPES, TRANSFORM_NAMES
from kernel_trace import assert_stage2_kernel, launched_kernels

pytestmark = pytest.mark.gpu

TOL_LINEAR = 1e-4
TOL_XYB = 2e-5


def _state(w, h, seed, p, **kw):
    qw, qo = qm_generate()
    return synth.make_state(w, h, seed=seed, params=p, qm_weights=qw, qm_offsets=qo, **kw)


def _single_type_state(t, p, seed):
    """A frame tiled with one TransformType."""
    H, W = p.height, p.width
    st = _state(W, H, seed, p, mix="dct8")
    _, _, ph, pw = TRANSFORM_TYPES[t]
    bh, bw = ph // 8, pw // 8
    hb, wb = H // 8, W // 8
    assert hb % bh == 0 and wb % bw == 0
    st["dct_select"][:] = t
    org = np.zeros((hb, wb), np.uint8)
    org[::bh, ::bw] = 1
    st["block_origin"] = org
    hm = st["hf_mul"][::bh, ::bw]
    st["hf_mul"] = np.ascontiguousarray(np.repeat(np.repeat(hm, bh, axis=0), bw, axis=1))
    rng = np.random.default_rng(seed + 99)
    # denser, small coefficients so every basis function is exercised
    q = (rng.integers(-3, 4, size=(3, H, W)) * (rng.random((3, H, W)) < 0.2)).astype(np.int32)
    st["qcoeff"] = q
    return st


@pytest.mark.parametrize("t", range(27))
def test_invert_every_transform_type(recon, orc, t):
    _, _, ph, pw = TRANSFORM_TYPES[t]
    H, W = max(256, ph), max(256, pw)
    p = default_frame_params(W, H, global_scale=32768)
    st = _single_type_state(t, p, seed=100 + t)
    ref = orc.vardct_invert(p, st, nthreads=8)
    got = recon.invertVarDCT(p, st)
    assert np.array_equal(got, ref), "%s: max abs err %g" % (TRANSFORM_NAMES[t], np.abs(got - ref).max())


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("shape", [(512, 512), (1280, 720), (264, 8), (8, 264), (776, 520)])
def test_invert_mixed_partition(recon, orc, shape, aligned):
    W, H = shape
    p = default_frame_params(W, H)
    st = _state(W, H, 7 + W + H, p, aligned=aligned)
    ref = orc.vardct_invert(p, st, nthreads=8)
    got = recon.invertVarDCT(p, st)
    assert np.array_equal(got, ref), "max abs err %g" % np.abs(got - ref).max()


def test_gaborish(recon, orc):
    p = default_frame_params(328, 200)
    rng = np.random.default_rng(3)
    planes = rng.random((3, 200, 328), dtype=np.float32)
    ref = orc.gab(p, planes)
    got = recon.performGabConvolution(p, planes)
    assert np.array_equal(got, ref)
    recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_STAGED)
    try:
        assert np.array_equal(recon.performGabConvolution(p, planes), ref)
    finally:
        recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)


@pytest.mark.parametrize("iters", [1, 2, 3])
def test_epf(recon, orc, iters):
    W, H = 328, 200
    p = default_frame_params(W, H, epf_iters=iters)
    rng = np.random.default_rng(4 + iters)
    planes = (rng.random((3, H, W), dtype=np.float32) * np.array([0.05, 1.0, 1.0], np.float32)[:, None, None])
    planes = planes * 0.2 + 0.4
    hm = rng.integers(1, 5, size=(H // 8, W // 8)).astype(np.int32)
    sh = rng.integers(0, 8, size=(H // 8, W // 8)).astype(np.int32)   # includes 0 = pass-through blocks
    ref = orc.epf(p, planes, hm, sh, nthreads=8)
    got = recon.performEdgePreservingFilter(p, planes, hm, sh)
    assert np.array_equal(got, ref), "max abs err %g" % np.abs(got - ref).max()
    for opt, exact in ((_lib.STAGE2_STAGED, True), (_lib.STAGE2_FUSED, False)):
        recon.set_option(_lib.OPT_STAGE2, opt)
        try:
            g2 = recon.performEdgePreservingFilter(p, planes, hm, sh)
        finally:
            recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)
        assert np.array_equal(g2, ref) if exact else np.abs(g2 - ref).max() <= 5e-6


@pytest.mark.parametrize("iters", [1, 3])
@pytest.mark.parametrize("stage2", ["stream", "tile", "staged"])
def test_epf_with_non_positive_hf_multipliers(recon, orc, iters, stage2):
    """HFMetadata takes the HF multiplier as 1 + a Modular-decoded value (HFMetadata.java:49): a crafted stream can make it zero or
    negative, sigma and 1/sigma then are infinite or negative and epfWeight's 1 - x exceeds 1.  Every stage-2 kernel must still follow
    the reference (the stream kernel clamps with a saturating subtract only in rows whose 1/sigma are all non-negative)."""
    W, H = 328, 200
    p = default_frame_params(W, H, epf_iters=iters)
    rng = np.random.default_rng(40 + iters)
    planes = (rng.random((3, H, W), dtype=np.float32) * np.array([0.05, 1.0, 1.0], np.float32)[:, None, None]) * 0.2 + 0.4
    hm = rng.integers(1, 5, size=(H // 8, W // 8)).astype(np.int32)
    sh = rng.integers(0, 8, size=(H // 8, W // 8)).astype(np.int32)
    hm[rng.random(hm.shape) < 0.2] = -3
    hm[rng.random(hm.shape) < 0.1] = 0
    sh[(hm < 0) & (sh == 0)] = 5          # sharpness 0 with a negative multiplier (1/sigma = -inf) breeds NaNs: out of this test's scope
    ref = orc.epf(p, planes, hm, sh, nthreads=8)
    assert np.isfinite(ref).all()
    recon.set_option(_lib.OPT_STAGE2, {"stream": _lib.STAGE2_STREAM, "tile": _lib.STAGE2_TILE, "staged": _lib.STAGE2_STAGED}[stage2])
    try:
        got, kernels = launched_kernels(lambda: recon.performEdgePreservingFilter(p, planes, hm, sh))
    finally:
        recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)
    assert_stage2_kernel(kernels, stage2, p)
    assert np.array_equal(got, ref), "max abs err %g" % np.abs(got - ref).max()


def test_stream_kernel_random_shapes(recon, orc):
    """The stream kernel (forced) against the oracle on thirty random frame shapes and filter settings, through the whole
    reconstruction: widths from one 8-pixel block to several column strips with a ragged last strip, heights from one block row to several
    chunks, every (gab, epf_iters >= 1).  The kernel trace shows that k2_stream, not its fallback, made each result."""
    rng = np.random.default_rng(20261017)
    qw, qo = qm_generate()
    recon.setWeights(qw, qo)
    for k in range(30):
        W = 8 * int(rng.integers(1, 64)) if k % 4 else 8 * int(rng.integers(100, 170))
        H = 8 * int(rng.integers(1, 48)) if k % 5 else 8 * int(rng.integers(60, 100))
        iters, gab = int(rng.integers(1, 4)), bool(rng.integers(0, 2))
        p = default_frame_params(W, H, epf_iters=iters, gab=gab)
        st = synth.make_state(W, H, seed=7000 + k, params=p, qm_weights=qw, qm_offsets=qo)
        recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_STREAM)
        try:
            got, kernels = launched_kernels(lambda: recon.reconstruct(p, st))
        finally:
            recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)
        assert_stage2_kernel(kernels, "stream", p)
        want = orc.vardct_reconstruct(p, st, nthreads=8)
        assert np.array_equal(got, want), "%dx%d gab %d epf %d: max abs err %g" % (W, H, gab, iters, np.abs(got - want).max())


def test_epf_rejects_bad_sharpness(recon):
    p = default_frame_params(64, 64, epf_iters=1)
    planes = np.zeros((3, 64, 64), np.float32)
    hm = np.ones((8, 8), np.int32)
    sh = np.full((8, 8), 9, np.int32)
    with pytest.raises(InvalidBitstreamError):
        recon.performEdgePreservingFilter(p, planes, hm, sh)


def test_color_transforms(recon, orc):
    W, H = 256, 64
    rng = np.random.default_rng(5)
    planes = rng.random((3, H, W), dtype=np.float32)
    planes[0] = (planes[0] - 0.5) * 0.05
    for mode in (0, 1, 2, 3):
        p = default_frame_params(W, H, color_mode=mode)
        ref = orc.color(p, planes)
        got = recon.performColorTransforms(p, planes)
        assert np.abs(got - ref).max() <= 2e-6 * max(1.0, np.abs(ref).max()), mode


def _srgb_quantise(lin, bits):
    """TransferFunction.TF_SRGB.fromLinearF (J/color/TransferFunction.java:39-43) + ImageBuffer.castToIntWithMax (:129-145)."""
    lin = lin.astype(np.float32)
    a = np.where(lin <= np.float32(0.0031308), lin * np.float32(12.92),
                 np.float32(1.055) * np.power(np.maximum(lin, 0), np.float32(1.0 / 2.4), dtype=np.float32) - np.float32(0.055))
    mx = (1 << bits) - 1
    v = (a.astype(np.float32) * np.float32(mx) + np.float32(0.5)).astype(np.int64)
    return np.clip(v, 0, mx)


@pytest.mark.parametrize("cfg", [
    dict(shape=(512, 512), iters=1, gab=True),      # lenna-like: gab on, EPF 1
    dict(shape=(1280, 720), iters=1, gab=True),     # bbb-like
    dict(shape=(1024, 768), iters=3, gab=True),     # 8K-config settings at a size the oracle does in seconds
    dict(shape=(520, 264), iters=2, gab=False),
    dict(shape=(264, 520), iters=0, gab=True),
    dict(shape=(256, 256), iters=0, gab=False),
])
@pytest.mark.parametrize("stage2", ["staged", "auto", "pair", "stream", "tile", "fast"])
def test_full_reconstruction(recon, orc, cfg, stage2):
    W, H = cfg["shape"]
    p = default_frame_params(W, H, epf_iters=cfg["iters"], gab=cfg["gab"])
    st = _state(W, H, 11 + W, p)
    ref = orc.vardct_reconstruct(p, st, nthreads=8)
    if stage2 == "fast" and not (cfg["gab"] or cfg["iters"]):
        pytest.skip("nothing to fuse")
    try:
        # auto = the faster of the two fused bit-exact kernels for the frame; stream = k2_stream wherever TMA applies; tile = k2_exact
        recon.set_option(_lib.OPT_STAGE2, {"staged": _lib.STAGE2_STAGED, "auto": _lib.STAGE2_AUTO, "pair": _lib.STAGE2_PAIR,
                                           "stream": _lib.STAGE2_STREAM, "tile": _lib.STAGE2_TILE, "fast": _lib.STAGE2_FUSED}[stage2])
    except NotImplementedError:
        pytest.skip("library built without this opt-in stage-2 variant (-DJXLB200_WITH_PAIR)")
    try:
        got, kernels = launched_kernels(lambda: recon.reconstruct(p, st))
    finally:
        recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)
    if stage2 in ("stream", "tile", "staged"):
        assert_stage2_kernel(kernels, stage2, p)
    if stage2 != "fast":
        assert np.array_equal(got, ref), "%s path must be bit-identical; max abs err %g" % (stage2, np.abs(got - ref).max())
    err = np.abs(got - ref).max()
    assert err <= TOL_LINEAR, "max abs err %g on linear planes" % err
    for bits in (8, 16):
        d = np.abs(_srgb_quantise(got, bits) - _srgb_quantise(ref, bits))
        # the opt-in re-associated EPF may move saturated dark pixels by 2 steps at 16 bits (documented in the header)
        lim = 2 if (stage2 == "fast" and bits == 16) else 1
        assert d.max() <= lim, "%d-bit sRGB differs by %d LSB" % (bits, d.max())
        assert (d > 1).mean() <= 1e-5


def test_invalid_transform_type_is_reported(recon):
    p = default_frame_params(64, 64)
    st = _state(64, 64, 1, p, mix="dct8")
    st["dct_select"][3, 3] = 31
    with pytest.raises(InvalidBitstreamError):
        recon.invertVarDCT(p, st)


def test_stage1_alone_rejects_chroma_subsampling(recon):
    p = default_frame_params(64, 64)
    p.shift_x[0] = 1
    st = _state(64, 64, 1, default_frame_params(64, 64), mix="dct8")
    with pytest.raises(NotImplementedError):
        recon.invertVarDCT(p, st)


def test_bad_arguments(recon):
    p = default_frame_params(64, 64)
    st = _state(64, 64, 1, p, mix="dct8")
    st["lf"] = st["lf"][:, :4]
    with pytest.raises(ValueError):
        recon.invertVarDCT(p, st)


# ---- chroma-subsampled frames (JPEG recompression; SURVEY.md 8f-2) ----
def _subsampled_state(W, H, shift_y, shift_x, seed):
    from jxlatte_b200 import synth
    p = default_frame_params(W, H, epf_iters=0, gab=False, color_mode=2)
    p.shift_y[:] = shift_y
    p.shift_x[:] = shift_x
    qw, qo = qm_generate()
    st = synth.make_state(W, H, seed=seed, mix=(1.0, 0.0, 0.0, 0.0, 0.0), params=p, qm_weights=qw, qm_offsets=qo)
    st = dict(st)
    st["qcoeff"] = [np.ascontiguousarray(st["qcoeff"][c][:H >> shift_y[c], :W >> shift_x[c]]) for c in range(3)]
    st["lf"] = [np.ascontiguousarray(st["lf"][c][:(H // 8) >> shift_y[c], :(W // 8) >> shift_x[c]]) for c in range(3)]
    return p, st, qw, qo


@pytest.mark.gpu
@pytest.mark.parametrize("shifts", [((1, 0, 1), (1, 0, 1)), ((0, 0, 0), (1, 0, 1)), ((1, 0, 1), (0, 0, 0)), ((0, 1, 1), (1, 1, 0))])
@pytest.mark.parametrize("filters", [(False, 0), (True, 2)])
def test_chroma_subsampled_frame_exact(recon, orc, shifts, filters):
    """4:2:0, 4:2:2, 4:4:0 and a mixed layout: stage 1 per channel on strided block maps + Frame.invertSubsampling."""
    W, H = 272, 144
    p, st, qw, qo = _subsampled_state(W, H, shifts[0], shifts[1], seed=0x4A584C00 + 77)
    p.gab, p.epf_iters = (1 if filters[0] else 0), filters[1]
    recon.setWeights(qw, qo)
    got = recon.reconstruct(p, st)
    want = orc.vardct_reconstruct(p, st, nthreads=4)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_chroma_subsampling_rejects_large_varblocks(recon):
    from jxlatte_b200 import synth
    W, H = 256, 256
    p = default_frame_params(W, H, epf_iters=0, gab=False, color_mode=2)
    p.shift_y[:] = (1, 0, 1)
    p.shift_x[:] = (1, 0, 1)
    qw, qo = qm_generate()
    st = dict(synth.make_state(W, H, seed=5, params=p, qm_weights=qw, qm_offsets=qo))
    st["qcoeff"] = [np.ascontiguousarray(st["qcoeff"][c][:H >> p.shift_y[c], :W >> p.shift_x[c]]) for c in range(3)]
    st["lf"] = [np.ascontiguousarray(st["lf"][c][:(H // 8) >> p.shift_y[c], :(W // 8) >> p.shift_x[c]]) for c in range(3)]
    recon.setWeights(qw, qo)
    with pytest.raises(NotImplementedError):
        recon.reconstruct(p, st)


@pytest.mark.gpu
def test_inconsistent_block_maps_are_rejected(recon):
    """A block_origin / dct_select pair that HFMetadata.placeBlock could never produce (a 64x64 varblock hanging over the
    frame edge, one crossing a group boundary) must come back as an invalid-stream error, not as out-of-bounds writes."""
    p = default_frame_params(320, 64)
    st = _state(320, 64, 1, p, mix="dct8")
    for (by, bx) in ((4, 0), (0, 36), (0, 28)):          # leaves the frame at the bottom / at the right / crosses x = 256
        bad = dict(st)
        bad["dct_select"] = st["dct_select"].copy()
        bad["dct_select"][by, bx] = 18                   # DCT64
        with pytest.raises(InvalidBitstreamError):
            recon.invertVarDCT(p, bad)
    assert np.isfinite(recon.invertVarDCT(p, st)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("H", [8, 264, 520, 776, 1032, 1288, 1544, 2056])
def test_host_entry_slab_schedule_exact(recon, orc, H):
    """The pipelined host entry point cuts tall frames into group-row slabs (the first two and the last two one group row
    high, 512 rows in between): every schedule shape must give the whole-frame result."""
    W = 72
    p = default_frame_params(W, H, epf_iters=3)
    st = _state(W, H, 100 + H, p, mix="small")
    assert np.array_equal(recon.reconstruct(p, st), orc.vardct_reconstruct(p, st, nthreads=8))


@pytest.mark.gpu
@pytest.mark.parametrize("H", [8, 520, 1288])
def test_host_entry_int16_coefficients_exact(recon, orc, H):
    """jxlb200_vardct_reconstruct_i16: coefficients narrowed to int16 by the caller, widened on the device -- the int32
    call's result bit for bit, on a single slab and on pipelined ones."""
    W = 72
    p = default_frame_params(W, H, epf_iters=3)
    st = _state(W, H, 300 + H, p, mix="small")
    want = orc.vardct_reconstruct(p, st, nthreads=8)
    assert np.array_equal(recon.reconstruct(p, st, narrow=True), want)
    st16 = dict(st)
    st16["qcoeff"] = [np.ascontiguousarray(st["qcoeff"][c], dtype=np.int16) for c in range(3)]
    assert np.array_equal(recon.reconstruct(p, st16, narrow=True), want)
    wide = dict(st)
    wide["qcoeff"] = [st["qcoeff"][c].copy() for c in range(3)]
    wide["qcoeff"][1][0, 1] = 40000
    with pytest.raises(ValueError):
        recon.reconstruct(p, wide, narrow=True)


@pytest.mark.gpu
def test_chroma_subsampled_frame_int16_coefficients_exact(recon, orc):
    W, H = 272, 144
    p, st, qw, qo = _subsampled_state(W, H, (1, 0, 1), (1, 0, 1), seed=0x4A584C00 + 78)
    p.gab, p.epf_iters = 1, 2
    recon.setWeights(qw, qo)
    assert np.array_equal(recon.reconstruct(p, st, narrow=True), orc.vardct_reconstruct(p, st, nthreads=4))


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [dict(W=520, H=264, bits=8, narrow=False, crop=(517, 259)), dict(W=328, H=1288, bits=16, narrow=True, crop=(328, 1288)),
                                 dict(W=72, H=776, bits=8, narrow=True, crop=(65, 770))])
def test_packed_output_matches_oracle_pack(recon, orc, cfg):
    """jxlb200_vardct_reconstruct_packed: sRGB transfer + 8/16-bit quantise + interleave on the device (single slab and the
    pipelined schedule) == the oracle's planes through the oracle's PNGWriter sample pipeline, byte for byte."""
    W, H = cfg["W"], cfg["H"]
    p = default_frame_params(W, H, epf_iters=3)
    st = _state(W, H, 500 + W, p, mix="small") if W < 100 else _state(W, H, 500 + W, p)
    planes = orc.vardct_reconstruct(p, st, nthreads=8)
    cw, ch = cfg["crop"]
    want = orc.pack_samples([np.ascontiguousarray(planes[c][:ch, :cw]) for c in range(3)], [cfg["bits"]] * 3, 3, True, cfg["bits"])
    got = recon.reconstruct_packed(p, st, bits=cfg["bits"], linear=True, crop=(cw, ch), narrow=cfg["narrow"])
    assert got.shape == want.shape and np.array_equal(got, want)
    # without the transfer function (an image that is already display-referred, e.g. JPEG-recompressed YCbCr)
    want2 = orc.pack_samples([np.ascontiguousarray(planes[c][:ch, :cw]) for c in range(3)], [cfg["bits"]] * 3, 3, False, cfg["bits"])
    assert np.array_equal(recon.reconstruct_packed(p, st, bits=cfg["bits"], linear=False, crop=(cw, ch)), want2)
    with pytest.raises(ValueError):
        recon.reconstruct_packed(p, st, bits=12)


@pytest.mark.gpu
def test_shared_reciprocal_divide(recon):
    """k2_exact divides a pixel's three channel sums by one sum of weights with a reciprocal refined once (the fast path of
    __fdiv_rn itself, shared): on 2^26 operand pairs per seed -- divisors 1..13, numerators image-like, tiny, huge, zero, denormal
    bit patterns -- every result must equal __fdiv_rn's bit for bit."""
    for seed in (1, 2, 3):
        assert recon.selftest_divide(1 << 26, seed) == 0


@pytest.mark.gpu
def test_registered_caller_buffers(recon, orc):
    """jxlb200_host_register: a caller's ordinary (pageable) buffers page-locked in place, used by the pipelined host entry
    point, then released -- same planes as ever."""
    W, H = 264, 1032
    p = default_frame_params(W, H, epf_iters=2)
    st = dict(_state(W, H, 77, p))
    st["qcoeff"] = np.array(st["qcoeff"], np.int32, order="C", copy=True)
    out = np.empty((3, H, W), np.float32)
    recon.host_register(st["qcoeff"]); recon.host_register(out)
    try:
        got = recon.reconstruct(p, st, out=out)
    finally:
        recon.host_unregister(st["qcoeff"]); recon.host_unregister(out)
    assert np.array_equal(got, orc.vardct_reconstruct(p, st, nthreads=8))
