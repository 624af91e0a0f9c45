"""Modular inverse transforms on the GPU (through the C ABI) against the oracle: bit-exact (int32, Java semantics)."""
import numpy as np
import pytest

from jxlatte_b200.host import ModularTransforms, RCT, PALETTE, SQUEEZE, default_squeeze_params, forward_channel_layout

pytestmark = pytest.mark.gpu


def _rand(rng, shape, lo=-70000, hi=70000):
    return rng.integers(lo, hi, size=shape, dtype=np.int64).astype(np.int32)


@pytest.mark.parametrize("rct_type", range(42))
def test_rct_all_types_and_permutations(recon, orc, rct_type):
    rng = np.random.default_rng(rct_type)
    ch = _rand(rng, (3, 37, 53))
    ch[0, 0, 0] = 2 ** 31 - 1          # wrap-around must match Java int arithmetic
    ch[2, 0, 0] = 2 ** 31 - 5
    ref = orc.modular_rct(ch, rct_type)
    got = np.stack(recon.inverseRCT(ch, rct_type))
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("shape", [(1, 1), (1, 2), (5, 9), (64, 64), (33, 100), (200, 7), (257, 511)])
@pytest.mark.parametrize("horizontal", [True, False])
def test_squeeze_round_trip_and_oracle(recon, orc, shape, horizontal):
    rng = np.random.default_rng(shape[0] * 7 + shape[1] + int(horizontal))
    x = _rand(rng, shape, -5000, 5000)
    avg, res = orc.modular_forward_squeeze(x, horizontal)
    ref = orc.modular_squeeze(avg, res, horizontal)
    assert np.array_equal(ref, x)      # the oracle inverts its own forward
    got = recon.inverseHorizontalSqueeze(avg, res) if horizontal else recon.inverseVerticalSqueeze(avg, res)
    assert np.array_equal(got, ref)
    # arbitrary residuals (not produced by a forward transform) still have to match
    res2 = _rand(rng, res.shape, -300, 300)
    ref2 = orc.modular_squeeze(avg, res2, horizontal)
    got2 = recon.inverseHorizontalSqueeze(avg, res2) if horizontal else recon.inverseVerticalSqueeze(avg, res2)
    assert np.array_equal(got2, ref2)


def test_squeeze_rejects_mismatched_channels(recon):
    with pytest.raises(ValueError):
        recon.inverseHorizontalSqueeze(np.zeros((4, 4), np.int32), np.zeros((4, 2), np.int32))


@pytest.mark.parametrize("d_pred", [0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12, 13])
@pytest.mark.parametrize("bit_depth", [8, 12])
def test_palette_with_deltas_every_predictor(recon, orc, d_pred, bit_depth):
    rng = np.random.default_rng(d_pred * 31 + bit_depth)
    h, w, num_c, nb_colors, nb_deltas = 45, 61, 3, 20, 6
    palette = _rand(rng, (num_c, nb_colors), 0, 1 << bit_depth)
    # indices: mostly plain colours, some synthetic (>= nb_colors, both ranges), some negative (delta palette), some < nb_deltas
    idx = rng.integers(0, nb_colors, size=(h, w)).astype(np.int32)
    m = rng.random((h, w))
    idx[m < 0.08] = rng.integers(nb_colors, nb_colors + 64, size=int((m < 0.08).sum()))
    idx[(m >= 0.08) & (m < 0.12)] = rng.integers(nb_colors + 64, nb_colors + 64 + 125, size=int(((m >= 0.08) & (m < 0.12)).sum()))
    idx[(m >= 0.12) & (m < 0.2)] = -rng.integers(1, 300, size=int(((m >= 0.12) & (m < 0.2)).sum()))
    ref = orc.modular_palette(idx, palette, nb_deltas, d_pred, bit_depth)
    got = np.stack(recon.inversePalette(idx, palette, nb_deltas, d_pred, bit_depth))
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("d_pred", [0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12, 13])
def test_palette_with_deltas_across_row_bands(recon, orc, d_pred):
    """k4_palette_delta runs as one 1024-thread CTA sweeping bands of 1024 rows: heights at, one past and two bands past the band
    size, and widths of 1, 2, 3 and 61 columns, where the predictors' north / west fallbacks decide most samples."""
    rng = np.random.default_rng(1000 + d_pred)
    num_c, nb_colors, nb_deltas = 3, 20, 6
    palette = _rand(rng, (num_c, nb_colors), 0, 256)
    for h in (1024, 1025, 2100):
        for w in (1, 2, 3, 61):
            idx = rng.integers(0, nb_colors, size=(h, w)).astype(np.int32)
            m = rng.random((h, w))
            idx[m < 0.3] = rng.integers(0, nb_deltas, size=int((m < 0.3).sum()))          # delta entries: predicted + palette
            idx[(m >= 0.3) & (m < 0.35)] = rng.integers(nb_colors, nb_colors + 64, size=int(((m >= 0.3) & (m < 0.35)).sum()))
            idx[(m >= 0.35) & (m < 0.4)] = -rng.integers(1, 300, size=int(((m >= 0.35) & (m < 0.4)).sum()))
            ref = orc.modular_palette(idx, palette, nb_deltas, d_pred, 8)
            got = np.stack(recon.inversePalette(idx, palette, nb_deltas, d_pred, 8))
            assert np.array_equal(got, ref), "%dx%d: first difference at %s" % (h, w, np.argwhere(got != ref)[:1].tolist())


def test_palette_without_deltas_is_a_gather(recon, orc):
    rng = np.random.default_rng(2)
    palette = _rand(rng, (4, 256), 0, 256)
    idx = rng.integers(0, 256, size=(300, 500)).astype(np.int32)
    ref = orc.modular_palette(idx, palette, 0, 0, 8)
    got = np.stack(recon.inversePalette(idx, palette, 0, 0, 8))
    assert np.array_equal(got, ref)


def test_palette_weighted_predictor_is_unsupported(recon):
    with pytest.raises(NotImplementedError):
        recon.inversePalette(np.zeros((4, 4), np.int32), np.zeros((1, 2), np.int32), 1, 6, 8)


def test_apply_transforms_default_squeeze_plus_rct(recon, orc):
    """ModularStream.applyTransforms on a decoded channel list: default squeeze pyramid (incl. the not-in-place chroma
    steps) undone on the GPU, then RCT -- against the same sequence applied with the oracle."""
    rng = np.random.default_rng(8)
    h, w = 40, 72
    img = _rand(rng, (3, h, w), 0, 256)
    sp = default_squeeze_params([(h, w)] * 3, 0)
    # forward: replay the constructor's channel bookkeeping with the oracle's forward squeeze
    ch = [img[c].copy() for c in range(3)]
    for (horizontal, in_place, begin, num_c) in sp:
        end = begin + num_c - 1
        offset = end + 1 if in_place else len(ch)
        for k in range(begin, end + 1):
            avg, res = orc.modular_forward_squeeze(ch[k], horizontal)
            ch[k] = avg
            ch.insert(offset + k - begin, res)
    assert [c.shape for c in ch] == forward_channel_layout([(h, w)] * 3, sp)
    mt = ModularTransforms(recon, bit_depth=8)
    out = mt.applyTransforms(ch, [{"tr": RCT, "begin_c": 0, "rct_type": 0}, {"tr": SQUEEZE, "sp": sp}])
    assert len(out) == 3
    for c in range(3):
        assert np.array_equal(out[c], img[c])
    # with a real RCT in front: decoded channels hold the forward-RCT'd image; undo squeeze then RCT type 6 perm 1
    out2 = mt.applyTransforms(ch, [{"tr": RCT, "begin_c": 0, "rct_type": 13}, {"tr": SQUEEZE, "sp": sp}])
    ref2 = orc.modular_rct(img, 13)
    for c in range(3):
        assert np.array_equal(out2[c], ref2[c])
