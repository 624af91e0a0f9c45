"""Float64 references for the stages after stage 1 (stage 1 itself: test_stage1_f64.py), each compared with the CPU oracle and the kernel.

The oracle was written from the same reading of the Java as the kernels, so "bit-identical to the oracle" cannot catch a misreading
the two share.  Each reference below restates one stage as mathematics -- whole-plane shifts of a mirror-padded float64 array, no
per-pixel loops -- and cites the Java lines the oracle cites (J/ = java/com/traneptora/jxlatte/ in the reference tree).

Tolerances.  A linear stage is held to a bound computed per output pixel from its own terms, c * 2^-24 * sum |w_i * x_i|, with c the
number of float32 operations on the longest chain from an input sample (or a float32 weight) to the output.  EPF and noise are not
linear; each has one stated constant, derived in its docstring.  Every comparison also evaluates the reference once with a plausible
bug and asserts that the same check rejects it by at least ten times the bound, so no check can pass by being blind.
"""
import numpy as np
import pytest

from jxlatte_b200 import _lib, default_frame_params
from jxlatte_b200.upsampling import up_weights

U = 2.0 ** -24                                   # unit roundoff of float32
FLOAT_MIN_VALUE = float(np.float32(1.401298464324817e-45))   # Java's Float.MIN_VALUE: the smallest POSITIVE float
SRGB_KNEE = float(np.float32(0.00313066844250063))           # TF_SRGB.fromLinearF's branch point, as the float literal it is


def frame_params(w, h, **kw):
    """default_frame_params at any size (a Modular frame has its own, not a multiple of 8)."""
    p = default_frame_params(8, 8, **kw)
    p.width, p.height = w, h
    return p


# ---- edges -------------------------------------------------------------------------------------------------------------
def mirror_index(n, lo, hi):
    """MathHelper.mirrorCoordinate (J/util/MathHelper.java:323-329) of every coordinate in [lo, hi): the plane reflected about
    its edges with the edge sample repeated, which is periodic with period 2n -- so a reach beyond the plane reflects again."""
    m = np.arange(lo, hi) % (2 * n)
    return np.where(m >= n, 2 * n - 1 - m, m)


def pad(a, r):
    """Mirror-pad the last two axes by r."""
    h, w = a.shape[-2:]
    return a[..., mirror_index(h, -r, h + r)[:, None], mirror_index(w, -r, w + r)[None, :]]


def shifted(P, r, dy, dx, h, w):
    """The plane P (padded by r) moved so that element [y, x] is the original's [y + dy, x + dx]."""
    return P[..., r + dy:r + dy + h, r + dx:r + dx + w]


def compare(got, ref, bound):
    """(largest |got - ref|, largest |got - ref| / bound)."""
    err = np.abs(np.asarray(got, np.float64) - ref)
    assert not np.isnan(err).any()
    return float(err.max()), float((err / np.maximum(bound, 1e-300)).max())


def assert_within(got, ref, bound, what):
    err, ratio = compare(got, ref, bound)
    assert ratio <= 1.0, "%s: max abs err %.3g is %.2f x its bound" % (what, err, ratio)


def assert_rejects(bug, ref, bound, what):
    """The check of assert_within, applied to the reference evaluated with a plausible bug, fails by 10 x or more."""
    err, ratio = compare(bug, ref, bound)
    assert ratio >= 10.0, "%s: the check does not see this bug (max abs diff %.3g, only %.2f x the bound)" % (what, err, ratio)


def test_mirror_padding_matches_oracle(orc):
    for n in (1, 2, 3, 10):
        assert list(mirror_index(n, -4 * n - 7, 5 * n + 7)) == [orc.mirror_coordinate(c, n) for c in range(-4 * n - 7, 5 * n + 7)]
    a = np.arange(6.0).reshape(2, 3)
    P = pad(a, 2)                                # a 5 x 5 reach on a 2 x 3 plane reflects more than once
    assert P.shape == (6, 7) and list(P[2]) == [1, 0, 0, 1, 2, 2, 1] and list(P[:, 2]) == [3, 0, 0, 3, 3, 0]


# ---- Gaborish: Frame.performGabConvolution (J/frame/Frame.java:505-542) ------------------------------------------------
GAB_OPS = 11     # weights: 1 + 4 (w1 + w2) (3), 1 / that (1), w * mult (1); 4-term sum (3); product (1); 3-term sum (2)
ADJ = ((0, -1), (0, 1), (-1, 0), (1, 0))
DIAG = ((-1, -1), (-1, 1), (1, -1), (1, 1))


def gab_ref(p, planes):
    """-> (out, bound).  The Java clamps a neighbour to the plane (y == 0 ? 0 : y - 1); for a reach of one that is mirroring."""
    x = np.asarray(planes, np.float64)
    h, w = x.shape[1:]
    P = pad(x, 1)
    adj = [shifted(P, 1, dy, dx, h, w) for dy, dx in ADJ]
    diag = [shifted(P, 1, dy, dx, h, w) for dy, dx in DIAG]
    out, bound = np.empty_like(x), np.empty_like(x)
    for c in range(3):
        w1, w2 = float(p.gab_w1[c]), float(p.gab_w2[c])
        m = 1.0 / (1.0 + 4.0 * (w1 + w2))
        out[c] = m * x[c] + w1 * m * sum(a[c] for a in adj) + w2 * m * sum(d[c] for d in diag)
        bound[c] = GAB_OPS * U * (abs(m) * np.abs(x[c]) + abs(w1 * m) * sum(np.abs(a[c]) for a in adj)
                                  + abs(w2 * m) * sum(np.abs(d[c]) for d in diag))
    return out, bound


def gab_bug(p, planes):
    """w1 and w2 swapped."""
    q = p.copy()
    q.gab_w1[:], q.gab_w2[:] = list(p.gab_w2), list(p.gab_w1)
    return gab_ref(q, planes)[0]


# ---- EPF: Frame.performEdgePreservingFilter (J/frame/Frame.java:544-679) -----------------------------------------------
CROSS = ((0, 0), (0, -1), (0, 1), (-1, 0), (1, 0))                                            # epfCross, Point(y, x)
DOUBLE_CROSS = CROSS + ((-1, 1), (1, 1), (1, -1), (-1, -1), (0, -2), (0, 2), (2, 0), (-2, 0))  # epfDoubleCross
TOL_EPF = 2e-6
"""EPF tolerance (absolute), for the inputs of epf_planes: samples |x| <= 0.5 whose range R over a 5 x 5 patch is <= 0.03.  One pass
is out = sum_k w_k x_k / sum_k w_k with w_k = max(0, 1 - s d_k), d_k a float32 sum of up to 15 scaled absolute differences.  The
centre tap has d = 0 and w = 1, so sum_k w_k >= 1 and d out / d w_k = (x_k - out) / sum w is at most R.  Float32 rounding gives d_k a
relative error <= 17u and w_k an absolute one <= 20u (s d_k < 1 wherever w_k > 0): 13 taps move the output by <= 13 * 20u * R =
4.6e-7; the two 13-term float32 sums and the divide add <= 16u * max |x| = 4.8e-7.  So one pass is off by <= 9.4e-7 in the worst
case.  Later passes carry the earlier error through weights that depend on it, which could amplify it a few times at worst, but the
roundings of neighbouring taps are independent and mostly cancel: the largest error measured against the oracle is 1.6e-7 over every
shape, sigma map and pass count here, and it grows by less than 2x from one pass to three.  2e-6 is twice the single-pass worst case
and 12x the largest measured error; each bug below moves some pixel by 10x it or more."""


def epf_inv_sigma(p, hf_mul, sharpness):
    """Per-pixel 1/sigma of a VarDCT frame: sigma = 65536 / globalScale * epfSharpLut[sharpness] / hfMul per 8 x 8 block."""
    sigma = 65536.0 / p.global_scale * np.array(list(p.epf_sharp_lut), np.float64)[sharpness] / hf_mul
    with np.errstate(divide="ignore"):
        inv = 1.0 / sigma
    # a sigma within float32 rounding of the pass-through threshold 0.3 could go either way: the inputs keep clear of it
    assert not (np.abs(sigma - 0.3) < 1e-4).any()
    return np.repeat(np.repeat(inv, 8, axis=0), 8, axis=1)[:p.height, :p.width]


def _on_border(y, x):
    return ((y & 7) == 0) | ((y & 7) == 7) | ((x & 7) == 0) | ((x & 7) == 7)


def epf_ref(p, planes, inv_sigma, bug=None):
    """-> (out, fraction of the non-centre weights strictly between 0 and 1).  inv_sigma: per-pixel 1/sigma.
    Passes 0 / 1 / 2 run for epf_iters 3 / >= 1 / >= 2 (SURVEY A13); a pixel whose 1/sigma is NaN or above 1 / 0.3 passes through
    (:604-609); the border SAD multiplier is keyed on the CENTRE pixel's (y & 7, x & 7) (epfWeight :671-679, SURVEY A12).
    bug = "neighbour": multiplier keyed on the neighbour's position; "swap12": passes 1 and 2 in the wrong order."""
    x = np.asarray(planes, np.float64)
    h, w = x.shape[1:]
    passes = ([0] if p.epf_iters == 3 else []) + [1] + ([2] if p.epf_iters >= 2 else [])
    if bug == "swap12" and 2 in passes:
        passes[-2:] = [2, 1]
    step = 1.65 * 4.0 * (1.0 - np.sqrt(0.5))
    scale = np.array(list(p.epf_channel_scale), np.float64)[:, None, None]
    yy, xx = np.mgrid[0:h, 0:w]
    through = ~(inv_sigma <= 1.0 / 0.3)
    inv = np.where(through, 0.0, inv_sigma)
    mid = total = 0
    for i in passes:
        s = step * {0: p.epf_pass0_sigma_scale, 1: 1.0, 2: p.epf_pass2_sigma_scale}[i] * inv
        P = pad(x, 3)

        def at(dy, dx):
            return shifted(P, 3, dy, dx, h, w)
        sw, sc = 0.0, 0.0
        for dy, dx in DOUBLE_CROSS if i == 0 else CROSS:
            if i == 2:                                               # epfDistance2 :657-669
                d = (scale * np.abs(x - at(dy, dx))).sum(0)
            else:                                                    # epfDistance1 :638-655
                d = sum((scale * np.abs(at(ey, ex) - at(dy + ey, dx + ex))).sum(0) for ey, ex in CROSS)
            border = _on_border(yy + dy, xx + dx) if bug == "neighbour" else _on_border(yy, xx)
            d = np.where(border, d * p.epf_border_sad_mul, d)
            wk = np.maximum(0.0, 1.0 - d * s)
            if (dy, dx) != (0, 0):
                mid += int(((wk > 0) & (wk < 1) & ~through).sum())
                total += int((~through).sum())
            sw = sw + wk
            sc = sc + wk * at(dy, dx)
        x = np.where(through, x, sc / sw)
    return x, mid / max(total, 1)


def epf_planes(h, w, seed):
    """Step edges plus noise, small enough that most EPF weights fall strictly between 0 and 1."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    step = ((xx * 3 + yy * 5) % 23 < 11).astype(np.float64)
    amp = np.array([0.0004, 0.004, 0.004])[:, None, None]
    x = np.array([0.0, 0.45, 0.4])[:, None, None] + amp * (step + 0.5 * rng.standard_normal((3, h, w)))
    return x.astype(np.float32)


SHAPES = [(1, 1), (1, 13), (13, 1), (7, 9), (67, 45), (264, 136)]     # (h, w)
MODULAR_SIGMA = 0.7


# ---- colour: JXLCodestreamDecoder.performColorTransforms (J/JXLCodestreamDecoder.java:256-283), OpsinInverseMatrix.invertXYB
# (J/color/OpsinInverseMatrix.java:81-84, 105-142), the YCbCr -> RGB of the same method ------------------------------------
YCC = (128.0 / 255.0, 1.402, 0.344136286201022, 0.714136286201022, 1.772)


def color_ref(p, planes, bug=None):
    """-> (out, bound).  color_mode bit 0: XYB -> linear RGB; bit 1: YCbCr -> RGB, after XYB when both are set.
    bug = "xsign": X enters L and M with the opposite signs; "cbcr": the 1.402 / 1.772 factors of Cr and Cb swapped."""
    x = np.asarray(planes, np.float64)
    e = np.zeros_like(x)                                             # error bound carried through the two steps
    if p.color_mode & 1:
        bias = np.array(list(p.opsin_bias), np.float64)
        m = np.array(list(p.opsin_matrix), np.float64).reshape(3, 3) * (255.0 / p.intensity_target)
        sx = -1.0 if bug == "xsign" else 1.0
        g = [x[1] + sx * x[0] - np.cbrt(bias[0]), x[1] - sx * x[0] - np.cbrt(bias[1]), x[2] - np.cbrt(bias[2])]
        eg = [e[1] + e[0] + 3 * U * (np.abs(x[1]) + np.abs(x[0]) + abs(np.cbrt(bias[0]))),    # cbrt, two adds
              e[1] + e[0] + 3 * U * (np.abs(x[1]) + np.abs(x[0]) + abs(np.cbrt(bias[1]))),
              e[2] + 2 * U * (np.abs(x[2]) + abs(np.cbrt(bias[2])))]
        mix = [g[k] ** 3 + bias[k] for k in range(3)]
        emix = [3 * g[k] ** 2 * eg[k] + 3 * U * (np.abs(g[k]) ** 3 + abs(bias[k])) for k in range(3)]   # two muls, one add
        x = np.stack([sum(m[r, k] * mix[k] for k in range(3)) for r in range(3)])
        # the matrix itself is rounded twice (255 / intensity_target, times it), then 3 muls and 2 adds
        e = np.stack([sum(abs(m[r, k]) * (emix[k] + 7 * U * np.abs(mix[k])) for k in range(3)) for r in range(3)])
    if p.color_mode & 2:
        half, kr, kgb, kgr, kb = YCC
        if bug == "cbcr":
            kr, kb = kb, kr
        cb, y, cr = x
        yh = y + half
        x = np.stack([yh + kr * cr, yh - kgb * cb - kgr * cr, yh + kb * cb])
        ay = np.abs(y) + half
        e = np.stack([e[1] + kr * e[2] + 3 * U * (ay + kr * np.abs(cr)),
                      e[1] + kgb * e[0] + kgr * e[2] + 4 * U * (ay + kgb * np.abs(cb) + kgr * np.abs(cr)),
                      e[1] + kb * e[0] + 3 * U * (ay + kb * np.abs(cb))])
    return x, e


def color_planes(h, w, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((3, h, w))
    x[0] = (x[0] - 0.5) * 0.05
    return x.astype(np.float32)


# ---- upsampling: Frame.performUpsampling (J/frame/Frame.java:217-260), ImageHeader.getUpWeights (J/bundle/ImageHeader.java:441-470)
UP_OPS = 25      # 25 products accumulated in order: the first product, then 24 adds (each add rounds once, each product once)


def upsample_ref(a, k, weights, edge="mirror"):
    """-> (out, bound).  Output phase (ky, kx) of input pixel (y, x) is the 5 x 5 correlation of the mirrored neighbourhood with
    weights[ky][kx], clamped to the window's [min, max] -- where max starts at Float.MIN_VALUE, the smallest POSITIVE float, so a
    window with no positive sample clamps at ~0 (the Java's quirk, kept by the oracle and the kernel; see k8_features.cuh)."""
    x = np.asarray(a, np.float64)
    h, w = x.shape
    P = pad(x, 2) if edge == "mirror" else np.pad(x, 2, mode="edge")
    win = np.stack([shifted(P, 2, iy - 2, ix - 2, h, w) for iy in range(5) for ix in range(5)])
    wt = np.asarray(weights, np.float64).reshape(k, k, 25)
    tot = np.einsum("abt,thw->hawb", wt, win).reshape(h * k, w * k)
    bound = UP_OPS * U * np.einsum("abt,thw->hawb", np.abs(wt), np.abs(win)).reshape(h * k, w * k)
    lo = np.repeat(np.repeat(win.min(0), k, axis=0), k, axis=1)
    hi = np.repeat(np.repeat(np.maximum(win.max(0), FLOAT_MIN_VALUE), k, axis=0), k, axis=1)
    return np.clip(tot, lo, hi), bound


def test_up_weights_facts():
    """Facts about the expanded tables that do not depend on how the expansion is written: every phase kernel sums to 1; the table
    is symmetric under ky -> k-1-ky with iy -> 4-iy (and the same in x), and under transposition."""
    for k in (2, 4, 8):
        w = up_weights(k).astype(np.float64)
        assert w.shape == (k, k, 5, 5)
        assert np.abs(w.sum(axis=(2, 3)) - 1.0).max() <= 1e-7, k
        assert np.array_equal(w, w[::-1, :, ::-1, :]) and np.array_equal(w, w[:, ::-1, :, ::-1])
        assert np.array_equal(w, w.transpose(1, 0, 3, 2))
        assert not np.array_equal(w, w.transpose(1, 0, 2, 3))      # so swapping the phases alone is a real bug


UP_SHAPES = [(1, 1), (1, 2), (2, 1), (2, 3), (1, 37), (37, 1), (37, 61), (64, 5)]


def up_plane(shape, seed):
    return np.random.default_rng(seed).uniform(-1.0, 1.5, shape).astype(np.float32)


# ---- chroma upsampling: Frame.invertSubsampling (J/frame/Frame.java:681-723) ---------------------------------------------
CHROMA_OPS = 6   # per doubling: 0.75 * x, 0.25 * neighbour, the add; at most two doublings


def _double(x, axis, near, far):
    """One 2x doubling along axis: sample 2i = near * x[i] + far * x[i - 1], 2i + 1 = near * x[i] + far * x[i + 1], edges clamped."""
    x = np.moveaxis(x, axis, -1)
    P = np.concatenate([x[..., :1], x, x[..., -1:]], axis=-1)       # clamp == mirror at a reach of one
    out = np.empty(x.shape[:-1] + (2 * x.shape[-1],))
    out[..., 0::2] = near * x + far * P[..., :-2]
    out[..., 1::2] = near * x + far * P[..., 2:]
    return np.moveaxis(out, -1, axis)


def chroma_ref(p, sub, near=0.75, far=0.25):
    """-> (out [3, H, W], bound).  Per channel: shift_x horizontal doublings, then shift_y vertical ones.  All weights are
    positive, so sum |w_i x_i| is the same operator applied to |x|."""
    out, bound = [], []
    for c in range(3):
        x = np.asarray(sub[c], np.float64)
        b = np.abs(x)
        for _ in range(p.shift_x[c]):
            x, b = _double(x, 1, near, far), _double(b, 1, 0.75, 0.25)
        for _ in range(p.shift_y[c]):
            x, b = _double(x, 0, near, far), _double(b, 0, 0.75, 0.25)
        out.append(x)
        bound.append(CHROMA_OPS * U * b)
    return np.stack(out), np.stack(bound)


CHROMA_SHIFTS = [((1, 0, 1), (1, 0, 1)), ((0, 0, 0), (1, 0, 1)), ((1, 0, 1), (0, 0, 0)), ((0, 1, 1), (1, 1, 0))]
CHROMA_SIZES = [(16, 16), (48, 32), (272, 144)]          # (W, H); 16 x 16 is the smallest subsampled frame the library takes


# ---- noise: XorShiro (J/frame/features/XorShiro.java), Frame.initializeNoise / synthesizeNoise (J/frame/Frame.java:748-835) --
M64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15


def splitmix64(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def xorshiro_batches(seed0, seed1, n):
    """n batches of 16 uint32 values: eight xorshift128+ lanes seeded by SplitMix64 chains; lane i gives values 2i (low half of
    its sum) and 2i + 1 (high half)."""
    s0, s1 = [splitmix64((seed0 + GOLDEN) & M64)], [splitmix64((seed1 + GOLDEN) & M64)]
    for _ in range(7):
        s0.append(splitmix64(s0[-1]))
        s1.append(splitmix64(s1[-1]))
    s0, s1 = np.array(s0, np.uint64), np.array(s1, np.uint64)
    out = np.empty((n, 8), np.uint64)
    for t in range(n):
        a, b = s1, s0
        out[t] = a + b
        s0 = a
        b = b ^ (b << np.uint64(23))
        s1 = b ^ a ^ (b >> np.uint64(18)) ^ (a >> np.uint64(5))
    return np.stack([out & np.uint64(0xFFFFFFFF), out >> np.uint64(32)], axis=-1).reshape(n, 16)


def noise_uniforms(h, w, group_dim, seed0, swap_xy=False):
    """[3, h, w] samples in [1, 2): per group of group_dim^2 pixels, an RNG seeded with (seed0, x0 << 32 | y0) fills channel by
    channel, row by row, 16 values at a time (the unused tail of a row's last batch is dropped); a value is 1 + (bits >> 9) / 2^23."""
    out = np.zeros((3, h, w))
    for y0 in range(0, h, group_dim):
        for x0 in range(0, w, group_dim):
            seed1 = (y0 << 32 | x0) if swap_xy else (x0 << 32 | y0)
            ys, xs = min(group_dim, h - y0), min(group_dim, w - x0)
            nbx = (xs + 15) // 16
            bits = xorshiro_batches(seed0, seed1, 3 * ys * nbx).reshape(3, ys, nbx * 16)[:, :, :xs]
            out[:, y0:y0 + ys, x0:x0 + xs] = 1.0 + (bits >> np.uint64(9)).astype(np.float64) / 2.0 ** 23
    return out


TOL_NOISE = 3e-5
"""Noise tolerance (absolute).  The Laplacian sums 25 float32 products of samples in [1, 2) with weights 0.16 and -3.84: error <=
26u * (24 * 0.16 + 3.84) * 2 ~ 2.4e-5 before the noise is scaled by at most 0.00171875 + 0.21828125 = 0.22 and by an intensity
factor <= 1, so ~5.3e-6 per channel term; nr + ng, then base_x * nrg + nr - ng add up to four of them (2.1e-5) plus roundings of
order u.  The intensity factor is a continuous piecewise-linear function of 3 (Y +- X) with slope < 1 here, so its own rounding
contributes below 1e-7.  3e-5 covers the sum; a wrong bit stream moves pixels by about 0.1."""


def noise_ref(planes, group_dim, seed0, lut, base_x, base_b, swap_xy=False):
    loc = noise_uniforms(planes.shape[1], planes.shape[2], group_dim, seed0, swap_xy)
    h, w = loc.shape[1:]
    P = pad(loc, 2)
    lap = np.full((5, 5), 0.16)
    lap[2, 2] = -3.84
    n = sum(lap[iy, ix] * shifted(P, 2, iy - 2, ix - 2, h, w) for iy in range(5) for ix in range(5))
    X, Y, B = np.asarray(planes, np.float64)
    lt = np.asarray(lut, np.float64)

    def strength(v):                                     # linear interpolation in the 8-entry LUT over [0, 7], clamped to [0, 1]
        v = 3.0 * np.maximum(v, 0.0)
        i = np.where(v >= 7, 6, np.floor(np.minimum(v, 7))).astype(int)
        f = np.where(v >= 7, 1.0, v - i)
        return np.clip(lt[i] + (lt[i + 1] - lt[i]) * f, 0.0, 1.0)
    nr = strength(Y + X) * (0.00171875 * n[0] + 0.21828125 * n[2])
    ng = strength(Y - X) * (0.00171875 * n[1] + 0.21828125 * n[2])
    return np.stack([X + base_x * (nr + ng) + nr - ng, Y + nr + ng, B + base_b * (nr + ng)])


NOISE_CASES = [(20, 1030, 1024), (40, 1100, 512), (9, 600, 512), (300, 530, 256), (257, 17, 256), (1, 1, 256), (130, 7, 128),
               (5, 13, 128), (64, 40, 128)]   # (h, w, group_dim)


def noise_inputs(h, w, seed):
    rng = np.random.default_rng(seed)
    pl = np.stack([rng.uniform(-0.02, 0.02, (h, w)), rng.uniform(0.05, 0.9, (h, w)), rng.uniform(0.0, 0.9, (h, w))]).astype(np.float32)
    lut = rng.uniform(0.05, 0.6, 8).astype(np.float32)
    return pl, lut, (5 << 32) | 2


# ---- LF dequantisation, LF chroma-from-luma, adaptive smoothing: LFCoefficients (J/frame/vardct/LFCoefficients.java:61-103,
# adaptiveSmooth :113-179), per LF group of 256 x 256 blocks ----------------------------------------------------------------
LF_W = (0.05226273532324128, 0.20345139757231578, 0.0334829185968739)     # centre, each adjacent, each diagonal


def lf_ref(q, ep, sd, kx, kb, cfl, smooth, cross_groups=False):
    """-> (out, bound).  Every group is dequantised with its own extraPrecision; smoothing sees only the group's own samples and
    copies the group's border ring (and groups smaller than 3 x 3 entirely).  cross_groups=True is the bug: one smoothing pass over
    the whole plane.  The bound is carried through the non-linear gap with the derivatives of (s - wv) * g + wv."""
    q = np.asarray(q, np.float64)
    hb, wb = q.shape[1:]
    gcols = (wb + 255) // 256
    sd = np.array([float(v) for v in sd])
    div = 2.0 ** np.asarray(ep, np.float64).reshape(-1, gcols)
    div = np.repeat(np.repeat(div, 256, axis=0), 256, axis=1)[:hb, :wb]
    co = q * sd[:, None, None] / div                                  # exact in float32 too: a power-of-two divide and one product
    e = U * np.abs(co)
    if cfl:
        co = np.stack([co[0] + kx * co[1], co[1], co[2] + kb * co[1]])
        e = np.stack([e[0] + abs(kx) * e[1] + 2 * U * (np.abs(co[0]) + 2 * abs(kx) * np.abs(co[1])), e[1],
                      e[2] + abs(kb) * e[1] + 2 * U * (np.abs(co[2]) + 2 * abs(kb) * np.abs(co[1]))])
    if not smooth:
        return co, e
    out, bound = co.copy(), e.copy()
    groups = [(0, 0, hb, wb)] if cross_groups else [(y0, x0, min(256, hb - y0), min(256, wb - x0))
                                                       for y0 in range(0, hb, 256) for x0 in range(0, wb, 256)]
    for y0, x0, h, w in groups:
        if h < 3 or w < 3:
            continue
        c, ce = co[:, y0:y0 + h, x0:x0 + w], e[:, y0:y0 + h, x0:x0 + w]
        s, se = c[:, 1:-1, 1:-1], ce[:, 1:-1, 1:-1]

        def around(a, taps):
            return sum(a[:, 1 + dy:h - 1 + dy, 1 + dx:w - 1 + dx] for dy, dx in taps)
        wv = LF_W[0] * s + LF_W[1] * around(c, ADJ) + LF_W[2] * around(c, DIAG)
        terms = LF_W[0] * np.abs(s) + LF_W[1] * around(np.abs(c), ADJ) + LF_W[2] * around(np.abs(c), DIAG)
        wve = LF_W[0] * se + LF_W[1] * around(ce, ADJ) + LF_W[2] * around(ce, DIAG) + 7 * U * terms   # 4-term sum (3), product (1), 3-term sum (2), + 1
        gap = np.maximum(0.5, (np.abs(s - wv) * sd[:, None, None]).max(0))
        gape = ((se + wve + U * np.abs(s - wv)) * sd[:, None, None]).max(0) + U * gap
        g = np.maximum(0.0, 3.0 - 4.0 * gap)
        ge = np.where(g > 0, 4.0 * gape + 2 * U * (3.0 + 4.0 * gap), 4.0 * gape)
        out[:, y0 + 1:y0 + h - 1, x0 + 1:x0 + w - 1] = (s - wv) * g + wv
        bound[:, y0 + 1:y0 + h - 1, x0 + 1:x0 + w - 1] = ((se + wve) * g + np.abs(s - wv) * ge + wve
                                                          + 3 * U * (np.abs(s - wv) * (1 + g) + np.abs(wv)))
    return out, bound


LF_SIZES = (1, 2, 3, 255, 256, 257, 513)


def lf_inputs(hb, wb):
    rng = np.random.default_rng(hb * 1000 + wb)
    # gap = max(0.5, |s - wv| * scaledDequant) must cross 0.5 and 0.75 somewhere, so that the smoothing factor 3 - 4 gap takes
    # every value in [0, 1]: small steps with occasional spikes
    base = rng.integers(-50, 50, size=(3, 1, 1))
    q = (base + rng.integers(-3, 4, size=(3, hb, wb)) + 6 * (rng.random((3, hb, wb)) < 0.05)).astype(np.int32)
    ng = ((hb + 255) // 256) * ((wb + 255) // 256)
    ep = (np.arange(ng) * 3 + 1) % 4                                  # a different extraPrecision for neighbouring groups
    sd = [np.float32(0.61), np.float32(1.3), np.float32(0.87)]
    return q, ep.astype(np.uint8), sd, np.float32(0.013), np.float32(1.0 + 3.0 / 84.0)


# ---- PNG samples: TF_SRGB.fromLinearF (J/color/TransferFunction.java:39-43), ImageBuffer.castToInt0 / clamp
# (J/util/ImageBuffer.java:129-160), PNGWriter's interleave (J/io/PNGWriter.java:191-203) -------------------------------------
def pack_ref(ch, is_int, depth, n_color, linear, bits, rounding=0.5):
    """-> (samples int64 [h, w, C], near [h, w, C]): the float64 sample and whether its pre-rounding value lies within a few float32
    ulps of an integer, where a float32 evaluation may round to the neighbouring sample.  rounding=0 is the bug (truncation)."""
    maxv = (1 << bits) - 1
    q, near = [], []
    for c, a in enumerate(ch):
        if is_int[c] and depth[c] == bits:
            v = np.asarray(a, np.int64)
            q.append(np.clip(v, 0, maxv))
            near.append(np.zeros(v.shape, bool))
            continue
        f = np.asarray(a, np.float64) / ((1 << depth[c]) - 1) if is_int[c] else np.asarray(a, np.float64)
        if linear and c < n_color:
            with np.errstate(invalid="ignore"):
                f = np.where(f < SRGB_KNEE, f * 12.92, 1.055 * np.power(np.where(f < SRGB_KNEE, 1.0, f), 1 / 2.4) - 0.055)
        v = f * maxv + rounding
        with np.errstate(invalid="ignore"):
            near.append(np.abs(v - np.round(v)) <= 8 * U * (np.abs(f) * maxv + 1.0))
            t = np.where(np.isnan(v), 0.0, np.clip(np.trunc(np.nan_to_num(v, posinf=2.0 ** 40, neginf=-2.0 ** 40)), 0, maxv))
        q.append(t.astype(np.int64))
    return np.stack(q, -1), np.stack(near, -1)


def unpack(buf, bits):
    b = np.asarray(buf).astype(np.int64)
    return b[..., 0::2] * 256 + b[..., 1::2] if bits > 8 else b


def assert_pack_close(got, ref, near, what):
    """Samples may differ by one step, and only where the float64 value sits on a rounding boundary; such places are rare."""
    d = np.abs(got - ref)
    assert d.max() <= 1, "%s: a sample differs by %d" % (what, d.max())
    assert not (d[~near] > 0).any(), "%s: %d samples differ away from a rounding boundary" % (what, int((d[~near] > 0).sum()))
    assert (d > 0).sum() <= max(2, d.size // 1000), what
    return int((d > 0).sum())


def pack_cases():
    """Float planes with NaN, +-inf, negatives, the knee and its float neighbours; int planes with depth != bits and == bits."""
    rng = np.random.default_rng(11)
    special = np.array([np.nan, np.inf, -np.inf, -0.5, -1e-9, 0.0, SRGB_KNEE, np.nextafter(np.float32(SRGB_KNEE), np.float32(0)),
                        np.nextafter(np.float32(SRGB_KNEE), np.float32(1)), 1.0, 1.0000001, 7.5, 1e-30, 0.5], np.float32)
    out = []
    for w in range(1, 8):
        h = 5
        f = rng.uniform(-0.05, 1.1, (3, h, w)).astype(np.float32)
        flat = f.reshape(-1)
        flat[:special.size] = special[:flat.size]
        ints = rng.integers(-20, 1100, size=(h, w)).astype(np.int32)
        out.append((w, [f[0], f[1], f[2], ints], [False, False, False, True]))
    return out


# ========================================================================================================================
# oracle vs reference (CPU) -- with the negative controls
# ========================================================================================================================
@pytest.mark.parametrize("shape", SHAPES)
def test_gaborish_oracle_vs_f64(orc, shape):
    h, w = shape
    p = frame_params(w, h, epf_iters=0)
    x = epf_planes(h, w, 1) * np.float32(8.0) - np.float32(2.0)
    ref, bound = gab_ref(p, x)
    assert_within(orc.gab(p, x), ref, bound, "oracle Gaborish")
    if h * w > 1:
        assert_rejects(gab_bug(p, x), ref, bound, "Gaborish with w1 and w2 swapped")


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("iters", [1, 2, 3])
def test_epf_uniform_oracle_vs_f64(orc, shape, iters):
    h, w = shape
    p = frame_params(w, h, epf_iters=iters, gab=False)
    x = epf_planes(h, w, 2 + iters)
    inv = np.full((h, w), 1.0 / np.float32(MODULAR_SIGMA))
    ref, mid = epf_ref(p, x, inv)
    assert_within(orc.epf_uniform(p, x, MODULAR_SIGMA), ref, TOL_EPF, "oracle EPF")
    if h * w >= 60:
        assert mid > 0.2, "the input leaves too few weights strictly between 0 and 1 (%.2f)" % mid
        assert_rejects(epf_ref(p, x, inv, bug="neighbour")[0], ref, TOL_EPF, "EPF border multiplier keyed on the neighbour")
        if iters >= 2:                                               # (pass 0 smooths first when iters == 3)
            assert_rejects(epf_ref(p, x, inv, bug="swap12")[0], ref, TOL_EPF, "EPF with passes 1 and 2 swapped")


def epf_vardct_case(w, h, iters, seed):
    p = default_frame_params(w, h, epf_iters=iters)
    rng = np.random.default_rng(seed)
    hm = rng.integers(1, 5, size=(h // 8, w // 8)).astype(np.int32)
    sh = rng.integers(1, 8, size=(h // 8, w // 8)).astype(np.int32)
    sh[rng.random(sh.shape) < 0.25] = 0                               # sharpness 0: sigma 0, the block passes through
    sh[0, 0] = 3
    return p, epf_planes(h, w, seed), hm, sh


EPF_VARDCT = [(8, 8), (120, 40), (232, 64), (344, 24)]     # (W, H): widths 8 + 112 k leave a ragged last column strip in k2_stream


@pytest.mark.parametrize("size", EPF_VARDCT)
@pytest.mark.parametrize("iters", [1, 2, 3])
def test_epf_vardct_oracle_vs_f64(orc, size, iters):
    w, h = size
    p, x, hm, sh = epf_vardct_case(w, h, iters, 7 * iters + w)
    ref, mid = epf_ref(p, x, epf_inv_sigma(p, hm, sh))
    assert_within(orc.epf(p, x, hm, sh), ref, TOL_EPF, "oracle VarDCT EPF")
    assert mid > 0.2
    assert_rejects(epf_ref(p, x, epf_inv_sigma(p, hm, sh), bug="neighbour")[0], ref, TOL_EPF, "EPF multiplier keyed on the neighbour")
    if iters >= 2:
        assert_rejects(epf_ref(p, x, epf_inv_sigma(p, hm, sh), bug="swap12")[0], ref, TOL_EPF, "EPF with passes 1 and 2 swapped")


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_color_oracle_vs_f64(orc, shape, mode):
    h, w = shape
    p = frame_params(w, h, color_mode=mode)
    x = color_planes(h, w, mode)
    ref, bound = color_ref(p, x)
    assert_within(orc.color(p, x), ref, bound, "oracle colour mode %d" % mode)
    if mode & 1:
        assert_rejects(color_ref(p, x, bug="xsign")[0], ref, bound, "XYB with the sign of X flipped")
    if mode & 2:
        assert_rejects(color_ref(p, x, bug="cbcr")[0], ref, bound, "YCbCr with the Cb and Cr factors swapped")


@pytest.mark.parametrize("k", [2, 4, 8])
def test_upsampling_oracle_vs_f64(orc, k):
    wts = up_weights(k)
    for i, shape in enumerate(UP_SHAPES):
        a = up_plane(shape, 10 * k + i)
        ref, bound = upsample_ref(a, k, wts)
        assert_within(orc.upsample(a, k, wts), ref, bound, "oracle x%d %s" % (k, shape))
        if min(shape) >= 3:
            assert_rejects(upsample_ref(a, k, wts.transpose(1, 0, 2, 3))[0], ref, bound, "upsampling with the phases transposed")
            assert_rejects(upsample_ref(a, k, wts, edge="nearest")[0], ref, bound, "upsampling with nearest edges")
    neg = -up_plane((9, 9), k) - np.float32(1.0)                      # every window negative: the Float.MIN_VALUE cap holds them at ~0
    ref, bound = upsample_ref(neg, k, wts)
    assert ref.max() == FLOAT_MIN_VALUE
    assert_within(orc.upsample(neg, k, wts), ref, bound, "oracle x%d, negative plane" % k)


def test_splitmix64_known_answer():
    # SplitMix64 with state 0 first adds the golden gamma, then mixes: its first output is this published constant
    assert splitmix64(GOLDEN) == 0xE220A8397B1DCDAF
    assert splitmix64(splitmix64(GOLDEN)) != 0xE220A8397B1DCDAF


@pytest.mark.parametrize("case", NOISE_CASES)
def test_noise_oracle_vs_f64(orc, case):
    h, w, gd = case
    pl, lut, seed0 = noise_inputs(h, w, h + w + gd)
    ref = noise_ref(pl, gd, seed0, lut, 0.0, 1.0)
    assert np.abs(ref - pl).max() > 0.01 or h * w < 25               # the noise is visible
    assert_within(orc.noise(pl, gd, seed0, lut, 0.0, 1.0), ref, TOL_NOISE, "oracle noise")
    if max(h, w) > gd:
        assert_rejects(noise_ref(pl, gd, seed0, lut, 0.0, 1.0, swap_xy=True), ref, TOL_NOISE, "noise with x0 and y0 swapped in seed1")


@pytest.mark.parametrize("hb", LF_SIZES)
@pytest.mark.parametrize("wb", LF_SIZES)
def test_lf_dequant_oracle_vs_f64(orc, hb, wb):
    q, ep, sd, kx, kb = lf_inputs(hb, wb)
    for cfl in (False, True):
        for smooth in (False, True):
            ref, bound = lf_ref(q, ep, sd, kx, kb, cfl, smooth)
            assert_within(orc.lf_dequant(q, ep, sd, kx, kb, cfl=cfl, smooth=smooth), ref, bound, "oracle LF cfl=%d smooth=%d" % (cfl, smooth))
            if smooth and (hb > 256 or wb > 256) and min(hb, wb) >= 3:
                assert_rejects(lf_ref(q, ep, sd, kx, kb, cfl, smooth, cross_groups=True)[0], ref, bound, "LF smoothing across a group border")


@pytest.mark.parametrize("shifts", CHROMA_SHIFTS)
@pytest.mark.parametrize("size", CHROMA_SIZES)
def test_chroma_upsampling_oracle_vs_f64(orc, shifts, size):
    W, H = size
    p = frame_params(W, H)
    p.shift_y[:], p.shift_x[:] = shifts
    rng = np.random.default_rng(W + H)
    sub = [rng.uniform(-1, 1, (H >> p.shift_y[c], W >> p.shift_x[c])).astype(np.float32) for c in range(3)]
    ref, bound = chroma_ref(p, sub)
    assert_within(orc.invert_subsampling(p, sub), ref, bound, "oracle chroma upsampling")
    assert_rejects(chroma_ref(p, sub, near=0.25, far=0.75)[0], ref, bound, "chroma upsampling with 0.25 and 0.75 swapped")


@pytest.mark.parametrize("bits", [8, 16])
@pytest.mark.parametrize("linear", [True, False])
def test_pack_samples_oracle_vs_f64(orc, bits, linear):
    depths = [bits, bits, bits, 10 if bits == 8 else 12]
    for w, ch, is_int in pack_cases():
        ref, near = pack_ref(ch, is_int, depths, 3, linear, bits)
        got = unpack(orc.pack_samples(ch, depths, 3, linear, bits), bits)
        assert_pack_close(got, ref, near, "oracle %d-bit, width %d" % (bits, w))
        # the int channel at its own depth passes through clamped
        same = [ch[0], ch[1], ch[2], ch[3]]
        r2, _ = pack_ref(same, is_int, [bits] * 4, 3, linear, bits)
        assert np.array_equal(unpack(orc.pack_samples(same, [bits] * 4, 3, linear, bits), bits)[..., 3], r2[..., 3])
    bug, _ = pack_ref(ch, is_int, depths, 3, linear, bits, rounding=0.0)
    assert ((bug != ref) & ~near).sum() >= 10 * max(2, ref.size // 1000), "truncating instead of rounding goes unseen"


# ========================================================================================================================
# kernel vs reference (GPU)
# ========================================================================================================================
def _stage2(recon, mode):
    return recon.set_option(_lib.OPT_STAGE2, {"stream": _lib.STAGE2_STREAM, "tile": _lib.STAGE2_TILE, "staged": _lib.STAGE2_STAGED,
                                              "auto": _lib.STAGE2_AUTO}[mode])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
def test_gaborish_kernel_vs_f64(recon, shape):
    h, w = shape
    p = frame_params(w, h, epf_iters=0, color_mode=0)
    x = epf_planes(h, w, 1) * np.float32(8.0) - np.float32(2.0)
    if min(h, w) < 4:
        with pytest.raises(NotImplementedError):
            recon.restoreModularFrame(p, x, MODULAR_SIGMA)
        return
    ref, bound = gab_ref(p, x)
    assert_within(recon.restoreModularFrame(p, x, MODULAR_SIGMA), ref, bound, "restore_uniform Gaborish")
    if h % 8 == 0 and w % 8 == 0:
        assert_within(recon.performGabConvolution(p, x), ref, bound, "jxlb200_gaborish")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("iters", [1, 2, 3])
def test_epf_uniform_kernel_vs_f64(recon, shape, iters):
    h, w = shape
    p = frame_params(w, h, epf_iters=iters, gab=False, color_mode=0)
    x = epf_planes(h, w, 2 + iters)
    if min(h, w) < 4:
        with pytest.raises(NotImplementedError):
            recon.restoreModularFrame(p, x, MODULAR_SIGMA)
        return
    ref, _ = epf_ref(p, x, np.full((h, w), 1.0 / np.float32(MODULAR_SIGMA)))
    assert_within(recon.restoreModularFrame(p, x, MODULAR_SIGMA), ref, TOL_EPF, "restore_uniform EPF")


@pytest.mark.gpu
@pytest.mark.parametrize("size", EPF_VARDCT)
@pytest.mark.parametrize("iters", [1, 2, 3])
@pytest.mark.parametrize("stage2", ["stream", "tile", "staged"])
def test_epf_vardct_kernel_vs_f64(recon, size, iters, stage2):
    from kernel_trace import assert_stage2_kernel, launched_kernels
    w, h = size
    p, x, hm, sh = epf_vardct_case(w, h, iters, 7 * iters + w)
    ref, _ = epf_ref(p, x, epf_inv_sigma(p, hm, sh))
    _stage2(recon, stage2)
    try:
        got, names = launched_kernels(lambda: recon.performEdgePreservingFilter(p, x, hm, sh))
    finally:
        _stage2(recon, "auto")
    assert_stage2_kernel(names, stage2, p)
    assert_within(got, ref, TOL_EPF, "%s EPF" % stage2)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_color_kernel_vs_f64(recon, shape, mode):
    h, w = shape
    p = frame_params(w, h, epf_iters=0, gab=False, color_mode=mode)
    x = color_planes(h, w, mode)
    ref, bound = color_ref(p, x)
    assert_within(recon.restoreModularFrame(p, x, MODULAR_SIGMA), ref, bound, "restore_uniform colour mode %d" % mode)
    if h % 8 or w % 8:
        with pytest.raises(ValueError):                               # the VarDCT entry point takes padded frames only
            recon.performColorTransforms(p, x)
    else:
        assert_within(recon.performColorTransforms(p, x), ref, bound, "jxlb200_color_transform mode %d" % mode)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 4, 8])
def test_upsampling_kernel_vs_f64(recon, k):
    wts = up_weights(k)
    for i, shape in enumerate(UP_SHAPES):
        a = up_plane(shape, 10 * k + i)
        ref, bound = upsample_ref(a, k, wts)
        assert_within(recon.performUpsampling(a, k, wts), ref, bound, "k8_upsample x%d %s" % (k, shape))


@pytest.mark.gpu
@pytest.mark.parametrize("case", NOISE_CASES)
def test_noise_kernel_vs_f64(recon, case):
    h, w, gd = case
    pl, lut, seed0 = noise_inputs(h, w, h + w + gd)
    assert_within(recon.synthesizeNoise(pl, gd, seed0, lut, 0.0, 1.0), noise_ref(pl, gd, seed0, lut, 0.0, 1.0), TOL_NOISE, "k8_noise")


@pytest.mark.gpu
@pytest.mark.parametrize("hb", LF_SIZES)
@pytest.mark.parametrize("wb", LF_SIZES)
def test_lf_dequant_kernel_vs_f64(recon, hb, wb):
    q, ep, sd, kx, kb = lf_inputs(hb, wb)
    for cfl in (False, True):
        for smooth in (False, True):
            ref, bound = lf_ref(q, ep, sd, kx, kb, cfl, smooth)
            assert_within(recon.dequantLF(q, ep, sd, kx, kb, cfl=cfl, smooth=smooth), ref, bound, "k8_lf_dequant cfl=%d smooth=%d" % (cfl, smooth))


@pytest.mark.gpu
@pytest.mark.parametrize("shifts", CHROMA_SHIFTS)
@pytest.mark.parametrize("size", CHROMA_SIZES)
def test_chroma_upsampling_kernel_vs_f64(recon, orc, shifts, size):
    """Through the whole reconstruction with the filters and the colour transform off: stage 1 (bit-identical to the oracle's,
    checked in test_vardct_gpu.py) followed by the upsampling of the subsampled channels."""
    from jxlatte_b200 import synth
    from jxlatte_b200.host import qm_generate
    W, H = size
    p = default_frame_params(W, H, epf_iters=0, gab=False, color_mode=0)
    p.shift_y[:], p.shift_x[:] = shifts
    qw, qo = qm_generate()
    st = dict(synth.make_state(W, H, seed=W * 7 + H, mix=(1.0, 0.0, 0.0, 0.0, 0.0), params=p, qm_weights=qw, qm_offsets=qo))
    st["qcoeff"] = [np.ascontiguousarray(st["qcoeff"][c][:H >> shifts[0][c], :W >> shifts[1][c]]) for c in range(3)]
    st["lf"] = [np.ascontiguousarray(st["lf"][c][:(H // 8) >> shifts[0][c], :(W // 8) >> shifts[1][c]]) for c in range(3)]
    sub = orc.vardct_invert(p, st, nthreads=4)
    ref, bound = chroma_ref(p, sub if isinstance(sub, list) else list(sub))
    recon.setWeights(qw, qo)
    assert_within(recon.reconstruct(p, st), ref, bound, "chroma upsampling")


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [8, 16])
@pytest.mark.parametrize("linear", [True, False])
def test_pack_samples_kernel_vs_f64(recon, bits, linear):
    depths = [bits, bits, bits, 10 if bits == 8 else 12]
    for w, ch, is_int in pack_cases():
        ref, near = pack_ref(ch, is_int, depths, 3, linear, bits)
        assert_pack_close(unpack(recon.packSamples(ch, depths, 3, linear, bits), bits), ref, near, "k8_pack_samples %d-bit, width %d" % (bits, w))


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [8, 16])
def test_packed_reconstruction_ragged_crops_vs_f64(recon, orc, bits):
    """k8_pack_rgb at crop widths 1 to 7 (a ragged last quad of four pixels) and a crop of a few rows."""
    from jxlatte_b200 import synth
    from jxlatte_b200.host import qm_generate
    W, H = 64, 16
    p = default_frame_params(W, H, epf_iters=1)
    qw, qo = qm_generate()
    st = synth.make_state(W, H, seed=404 + bits, params=p, qm_weights=qw, qm_offsets=qo)
    recon.setWeights(qw, qo)
    planes = orc.vardct_reconstruct(p, st, nthreads=4)
    for cw, chh in [(c, H) for c in range(1, 8)] + [(5, 3), (61, 9)]:
        crop = [planes[c][:chh, :cw] for c in range(3)]
        for linear in (True, False):
            ref, near = pack_ref(crop, [False] * 3, [bits] * 3, 3, linear, bits)
            got = unpack(recon.reconstruct_packed(p, st, bits=bits, linear=linear, crop=(cw, chh)), bits)
            assert_pack_close(got, ref, near, "k8_pack_rgb %d-bit crop %dx%d" % (bits, cw, chh))
