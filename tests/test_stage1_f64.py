"""Stage 1 (dequantisation, chroma-from-luma, LLF and the 27 inverse transforms) against an independent float64 reference.

The oracle and the kernels were written from the same reading of the Java, so bit equality between them cannot catch a misreading
they share.  stage1_ref restates stage 1 as mathematics: whole-plane dequantisation, the chroma-from-luma rule stated per pixel, the
LLF corner as a forward DCT matrix, and one explicit float64 linear map per TransformType applied to every varblock of that type at
once.  It cites the Java lines the oracle cites (oracle/vardct_oracle.c:616-775, 820-928; J/ = java/com/traneptora/jxlatte/).

The QM tables are an input (the product's qm_generate() output, pinned elsewhere), and so is the AFV basis (orc.afv_basis(), whose
orthonormality test_oracle.py pins).  Everything else -- the cosines, the LLF scales, the Haar levels, the placements -- is computed
here from its definition, and each 8 x 8-class matrix is checked for a structural property before it is trusted.

Tolerances follow test_f64_reference.py: per output pixel, bound = c_t * U * (|A| |d|) + |A| e_d, with d the coefficient block after
dequantisation, chroma-from-luma and LLF, e_d its own bound carried through those steps, A the type's map (as the product of the
absolute values of its stages, which bounds the absolute value of the product) and c_t the float32 operations on its longest chain.
Every comparison also evaluates the reference with plausible bugs and asserts the same check rejects each by ten times the bound.
"""
import numpy as np
import pytest
import scipy.fft

from jxlatte_b200 import default_frame_params, synth
from jxlatte_b200.host import qm_generate
from jxlatte_b200.params import COLOR_NONE, TRANSFORM_NAMES, TRANSFORM_TYPES
from test_f64_reference import U, assert_rejects, assert_within, chroma_ref, compare

CLASS8 = (0, 1, 2, 3, 12, 13, 14, 15, 16, 17)
M_DCT, M_DCT2, M_DCT4, M_HORNUSS, M_DCT8_4, M_DCT4_8, M_AFV = range(7)      # TransformType.transformMethod


def _dims(t):
    return TRANSFORM_TYPES[t][2], TRANSFORM_TYPES[t][3]


# ---- the 1-D DCTs (J/util/MathHelper.java:68-94) ------------------------------------------------------------------------
def idct_mat(n):
    """MathHelper.inverseDCTHorizontal as a matrix [pixel k, frequency m]: in[0] + sum_m in[m] sqrt2 cos(pi m (k + 1/2) / n), which
    is the orthonormal DCT-III times sqrt(n)."""
    k, m = np.mgrid[0:n, 0:n]
    return np.where(m == 0, 1.0, np.sqrt(2.0) * np.cos(np.pi * m * (k + 0.5) / n))


def fdct_mat(n):
    """MathHelper.forwardDCTHorizontal [frequency m, sample k]: the orthonormal DCT-II divided by sqrt(n), the inverse of idct_mat."""
    return idct_mat(n).T / n


def idct_ops(n):
    """One inverse DCT of length n: out[k] = in[0] + sum fl(in[m] * fl(lut)) in m order -- the rounding of the LUT entry, one
    multiply and n - 1 adds on the longest chain (in[1]'s)."""
    return 0 if n == 1 else n + 1


def llf_scale(i):
    """LLFScale's closed form (J/frame/vardct/LLFScale.java:7-23)."""
    return 1.0 / (np.cos(np.pi * i / 512) * np.cos(np.pi * i / 256) * np.cos(np.pi * i / 128))


# ---- the 8 x 8-class transforms (J/frame/group/PassGroup.java:88-331), as stages acting on [n, 8, 8] float64 blocks ------------
def haar(b, s):
    """PassGroup.auxDCT2 at size s: each 2 x 2 group of the top-left s x s coefficients (c00 c01 / c10 c11, taken s/2 apart) becomes
    the 2 x 2 pixels (00, 01, 10, 11) = (sum, c00 + c01 - c10 - c11, c00 - c01 + c10 - c11, the alternating sum)."""
    out, h = b.copy(), s // 2
    c00, c01, c10, c11 = b[:, :h, :h], b[:, :h, h:s], b[:, h:s, :h], b[:, h:s, h:s]
    out[:, 0:s:2, 0:s:2] = c00 + c01 + c10 + c11
    out[:, 0:s:2, 1:s:2] = c00 + c01 - c10 - c11
    out[:, 1:s:2, 0:s:2] = c00 - c01 + c10 - c11
    out[:, 1:s:2, 1:s:2] = c00 - c01 - c10 + c11
    return out


def sep(Mh, x, Mw):
    """Mh x Mw^T for every block of x [n, h, w]: a separable 2-D map."""
    return Mh @ x @ Mw.T


def _idct2(s, flipped=False):
    """The 2-D inverse DCT of [n, h, w] blocks; flipped = MathHelper.inverseDCT2D's transposed output."""
    r = sep(idct_mat(s.shape[1]), s, idct_mat(s.shape[2]))
    return r.transpose(0, 2, 1) if flipped else r


def hornuss_quadrants(h, bug=None):
    """Hornuss after its Haar level: quadrant (y, x) gathers the coefficients h[y + 2 iy, x + 2 ix]; its centre pixel (1, 1) is the
    quadrant's LF minus 1/16 of the other fifteen, every other pixel is its coefficient plus the centre, and pixel (0, 0) takes
    coefficient (1, 1).  So each quadrant's mean is its LF."""
    out = np.empty_like(h)
    for y in range(2):
        for x in range(2):
            sub = h[:, y::2, x::2]
            lf = sub[:, 0, 0]
            res = sub.sum(axis=(1, 2)) - lf
            centre = lf if bug == "hornuss_nores" else lf - res / 16.0
            q = sub + centre[:, None, None]
            q[:, 1, 1] = centre
            q[:, 0, 0] = sub[:, 1, 1] + centre
            out[:, 4 * y:4 * y + 4, 4 * x:4 * x + 4] = q
    return out


def dct4_quadrants(h):
    """DCT4 after its Haar level: quadrant (y, x) is the 4 x 4 inverse DCT (output transposed) of h[y + 2 iy, x + 2 ix]."""
    out = np.empty_like(h)
    for y in range(2):
        for x in range(2):
            out[:, 4 * y:4 * y + 4, 4 * x:4 * x + 4] = _idct2(h[:, y::2, x::2], flipped=True)
    return out


def halves_mix(b):
    """DCT8_4 / DCT4_8: the two halves' DCs are c00 + c10 and c00 - c10, read from positions (0, 0) and (1, 0)."""
    out = b.copy()
    out[:, 0, 0], out[:, 1, 0] = b[:, 0, 0] + b[:, 1, 0], b[:, 0, 0] - b[:, 1, 0]
    return out


def halves(m, t, bug=None):
    """Half i takes coefficient rows i, i + 2, i + 4, i + 6 as a 4 x 8 block; DCT4_8 stacks the halves' 4 x 8 inverse DCTs top /
    bottom, DCT8_4 places their transposes (8 x 4) left / right."""
    out = np.empty_like(m)
    for i in range(2):
        j = 1 - i if bug == "halves_swap" else i
        if t == 12:
            out[:, 4 * j:4 * j + 4, :] = _idct2(m[:, i::2, :])
        else:
            out[:, :, 4 * j:4 * j + 4] = _idct2(m[:, i::2, :], flipped=True)
    return out


def afv_mix(b):
    """AFV's three DCs from c00, c10 = (1, 0) and c01 = (0, 1): the corner's 4 (c00 + c10 + c01) at (0, 0), the 4 x 4 block's
    c00 + c10 - c01 at (0, 1), the 4 x 8 half's c00 - c10 at (1, 0)."""
    out = b.copy()
    c00, c10, c01 = b[:, 0, 0], b[:, 1, 0], b[:, 0, 1]
    out[:, 0, 0], out[:, 0, 1], out[:, 1, 0] = 4.0 * (c00 + c10 + c01), c00 + c10 - c01, c00 - c10
    return out


def afv_place(m, t, basis, bug=None):
    """AFV0-3: a 4 x 4 corner in the AFV basis (coefficients m[2 iy, 2 ix]), mirrored into the block's corner (flip x for AFV1 and
    AFV3, flip y for AFV2 and AFV3); beside it a 4 x 4 inverse DCT (output transposed) of m[2 iy, 2 ix + 1]; the other half a 4 x 8
    inverse DCT of the odd rows m[2 iy + 1, :]."""
    if bug == "afv12" and t in (15, 16):
        t = 31 - t
    fy, fx = int(t in (16, 17)), int(t in (15, 17))
    n = m.shape[0]
    out = np.empty_like(m)
    corner = (m[:, 0::2, 0::2].reshape(n, 16) @ basis).reshape(n, 4, 4)
    corner = corner[:, ::-1, :] if fy else corner
    corner = corner[:, :, ::-1] if fx else corner
    out[:, 4 * fy:4 * fy + 4, 4 * fx:4 * fx + 4] = corner
    out[:, 4 * fy:4 * fy + 4, 4 * (1 - fx):4 * (1 - fx) + 4] = _idct2(m[:, 0::2, 1::2], flipped=True)
    out[:, 4 * (1 - fy):4 * (1 - fy) + 4, :] = _idct2(m[:, 1::2, :])
    return out


# float32 operations on the longest chain of each stage, summed over the stages of a method:
#   Haar level: a 4-term sum (3)
#   Hornuss quadrant: 15-term residual (14 adds; the first add is to 0), * 1/16 (exact), LF - that (1), + coefficient (1): 16
#   4 x 4 / 4 x 8 inverse DCT: idct_ops(4) + idct_ops(4) = 10 / idct_ops(4) + idct_ops(8) = 14
#   halves' DCs: one add (1); AFV's DCs: two adds, * 4 exact (2)
#   AFV corner: 16 products with the float32 basis as given, summed from 0 (1 + 15); the corner is the longest of the three parts
CLASS8_OPS = {M_DCT2: 3 + 3 + 3, M_HORNUSS: 3 + 16, M_DCT4: 3 + 10, M_DCT8_4: 1 + 14, M_DCT4_8: 1 + 14, M_AFV: 2 + 16}


def class8_stages(t, basis, bug=None):
    """The stages of an 8 x 8-class type, each a function of [n, 8, 8] blocks, in the order they apply."""
    method = TRANSFORM_TYPES[t][1]
    if method == M_DCT2:
        return [lambda b, s=s: haar(b, s) for s in ((8, 4, 2) if bug == "dct2_reverse" else (2, 4, 8))]
    if method == M_HORNUSS:
        return [lambda b: haar(b, 2), lambda b: hornuss_quadrants(b, bug)]
    if method == M_DCT4:
        return [lambda b: haar(b, 2), dct4_quadrants]
    if method in (M_DCT8_4, M_DCT4_8):
        return [halves_mix, lambda b: halves(b, t, bug)]
    assert method == M_AFV
    return [afv_mix, lambda b: afv_place(b, t, basis, bug)]


def _matrix(f):
    """A linear function of [n, 8, 8] blocks as a 64 x 64 matrix [pixel, coefficient]."""
    return f(np.eye(64).reshape(64, 8, 8)).reshape(64, 64).T


def class8_maps(t, basis, bug=None):
    """-> (A, |A|): the type's 64 x 64 matrix and the product of its stages' absolute values."""
    A, absA = np.eye(64), np.eye(64)
    for f in class8_stages(t, basis, bug):
        S = _matrix(f)
        A, absA = S @ A, np.abs(S) @ absA
    return A, absA


def ops(t):
    """c_t: float32 operations on the longest chain of type t's inverse transform."""
    ph, pw = _dims(t)
    method = TRANSFORM_TYPES[t][1]
    return idct_ops(ph) + idct_ops(pw) if method == M_DCT else CLASS8_OPS[method]


# ---- the reference -------------------------------------------------------------------------------------------------------
def cell_origins(ds, bo):
    """(oy, ox): the block position of the origin of the varblock covering each 8 x 8 cell."""
    oy = np.full(ds.shape, -1, np.int64)
    ox = np.full(ds.shape, -1, np.int64)
    for t in np.unique(ds[bo != 0]):
        ys, xs = np.nonzero((bo != 0) & (ds == t))
        bh, bw = _dims(t)[0] >> 3, _dims(t)[1] >> 3
        Y = ys[:, None, None] + np.arange(bh)[None, :, None]
        X = xs[:, None, None] + np.arange(bw)[None, None, :]
        oy[Y, X], ox[Y, X] = ys[:, None, None], xs[:, None, None]
    assert (oy >= 0).all(), "the partition leaves a cell uncovered"
    return oy, ox


def quirk_count(st):
    """Varblocks with a pixel in a 64 x 64 tile whose gate varblock (the one covering the tile's top-left pixel) comes later in
    raster order of origins: chroma-from-luma gives those pixels a factor of 0."""
    ds, bo = st["dct_select"], st["block_origin"]
    oy, ox = cell_origins(ds, bo)
    wb = ds.shape[1]
    idx = oy * wb + ox
    gate = idx[::8, ::8]
    early = idx < np.repeat(np.repeat(gate, 8, 0), 8, 1)[:idx.shape[0], :idx.shape[1]]
    return len(np.unique(idx[early]))


def _px(a):
    return np.repeat(np.repeat(a, 8, axis=0), 8, axis=1)


def channel_maps(p, st, c):
    """The varblocks of channel c as cell maps of its own plane: (type, origin y, origin x, hf_mul, full-resolution origin y, x).
    A subsampled channel takes a varblock only where its block position is a multiple of the shift, at the shifted position
    (oracle/vardct_oracle.c:812-818); only 8 x 8-class types can be subsampled."""
    ds, bo = st["dct_select"].astype(np.int64), st["block_origin"]
    sy, sx = p.shift_y[c], p.shift_x[c]
    oy, ox = cell_origins(ds, bo)
    hm = st["hf_mul"].astype(np.int64)
    if not (sy or sx):
        return ds, oy, ox, hm[oy, ox], oy, ox
    keep = (bo != 0) & (np.arange(ds.shape[0])[:, None] % (1 << sy) == 0) & (np.arange(ds.shape[1])[None, :] % (1 << sx) == 0)
    assert np.isin(ds[keep], CLASS8).all(), "a subsampled frame holds only 8 x 8-class varblocks (DESIGN §8)"
    fy, fx = np.nonzero(keep)
    hc, wc = ds.shape[0] >> sy, ds.shape[1] >> sx
    shape = (hc, wc)
    t, hmc, gy, gx = (np.empty(shape, np.int64) for _ in range(4))
    t[fy >> sy, fx >> sx], hmc[fy >> sy, fx >> sx] = ds[fy, fx], hm[fy, fx]
    gy[fy >> sy, fx >> sx], gx[fy >> sy, fx >> sx] = fy, fx
    cy, cx = np.mgrid[0:hc, 0:wc]
    return t, cy, cx, hmc, gy, gx


def dequant(p, st, c, maps, bug=None):
    """HFCoefficients.dequantizeHFCoefficients (:267-319) of channel c -> (d, e_d); the LLF corners are left at zero."""
    t, oy, ox, hm, _, _ = (_px(a) for a in maps)
    hc, wc = t.shape
    yy, xx = np.mgrid[0:hc, 0:wc]
    tt = np.array(TRANSFORM_TYPES, np.int64)
    param, method, ph, pw = tt[t, 0], tt[t, 1], tt[t, 2], tt[t, 3]
    ly, lx = yy - oy * 8, xx - ox * 8
    flip = (ph > pw) | ((method == M_DCT) & (ph == pw))                  # TransformType.flip :129-131
    if bug == "noflip":
        flip = np.zeros_like(flip)
    wy, wx = np.where(flip, lx, ly), np.where(flip, ly, lx)
    qw = np.asarray(st["qm_weights"], np.float64)
    widx = wy * np.maximum(ph, pw) + wx
    if bug == "noflip":
        # a stand-in, not the Java's behaviour: a real dropped flip on a tall block reads past its matrix into the next one; the
        # wrap keeps the planted read inside the parameter's own matrix, still at the wrong weights
        widx = widx % (ph * pw)
    w = qw[np.asarray(st["qm_offsets"])[param * 3 + c] + widx]
    xqm, bqm = (p.bqm_scale, p.xqm_scale) if bug == "xb_swap" else (p.xqm_scale, p.bqm_scale)
    sf = 65536.0 / p.global_scale * (0.8 ** (xqm - 2.0), 1.0, 0.8 ** (bqm - 2.0))[c]
    q = np.asarray(st["qcoeff"][c], np.int64).astype(np.float64)
    qb, qbn = float(np.float32(p.quant_bias[c])), float(np.float32(p.quant_bias_numerator))
    safe = np.where(np.abs(q) < 2, 2.0, q)
    tail = q + qbn / safe if bug == "qbn_add" else q - qbn / safe
    neg1 = qb if bug == "qb_sign" else -qb
    quant = np.where(q == -1, neg1, np.where(q == 1, qb, np.where(q == 0, 0.0, tail)))
    scale = sf / hm * w
    d = quant * scale
    # float32: |q| > 2^24 converts with one rounding, qbn / q is one more, the subtraction one (3 on the tail's terms); sf is
    # 65536 / global_scale (1), the float pow (1), their product (1), / hf_mul (1, and 1 more for a multiplier above 2^24); then
    # quant * sf and * weight (2).  qb and the weight are float32 inputs used as given.
    e_quant = np.where(np.abs(q) < 2, 0.0, 3 * U * (np.abs(q) + np.abs(qbn / safe)))
    sf_ops = 4 + (np.abs(hm) > 2 ** 24)
    e = np.abs(scale) * e_quant + (2 + sf_ops) * U * np.abs(d)
    corner = (ly < ph >> 3) & (lx < pw >> 3)
    return np.where(corner, 0.0, d), np.where(corner, 0.0, e)


def cfl(p, st, d, e, bug=None):
    """HFCoefficients.chromaFromLuma (:146-192), stated per pixel: the pixel's 64 x 64 tile gives k = base + factor / color_factor,
    which applies only when the pixel's varblock origin is at or after (raster order of origins) the origin of the varblock covering
    the tile's top-left pixel -- before that the Java's per-group factor cache still holds 0.  X += kX Y, B += kB Y."""
    ds, bo = st["dct_select"], st["block_origin"]
    oy, ox = cell_origins(ds, bo)
    wb = ds.shape[1]
    idx = oy * wb + ox
    H, W = d.shape[1:]
    ty, tx = np.mgrid[0:H, 0:W]
    ty, tx = ty >> 6, tx >> 6
    if bug == "cfl_per_block":                                            # the tile of the varblock's origin
        ty, tx = _px(oy * 8 >> 6), _px(ox * 8 >> 6)
    gate = idx[::8, ::8][ty, tx]
    on = (_px(idx) >= gate) | (bug == "cfl_always")
    out, err = d.copy(), e.copy()
    for c, base, fac in ((0, p.base_corr_x, st["x_from_y"]), (2, p.base_corr_b, st["b_from_y"])):
        f = np.asarray(fac, np.float64)[ty, tx] / p.color_factor
        k = np.where(on, float(np.float32(base)) + f, 0.0)
        K = np.where(on, abs(float(np.float32(base))) + np.abs(f), 0.0)
        # k: one divide, one add (2 u K); k * Y and the add (2 u): |k Y| carries 4 u K |Y| in all, the sum u |X|
        out[c] = d[c] + k * d[1]
        err[c] = e[c] + K * e[1] + U * (np.abs(d[c]) + 4 * K * np.abs(d[1]))
    return out, err


def llf(p, st, c, maps, d, e, bug=None):
    """HFCoefficients.finalizeLLF (:194-229): the dsH x dsW corner of each varblock is the forward 2-D DCT of the LF sub-grid at its
    position (at pos >> shift in a subsampled channel) times scale(ky) scale(kx), scale at index k << (5 - log2 ds).
    bug = "llf_transpose": the LF sub-grid gathered with its axes swapped (element (ky, kx) from row x + kx, column y + ky), the
    misreading of a rectangular corner an implementation can make -- swapping the scale indices instead would read past LLFScale's
    32-entry table, and swapping the DCT axes of a separable map with the transposes that make the shapes fit changes nothing."""
    t, oy, ox = maps[:3]
    lf = np.asarray(st["lf"][c], np.float64)
    for tv in np.unique(t):
        ph, pw = _dims(tv)
        dh, dw = ph >> 3, pw >> 3
        ys, xs = np.nonzero((t == tv) & (oy == np.arange(t.shape[0])[:, None]) & (ox == np.arange(t.shape[1])[None, :]))
        ly, lx = ys, xs
        if bug == "sub_lf_unshifted":                                     # the full-resolution position
            ly, lx = np.minimum(maps[4][ys, xs], lf.shape[0] - dh), np.minimum(maps[5][ys, xs], lf.shape[1] - dw)
        if bug == "llf_transpose":
            rows = np.minimum(ly[:, None, None] + np.arange(dw)[None, None, :], lf.shape[0] - 1)
            cols = np.minimum(lx[:, None, None] + np.arange(dh)[None, :, None], lf.shape[1] - 1)
            sub = lf[rows, cols]
        else:
            sub = lf[(ly[:, None] + np.arange(dh))[:, :, None], (lx[:, None] + np.arange(dw))[:, None, :]]
        Fh, Fw = fdct_mat(dh), fdct_mat(dw)
        lh, lw = int(np.log2(dh)), int(np.log2(dw))
        sc = np.outer(llf_scale(np.arange(dh) << (5 - lh)), llf_scale(np.arange(dw) << (5 - lw)))
        val = sep(Fh, sub, Fw) * sc
        # float32: each forward DCT of length n > 1 is a product with a rounded LUT entry and n - 1 adds (n + 1); the scale is two
        # rounded table entries and their product, and the final multiply (4)
        n_ops = idct_ops(dh) + idct_ops(dw) + (4 if dh * dw > 1 else 0)
        bnd = n_ops * U * sep(np.abs(Fh), np.abs(sub), np.abs(Fw)) * sc
        Y = (ys * 8)[:, None, None] + np.arange(dh)[None, :, None]
        X = (xs * 8)[:, None, None] + np.arange(dw)[None, None, :]
        d[Y, X], e[Y, X] = val, bnd


def invert(t_map, oy, ox, d, e, basis, bug=None):
    """PassGroup.invertVarDCT (:209-330) of one channel: every varblock's map applied to its coefficients, in place -> (pixels, bound)."""
    out, bound = np.zeros_like(d), np.zeros_like(d)
    for tv in np.unique(t_map):
        ph, pw = _dims(tv)
        ys, xs = np.nonzero((t_map == tv) & (oy == np.arange(t_map.shape[0])[:, None]) & (ox == np.arange(t_map.shape[1])[None, :]))
        Y = (ys * 8)[:, None, None] + np.arange(ph)[None, :, None]
        X = (xs * 8)[:, None, None] + np.arange(pw)[None, None, :]
        blk, eb = d[Y, X], e[Y, X]
        if TRANSFORM_TYPES[tv][1] == M_DCT:
            if bug == "transpose_rect" and ph != pw:                        # the stored block read as a pw x ph one
                Ch, Cw = idct_mat(pw), idct_mat(ph)
                px = sep(Ch, blk.reshape(-1, pw, ph), Cw).reshape(-1, ph, pw)
            else:
                Ch, Cw = idct_mat(ph), idct_mat(pw)
                px = sep(Ch, blk, Cw)
            aCh, aCw = np.abs(idct_mat(ph)), np.abs(idct_mat(pw))
            bnd = (ops(tv) * U * sep(aCh, np.abs(blk), aCw) + sep(aCh, eb, aCw))
        else:
            A, absA = class8_maps(tv, basis, bug)
            n = len(ys)
            px = (blk.reshape(n, 64) @ A.T).reshape(n, 8, 8)
            _, absA = class8_maps(tv, basis)
            bnd = ((ops(tv) * U * np.abs(blk).reshape(n, 64) + eb.reshape(n, 64)) @ absA.T).reshape(n, 8, 8)
        out[Y, X], bound[Y, X] = px, bnd
    return out, bound


def stage1_ref(p, st, basis, bug=None, want_dequant=False):
    """-> (planes, bound) [, (d, e_d)]: per channel, the (H >> sy) x (W >> sx) plane.  Chroma-from-luma is skipped entirely when any
    channel is subsampled (:149-151) -- unless bug == "sub_cfl", which applies it with Y read at the same image position."""
    maps = [channel_maps(p, st, c) for c in range(3)]
    de = [dequant(p, st, c, maps[c], bug) for c in range(3)]
    subsampled = any(p.shift_x[c] or p.shift_y[c] for c in range(3))
    if not subsampled:
        d, e = cfl(p, st, np.stack([a for a, _ in de]), np.stack([b for _, b in de]), bug)
        de = [(d[c], e[c]) for c in range(3)]
    elif bug == "sub_cfl":
        for c in (0, 2):
            hc, wc = de[c][0].shape
            yy, xx = np.mgrid[0:hc, 0:wc]
            y = de[1][0][(yy << p.shift_y[c]) >> p.shift_y[1], (xx << p.shift_x[c]) >> p.shift_x[1]]
            f = np.asarray((st["x_from_y"], None, st["b_from_y"])[c], np.float64)[(yy << p.shift_y[c]) >> 6, (xx << p.shift_x[c]) >> 6]
            de[c] = (de[c][0] + ((p.base_corr_x, 0, p.base_corr_b)[c] + f / p.color_factor) * y, de[c][1])
    planes, bounds = [], []
    for c in range(3):
        d, e = de[c][0].copy(), de[c][1].copy()
        llf(p, st, c, maps[c], d, e, bug)
        de[c] = (d, e)
        o, b = invert(maps[c][0], maps[c][1], maps[c][2], d, e, basis, bug)
        planes.append(o)
        bounds.append(b)
    if not subsampled:
        planes, bounds = np.stack(planes), np.stack(bounds)
    if want_dequant:
        return planes, bounds, de
    return planes, bounds


# ---- frames -----------------------------------------------------------------------------------------------------------
QW, QO = qm_generate()


def single_type_state(t, W, H, seed, hf_zero=False):
    """A frame tiled with one TransformType, dense small coefficients (or none), every hf_mul and CfL factor drawn."""
    p = default_frame_params(W, H, global_scale=32768)
    st = dict(synth.make_state(W, H, seed=seed, mix="dct8", params=p, qm_weights=QW, qm_offsets=QO))
    ph, pw = _dims(t)
    bh, bw = ph // 8, pw // 8
    hb, wb = H // 8, W // 8
    st["dct_select"] = np.full((hb, wb), t, np.uint8)
    org = np.zeros((hb, wb), np.uint8)
    org[::bh, ::bw] = 1
    st["block_origin"] = org
    st["hf_mul"] = np.ascontiguousarray(np.repeat(np.repeat(st["hf_mul"][::bh, ::bw], bh, 0), bw, 1))
    rng = np.random.default_rng(seed + 99)
    q = rng.integers(-3, 4, size=(3, H, W)) * (rng.random((3, H, W)) < 0.3)
    st["qcoeff"] = np.zeros((3, H, W), np.int32) if hf_zero else q.astype(np.int32)
    return p, st


def single_size(t):
    ph, pw = _dims(t)
    return max(256, pw), max(256, ph)


def mixed_state(W, H, aligned, seed):
    p = default_frame_params(W, H)
    return p, dict(synth.make_state(W, H, seed=seed, params=p, qm_weights=QW, qm_offsets=QO, aligned=aligned))


def extremes_state(seed):
    """int32 extremes in a few varblocks, q = 0, +-1, +-2 elsewhere; hf_mul 1 and 2^20; CfL factors -128 and 127; xqm != bqm."""
    W, H = 256, 128
    p = default_frame_params(W, H, global_scale=1, xqm_scale=5, bqm_scale=1)
    st = dict(synth.make_state(W, H, seed=seed, params=p, qm_weights=QW, qm_offsets=QO, mix="small"))
    rng = np.random.default_rng(seed)
    q = rng.choice(np.array([0, 1, -1, 2, -2], np.int64), size=(3, H, W))
    big = np.array([2 ** 24 + 1, -(2 ** 24 + 1), 2 ** 31 - 1, -2 ** 31], np.int64)
    q[:, :16, :64] = rng.choice(big, size=(3, 16, 64))                   # only the top band: other blocks keep small bounds
    st["qcoeff"] = q.astype(np.int32)
    hm = st["hf_mul"].copy()
    hm[:, ::2] = 1
    hm[:, 1::2] = 1 << 20
    oy, ox = cell_origins(st["dct_select"], st["block_origin"])
    st["hf_mul"] = np.ascontiguousarray(hm[oy, ox])
    xf = st["x_from_y"]
    xf.flat[::2], xf.flat[1::2] = -128, 127
    bf = st["b_from_y"]
    bf.flat[::2], bf.flat[1::2] = 127, -128
    return p, st


def scaled_params(global_scale):
    def make(seed):
        p, st = extremes_state(seed)
        p.global_scale = global_scale
        return p, st
    return make


def random_table(seed):
    """Random positive QM weights, asymmetric in every matrix, at the default offsets."""
    rng = np.random.default_rng(seed)
    return rng.uniform(0.25, 2.0, QW.size).astype(np.float32), QO.copy()


def subsampled_state(W, H, shifts, seed):
    """Only 8 x 8-class varblocks; each channel's coefficients and LF cut to its own plane."""
    sy, sx = shifts
    p = default_frame_params(W, H, epf_iters=0, gab=False, color_mode=COLOR_NONE)
    p.shift_y[:], p.shift_x[:] = sy, sx
    st = dict(synth.make_state(W, H, seed=seed, mix=(1.0, 0.0, 0.0, 0.0, 0.0), params=p, qm_weights=QW, qm_offsets=QO))
    rng = np.random.default_rng(seed)
    st["dct_select"] = np.asarray(CLASS8, np.uint8)[rng.integers(0, 10, size=st["dct_select"].shape)]
    st["qcoeff"] = [np.ascontiguousarray(st["qcoeff"][c][:H >> sy[c], :W >> sx[c]]) for c in range(3)]
    st["lf"] = [np.ascontiguousarray(st["lf"][c][:(H // 8) >> sy[c], :(W // 8) >> sx[c]]) for c in range(3)]
    return p, st


SUB_SHIFTS = {"420": ((1, 0, 1), (1, 0, 1)), "422": ((0, 0, 0), (1, 0, 1)), "440": ((1, 0, 1), (0, 0, 0))}


# ---- which planted bugs each case exercises ---------------------------------------------------------------------------------
def hornuss_residuals(st):
    """Whether some Hornuss block has a non-zero coefficient outside its 2 x 2 LF: without one, dropping the residual changes nothing."""
    hb, wb = st["dct_select"].shape
    ly, lx = np.mgrid[0:hb * 8, 0:wb * 8] & 7
    where = (_px(st["dct_select"]) == 1) & ((ly >= 2) | (lx >= 2))
    return any((np.asarray(st["qcoeff"][c]) != 0)[where].any() for c in range(3))


def bugs_for(p, st):
    ds = st["dct_select"]
    present = set(np.unique(ds[st["block_origin"] != 0]).tolist())
    q = np.asarray(st["qcoeff"][1])
    out = []
    if (np.asarray(st["qcoeff"][0]) != 0).any() or (q != 0).any():
        if any(_dims(t)[0] > _dims(t)[1] for t in present):
            out.append("noflip")
        if (q == -1).any():
            out.append("qb_sign")
        if (np.abs(q) >= 2).any():
            out.append("qbn_add")
        if p.xqm_scale != p.bqm_scale:
            out.append("xb_swap")
    if quirk_count(st) > 0 and (q != 0).any():
        out.append("cfl_always")
    if present & {21, 22, 23, 24, 25, 26} and (q != 0).any() and len(np.unique(st["x_from_y"])) > 1:
        out.append("cfl_per_block")
    rect = {t for t in present if TRANSFORM_TYPES[t][1] == M_DCT and _dims(t)[0] != _dims(t)[1]}
    if rect:
        out += ["llf_transpose", "transpose_rect"] if (q != 0).any() else ["llf_transpose"]
    if present & {12, 13}:
        out.append("halves_swap")
    if present & {15, 16}:
        out.append("afv12")
    if 1 in present and hornuss_residuals(st):
        out.append("hornuss_nores")
    if 2 in present:
        out.append("dct2_reverse")
    return out


def assert_rejects_any(bugged, ref, bound, channels, what):
    """assert_rejects on the channel where the bug shows most (a bug may touch only some channels)."""
    c = max(channels, key=lambda k: compare(bugged[k], ref[k], bound[k])[1])
    assert_rejects(bugged[c], ref[c], bound[c], "%s, channel %d" % (what, c))


def check_against(got, p, st, basis, what, bugs=None, got_dequant=None):
    """got (and the oracle's dequantised planes) against the reference; then every planted bug of the case is rejected."""
    ref, bound, de = stage1_ref(p, st, basis, want_dequant=True)
    if got_dequant is not None:
        for c in range(3):
            assert_within(got_dequant[c], de[c][0], de[c][1], "%s: coefficients of channel %d" % (what, c))
    for c in range(3):
        assert_within(got[c], ref[c], bound[c], "%s: channel %d" % (what, c))
    for bug in (bugs_for(p, st) if bugs is None else bugs):
        assert_rejects_any(stage1_ref(p, st, basis, bug=bug)[0], ref, bound, range(3), "%s, planted bug %r" % (what, bug))
    return ref, bound


# ========================================================================================================================
# the reference's own pieces (CPU)
# ========================================================================================================================
def test_dct_matrices_match_scipy():
    for n in (1, 2, 4, 8, 16, 32, 64, 128, 256):
        x = np.random.default_rng(n).standard_normal((n, 3))
        assert np.allclose(idct_mat(n) @ x, scipy.fft.idct(x, type=2, axis=0, norm="ortho") * np.sqrt(n), rtol=0, atol=1e-9)
        assert np.allclose(fdct_mat(n) @ x, scipy.fft.dct(x, type=2, axis=0, norm="ortho") / np.sqrt(n), rtol=0, atol=1e-9)
        assert np.allclose(fdct_mat(n) @ idct_mat(n), np.eye(n), atol=1e-12)
    b = np.random.default_rng(5).standard_normal((2, 16, 8))
    assert np.allclose(_idct2(b), scipy.fft.idctn(b, axes=(1, 2), norm="ortho") * np.sqrt(128), atol=1e-12)


def test_llf_scale_closed_form():
    """scale(0) = 1, it grows with the index, and index 31 is the table's last entry (1.5143734..., its decimal literal within
    1e-13 -- a millionth of a float32 ulp)."""
    s = llf_scale(np.arange(32))
    assert s[0] == 1.0 and (np.diff(s) > 0).all() and abs(s[31] - 1.5143734423313919909) < 1e-12


@pytest.mark.parametrize("t", CLASS8[1:])
def test_class8_matrix_structure(orc, t):
    """What each 64 x 64 map must be regardless of how its loops are written: a DC alone gives a flat block of that value; the
    columns are mutually orthogonal for every type but Hornuss (Haar levels, scaled orthonormal DCTs, an orthonormal basis, and
    DC mixes whose combined columns are orthogonal), and Hornuss keeps every quadrant's mean at its Haar LF (its residual columns sum
    to 0 over each quadrant).  The planted variants break the property they touch or at least move the map."""
    basis = orc.afv_basis().astype(np.float64)
    A, absA = class8_maps(t, basis)
    dc = A @ np.eye(64)[0]
    assert np.allclose(dc, 1.0, atol=1e-12), TRANSFORM_NAMES[t]
    assert (absA >= np.abs(A) - 1e-12).all()
    G = A.T @ A
    method = TRANSFORM_TYPES[t][1]
    if method == M_HORNUSS:
        quad = np.zeros((4, 64))
        for k, (y, x) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
            m = np.zeros((8, 8))
            m[4 * y:4 * y + 4, 4 * x:4 * x + 4] = 1.0 / 16
            quad[k] = m.reshape(64)
        means = quad @ A                                                  # columns 0, 1, 8, 9: the Haar LF coefficients
        assert np.allclose(np.delete(means, [0, 1, 8, 9], axis=1), 0.0, atol=1e-12)
        assert np.allclose(means[:, [0, 1, 8, 9]], haar(np.eye(64).reshape(64, 8, 8), 2).reshape(64, 64)[[0, 1, 8, 9]][:, [0, 1, 8, 9]].T)
        assert np.linalg.matrix_rank(A) == 64
        bugged = class8_maps(t, basis, "hornuss_nores")[0]
        assert not np.allclose(np.delete(quad @ bugged, [0, 1, 8, 9], axis=1), 0.0)
    else:
        # the AFV basis is a float32 table, orthonormal to ~1e-7; everything else is built in float64 here
        tol = 1e-6 if method == M_AFV else 1e-9
        assert np.allclose(G - np.diag(np.diag(G)), 0.0, atol=tol), TRANSFORM_NAMES[t]
        assert np.linalg.matrix_rank(A) == 64
    for bug in ("dct2_reverse", "halves_swap", "afv12"):
        B = class8_maps(t, basis, bug)[0]
        if (bug, t) in (("dct2_reverse", 2), ("halves_swap", 12), ("halves_swap", 13), ("afv12", 15), ("afv12", 16)):
            assert not np.allclose(A, B)


def test_dct_method_is_orthogonal_up_to_scale():
    for t in range(27):
        if TRANSFORM_TYPES[t][1] == M_DCT and max(_dims(t)) <= 32:
            ph, pw = _dims(t)
            A = np.kron(idct_mat(ph), idct_mat(pw))
            assert np.allclose(A.T @ A, ph * pw * np.eye(ph * pw), atol=1e-8)
            assert np.allclose(A[:, 0], 1.0)


def test_quirk_counter():
    st = synth.make_state(520, 264, seed=31, aligned=False)
    assert quirk_count(st) > 0
    assert quirk_count(synth.make_state(256, 256, seed=31, mix="dct8")) == 0


# ========================================================================================================================
# oracle vs reference (CPU), with the planted bugs
# ========================================================================================================================
@pytest.fixture(scope="module")
def basis(orc):
    return orc.afv_basis().astype(np.float64)


@pytest.mark.parametrize("t", range(27))
@pytest.mark.parametrize("hf", ["dense", "zero"])
def test_single_type_oracle_vs_f64(orc, basis, t, hf):
    W, H = single_size(t)
    p, st = single_type_state(t, W, H, 100 + t, hf_zero=hf == "zero")
    out, dq = orc.vardct_invert(p, st, nthreads=8, want_dequant=True)
    bugs = None if hf == "dense" else [b for b in bugs_for(p, st) if b in ("llf_transpose",)]
    check_against(out, p, st, basis, "%s %s" % (TRANSFORM_NAMES[t], hf), bugs, got_dequant=dq)


@pytest.mark.parametrize("t", [0, 4, 5, 18, 21, 24])
def test_square_dct_weight_orientation_oracle_vs_f64(orc, basis, t):
    """Every default square DCT matrix is symmetric, so only an asymmetric table shows a dropped flip on square blocks."""
    W, H = single_size(t)
    p, st = single_type_state(t, W, H, 300 + t)
    st["qm_weights"], st["qm_offsets"] = random_table(t)
    out, dq = orc.vardct_invert(p, st, nthreads=8, want_dequant=True)
    check_against(out, p, st, basis, "%s, random table" % TRANSFORM_NAMES[t], ["noflip"], got_dequant=dq)


MIXED = [(8, 264), (264, 8), (520, 776), (1280, 720), (776, 520)]     # (W, H); 520 x 776 is wider and taller than 512 both ways


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("size", MIXED)
def test_mixed_partition_oracle_vs_f64(orc, basis, size, aligned):
    W, H = size
    p, st = mixed_state(W, H, aligned, 7 + W + H)
    if not aligned and W * H > 64 * 64:
        assert quirk_count(st) > 0
    out, dq = orc.vardct_invert(p, st, nthreads=8, want_dequant=True)
    check_against(out, p, st, basis, "%dx%d aligned=%d" % (W, H, aligned), got_dequant=dq)


EXTREMES = {"gs1": scaled_params(1), "gs65535": scaled_params(65535)}


@pytest.mark.parametrize("case", sorted(EXTREMES))
def test_extremes_oracle_vs_f64(orc, basis, case):
    p, st = EXTREMES[case](61)
    out, dq = orc.vardct_invert(p, st, nthreads=8, want_dequant=True)
    bugs = bugs_for(p, st)
    assert {"qb_sign", "qbn_add", "xb_swap"} <= set(bugs)
    check_against(out, p, st, basis, "extremes " + case, bugs, got_dequant=dq)


@pytest.mark.parametrize("layout", sorted(SUB_SHIFTS))
def test_subsampled_oracle_vs_f64(orc, basis, layout):
    p, st = subsampled_state(272, 144, SUB_SHIFTS[layout], 0x4A584C00 + 79)
    out, dq = orc.vardct_invert(p, st, nthreads=8, want_dequant=True)
    ref, bound, de = stage1_ref(p, st, basis, want_dequant=True)
    present = set(np.unique(st["dct_select"]).tolist())
    assert present == set(CLASS8)
    for c in range(3):
        assert_within(dq[c], de[c][0], de[c][1], "%s coefficients, channel %d" % (layout, c))
        assert_within(out[c], ref[c], bound[c], "%s channel %d" % (layout, c))
    for bug in ("sub_lf_unshifted", "sub_cfl"):
        assert_rejects_any(stage1_ref(p, st, basis, bug=bug)[0], ref, bound, (0, 2), "%s, planted bug %r" % (layout, bug))


# (W, H, aligned, mix): a narrow frame of 8 x 8 / 16-32 classes at every slab-schedule shape (one slab; the pipelined schedule's
# first two and last two slabs one group row high, 512 rows between), and a frame of every class, first-fit placed, over several
# 512-row slabs -- varblocks of 64 to 256 pixels and chroma-from-luma quirk varblocks inside the pipeline
FILTERLESS = [(72, h, True, "small") for h in (8, 264, 520, 1288, 2056)] + [(264, 1544, False, "mixed")]


def filterless_state(case):
    W, H, aligned, mix = case
    p = default_frame_params(W, H, epf_iters=0, gab=False, color_mode=COLOR_NONE)
    st = dict(synth.make_state(W, H, seed=100 + H, params=p, qm_weights=QW, qm_offsets=QO, mix=mix, aligned=aligned))
    if mix == "mixed":
        assert (st["dct_select"][st["block_origin"] != 0] >= 18).any() and quirk_count(st) > 0
    return p, st


@pytest.mark.parametrize("case", FILTERLESS, ids=lambda c: "%dx%d" % c[:2])
def test_filterless_reconstruct_is_stage1(orc, case):
    """With Gaborish, EPF and the colour transform off the whole reconstruction is stage 1 alone, bit for bit (in the oracle)."""
    p, st = filterless_state(case)
    assert np.array_equal(orc.vardct_reconstruct(p, st, nthreads=8), orc.vardct_invert(p, st, nthreads=8))


# ========================================================================================================================
# kernel vs reference (GPU)
# ========================================================================================================================
def _weights(recon, st):
    recon.setWeights(st["qm_weights"], st["qm_offsets"])


@pytest.mark.gpu
@pytest.mark.parametrize("t", range(27))
@pytest.mark.parametrize("hf", ["dense", "zero"])
def test_single_type_kernel_vs_f64(recon, basis, t, hf):
    W, H = single_size(t)
    p, st = single_type_state(t, W, H, 100 + t, hf_zero=hf == "zero")
    _weights(recon, st)
    check_against(recon.invertVarDCT(p, st), p, st, basis, "kernel %s %s" % (TRANSFORM_NAMES[t], hf), bugs=[])


@pytest.mark.gpu
@pytest.mark.parametrize("t", [0, 4, 5, 18, 21, 24, 6, 19])
def test_random_table_kernel_vs_f64(recon, basis, t):
    W, H = single_size(t)
    p, st = single_type_state(t, W, H, 300 + t)
    st["qm_weights"], st["qm_offsets"] = random_table(t)
    try:
        recon.setWeights(st["qm_weights"], st["qm_offsets"])
        got = recon.invertVarDCT(p, st)
    finally:
        recon.generateWeights()
    check_against(got, p, st, basis, "kernel %s, random table" % TRANSFORM_NAMES[t], ["noflip"])


@pytest.mark.gpu
@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("size", MIXED)
def test_mixed_partition_kernel_vs_f64(recon, basis, size, aligned):
    W, H = size
    p, st = mixed_state(W, H, aligned, 7 + W + H)
    _weights(recon, st)
    check_against(recon.invertVarDCT(p, st), p, st, basis, "kernel %dx%d aligned=%d" % (W, H, aligned), bugs=[])


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(EXTREMES))
def test_extremes_kernel_vs_f64(recon, basis, case):
    p, st = EXTREMES[case](61)
    _weights(recon, st)
    check_against(recon.invertVarDCT(p, st), p, st, basis, "kernel extremes " + case, bugs=[])


FAMILY = {t: "k1_small" for t in (0, 1, 2, 3, 12, 13, 14, 15, 16, 17)}
FAMILY.update({t: "k1_medium" for t in range(4, 12)})
FAMILY.update({t: "k1_big" for t in range(18, 27)})


def expected_work(t, n):
    """The stage-1 kernels that must have work for a frame of n varblocks of type t, and no other: k1_small or k1_medium (batches,
    any positive count), or exactly two k1_big instantiations -- pass 0 walks the 32-column strips of each varblock (columns of
    pixelHeight: class N = pixelHeight), pass 1 its 32-row strips (class N = pixelWidth), one item per strip and channel."""
    fam = FAMILY[t]
    if fam != "k1_big":
        return {fam: None}
    ph, pw = _dims(t)
    return {"k1_big<%d,0>" % ph: n * (pw // 32) * 3, "k1_big<%d,1>" % pw: n * (ph // 32) * 3}


@pytest.mark.gpu
@pytest.mark.parametrize("t", range(27))
def test_single_type_kernel_family(recon, basis, t):
    """Which stage-1 kernels had work.  Every stage-1 kernel is launched on every call (persistent grids read their work sizes on the
    device), so a kernel trace cannot show routing; the plan k0_count / k0_plan wrote (jxlb200_stage1_plan) can.  On a frame tiled
    with one type, only that type's family may have work: k1_small for types 0-3 and 12-17, k1_medium for 4-11, and for 18-26
    k1_big's column pass in the class of pixelHeight and its row pass in the class of pixelWidth.  The result is then held to the
    reference, so the kernel that had the work is the one that produced it."""
    W, H = single_size(t)
    p, st = single_type_state(t, W, H, 100 + t)
    _weights(recon, st)
    got = recon.invertVarDCT(p, st)
    counts, work = recon.stage1_plan()
    n = int(st["block_origin"].sum())
    assert counts[t] == n and counts.sum() == n, "%s: the plan counts %s" % (TRANSFORM_NAMES[t], counts.tolist())
    want = expected_work(t, n)
    for k, v in work.items():
        if k not in want:
            assert v == 0, "%s: %s has %d work items, but the type belongs to %s" % (TRANSFORM_NAMES[t], k, v, sorted(want))
        elif want[k] is None:
            assert v > 0, "%s: %s has no work" % (TRANSFORM_NAMES[t], k)
        else:
            assert v == want[k], "%s: %s has %d work items, not %d" % (TRANSFORM_NAMES[t], k, v, want[k])
    check_against(got, p, st, basis, "kernel family %s" % TRANSFORM_NAMES[t], bugs=[])


def test_expected_work_covers_every_big_instantiation():
    """The 9 big types reach all 8 k1_big instantiations (4 line-length classes x 2 passes), so no instantiation goes unchecked."""
    seen = set()
    for t in range(18, 27):
        seen |= set(expected_work(t, 1))
    assert seen == {"k1_big<%d,%d>" % (32 << k, pas) for k in range(4) for pas in (0, 1)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", FILTERLESS, ids=lambda c: "%dx%d" % c[:2])
@pytest.mark.parametrize("narrow", [False, True])
def test_filterless_reconstruct_kernel_vs_f64(recon, basis, case, narrow):
    """The slab-pipelined host entry point (int32, and the int16 call) with every filter and the colour transform off."""
    p, st = filterless_state(case)
    _weights(recon, st)
    check_against(recon.reconstruct(p, st, narrow=narrow), p, st, basis, "reconstruct %dx%d narrow=%d" % (case[0], case[1], narrow),
                  bugs=[])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", sorted(SUB_SHIFTS))
def test_subsampled_reconstruct_kernel_vs_f64(recon, basis, layout):
    """Per-channel stage 1 at the shifted positions, then the chroma upsampling (chroma_ref), with the stage-1 bound carried through
    the upsampling's positive weights."""
    p, st = subsampled_state(272, 144, SUB_SHIFTS[layout], 0x4A584C00 + 79)
    ref, bound = stage1_ref(p, st, basis)
    up, up_bound = chroma_ref(p, ref)
    carried, _ = chroma_ref(p, bound)
    _weights(recon, st)
    got = recon.reconstruct(p, st)
    for c in range(3):
        assert_within(got[c], up[c], up_bound[c] + carried[c], "%s subsampled reconstruct, channel %d" % (layout, c))


@pytest.mark.gpu
@pytest.mark.parametrize("pitch", [296, 270])
def test_invert_dev_pitched_output(recon, basis, pitch):
    """jxlb200_vardct_invert_dev into planes wider than the frame: the frame matches, the padding columns keep their NaN.  A pitch
    that is a multiple of 4 takes the kernels' vector stores, 270 the scalar ones."""
    import torch
    W, H = 264, 136
    p, st = mixed_state(W, H, False, 17)
    _weights(recon, st)
    dev = torch.device("cuda", 0)
    d = {k: torch.from_numpy(np.ascontiguousarray(st[k])).to(dev)
         for k in ("qcoeff", "lf", "dct_select", "block_origin", "hf_mul", "x_from_y", "b_from_y")}
    out = torch.full((3, H, pitch), float("nan"), dtype=torch.float32, device=dev)
    recon.invert_dev(p, [d["qcoeff"][c].data_ptr() for c in range(3)], [d["lf"][c].data_ptr() for c in range(3)],
                     d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(),
                     d["x_from_y"].data_ptr(), d["b_from_y"].data_ptr(), [out[c].data_ptr() for c in range(3)], pitch)
    recon.sync()
    got = out.cpu().numpy()
    assert np.isnan(got[:, :, W:]).all(), "invert_dev wrote into the padding columns"
    check_against(got[:, :, :W], p, st, basis, "invert_dev pitch %d" % pitch, bugs=[])


@pytest.mark.gpu
def test_batch_stack_kernel_vs_f64(recon, basis):
    """jxlb200_vardct_reconstruct_batch_dev with the filters off: stage 1 runs once over the stack, and every frame must match its
    own reference (a varblock or CfL tile leaking across a frame boundary would show)."""
    import torch
    W, H, n = 264, 128, 3
    p = default_frame_params(W, H, epf_iters=0, gab=False, color_mode=COLOR_NONE)
    sts = [dict(synth.make_state(W, H, seed=930 + f, params=p, qm_weights=QW, qm_offsets=QO, aligned=f != 1)) for f in range(n)]
    _weights(recon, sts[0])
    dev = torch.device("cuda", 0)
    keys = ("qcoeff", "lf", "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y")
    d = {k: torch.from_numpy(np.ascontiguousarray(np.concatenate([s[k] for s in sts], axis=-2))).to(dev) for k in keys}
    out = torch.full((3, H * n, W), float("nan"), dtype=torch.float32, device=dev)
    recon.reconstruct_batch_dev(p, n, [d["qcoeff"][c].data_ptr() for c in range(3)], [d["lf"][c].data_ptr() for c in range(3)],
                                d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(),
                                d["x_from_y"].data_ptr(), d["b_from_y"].data_ptr(), d["sharpness"].data_ptr(),
                                [out[c].data_ptr() for c in range(3)])
    recon.sync()
    got = out.cpu().numpy()
    for f in range(n):
        check_against(got[:, f * H:(f + 1) * H], p, sts[f], basis, "batch frame %d" % f, bugs=[])


@pytest.mark.gpu
@pytest.mark.parametrize("t", range(27))
def test_flat_lf_gives_flat_block_kernel(recon, basis, t):
    """Free of any reading: with no HF and a constant LF v per channel, every varblock of every type is flat at v."""
    W, H = single_size(t)
    p, st = single_type_state(t, W, H, 500 + t, hf_zero=True)
    v = (0.0123, 0.61, -0.37)
    st["lf"] = np.stack([np.full(st["lf"][0].shape, v[c], np.float32) for c in range(3)])
    _weights(recon, st)
    got = recon.invertVarDCT(p, st)
    _, bound = stage1_ref(p, st, basis)
    for c in range(3):
        assert_within(got[c], np.full((H, W), float(np.float32(v[c]))), bound[c], "%s flat LF, channel %d" % (TRANSFORM_NAMES[t], c))
