"""The group-row split (SURVEY.md 8(e)) on ONE GPU: a frame processed as slabs with explicit halo rows must be
bit-identical to the frame processed whole.  This is the same device path the multi-GPU split uses; only the halo
transport (NCCL there, a device copy here) differs."""
import numpy as np
import pytest

from jxlatte_b200 import synth, default_frame_params, _lib
from jxlatte_b200.host import qm_generate, Slab
from jxlatte_b200.multigpu import slab_rows, split_state
from kernel_trace import assert_stage2_kernel, launched_kernels

pytestmark = pytest.mark.gpu
HALO = _lib.HALO_ROWS
FORCED = {_lib.STAGE2_STREAM: "stream", _lib.STAGE2_TILE: "tile", _lib.STAGE2_STAGED: "staged"}


@pytest.mark.parametrize("cfg", [dict(W=328, H=776, parts=3, iters=3, gab=True), dict(W=512, H=512, parts=2, iters=1, gab=True),
                                 dict(W=264, H=1032, parts=4, iters=2, gab=False)])
@pytest.mark.parametrize("stage2", [_lib.STAGE2_AUTO, _lib.STAGE2_STREAM, _lib.STAGE2_TILE, _lib.STAGE2_STAGED])
def test_slabs_match_whole_frame(recon, cfg, stage2):
    import torch
    W, H, parts = cfg["W"], cfg["H"], cfg["parts"]
    p = default_frame_params(W, H, epf_iters=cfg["iters"], gab=cfg["gab"])
    qw, qo = qm_generate()
    st = synth.make_state(W, H, seed=5 + W, params=p, qm_weights=qw, qm_offsets=qo)
    recon.set_option(_lib.OPT_STAGE2, stage2)
    try:
        whole, kernels = launched_kernels(lambda: recon.reconstruct(p, st))
        if stage2 in FORCED:
            assert_stage2_kernel(kernels, FORCED[stage2], p)
        dev = torch.device("cuda", 0)
        spans = [slab_rows(H, parts, r) for r in range(parts)]
        wb = W // 8
        xybs, maps, outs, ps, dsts = [], [], [], [], []
        # stage 1 per slab (independent: varblocks never cross a group row)
        for (y0, rows) in spans:
            s = split_state(st, y0, rows)
            ps_ = default_frame_params(W, rows, epf_iters=cfg["iters"], gab=cfg["gab"])
            d = {k: torch.from_numpy(np.ascontiguousarray(s[k])).to(dev) for k in
                 ("qcoeff", "lf", "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y")}
            xyb = torch.zeros((3, rows + 2 * HALO, W), dtype=torch.float32, device=dev)
            base = [xyb[c].data_ptr() + HALO * W * 4 for c in range(3)]
            recon.invert_dev(ps_, [d["qcoeff"][c].data_ptr() for c in range(3)], [d["lf"][c].data_ptr() for c in range(3)],
                             d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(),
                             d["x_from_y"].data_ptr(), d["b_from_y"].data_ptr(), base, W)
            m = torch.ones((2, rows // 8 + 2, wb), dtype=torch.int32, device=dev)
            m[0, 1:-1] = d["hf_mul"]
            m[1, 1:-1] = d["sharpness"]
            xybs.append(xyb); maps.append(m); ps.append(ps_); dsts.append(d)
        recon.sync()
        # halo transport: neighbours' boundary rows and block rows
        for i, (y0, rows) in enumerate(spans):
            if i > 0:
                pr = spans[i - 1][1]
                xybs[i][:, :HALO] = xybs[i - 1][:, pr:pr + HALO]
                maps[i][:, 0] = maps[i - 1][:, -2]
            if i < parts - 1:
                xybs[i][:, HALO + rows:] = xybs[i + 1][:, HALO:2 * HALO]
                maps[i][:, -1] = maps[i + 1][:, 1]
        torch.cuda.synchronize()
        got = np.empty((3, H, W), np.float32)
        for i, (y0, rows) in enumerate(spans):
            out = torch.empty((3, rows, W), dtype=torch.float32, device=dev)
            slab = Slab(y0, rows, H, 1 if i > 0 else 0, 1 if i < parts - 1 else 0)
            base = [xybs[i][c].data_ptr() + HALO * W * 4 for c in range(3)]
            _, kernels = launched_kernels(lambda: (recon.restore_dev(ps[i], slab, base, W, maps[i][0].data_ptr() + wb * 4,
                                                                     maps[i][1].data_ptr() + wb * 4, [out[c].data_ptr() for c in range(3)]),
                                                   recon.sync()))
            if stage2 in FORCED:
                assert_stage2_kernel(kernels, FORCED[stage2], ps[i])
            got[:, y0:y0 + rows] = out.cpu().numpy()
    finally:
        recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)
    assert np.array_equal(got, whole), "max abs diff %g" % np.abs(got - whole).max()


@pytest.mark.parametrize("cfg", [dict(W=512, H=256, n=3, iters=1, gab=True), dict(W=264, H=320, n=4, iters=3, gab=True),
                                 dict(W=256, H=64, n=5, iters=2, gab=False), dict(W=384, H=512, n=1, iters=0, gab=True)])
@pytest.mark.parametrize("stage2", [_lib.STAGE2_AUTO, _lib.STAGE2_STREAM])
def test_batch_of_stacked_frames_matches_single_frames(recon, orc, cfg, stage2):
    """jxlb200_vardct_reconstruct_batch_dev: n equally sized frames stacked vertically, stage 1 once over the stack, stage 2
    per frame.  Every frame must equal its own reconstruction (oracle for frame 0, the single-frame CUDA call for all): a
    varblock, chroma-from-luma tile or filter tap leaking across a frame boundary would show."""
    import torch
    W, H, n = cfg["W"], cfg["H"], cfg["n"]
    p = default_frame_params(W, H, epf_iters=cfg["iters"], gab=cfg["gab"])
    qw, qo = qm_generate()
    sts = [synth.make_state(W, H, seed=900 + 7 * f + W, params=p, qm_weights=qw, qm_offsets=qo) for f in range(n)]
    singles = [recon.reconstruct(p, s) for s in sts]
    assert np.array_equal(singles[0], orc.vardct_reconstruct(p, sts[0], nthreads=8))
    dev = torch.device("cuda", 0)
    keys = ("qcoeff", "lf", "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y")
    d = {k: torch.from_numpy(np.ascontiguousarray(np.concatenate([s[k] for s in sts], axis=-2))).to(dev) for k in keys}
    out = torch.full((3, H * n, W), np.nan, dtype=torch.float32, device=dev)
    recon.set_option(_lib.OPT_STAGE2, stage2)      # the stack goes through the stream kernel as one launch when forced (or large enough)
    try:
        _, kernels = launched_kernels(lambda: (
            recon.reconstruct_batch_dev(p, n, [d["qcoeff"][c].data_ptr() for c in range(3)], [d["lf"][c].data_ptr() for c in range(3)],
                                        d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(),
                                        d["x_from_y"].data_ptr(), d["b_from_y"].data_ptr(), d["sharpness"].data_ptr(),
                                        [out[c].data_ptr() for c in range(3)]),
            recon.sync()))
    finally:
        recon.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)
    if stage2 == _lib.STAGE2_STREAM:
        assert_stage2_kernel(kernels, "stream", p)
    got = out.cpu().numpy()
    for f in range(n):
        assert np.array_equal(got[:, f * H:(f + 1) * H], singles[f]), "frame %d of the stack differs" % f


def test_batch_rejects_bad_shapes(recon):
    p = default_frame_params(64, 72)        # height not a multiple of 64: chroma-from-luma tiles of two frames would mix
    with pytest.raises(ValueError):
        recon.reconstruct_batch_dev(p, 2, [0, 0, 0], [0, 0, 0], 0, 0, 0, 0, 0, 0, [0, 0, 0])
