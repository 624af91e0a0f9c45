"""Which CUDA kernels a call launched, read from a torch.profiler trace (CUDA activity records, cat == "kernel").

Used to prove that a test which forces a stage-2 kernel ran that kernel: JXLB200_OPT_STAGE2 = 5 (stream) takes k2_exact instead
wherever k2_stream cannot take the frame, and a result that matches the oracle cannot tell the two apart."""
import json
import os
import tempfile


def launched_kernels(fn):
    """-> (fn(), names of the kernels launched while fn ran)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    fd, path = tempfile.mkstemp(suffix=".json")
    os.close(fd)
    try:
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    finally:
        os.unlink(path)
    return result, [e.get("name", "") for e in events if e.get("cat") == "kernel"]


def expected_stage2(mode, p):
    """The fused stage-2 kernel a frame with params p must run under a forced mode ("stream", "tile" or "staged"), or None.
    k2_stream takes frames whose sizes are multiples of 8 with 16-byte aligned planes and epf_iters >= 1 (the library's planes always
    are aligned); k2_exact takes any frame with Gaborish or EPF on; "staged" runs one kernel per stage and neither fused one."""
    filters = bool(p.gab) or p.epf_iters > 0
    if mode == "staged" or not filters:
        return None
    if mode == "stream" and p.epf_iters >= 1 and p.width % 8 == 0 and p.height % 8 == 0:
        return "k2_stream"
    return "k2_exact"


def assert_stage2_kernel(names, mode, p):
    want = expected_stage2(mode, p)
    ran = sorted({n for n in names if "k2_stream" in n or "k2_exact" in n})
    if want is None:
        assert not ran, "stage 2 %r must run no fused kernel, but ran %s" % (mode, ran)
    else:
        other = "k2_exact" if want == "k2_stream" else "k2_stream"
        assert any(want in n for n in ran) and not any(other in n for n in ran), (
            "stage 2 %r on a %dx%d frame (epf_iters %d, gab %d) must run %s, but ran %s"
            % (mode, p.width, p.height, p.epf_iters, p.gab, want, ran or "no fused stage-2 kernel"))
