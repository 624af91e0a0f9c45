#!/usr/bin/env python
"""tools/stage1_ab.py -- stage 1 (dequantisation, chroma-from-luma, LLF, inverse transforms) of the 8K benchmark frame, timed for
one build of the library, so that two builds can be compared run against run.

    JXLB200_LIB=/path/to/libjxlb200.so python tools/stage1_ab.py [--reps 5] [--n 20] [--out FILE.json]

The library is the one JXLB200_LIB names (default: the in-tree jxlatte_b200/libjxlb200.so).  Inputs are bench.py's: the 8K
workload's frame state (7680x4320, default synthetic density) and the same frame with coefficients drawn at SURVEY.md 8(d)'s 15 %
density.  For each it reports

  * rec.invert_dev timed by CUDA events (n calls per repetition, `reps` repetitions: median, min, max in ms),
  * a full rec.reconstruct_dev step (stage 1 + stage 2) at the default density, timed the same way,
  * each k1_* / k0_* kernel's mean duration per invert_dev call from a torch.profiler CUDA trace, taken in a separate pass,
  * the CRC32 of the three stage-1 planes (and of the reconstructed planes), to show that two builds compute the same thing,

together with the GPU's name and power limit.  One JSON object goes to stdout (and to --out).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    import torch
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except Exception as e:      # the name still identifies the card
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


def crc(t):
    return "%08x" % (zlib.crc32(t.detach().cpu().numpy().tobytes()) & 0xffffffff)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n", type=int, default=20, help="calls per timed repetition")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from bench import Workload, make_inputs
    from jxlatte_b200 import _lib
    from jxlatte_b200.host import Reconstructor

    if not torch.cuda.is_available():
        sys.exit("stage1_ab.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rec = Reconstructor(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    rec.set_stream(stream.cuda_stream)

    wl = Workload("8k", rec, dev, 0, 1)
    W, H, p, d = wl.W, wl.H, wl.p, wl.first
    xyb = torch.empty((3, H, W), dtype=torch.float32, device=dev)
    lf = [d["lf"][c].data_ptr() for c in range(3)]
    _, st_s, _, _ = make_inputs(W, H, 0x4A584C00 + 2, wl.iters, survey_spec=True)
    spec = {"qcoeff": torch.from_numpy(np.ascontiguousarray(st_s["qcoeff"])).to(dev),
            "x_from_y": torch.from_numpy(st_s["x_from_y"]).to(dev), "b_from_y": torch.from_numpy(st_s["b_from_y"]).to(dev)}
    del st_s

    def invert(src):
        q = [src["qcoeff"][c].data_ptr() for c in range(3)]
        rec.invert_dev(p, q, lf, d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(),
                       src["x_from_y"].data_ptr(), src["b_from_y"].data_ptr(), [xyb[c].data_ptr() for c in range(3)], W)

    cases = {"invert_dev_default_density": lambda: invert(d), "invert_dev_15pct_density": lambda: invert(spec),
             "reconstruct_dev_step": wl.step}

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        out = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(args.n):
                fn()
            b.record(stream)
            torch.cuda.synchronize()
            out.append(a.elapsed_time(b) / args.n)
        return {"median_ms": statistics.median(out), "min_ms": min(out), "max_ms": max(out), "runs_ms": out}

    res = {"library": _lib.SO_PATH, "gpu": gpu_info(0), "frame": [W, H], "calls_per_rep": args.n, "reps": args.reps,
           "timing": {}, "crc32": {}, "kernels_us_per_invert_dev": {}}
    for name, fn in cases.items():
        res["timing"][name] = timed(fn)

    # CRCs: stage-1 planes of both densities, the reconstructed planes of the default one
    invert(spec); torch.cuda.synchronize()
    res["crc32"]["stage1_planes_15pct_density"] = crc(xyb)
    invert(d); torch.cuda.synchronize()
    res["crc32"]["stage1_planes_default_density"] = crc(xyb)
    wl.step(); torch.cuda.synchronize()
    res["crc32"]["reconstructed_planes"] = crc(d["out"])

    # kernel durations from a CUDA trace, in a pass of its own (tracing slows the host)
    from torch.profiler import profile, ProfilerActivity
    for label, src in (("default_density", d), ("15pct_density", spec)):
        calls = 10
        invert(src); torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                invert(src)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            if ev.key.startswith(("void k1_", "k1_", "void k0_", "k0_")):
                us = getattr(ev, "device_time_total", None)
                if us is None:
                    us = ev.cuda_time_total
                per[ev.key.split("(")[0].replace("void ", "")] = round(us / calls, 2)
        res["kernels_us_per_invert_dev"][label] = dict(sorted(per.items(), key=lambda kv: -kv[1]))
    rec.close()

    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
