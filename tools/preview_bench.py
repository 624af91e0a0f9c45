"""Per-sample times of the 1:8 preview (JXLOptions(preview=True)) against the full decode, on both engines.

    python tools/preview_bench.py OUT_DIR [--repeat N] [--samples a,b,...]

For each sample in tests/golden/samples it reports, in OUT_DIR/preview.json:
  route                    the preview's route: "lf" (rendered from the LF images, no HF entropy decoding) or "full"
  full_front_end_ms        full decode: entropy decoding and headers on the host
  preview_front_end_ms     preview: the same span (the LF-only parse; on the "full" route both parses)
  {host,device}_full_ms    "reconstruction + glue" of the full decode on CudaEngine / DeviceEngine: from the end of the front end to
                           the returned image (DeviceEngine: ending in the decoder's synchronise)
  {host,device}_preview_ms the same span of the preview
  psnr_lf_vs_full_db       "lf" samples: PSNR of the LF-route preview against the full-route preview of the same file (every channel
                           averaged over 8 x 8 areas), both as 8-bit sRGB samples (to_int(8)) on CudaEngine
Each figure is the best of N decodes after a warm-up decode of the same file, the four decodes alternating.  Animations are decoded
to their last image, the device figures summed over images.  The GPU's name and power limit are read in the same run (nvidia-smi,
read-only query)."""
import argparse
import json
import os
import sys
from unittest import mock

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from device_decode_bench import SAMPLES, gpu_info  # noqa: E402


def decode_all(path, engine, preview):
    """-> (front end s, reconstruction + glue s summed over the displayed images, route)."""
    from jxlatte_b200.decoder import JXLDecoder, JXLOptions
    d = JXLDecoder(path, engine=engine, options=JXLOptions(preview=preview))
    glue = 0.0
    while True:
        img = d.decode()
        if img is None:
            break
        glue += d.timings["reconstruct_s"]
    return d.timings["front_end_s"], glue, d.preview_route


def route_psnr(path, engine):
    """8-bit PSNR of the LF-route preview against the full-route preview (the route forced), over every displayed image."""
    from jxlatte_b200 import decoder

    def images():
        d = decoder.JXLDecoder(path, engine=engine, options=decoder.JXLOptions(preview=True))
        out = []
        while True:
            img = d.decode()
            if img is None:
                return out
            out.append(img.to_int(8).astype(np.float64))
    lf = images()
    with mock.patch.object(decoder, "preview_route", lambda info: "full"):
        full = images()
    mse = float(np.mean(np.concatenate([(a - b).ravel() ** 2 for a, b in zip(lf, full)])))
    return None if mse == 0 else round(10.0 * np.log10(255.0 ** 2 / mse), 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--samples", default="")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("preview_bench: no CUDA device")
    from jxlatte_b200.decoder import CudaEngine, DeviceEngine
    names = a.samples.split(",") if a.samples else sorted(f[:-4] for f in os.listdir(SAMPLES) if f.endswith(".jxl"))
    engines = dict(host=CudaEngine(), device=DeviceEngine())
    rows = {}
    for name in names:
        path = os.path.join(SAMPLES, name + ".jxl")
        for e in engines.values():                     # warm-up of the four decodes on this file
            decode_all(path, e, False)
            decode_all(path, e, True)
        t = {k: [] for k in ("full_fe", "preview_fe", "host_full", "host_preview", "device_full", "device_preview")}
        route = None
        for _ in range(a.repeat):
            for ename, e in engines.items():
                fe, g, _ = decode_all(path, e, False)
                t["full_fe"].append(fe)
                t[ename + "_full"].append(g)
                fe, g, route = decode_all(path, e, True)
                t["preview_fe"].append(fe)
                t[ename + "_preview"].append(g)
        best = {k: round(min(v) * 1e3, 3) for k, v in t.items()}
        rows[name] = dict(route=route, full_front_end_ms=best["full_fe"], preview_front_end_ms=best["preview_fe"],
                          host_full_ms=best["host_full"], host_preview_ms=best["host_preview"],
                          device_full_ms=best["device_full"], device_preview_ms=best["device_preview"])
        if route == "lf":
            rows[name]["psnr_lf_vs_full_db"] = route_psnr(path, engines["host"])     # None: identical samples
        print(name, json.dumps(rows[name]), flush=True)
    for e in engines.values():
        e.close()
    out = dict(gpu=gpu_info(), torch=torch.__version__, repeat=a.repeat, statistic="best of repeat after one warm-up decode",
               samples=rows)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "preview.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(gpu=out["gpu"])))


if __name__ == "__main__":
    main()
