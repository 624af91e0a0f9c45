"""Per-sample decode times of the host-buffer path (CudaEngine) against the device-resident path (DeviceEngine).

    python tools/device_decode_bench.py OUT_DIR [--repeat N] [--samples a,b,...]

For each sample in tests/golden/samples it reports, in OUT_DIR/device_decode.json:
  front_end_ms        entropy decoding and headers on the host (the same for both paths)
  host_glue_ms        host path: "reconstruction + glue", from the end of the front end to the returned numpy image
  device_glue_ms      device path: the same span, ending in the decoder's synchronise (the image is complete on the device)
  device_to_u8_ms     device path: front end excluded, to an 8-bit [C, H, W] CUDA tensor (to_int(8) and a synchronise)
Each figure is the best of N decodes after a warm-up decode of the same file.  Animations are decoded to their last image and
the figures summed over images.  The GPU's name and power limit are read in the same run (nvidia-smi, read-only query)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SAMPLES = os.path.join(ROOT, "tests", "golden", "samples")


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return ["unavailable: %s" % e]


def decode_all(path, engine, to_u8=False):
    """-> (front end s, reconstruction + glue s summed over the displayed images, to-u8 s or None, images)."""
    import torch
    from jxlatte_b200.decoder import JXLDecoder
    d = JXLDecoder(path, engine=engine)
    glue, n, u8 = 0.0, 0, None
    while True:
        img = d.decode()
        if img is None:
            break
        glue += d.timings["reconstruct_s"]
        n += 1
        if to_u8:
            t0 = time.perf_counter()
            img.to_int(8)
            torch.cuda.synchronize()
            u8 = (u8 or 0.0) + d.timings["reconstruct_s"] + time.perf_counter() - t0
    return d.timings["front_end_s"], glue, u8, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--samples", default="")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("device_decode_bench: no CUDA device")
    from jxlatte_b200.decoder import CudaEngine, DeviceEngine
    names = a.samples.split(",") if a.samples else sorted(f[:-4] for f in os.listdir(SAMPLES) if f.endswith(".jxl"))
    host, dev = CudaEngine(), DeviceEngine()
    rows = {}
    for name in names:
        path = os.path.join(SAMPLES, name + ".jxl")
        decode_all(path, host)
        decode_all(path, dev, to_u8=True)            # warm-up of both paths on this file
        fe, hg, dg, du = [], [], [], []
        for _ in range(a.repeat):                      # alternate the two paths
            f, g, _, n = decode_all(path, host)
            fe.append(f)
            hg.append(g)
            f, g, _, _ = decode_all(path, dev)
            fe.append(f)
            dg.append(g)
            _, _, u, _ = decode_all(path, dev, to_u8=True)
            du.append(u)
        rows[name] = dict(images=n, front_end_ms=round(min(fe) * 1e3, 3), host_glue_ms=round(min(hg) * 1e3, 3),
                          device_glue_ms=round(min(dg) * 1e3, 3), device_to_u8_ms=round(min(du) * 1e3, 3))
        rows[name]["speedup_glue"] = round(rows[name]["host_glue_ms"] / max(rows[name]["device_glue_ms"], 1e-9), 2)
        print(name, json.dumps(rows[name]), flush=True)
    host.close()
    dev.close()
    out = dict(gpu=gpu_info(), torch=torch.__version__, repeat=a.repeat, statistic="best of repeat after one warm-up decode",
               samples=rows)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "device_decode.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(gpu=out["gpu"])))


if __name__ == "__main__":
    main()
