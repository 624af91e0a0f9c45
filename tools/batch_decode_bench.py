"""Throughput of decode_batch against a loop of single-file decodes, on DeviceEngine.

    python tools/batch_decode_bench.py OUT_JSON [--repeat N] [--copies K] [--workers W]

Two lists: the 12 samples of tests/golden/samples, and K (default 8) copies of them in a row.  Each list is decoded two ways, the
two alternating in one run:
  loop    JXLDecoder(path, engine=DeviceEngine).decode().to_int(8) per file, then one synchronise
  batch   decode_batch(paths, engine, bits=8, mode="rgb", workers=W) (W: decode_batch's default when not given)
Each figure is the best of N runs after a warm-up run of both ways.  Reported per list: images/s of each way, and for the best batch
run its timings (host parse time summed over files, parse wall, device wall, total) and parse / device overlap = parse wall +
device wall - total.  The GPU's name and power limit, the CPU count and the workers value used are read in the same run (nvidia-smi,
read-only query)."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from device_decode_bench import SAMPLES, gpu_info  # noqa: E402


def run_loop(paths, engine):
    import torch
    from jxlatte_b200.decoder import JXLDecoder
    t0 = time.perf_counter()
    out = [JXLDecoder(p, engine=engine).decode().to_int(8) for p in paths]
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def run_batch(paths, engine, workers):
    from jxlatte_b200.decoder import decode_batch
    t0 = time.perf_counter()
    r = decode_batch(paths, engine, bits=8, mode="rgb", workers=workers)
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_json")
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--copies", type=int, default=8)
    ap.add_argument("--workers", type=int, default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_decode_bench: no CUDA device")
    from jxlatte_b200.decoder import DeviceEngine
    names = sorted(f[:-4] for f in os.listdir(SAMPLES) if f.endswith(".jxl"))
    base = [os.path.join(SAMPLES, n + ".jxl") for n in names]
    dev = DeviceEngine()
    cores = os.cpu_count() or 1
    lists = {"samples_x1": base, "samples_x%d" % a.copies: base * a.copies}
    rows = {}
    for key, paths in lists.items():
        workers = a.workers or max(1, min(len(paths), cores // 2))          # decode_batch's default
        run_loop(paths, dev)
        _, r = run_batch(paths, dev, workers)                                  # warm-up of both ways
        del r
        loop_t, batch_t, best = [], [], None
        for _ in range(a.repeat):                                              # alternate the two ways
            t, out = run_loop(paths, dev)
            loop_t.append(t)
            del out
            t, r = run_batch(paths, dev, workers)
            batch_t.append(t)
            if best is None or t < best[0]:
                best = (t, dict(r.timings))
            del r
        tm = best[1]
        rows[key] = dict(files=len(paths), workers=workers, loop_s=round(min(loop_t), 4), batch_s=round(min(batch_t), 4),
                         loop_images_per_s=round(len(paths) / min(loop_t), 2), batch_images_per_s=round(len(paths) / min(batch_t), 2),
                         batch_parse_sum_s=round(tm["parse_s"], 4), batch_parse_wall_s=round(tm["parse_wall_s"], 4),
                         batch_device_wall_s=round(tm["device_wall_s"], 4), batch_total_s=round(tm["total_s"], 4),
                         batch_overlap_s=round(tm["parse_wall_s"] + tm["device_wall_s"] - tm["total_s"], 4))
        rows[key]["speedup"] = round(rows[key]["loop_s"] / rows[key]["batch_s"], 2)
        print(key, json.dumps(rows[key]), flush=True)
    dev.close()
    out = dict(gpu=gpu_info(), cpu_count=cores, torch=torch.__version__, repeat=a.repeat,
               statistic="best of repeat after one warm-up run of each way, the two ways alternating", samples=names, lists=rows)
    d = os.path.dirname(os.path.abspath(a.out_json))
    os.makedirs(d, exist_ok=True)
    with open(a.out_json, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(gpu=out["gpu"], cpu_count=cores)))


if __name__ == "__main__":
    main()
