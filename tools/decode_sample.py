"""CLI in the spirit of `java -jar jxlatte.jar input.jxl output.png` (J/JXLatte.java): decodes a .jxl file with the C++
front end + the CUDA reconstruction and writes PNG (8/16 bit) or PFM.  Prints the host front-end time (entropy decoding,
headers) and the reconstruction time separately, as the north star asks.

    python tools/decode_sample.py input.jxl [output.png|output.pfm] [--bits 8|16] [--repeat N] [--device] [--preview]

--device decodes through DeviceEngine: the image stays on the GPU until the output file is written from it.
--preview decodes at 1:8 (JXLOptions(preview=True)) and prints the route it took: "lf" (from the LF images alone) or "full".

There is no CPU engine here: the checker's decode of the same file is tests/tools/decode_with_oracle.py."""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("input")
    ap.add_argument("output", nargs="?")
    ap.add_argument("--bits", type=int, default=8)
    ap.add_argument("--repeat", type=int, default=1)
    ap.add_argument("--device", action="store_true", help="keep the frame loop and the image on the GPU (DeviceEngine)")
    ap.add_argument("--preview", action="store_true", help="decode at 1:8 and print the route taken")
    a = ap.parse_args()
    from jxlatte_b200.decoder import CudaEngine, DeviceEngine, JXLDecoder, JXLOptions
    engine = DeviceEngine() if a.device else CudaEngine()
    best = None
    for _ in range(a.repeat):
        d = JXLDecoder(a.input, engine=engine, options=JXLOptions(preview=a.preview))
        t0 = time.perf_counter()
        img = d.decode()
        total = time.perf_counter() - t0
        if best is None or total < best[0]:
            best = (total, dict(d.timings))
    mp = img.width * img.height / 1e6
    print("%s: %dx%d, %d channel(s), engine=%s: front end %.1f ms, reconstruction + glue %.1f ms, total %.1f ms (%.1f MP/s end to end)" % (
        os.path.basename(a.input), img.width, img.height, len(img.channels), "device" if a.device else "cuda", best[1]["front_end_s"] * 1e3,
        best[1]["reconstruct_s"] * 1e3, best[0] * 1e3, mp / best[0]))
    if a.preview:
        print("preview route: %s" % d.preview_route)
    if a.output:
        if a.output.endswith(".pfm"):
            img.write_pfm(a.output)
        else:
            img.write_png(a.output, a.bits, engine=engine)
    engine.close()


if __name__ == "__main__":
    main()
