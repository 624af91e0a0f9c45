#!/usr/bin/env python
"""bench.py -- reconstructed MP/s of the VarDCT reconstruction path (dequant -> IDCT -> CfL/LLF -> Gaborish -> EPF ->
XYB->linear) on B200, with the roofline of the dominant kernel and the CPU restatement timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 8k|batch2048|split16k]
                    [--dump-outputs DIR]

A "step" = one pass of the hot path over one batch of synthetic post-entropy frame state (SURVEY.md 8(d)).
  8k        (default) one 7680x4320 frame per GPU, mixed varblocks DCT8..DCT256+AFV, gab on, EPF 3 iterations; N GPUs
            = a batch of N frames sharded per image, no communication (weak scaling)
  batch2048 sixteen 2048x2048 frames per GPU per step, EPF 1 iteration (per-image sharding, weak scaling), handed over as
            one vertically stacked batch (jxlb200_vardct_reconstruct_batch_dev: stage 1 once over the stack, stage 2 one
            launch with a frame dimension)
  split16k  one 16384x16384 frame split by group rows over the N GPUs, 7 halo rows exchanged with NCCL (strong scaling)
Prints ONE JSON line on rank 0.  Under torchrun one process per GPU; barrier + synchronize around the timed region,
device time by CUDA events, max over ranks.

--dump-outputs DIR writes the float32 linear planes the last timed step produced (what the caller of the timed entry point
receives) as DIR/planes.npy, shape (3, rows, width); under torchrun each rank writes DIR/planes_rank<R>.npy.  Inputs are
drawn from fixed seeds, so two builds run with the same arguments can be compared file for file.  Outputs larger than
64 MB in all are cut to a sample of whole rows drawn with a fixed seed (the same rows for the same shape).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_PX = 24.35      # SURVEY.md 8(d): 12 coeff + 12 out + 0.1875 LF + 0.1563 maps + ~0.002
BYTES_PER_PX_K2 = 24.13   # stage 2 alone: XYB in, linear out, sigma maps
METRIC = "reconstructed MP/s (VarDCT dequant->XYB)"
BATCH_FRAMES = 16         # frames per GPU per step of the batch2048 workload
DUMP_BYTES = 64 * 10**6   # --dump-outputs: at most this much in all, .npy headers included
DUMP_SEED = 0x4A584C00    # --dump-outputs: which rows a sample keeps


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append([s.strip() for s in o])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = [int(s[0]) for s in self.samples if s and s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples if len(s) >= 6 for i in range(4) if s[2 + i].lower().startswith("active")})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def make_inputs(W, H, seed, epf_iters, oracle_tables=False, survey_spec=False):
    from jxlatte_b200 import synth, default_frame_params
    p = default_frame_params(W, H, epf_iters=epf_iters, gab=True)
    if oracle_tables:       # the reference arm must not touch the product library: tables from the CPU restatement
        from oracle import oracle
        qw, qo = oracle.qm_default_weights()
    else:
        from jxlatte_b200.host import qm_generate
        qw, qo = qm_generate()
    st = synth.make_state(W, H, seed=seed, params=p, qm_weights=qw, qm_offsets=qo, survey_spec=survey_spec)
    return p, st, qw, qo


def dump_planes(dirname, name, planes, parts=1):
    """--dump-outputs: planes (3, rows, width), a device tensor or a numpy array, as float32 to dirname/name.npy; when that
    would pass DUMP_BYTES / parts, a sample of whole rows drawn with DUMP_SEED, kept in increasing order."""
    rows, width = planes.shape[1], planes.shape[2]
    keep = min(rows, (DUMP_BYTES // parts - 4096) // (3 * width * 4))     # 4096: room for the .npy header
    if keep < rows:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(rows, keep, replace=False))
        if isinstance(planes, np.ndarray):
            planes = planes[:, idx]
        else:
            import torch
            planes = planes[:, torch.from_numpy(idx).to(planes.device)]
    if not isinstance(planes, np.ndarray):
        planes = planes.cpu().numpy()
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(planes, dtype=np.float32))


def cpu_baseline(nthreads, sample=(2048, 2048), epf_iters=3, reps=1):
    """The CPU restatement of jxlatte's algorithm (oracle 'port'; not the JVM) on a bounded sample of the workload."""
    from oracle import oracle
    W, H = sample
    p, st, _, _ = make_inputs(W, H, 0x4A584C00 + 77, epf_iters, oracle_tables=True)
    t0 = time.perf_counter()
    for _ in range(reps):
        oracle.vardct_reconstruct(p, st, nthreads=nthreads)
    dt = (time.perf_counter() - t0) / reps
    return W * H / 1e6 / dt, dt


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  jxlatte is pure Java and no JVM exists in
    this image, so this arm times the C restatement (oracle/, kind 'port') on all host cores, each step a bounded sample of
    the workload; jxlatte itself runs this path on ONE thread, so the single-thread figure is reported beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle
    cores = os.cpu_count() or 1
    iters = 3 if args.workload != "batch2048" else 1
    W, H = 2048, 2048       # 64 groups: enough parallel work for every host core in both stages
    p, st, _, _ = make_inputs(W, H, 0x4A584C00 + 78, iters, oracle_tables=True)
    for _ in range(min(args.warmup, 2)):
        oracle.vardct_reconstruct(p, st, nthreads=cores)
    steps = max(1, args.steps)
    t0 = time.perf_counter()
    for _ in range(steps):
        planes = oracle.vardct_reconstruct(p, st, nthreads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_planes(args.dump_outputs, "planes", planes)
    v = W * H * steps / 1e6 / dt
    t0 = time.perf_counter()
    p1, st1, _, _ = make_inputs(1024, 1024, 0x4A584C00 + 79, iters, oracle_tables=True)
    t0 = time.perf_counter()
    oracle.vardct_reconstruct(p1, st1, nthreads=1)
    v1 = 1024 * 1024 / 1e6 / (time.perf_counter() - t0)
    sample = "one %dx%d frame of the workload per step (same varblock mix / gab / EPF %d iterations), not the full %s" % (
        W, H, iters, "7680x4320 frame" if args.workload == "8k" else "workload")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "MP/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, iters),
            "cpu_baseline": {"value": v, "unit": "MP/s", "cores": cores, "kind": "port", "sample": sample,
                             "single_thread": {"value": v1, "unit": "MP/s", "cores": 1,
                                               "sample": "one 1024x1024 frame; jxlatte runs this path on one thread"}},
            "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(args, iters):
    names = {"8k": "synthetic 7680x4320 VarDCT frame per GPU (batch of N frames sharded per image), mixed varblocks DCT8-DCT256+AFV, gab on, EPF 3 iterations",
             "batch2048": "%d synthetic 2048x2048 VarDCT frames per GPU per step (per-image sharding, one stacked batch call), mixed varblocks, gab on, EPF 1 iteration" % BATCH_FRAMES,
             "split16k": "synthetic 16384x16384 VarDCT frame split by group rows over N GPUs, NCCL halo rows, mixed varblocks, gab on, EPF 3 iterations"}
    return {"workload": names[args.workload], "epf_iters": iters, "parallelism": "per-image shard x%d" % args.gpus if args.workload != "split16k" else "group-row split x%d" % args.gpus,
            "l2": "inputs per step exceed the 126 MB L2 (no flush needed)"}


def note(msg):
    """progress on stderr (the JSON line alone goes to stdout)"""
    sys.stderr.write("[bench %s r%s] %s\n" % (time.strftime("%H:%M:%S"), os.environ.get("RANK", "0"), msg))
    sys.stderr.flush()


def bind_to_gpu_numa_node(local):
    """One process per GPU: keep the process (and with it the pinned host buffers it allocates, first touch) on the NUMA node the
    GPU hangs off, so that eight ranks' host<->device copies use both sockets' memory controllers and PCIe roots instead of
    crossing the socket link.  Best effort; returns what it did for the bench line."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return "single NUMA node"
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no usable CPU on node %d" % node
        os.sched_setaffinity(0, cpus)
        return "node %d (%d CPUs)" % (node, len(cpus))
    except Exception as e:
        return "not bound (%s)" % type(e).__name__


class Workload:
    """One workload's device-resident inputs and its step (one pass of the hot path over one batch)."""

    def __init__(self, name, rec, dev, rank, world):
        import torch
        from jxlatte_b200.multigpu import slab_rows, SplitFrame
        self.name, self.rec, self.world = name, rec, world
        self.iters = 1 if name == "batch2048" else 3
        if name == "8k":
            W, H, nframes = 7680, 4320, 1
        elif name == "batch2048":
            W, H, nframes = 2048, 2048, BATCH_FRAMES
        else:
            W, H, nframes = 16384, 16384, 1
        self.W, self.H, self.nframes = W, H, nframes
        rows = H
        if name == "split16k":      # contiguous group rows per rank; the rank's seed differs, the frame is "one frame" by shape
            y0, rows = slab_rows(H, world, rank)
        self.p, self.st, self.qw, self.qo = make_inputs(W, rows, 0x4A584C00 + 2 + rank, self.iters)
        rec.setWeights(self.qw, self.qo)
        keys = ("qcoeff", "lf", "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y")

        def dev_t(a):
            return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

        first = {k: dev_t(self.st[k]) for k in keys}
        first["out"] = torch.empty((3, rows, W), dtype=torch.float32, device=dev)
        self.first, self.stack, self.halo = first, None, None
        if nframes > 1:
            parts = [first]
            for f in range(1, nframes):
                _, stf, _, _ = make_inputs(W, H, 0x4A584C00 + 100 * f + rank, self.iters)
                parts.append({k: dev_t(stf[k]) for k in keys})
            self.stack = {k: torch.cat([d[k] for d in parts], dim=-2).contiguous() for k in keys}
            self.stack["out"] = torch.empty((3, H * nframes, W), dtype=torch.float32, device=dev)
            del parts
        if name == "split16k":
            self.halo = SplitFrame(rec, self.p, first, y0, rows, H, rank, world, dev)
        self.px_per_step_all = W * H if name == "split16k" else W * H * nframes * world

    def step(self):
        rec, p = self.rec, self.p
        if self.halo is not None:
            self.halo.step()
            return
        d = self.stack if self.stack is not None else self.first
        q, lf = [d["qcoeff"][c].data_ptr() for c in range(3)], [d["lf"][c].data_ptr() for c in range(3)]
        out = [d["out"][c].data_ptr() for c in range(3)]
        args = (d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(), d["x_from_y"].data_ptr(),
                d["b_from_y"].data_ptr(), d["sharpness"].data_ptr(), out)
        if self.stack is not None:
            rec.reconstruct_batch_dev(p, self.nframes, q, lf, *args)
        else:
            rec.reconstruct_dev(p, q, lf, *args)


def timed_steps(wl, stream, steps, warmup, barrier, dev, world):
    """W warm-up steps, then exactly K steps between two events on the launching stream, barrier + synchronize on both sides;
    returns (max-over-ranks ms for the K steps, launches)."""
    import torch
    import torch.distributed as dist
    for _ in range(max(warmup, 3)):
        wl.step()
    wl.rec.sync()
    barrier()
    l0 = wl.rec.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        wl.step()
    e1.record(stream)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), wl.rec.launch_count() - l0


def run_ours(args):
    import torch
    import torch.distributed as dist
    from jxlatte_b200 import _lib
    from jxlatte_b200.host import Reconstructor

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the ONE JSON line and nothing else: native libraries (NCCL's version banner) write to file descriptor 1
    # directly, so it points at stderr until the line is printed
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if numa:
        note("NUMA: " + numa)

    rec = Reconstructor(local)
    if os.environ.get("JXLB200_STAGE2"):      # kernel-variant experiments (include/jxlb200.h: JXLB200_OPT_STAGE2); default 0
        rec.set_option(_lib.OPT_STAGE2, int(os.environ["JXLB200_STAGE2"]))
    # a real (non-legacy) stream shared by torch's events and the library's kernels: a NULL handle would mean
    # "the context's own stream" to jxlb200_set_stream and the events would time nothing
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    rec.set_stream(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    note("building the %s workload" % args.workload)
    wl = Workload(args.workload, rec, dev, rank, world)
    W, H, iters, p, st = wl.W, wl.H, wl.iters, wl.p, wl.st
    note("timing %d steps" % args.steps)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        wl.step()
    rec.sync()
    barrier()
    if sampler:
        sampler.start()
    ms_max, launches = timed_steps(wl, stream, args.steps, 0, barrier, dev, world)
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=3)
    if args.dump_outputs:       # before the stage timings below write into the same planes
        out = (wl.stack if wl.stack is not None else wl.first)["out"]
        dump_planes(args.dump_outputs, "planes" if world == 1 else "planes_rank%d" % rank, out, world)
    value = wl.px_per_step_all * args.steps / 1e6 / (ms_max / 1e3)

    # ---- stage timing for the roofline of the dominant kernel (rank 0, same process, CUDA events on the same stream) ----
    roof = None
    cpu = None
    note("%.3f ms per step; stage timings" % (ms_max / args.steps))
    if rank == 0 and wl.halo is None:
        d = wl.first
        plane = torch.empty((3, H, W), dtype=torch.float32, device=dev)
        q = [d["qcoeff"][c].data_ptr() for c in range(3)]
        lf = [d["lf"][c].data_ptr() for c in range(3)]
        xyb = [plane[c].data_ptr() for c in range(3)]
        out1 = torch.empty((3, H, W), dtype=torch.float32, device=dev) if wl.stack is not None else d["out"]
        out = [out1[c].data_ptr() for c in range(3)]

        def timed(fn, n=10):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(n):
                fn()
            b.record(stream)
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n

        def stage2():
            rec.restore_dev(p, None, xyb, W, d["hf_mul"].data_ptr(), d["sharpness"].data_ptr(), out)

        t1 = timed(lambda: rec.invert_dev(p, q, lf, d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(),
                                          d["x_from_y"].data_ptr(), d["b_from_y"].data_ptr(), xyb, W))
        t2 = timed(stage2)
        # stage 1 again on coefficients drawn exactly as SURVEY.md 8(d) says (15 % non-zero everywhere, +-63, CfL +-32): k1_big's column
        # walk skips zero coefficients, so its time depends on the density; real files are far sparser (profiles/r2_coefficient_density.md)
        t1_spec = None
        if (W, H) == (7680, 4320) and not args.no_sub_records:
            _, st_s, _, _ = make_inputs(W, H, 0x4A584C00 + 2, iters, survey_spec=True)
            qs = torch.from_numpy(np.ascontiguousarray(st_s["qcoeff"])).to(dev)
            xs, bs = torch.from_numpy(st_s["x_from_y"]).to(dev), torch.from_numpy(st_s["b_from_y"]).to(dev)
            t1_spec = timed(lambda: rec.invert_dev(p, [qs[c].data_ptr() for c in range(3)], lf, d["dct_select"].data_ptr(), d["block_origin"].data_ptr(),
                                                   d["hf_mul"].data_ptr(), xs.data_ptr(), bs.data_ptr(), xyb, W))
            del qs, xs, bs, st_s
            # the spec-density planes are not image-like: put the workload's own stage-1 planes back before anything reads xyb again
            rec.invert_dev(p, q, lf, d["dct_select"].data_ptr(), d["block_origin"].data_ptr(), d["hf_mul"].data_ptr(),
                           d["x_from_y"].data_ptr(), d["b_from_y"].data_ptr(), xyb, W)
            rec.sync()
        peak, which = peaks()
        # stage 2 of a frame this size with Gaborish on is the stream kernel (csrc/jxlb200.cu: stream_pays), else the tile kernel
        k2_name = ("k2_stream (persistent, TMA-fed row rings: fused Gaborish+EPF+colour, bit-exact)" if (W * H >= 600000 and (p.gab or iters == 3) and iters >= 1)
                   else "k2_exact (fused Gaborish+EPF+colour, bit-exact)")
        if os.environ.get("JXLB200_STAGE2"):
            k2_name = "stage 2 as selected by JXLB200_STAGE2=%s" % os.environ["JXLB200_STAGE2"]
        dom = k2_name if t2 >= t1 else "stage 1 (k1_small/medium/big: dequant+CfL+LLF+IDCT)"
        bpp = BYTES_PER_PX_K2 if t2 >= t1 else BYTES_PER_PX
        ach = bpp * W * H / (max(t1, t2) / 1e3) / 1e9
        traffic = None
        try:   # dram__bytes_read + dram__bytes_write of the dominant kernel from the committed ncu --set full capture
            with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
                tj = json.load(f)
            if t2 >= t1 and iters == 3 and (W, H) == (7680, 4320):
                traffic = tj["traffic_bytes_per_launch"]
        except Exception:
            pass
        roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "kernel": dom, "peak_source": which, "algorithmic_bytes_per_px": bpp,
                "stage_ms": {"stage1_dequant_idct": t1, "stage2_gab_epf_color": t2, "stage1_at_survey_spec_density_15pct": t1_spec},
                "pipeline_frac": BYTES_PER_PX * W * H / ((t1 + t2) / 1e3) / 1e9 / peak}
        # the tolerance mode (JXLB200_OPT_STAGE2 = 2: re-associated, FMA-contracted EPF sums; inside 1e-4 / 1 LSB at 8 bits, what a
        # caller that quantises to 8 bits may select) timed beside the bit-exact default, with its error against it
        if not os.environ.get("JXLB200_STAGE2"):
            try:
                stage2()
                rec.sync()
                exact = out1.clone()
                rec.set_option(_lib.OPT_STAGE2, _lib.STAGE2_FUSED)
                t2f = timed(stage2)
                rec.sync()
                err = float((out1 - exact).abs().max().item())
                ach_f = BYTES_PER_PX_K2 * W * H / (t2f / 1e3) / 1e9
                roof["tolerance_mode"] = {"kernel": "k2_fused (JXLB200_OPT_STAGE2 = 2)", "stage2_ms": t2f, "achieved": ach_f, "frac": ach_f / peak,
                                          "max_abs_err_vs_exact": err,
                                          "pipeline_frac": BYTES_PER_PX * W * H / ((t1 + t2f) / 1e3) / 1e9 / peak}
                del exact
            finally:
                rec.set_option(_lib.OPT_STAGE2, _lib.STAGE2_AUTO)
        del plane

    # ---- e2e: the host-buffer C-ABI call a reference-side shim makes; pinned host memory, H2D + D2H inside.  EVERY rank
    # runs it at the same time (each on its own GPU and PCIe link); the aggregate is what N GPUs deliver to N callers ----
    e2e = None
    note("e2e")
    if wl.halo is None and args.workload == "8k":
        keys = ("qcoeff", "lf", "dct_select", "block_origin", "hf_mul", "sharpness", "x_from_y", "b_from_y")
        hst = {k: torch.from_numpy(np.ascontiguousarray(st[k])).pin_memory() for k in keys}
        hout = torch.empty((3, H, W), dtype=torch.float32).pin_memory()
        hnp = {k: v.numpy() for k, v in hst.items()}
        houtn = hout.numpy()
        rec.set_stream(None)
        n_e2e = max(3, min(args.steps, 10))

        def wall(fn):
            for _ in range(2):
                fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                fn()
            dt = (time.perf_counter() - t0) / n_e2e
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        dt = wall(lambda: rec.reconstruct(p, hnp, out=houtn))
        h2d = sum(int(v.numel() * v.element_size()) for v in hst.values())
        e2e = {"value": W * H * world / 1e6 / dt, "unit": "MP/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(hout.numel() * 4),
               "ms_per_step": dt * 1e3, "api": "jxlb200_vardct_reconstruct (host buffers, pinned; int32 coefficients in, float32 planes out: the reference's own layout)",
               "ranks": world, "numa": numa,
               "note": "every rank makes the call at once on its own GPU; value = all ranks' pixels / slowest rank's time"}
        # the same call with the coefficients narrowed to int16 by the caller (jxlb200_vardct_reconstruct_i16: half the upload,
        # identical planes); reported beside e2e, which stays on the reference's own int32 layout
        h16 = dict(hnp)
        q16 = torch.from_numpy(np.ascontiguousarray(st["qcoeff"]).astype(np.int16)).pin_memory()
        h16["qcoeff"] = q16.numpy()
        ref_planes = houtn.copy() if rank == 0 else None
        dt16 = wall(lambda: rec.reconstruct(p, h16, out=houtn, narrow=True))
        same = bool(np.array_equal(ref_planes, houtn)) if rank == 0 else None
        e2e["int16_coefficients"] = {"value": W * H * world / 1e6 / dt16, "unit": "MP/s", "ms_per_step": dt16 * 1e3,
                                     "h2d_bytes_per_step": h2d - int(q16.numel() * 2), "planes_equal_int32_call": same,
                                     "api": "jxlb200_vardct_reconstruct_i16 (host buffers, pinned)"}
        # PNG-ready samples: sRGB transfer + quantise + interleave on the device, 3 (6) bytes per pixel back
        for bits in (8, 16):
            hpk = torch.empty((H, W, 3 * bits // 8), dtype=torch.uint8).pin_memory()
            hpkn = hpk.numpy()
            dtp = wall(lambda: rec.reconstruct_packed(p, h16, bits=bits, linear=True, out=hpkn, narrow=True))
            e2e["png%d" % bits] = {"value": W * H * world / 1e6 / dtp, "unit": "MP/s", "ms_per_step": dtp * 1e3,
                                   "h2d_bytes_per_step": h2d - int(q16.numel() * 2), "d2h_bytes_per_step": int(hpk.numel()),
                                   "api": "jxlb200_vardct_reconstruct_packed (int16 coefficients in, interleaved %d-bit sRGB samples out, pinned)" % bits}
            del hpk
        if rank == 0:
            # what pinning buys: the same int32 / float32 call on pageable numpy arrays (a Panama Arena segment is pageable)
            pg = {k: np.array(v, copy=True) for k, v in hnp.items()}
            pout = np.empty((3, H, W), np.float32)
            for _ in range(2):
                rec.reconstruct(p, pg, out=pout)
            t0 = time.perf_counter()
            for _ in range(3):
                rec.reconstruct(p, pg, out=pout)
            e2e["pageable_host_buffers_ms_per_step"] = (time.perf_counter() - t0) / 3 * 1e3
            del pg, pout
        del q16, hst, hout
        rec.set_stream(stream.cuda_stream)

    if rank == 0 and world == 1 and wl.halo is None:
        cores = os.cpu_count() or 1
        v, dt_cpu = cpu_baseline(cores, sample=(2048, 2048), epf_iters=iters)
        cpu = {"value": v, "unit": "MP/s", "cores": cores, "kind": "port",
               "sample": "one 2048x2048 frame of the same synthetic workload (%.1f s), C restatement of jxlatte's algorithm, not the JVM" % dt_cpu}

    # ---- the other two configurations of BASELINE.json configs[4], as sub-records of the default line ----
    sub = {}
    if args.workload == "8k" and not args.no_sub_records:
        names = ["batch2048"] + (["split16k"] if world > 1 else [])
        del wl
        torch.cuda.empty_cache()
        for name in names:
            try:
                note("sub-record " + name)
                w2 = Workload(name, rec, dev, rank, world)
                k = max(3, min(args.steps, 10))
                ms2, _ = timed_steps(w2, stream, k, 3, barrier, dev, world)
                sub[name] = {"value": w2.px_per_step_all * k / 1e6 / (ms2 / 1e3), "unit": "MP/s", "ms_per_step": ms2 / k, "steps": k,
                             "scaling": "strong" if name == "split16k" else "weak",
                             "config": workload_config(argparse.Namespace(workload=name, gpus=world), w2.iters)}
                del w2
                torch.cuda.empty_cache()
            except Exception as e:      # a sub-record must never break the bench line
                sub[name] = {"error": repr(e)}

    front = None
    if rank == 0 and world == 1 and args.workload == "8k":
        # the sequential host half (entropy decoding, headers) is reported separately, as the north star asks: a real
        # sample through libjxlfront.so, then the same file end to end through the public JXLDecoder API on this GPU
        try:
            from jxlatte_b200 import frontend
            from jxlatte_b200.decoder import CudaEngine, JXLDecoder
            path = os.path.join(ROOT, "tests", "golden", "samples", "bbb.jxl")
            data = open(path, "rb").read()
            t_fe = []
            for _ in range(5):
                t0 = time.perf_counter()
                pr = frontend.parse(data)
                t_fe.append(time.perf_counter() - t0)
                pr.close()
            eng = CudaEngine()
            t_all = []
            for _ in range(4):
                t0 = time.perf_counter()
                img = JXLDecoder(data, engine=eng).decode()
                t_all.append(time.perf_counter() - t0)
            eng.close()
            mp = img.width * img.height / 1e6
            front = {"file": "tests/golden/samples/bbb.jxl (1280x720 VarDCT, gab, EPF 1)", "front_end_ms": min(t_fe) * 1e3,
                     "front_end_MP_per_s": mp / min(t_fe), "decode_total_ms": min(t_all[1:]) * 1e3,
                     "note": "front end = C++ host code (container, headers, ANS, MA trees, coefficient decode); total = JXLDecoder.decode() incl. Python glue"}
        except Exception as e:          # never let the side measurement break the bench line
            front = {"error": repr(e)}

    note("done")
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "MP/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": "strong" if args.workload == "split16k" else "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": workload_config(args, iters), "gpu_launches": int(launches),
                "clocks": sampler.summary() if sampler else None}
        if roof:
            line["roofline"] = roof
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if sub:
            line["sub_records"] = sub
        if front:
            line["front_end"] = front
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    rec.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="8k", choices=["8k", "batch2048", "split16k"])
    ap.add_argument("--no-sub-records", action="store_true", help="skip the batch2048 / split16k sub-records of the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the planes of the last timed step to DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
