#!/usr/bin/env python
"""bench.py — headline benchmark of the PCM -> spectrum -> pixels hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]

Default workload (BASELINE.json configs[1], `--config headline`): module `bars`, setbufsize 4096 ("4096-pt FFT"),
1920x1080 RGBA8, 1024 independent synthetic 22050 Hz stereo streams PER GPU (weak scaling: the batch is sharded
stream-wise, no inter-GPU collective on the data path).  Other BASELINE configurations through --config (same JSON line):
  radial4k   configs[2]: radial, setbufsize 8192, 3840x2160, 4096 streams over 8 GPUs = 512 per GPU
  graph720 / wave720   configs[3]'s modules: setbufsize 2048, 1280x720, 256 streams (throughput; the 240 fps cadence is
             tools/cadence.py)
  sweep:<n>:<w>x<h>    one point of configs[4] (bars, 8192 streams over 8 GPUs = 1024 per GPU; framebuffer ring when
             1024 frames exceed the HBM budget); tools/sweep_configs.py runs the whole grid

One step = one rd_update(modified=true) for every stream of the batch: the spectrum path (window + FFT + log + gravity
+ average + smoothing: one kernel below setbufsize 4096, three from there up — DESIGN 4.1a) and one frame per stream.

  value  frames/s, inputs already resident in HBM (glava_b200_update_device)
  e2e    frames/s through the reference-facing C ABI with HOST buffers, the way GLava's FIFO backend feeds it (fifo.c:89-110):
         every step the new int16 chunk of every stream crosses PCIe (glava_b200_ingest_fifo, rings stay in HBM), the update
         runs (glava_b200_update_rings) and one stream's frame comes back to pinned host memory (the "optional cudaMemcpy
         readback for inspection").  e2e.full_ring_path = the same through glava_b200_update with whole [batch][n] float
         rings (what glava.c:528-537 hands rd_update; 33.5 MB per step at the headline)
  roofline  raster kernel: W*H*4 algorithmic bytes per frame / its CUDA-event duration, vs MEASURED_PEAKS.json
  cpu_baseline  the REFERENCE ITSELF on the host cores — its rd_update on Mesa llvmpipe (oracle/cpu_baseline.py)

`--impl reference` times that same reference path as its own arm.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HOP = 256
UNIT = "frames/s"
FB_BUDGET = 48e9          # bytes of framebuffer kept resident per GPU; beyond that a ring of slots (8K sweeps)


def workload(name):
    """-> dict(module, n, w, h, batch, metric, label)"""
    if name == "headline":
        return dict(module="bars", n=4096, w=1920, h=1080, batch=1024,
                    metric="spectrum frames/sec @4096-pt FFT, 1920x1080 bars", label="BASELINE configs[1]")
    if name == "radial4k":
        return dict(module="radial", n=8192, w=3840, h=2160, batch=512,
                    metric="spectrum frames/sec @8192-pt FFT, 3840x2160 radial", label="BASELINE configs[2] (4096 streams / 8 GPUs)")
    if name in ("graph720", "wave720"):
        m = name[:-3]
        return dict(module=m, n=2048, w=1280, h=720, batch=256,
                    metric=f"spectrum frames/sec @2048-pt FFT, 1280x720 {m}", label="BASELINE configs[3] module, throughput")
    if name in ("circle1080", "radial1080", "graph1080", "wave1080"):
        m = name[:-4]
        return dict(module=m, n=4096, w=1920, h=1080, batch=1024,
                    metric=f"spectrum frames/sec @4096-pt FFT, 1920x1080 {m}", label="other module at the headline geometry")
    if name.startswith("sweep:"):
        _, n, geo = name.split(":")
        w, h = (int(v) for v in geo.split("x"))
        return dict(module="bars", n=int(n), w=w, h=h, batch=1024,
                    metric=f"spectrum frames/sec @{n}-pt FFT, {w}x{h} bars", label="BASELINE configs[4] point (8192 streams / 8 GPUs)")
    raise SystemExit(f"unknown --config {name}")


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        sm.sort()
        # "under load": upper half of the samples (the sampler also sees the idle gaps around the region)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the raster kernel from the committed ncu capture, if any"""
    try:
        with open(os.path.join(ROOT, "profiles", "raster_bars_traffic.json")) as f:
            return float(json.load(f)["dram_bytes_per_launch"])
    except Exception:
        return None


def config_block(wl, batch, world, p=None, fb_slots=None):
    return {"workload": f"{wl['module']} module, {wl['n']}-sample buffer ({wl['n'] // 2}-pt complex FFT), {wl['w']}x{wl['h']} RGBA8, "
                        f"batch={batch} streams per GPU ({wl['label']})",
            "module": wl["module"], "bufsize": wl["n"], "width": wl["w"], "height": wl["h"],
            "batch_per_gpu": batch, "streams_total": batch * world, "parallelism": f"stream-sharded x{world}, no collective"}


DUMP_STREAMS = 16          # streams whose outputs --dump-outputs writes
DUMP_PIXELS = 1 << 17      # pixels per dumped frame (the same seeded positions in every stream)


def dump_outputs(out_dir, r, batch):
    """What the last timed update handed its caller, for output-by-output comparison of two builds: the frames of a seeded
    sample of streams at a seeded sample of pixel positions.  With a framebuffer ring (fb_slots < batch) only the last
    `slots` streams still hold their frame, so the sample is drawn from those.  The timed path runs with lazy_smooth = 1,
    where glava_b200_spectrum() / _textures() hold only the bins the module samples and the rest is stale (glava_b200.h):
    those are not outputs of this path, and two builds may differ there without any pixel differing, so they are not
    written.  float32 / float64 only, about 34 MB at the headline configuration."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    p = r.params
    slots = p.fb_slots if 0 < p.fb_slots < batch else batch
    rng = np.random.default_rng(0)
    streams = np.sort(rng.choice(np.arange(batch - slots, batch), size=min(DUMP_STREAMS, slots), replace=False))
    pixels = np.sort(rng.choice(p.h * p.w, size=min(DUMP_PIXELS, p.h * p.w), replace=False))
    frames = np.stack([r.readback(int(s)).reshape(-1, 4)[pixels] for s in streams]).astype(np.float32)
    out = {"stream_index": streams.astype(np.float64), "frame_pixel_index": pixels.astype(np.float64), "frames_rgba8": frames}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args, wl, rank, world):
    """reference arm: the reference's own rd_update (CPU FFT + its GL passes and module shaders on Mesa llvmpipe) on all host
    cores, one GLava renderer per core; a step = every core renders FPW frames of the same workload"""
    if rank != 0:
        return
    from oracle.cpu_baseline import CpuBaseline, describe
    pd = dict(module=wl["module"], n=wl["n"], w=wl["w"], h=wl["h"])
    fpw = max(1, int(round(2 * (1920 * 1080) / (wl["w"] * wl["h"]))))      # ~0.15 s of CPU work per worker and step
    base = CpuBaseline(pd, frames_per_worker=fpw)
    for _ in range(args.warmup):
        base.step()
    t, frames = 0.0, 0
    for _ in range(args.steps):
        dt, f = base.step()
        t += dt; frames += f
    base.close()
    value = frames / t
    sample = f"{base.cores * fpw} frames per step ({fpw} per core) x {args.steps} steps; " + describe(base.kind)
    cfg = config_block(wl, 1, 1)
    cfg.update({"frames_per_step": frames // args.steps, "device": "host CPU", "batch_per_gpu": None, "streams_total": base.cores,
                "parallelism": f"one renderer per host core x{base.cores}"})
    line = {
        "impl": "reference", "metric": wl["metric"], "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": base.cores, "kind": base.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("GLAVA_BENCH_CONFIG", "headline"))
    ap.add_argument("--batch", type=int, default=env_int("GLAVA_BENCH_BATCH", 0), help="streams per GPU (0: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the lazy_smooth=0 and full-ring legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what their last step computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    wl = workload(args.config)

    rank = env_int("RANK", 0); world = env_int("WORLD_SIZE", 1); local = env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import glava_b200 as g
    from glava_b200.synth import synth_batch_int16

    MODULE, N, W, H = wl["module"], wl["n"], wl["w"], wl["h"]
    torch.cuda.set_device(local)
    # one process per GPU: run on the CPUs of the GPU's own NUMA node and keep every pinned buffer there (capi.cu)
    numa = g.lib().glava_b200_bind_thread_to_device(local)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL writes its banner ("NCCL version ...") straight to fd 1 when the communicator is created; stdout must
        # carry the one JSON line only, so communicator creation (init + first collective) runs with fd 1 -> fd 2
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier(device_ids=[local])
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    batch, K, Wm = (args.batch or wl["batch"]), args.steps, args.warmup
    p = g.default_params(MODULE, n=N, w=W, h=H)
    p.lazy_smooth = 1
    frame_bytes = W * H * 4
    if batch * frame_bytes > FB_BUDGET:
        p.fb_slots = max(1, int(FB_BUDGET // frame_bytes))
    r = g.Renderer(p, batch=batch, device=local)
    stream = torch.cuda.ExternalStream(r.cuda_stream, device=local)

    # ---- synthetic input: this rank's shard of the global stream set -----------------------------
    nsnap = min(K + Wm, 4)                                   # distinct ring snapshots cycled through
    total = N + nsnap * HOP
    pcm = synth_batch_int16(rank * batch, batch, 0, total)  # [batch][total][2] int16
    pcm_f = pcm.astype(np.float32) / np.float32(65535)      # fifo.c:104-107
    host_l = [g.pinned_empty((batch, N), np.float32, local) for _ in range(nsnap)]
    host_r = [g.pinned_empty((batch, N), np.float32, local) for _ in range(nsnap)]
    dev_l, dev_r = [], []
    for i in range(nsnap):
        host_l[i][:] = pcm_f[:, (i + 1) * HOP:(i + 1) * HOP + N, 0]
        host_r[i][:] = pcm_f[:, (i + 1) * HOP:(i + 1) * HOP + N, 1]
        dev_l.append(torch.from_numpy(host_l[i]).to(f"cuda:{local}"))
        dev_r.append(torch.from_numpy(host_r[i]).to(f"cuda:{local}"))
    torch.cuda.synchronize()

    def barrier():
        if distributed:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if not distributed:
            return ms
        t = torch.tensor([ms], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def device_leg(rr, steps):
        """K updates with the rings resident in HBM; -> (ms, kernel times, launches)"""
        st = torch.cuda.ExternalStream(rr.cuda_stream, device=local)
        for i in range(Wm):
            rr.update_device(dev_l[i % nsnap].data_ptr(), dev_r[i % nsnap].data_ptr(), True)
        rr.sync()
        rr.set_timing(True)
        l0 = rr.launch_count
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record(st)
        for i in range(steps):
            rr.update_device(dev_l[(Wm + i) % nsnap].data_ptr(), dev_r[(Wm + i) % nsnap].data_ptr(), True)
        b.record(st)
        rr.sync()
        barrier()
        ms = max_over_ranks(a.elapsed_time(b))
        kt = rr.kernel_times()
        rr.set_timing(False)
        return ms, kt, rr.launch_count - l0

    # ---- device-resident leg ("value") --------------------------------------------------------------
    sampler = ClockSampler(local); sampler.start()
    t_sampler = time.perf_counter()
    time.sleep(0.25)
    ms_dev, kt, launches = device_leg(r, K)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r, batch)
    # the raster kernel alone (no spectrum kernel co-running): modified=0 re-rasters the last spectrum
    r.set_timing(True)
    for _ in range(10):
        r.update_device(dev_l[0].data_ptr(), dev_r[0].data_ptr(), False)
    kt_iso = r.kernel_times()
    r.set_timing(False)

    # ---- end-to-end leg: the FIFO backend's data flow (fifo.c:89-110) — per step the new int16 chunk of every stream in,
    #      rings resident in HBM, one stream's frame out to pinned host memory ------------------------------------------
    frame = np.empty((H, W, 4), np.uint8)
    frame_pinned = g.pinned_empty((H, W, 4), np.uint8, local)
    fifo_chunks = [g.pinned_empty((batch, HOP * 2), np.int16, local) for _ in range(nsnap)]
    for i in range(nsnap):
        fifo_chunks[i][:] = pcm[:, N + i * HOP:N + (i + 1) * HOP, :].reshape(batch, HOP * 2)
    for i in range(3):
        r.ingest_fifo(fifo_chunks[i % nsnap]); r.update_rings(True); r.readback_async(i % batch, frame_pinned)
    r.sync()
    barrier()
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e4.record(stream)
    for i in range(K):
        r.ingest_fifo(fifo_chunks[i % nsnap])                     # H2D of batch * 256 frames * 2 ch * int16 + ring slide
        r.update_rings(True)                                      # spectrum + raster
        r.readback_async(i % batch, frame_pinned)                 # D2H of one stream's frame (snapshot + separate copy-out stream)
    r.readback_fence()                                            # e5 is ordered after the last frame's D2H
    e5.record(stream)
    r.sync()
    barrier()
    ms_fifo = max_over_ranks(e4.elapsed_time(e5))
    frame[:] = frame_pinned
    checksum = int(frame.astype(np.uint32).sum())

    # ---- the same with whole float rings through glava_b200_update (what glava.c:528-537 hands rd_update) ---------------
    ms_ring = None
    if not args.no_extras:
        r.set_async_input(True)                                   # double-buffer contract: no host block per update
        for i in range(2):
            r.update(host_l[i % nsnap], host_r[i % nsnap], True); r.readback_async(i % batch, frame_pinned)
        r.sync()
        barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record(stream)
        for i in range(K):
            r.update(host_l[i % nsnap], host_r[i % nsnap], True)  # H2D (copy stream) + kernels
            r.readback_async(i % batch, frame_pinned)
        r.readback_fence()
        e3.record(stream)
        r.sync()
        barrier()
        ms_ring = max_over_ranks(e2.elapsed_time(e3))
        r.set_async_input(False)

    # nvidia-smi samples every 100 ms and short runs (small --steps) end sooner than that: keep the SAME load
    # running, untimed, until the sampler has seen about 2 s of it, so the clocks line describes the load
    soak = 0
    while time.perf_counter() - t_sampler < 2.25:
        for i in range(16):
            r.update_device(dev_l[i % nsnap].data_ptr(), dev_r[i % nsnap].data_ptr(), True)
        r.sync(); soak += 16
    time.sleep(0.1)
    clocks = sampler.stop()
    clocks["untimed_soak_steps"] = soak
    fb_slots = int(p.fb_slots) or batch
    r.close()

    # ---- the API default (lazy_smooth = 0: K5 evaluates every texel, textures() / spectrum() are complete) ----------------
    lazy0 = None
    if not args.no_extras:
        p0 = p.copy(); p0.lazy_smooth = 0
        r0 = g.Renderer(p0, batch=batch, device=local)
        ms0, kt0, _ = device_leg(r0, max(K // 2, 10))
        r0.close()
        k0 = max(K // 2, 10)
        lazy0 = {"value": batch * world * k0 / (ms0 / 1e3), "unit": UNIT, "ms_per_step": ms0 / k0,
                 "note": "same workload with lazy_smooth = 0 (the C ABI's default): full-plane K5 as its own kernel"}

    total_frames = batch * world * K
    value = total_frames / (ms_dev / 1e3)
    peak, peak_src = hbm_peak()
    ras_ms = kt["raster_ms"] / max(kt["raster_launches"], 1)
    spec_ms = kt["spectrum_ms"] / max(kt["spectrum_launches"], 1)
    ras_iso_ms = kt_iso["raster_ms"] / max(kt_iso["raster_launches"], 1)
    alg_bytes = batch * W * H * 4
    achieved = alg_bytes / (ras_ms / 1e3) / 1e9

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle.cpu_baseline import CpuBaseline, describe
        try:                                                     # this process was pinned to the GPU's NUMA node: the reference gets
            os.sched_setaffinity(0, range(os.cpu_count()))       # every host core of the box
        except OSError:
            pass
        fpw = max(1, int(round(2 * (1920 * 1080) / (W * H))))
        base = CpuBaseline(dict(module=MODULE, n=N, w=W, h=H), frames_per_worker=fpw)
        base.step()
        t, f = 0.0, 0
        t_end = time.perf_counter() + 12.0
        steps = 0
        while steps < 3 or (time.perf_counter() < t_end and steps < 60):
            dt, fr = base.step(); t += dt; f += fr; steps += 1
        base.close()
        cpu = {"value": f / t, "unit": UNIT, "cores": base.cores, "kind": base.kind,
               "sample": f"{f} frames ({base.cores * fpw} per step, {steps} steps, {t:.1f} s) of the same workload; " + describe(base.kind)}

    if rank == 0:
        cfg = config_block(wl, batch, world)
        cfg.update({"pipeline": "B (setaccelfft true: R16 gravity/average/smooth passes)", "lazy_smooth": 1, "fb_slots": fb_slots,
                    "numa_node": numa,
                    "l2": f"every step writes {fb_slots if fb_slots < batch else batch} x {frame_bytes / 1e6:.2f} MB of framebuffer (>> 126 MB L2) "
                          "and cycles 4 input snapshots; no flush needed"})
        kern = {"bars": "raster_bars_kernel", "radial": "raster_radial_geo_kernel", "graph": "raster_graph_kernel",
                "wave": "raster_wave_kernel", "circle": "raster_circle_kernel"}.get(MODULE, "raster kernel")
        e2e = {"value": total_frames / (ms_fifo / 1e3), "unit": UNIT, "h2d_bytes_per_step": batch * HOP * 2 * 2,
               "d2h_bytes_per_step": frame_bytes, "ms_per_step": ms_fifo / K, "readback_checksum": checksum,
               "path": "glava_b200_ingest_fifo (int16 FIFO chunks, fifo.c:89-110; rings resident in HBM) + glava_b200_update_rings + "
                       "glava_b200_readback_async of one stream's frame"}
        if ms_ring is not None:
            e2e["full_ring_path"] = {"value": total_frames / (ms_ring / 1e3), "unit": UNIT, "h2d_bytes_per_step": 2 * batch * N * 4,
                                     "d2h_bytes_per_step": frame_bytes, "ms_per_step": ms_ring / K,
                                     "note": "glava_b200_update with whole [batch][n] float rings (glava.c:528-537 semantics), async-input "
                                             "double buffering, NUMA-local pinned rings"}
        line = {
            "metric": wl["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "roofline": {"bound": "hbm", "kernel": kern, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic() if args.config == "headline" else None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": ras_ms,
                         "spectrum_kernel_ms": spec_ms, "raster_share_of_step": ras_ms / (ms_dev / K),
                         "note": "kernel_ms is measured inside the timed steps, where the spectrum kernel of update i+1 "
                                 "co-runs with the raster kernel of update i (two streams); *_isolated = the raster kernel alone",
                         "kernel_ms_isolated": ras_iso_ms, "achieved_isolated": alg_bytes / (ras_iso_ms / 1e3) / 1e9,
                         "frac_isolated": alg_bytes / (ras_iso_ms / 1e3) / 1e9 / peak,
                         "whole_step_frac": alg_bytes / (ms_dev / K / 1e3) / 1e9 / peak},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "lazy_smooth_0": lazy0,
            "gpu_launches": launches,
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
