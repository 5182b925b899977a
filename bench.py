#!/usr/bin/env python
"""Benchmark of the hot path: Mpixels/s of REBLUR_DIFFUSE_SPECULAR at 3840x2160 (BASELINE.json metric), one frame per step.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--width 3840 --height 2160] [--dump-outputs DIR]

Runs on the tree as `python -m raytracingdenoiser_b200.build` left it and writes nothing there.

value     whole chain, inputs already resident in HBM (each frame's inputs are separate 265 MB buffers, i.e. larger than
          the 126 MB L2, so no flush is needed between steps), CUDA events on the launching stream, max over ranks.
          N > 1 (torchrun, one process per GPU): strong scaling of the same frames -- every rank denoises one horizontal strip
          (raytracingdenoiser_b200/strips.py: CUDA-IPC arenas, NVLink ghost rows, device-side barriers; no collective on the
          data path); the device-to-device copy of a rank's input strip into its IPC arena is inside the timed region.
e2e       the same metric through the C-ABI with HOST buffers: pinned host -> H2D -> nrdCudaDenoise -> D2H of both outputs for
          every step, pipelined over three streams with double-buffered staging (what an application would do).
roofline  Blur + PostBlur (the north-star kernels): algorithmic bytes (92 B/px, SURVEY.md 8(d)) / measured CUDA-event time,
          against MEASURED_PEAKS.json hbm_gbs; per_pass_frac gives the same for every pass.  At N > 1 the per-pass times of
          rank 0 include the wait for the slowest peer.
cpu_baseline / --impl reference   the CPU restatement of the reference shaders (oracle/, OpenMP over all host cores) on a
          bounded sample of the same frames.  It is a reported baseline; the oracle is never on the product path.
--dump-outputs DIR   after the timed steps, the outputs of the last timed step (OUT_DIFF_RADIANCE_HITDIST, OUT_SPEC_RADIANCE_HITDIST
          as float32) go to DIR/<name>.npy: whole (height, width, 4) arrays when all of them fit into 64 MB, otherwise the same fixed,
          seeded sample of texels of each, (texels, 4).  The inputs depend only on the arguments, so two builds can be compared
          output for output.  One GPU only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

ALGO_BYTES_PER_PIXEL = {  # SURVEY.md Appendix A, REBLUR_DIFFUSE_SPECULAR defaults
    "Classify tiles": 4, "Pre-pass": 42, "Temporal accumulation": 94, "History fix": 50, "Blur": 46, "Post-blur": 46, "Temporal stabilization": 66,
}
FALLBACK_HBM_GBS = 6650.0


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback"


def measured_traffic(width, height, world):
    """DRAM bytes of the Blur + PostBlur launch pair from the committed ncu capture of this workload (profiles/r2_reblur_traffic.json,
    written from an `ncu --set full` report; ncu cannot run inside a timed bench).  None when no capture matches the workload."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_reblur_traffic.json")))
        if world == 1 and list(t["size"]) == [width, height]:
            return float(t["bytes_per_launch"]["Blur"] + t["bytes_per_launch"]["Post-blur"])
    except Exception:
        pass
    return None


class ClockSampler(object):
    """nvidia-smi SM clock / throttle-reason sampler running beside the timed region."""

    def __init__(self, index=0):
        self.index, self.samples, self.reasons, self.max_mhz, self.proc = index, [], set(), None, None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            try:
                self.samples.append(float(parts[0]))
                self.max_mhz = float(parts[1])
                for n, v in zip(names, parts[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        s = sorted(self.samples)
        # median of the upper half: samples taken while the GPU was busy
        busy = s[len(s) // 2:] if s else []
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def host_threads():
    """Threads the CPU legs may really use: the affinity mask capped by the cgroup CPU quota (a container that sees 128 cores
    through sched_getaffinity may be throttled to a fraction of them; oversubscribing the quota makes the OpenMP team thrash).
    Returns (threads, affinity cores, quota in cores or None)."""
    import math
    affinity = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        parts = open("/sys/fs/cgroup/cpu.max").read().split()  # cgroup v2: "<quota|max> <period>"
        if parts and parts[0] != "max":
            quota = float(parts[0]) / float(parts[1])
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    threads = affinity if quota is None else max(1, min(affinity, int(math.ceil(quota))))
    return threads, affinity, quota


def generate_frames(width, height, count, device):
    from raytracingdenoiser_b200 import scene
    sc = scene.Scene(width, height, device=device)
    return [sc.frame(f) for f in range(count)]


def run_cpu_reference(width, height, frames, steps, warmup):
    """Times the oracle chain (all host threads) on `frames`; returns (Mpx/s, ms per step, threads)."""
    import oracle_runner as orr
    from raytracingdenoiser_b200 import harness, nrd
    # every host core the cgroup grants, also under torchrun (which exports OMP_NUM_THREADS=1 to every rank)
    orr.oracle_lib().oracle_set_num_threads(host_threads()[0])
    cpu = orr.CpuDenoiser(nrd.Denoiser.REBLUR_DIFFUSE_SPECULAR, width, height)
    host = [{k: (v.cpu() if hasattr(v, "cpu") else v) for k, v in fr.items()} for fr in frames]
    times = []
    for i in range(warmup + steps):
        fr = host[i % len(host)]
        cs = harness.make_common_settings(fr, width, height, i)
        cpu.set_inputs(fr)
        t0 = time.perf_counter()
        cpu.denoise(cs)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    threads, affinity, quota = host_threads()
    info = {"cores": orr.oracle_lib().oracle_num_threads(), "affinity_cores": affinity, "cgroup_quota_cores": quota,
            "frame_ms": [round(1e3 * t, 1) for t in times]}
    return width * height * len(times) / total / 1e6, 1e3 * total / len(times), info


DUMP_BYTES = 64 * 1000 * 1000  # all files together, .npy headers included


def dump_outputs(directory, outputs):
    """Writes {name: (H, W, C) tensor} as float32 DIR/<name>.npy: whole when everything fits into DUMP_BYTES, otherwise the texels
    of one fixed, seeded sample (the same texels for every output, in raster order)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    arrays = {n: t.float().cpu().numpy() for n, t in outputs.items()}
    data_bytes = DUMP_BYTES - 1024 * len(arrays)
    sample = None
    if sum(a.size * 4 for a in arrays.values()) > data_bytes:
        h, w = next(iter(arrays.values())).shape[:2]
        texels = data_bytes // sum(a[0, 0].size * 4 for a in arrays.values())
        sample = np.sort(np.random.default_rng(20240917).choice(h * w, size=texels, replace=False))
    for n, a in arrays.items():
        if sample is not None:
            a = a.reshape((a.shape[0] * a.shape[1],) + a.shape[2:])[sample]
        np.save(os.path.join(directory, n + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.gpus != 1:
        ap.error("--dump-outputs needs --gpus 1")

    import torch
    from raytracingdenoiser_b200 import harness, nrd  # nrd raises if the library is not built

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    W, H, K, Wm = args.width, args.height, args.steps, max(args.warmup, 3)
    workload = "REBLUR_DIFFUSE_SPECULAR %dx%d, %d-frame synthetic sequence with motion vectors, default settings" % (W, H, K + Wm)
    base = {"metric": "Mpixels/s REBLUR_DIFFUSE_SPECULAR @4K", "unit": "Mpixels/s", "n_gpus": args.gpus, "steps": K, "warmup": Wm, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "l2": "per-frame inputs are distinct 265 MB buffers (> 126 MB L2), no flush needed"}}

    # ------------------------------------------------------------------ reference arm: CPU restatement on host cores
    if args.impl == "reference":
        if rank != 0:
            return
        gen_dev = "cuda" if torch.cuda.is_available() else "cpu"
        nframes = min(K + Wm, 6)
        frames = generate_frames(W, H, nframes, gen_dev)
        mpx, ms, info = run_cpu_reference(W, H, frames, K, Wm)
        out = dict(base)
        cb = {"value": mpx, "unit": "Mpixels/s", "kind": "port",
              "sample": "%d timed frames of the %dx%d sequence (inputs cycle over %d generated frames)" % (K, W, H, nframes)}
        cb.update(info)
        out.update({"impl": "reference", "value": mpx, "ms_per_step": ms, "gpu_launches": 0,
                    "cpu_baseline": cb,
                    "e2e": {"value": mpx, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(out))
        return

    # ------------------------------------------------------------------ B200 arm
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback for the product path)"
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    frames = generate_frames(W, H, K + Wm, dev)
    stream = torch.cuda.current_stream(dev)
    den = nrd.Denoiser.REBLUR_DIFFUSE_SPECULAR
    in_names = [n for n in harness.DENOISER_RESOURCES[den] if n.startswith("IN_")]
    out_names = [n for n in harness.DENOISER_RESOURCES[den] if n.startswith("OUT_")]
    if world == 1:
        gpu = harness.GpuDenoiser(den, W, H, device=local_rank)
        y0, y1 = 0, H

        def bind(fr):
            # inputs are device resident: bind this frame's own buffers (what an application's ring of G-buffers looks like)
            for n in in_names:
                t = fr[n]
                gpu.ctx.set_user_texture(getattr(nrd.ResourceType, n), t.data_ptr(), t.stride(0) * t.element_size(), harness.USER_FORMATS[n][0])
    else:
        # strong scaling: one strip of whole 16-row tiles per rank, foreign rows are NVLink peer loads (strips.py).  The strip
        # textures live in the context's IPC arena, so "binding" a frame is a device-to-device copy of this rank's rows --
        # it is inside the timed region.
        from raytracingdenoiser_b200 import strips
        # cost-balanced partition from the sky mask of the first frame (every rank computes the same one): tiles beyond the
        # denoising range are skipped by every pass, so uniform strips would leave the rank that owns the sky idle
        cost = strips.tile_row_cost_from_viewz(frames[0]["IN_VIEWZ"])
        partition = strips.partition_rows_weighted(H, world, cost, min_rows=strips.DEFAULT_HALO_ROWS)
        # measured re-balancing (set-up, untimed): the first frames are denoised on the trial partition with per-dispatch timing on
        # (nrdCudaSetTiming: kernel time without barrier waits), the per-strip kernel times correct the cost of the tile rows and the
        # strips are cut again; the contexts are then rebuilt, so the benchmark itself starts from an empty history on the final strips
        balance = []
        for trial in range(int(os.environ.get("NRD_B200_BALANCE_TRIALS", "2"))):
            gpu = strips.StripDenoiser(den, W, H, rank, world, device=local_rank, partition=partition)
            gpu.connect()
            gpu.ctx.set_timing(True)
            mine = 0.0
            ncal = min(6, len(frames))
            for i in range(ncal):
                gpu.set_input_strips({n: frames[i][n][gpu.y0:gpu.y1].contiguous() for n in in_names}, stream)
                gpu.denoise(harness.make_common_settings(frames[i], W, H, i))
                gpu.synchronize()
                kernel_ms, _ = gpu.ctx.get_timing()
                if i >= ncal - 3:
                    mine += sum(kernel_ms)
            t = torch.tensor([mine], device=dev)
            every = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(every, t)
            ms = [float(e.item()) for e in every]
            balance.append({"strips": [list(p) for p in partition[1]], "kernel_ms_per_rank": [round(m / 3.0, 4) for m in ms]})
            gpu.destroy()
            del gpu
            torch.cuda.empty_cache()
            dist.barrier()
            if max(ms) <= 1.03 * min(ms):
                break
            cost = strips.rebalance_tile_row_cost(cost, partition[1], ms)
            partition = strips.partition_rows_weighted(H, world, cost, min_rows=strips.DEFAULT_HALO_ROWS)
        gpu = strips.StripDenoiser(den, W, H, rank, world, device=local_rank, partition=partition)
        base["config"]["strips"] = [list(p) for p in partition[1]]
        base["config"]["strip_balance"] = {"method": "sky-tile cost model, then strips re-cut from measured per-rank kernel time (set-up, untimed)", "trials": balance}
        gpu.connect()
        y0, y1 = gpu.y0, gpu.y1
        full_frames = frames if rank == 0 else None   # rank 0 re-denoises the sequence on one GPU afterwards: the N-GPU output is checked, not assumed
        frames = [{k: (v[y0:y1].contiguous() if k in in_names else v) for k, v in fr.items() if k in in_names or not k.startswith("IN_")} for fr in frames]
        torch.cuda.empty_cache()

        def bind(fr):
            gpu.set_input_strips({n: fr[n] for n in in_names}, stream)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    # IN_MV is bound as a storage texture by the chain (frame 0 clears it): keep pristine copies out of the way
    mv0 = frames[0]["IN_MV"].clone()
    # ONE clock sampler per job, on rank 0, started before the warm-up: its fork/exec + NVML initialisation must be nowhere near
    # a timed region (eight of them started between the barrier and the first event cost round 1 its N=8 number)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    for i in range(Wm):
        bind(frames[i])
        gpu.denoise(harness.make_common_settings(frames[i], W, H, i))
        if i == 0 and world == 1:
            frames[0]["IN_MV"].copy_(mv0)
    barrier()
    l0 = nrd.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(Wm, Wm + K):
        bind(frames[i])
        gpu.denoise(harness.make_common_settings(frames[i], W, H, i))
    e1.record(stream)
    barrier()
    if args.dump_outputs:  # before the per-pass and end-to-end runs below denoise further frames into the same textures
        dump_outputs(args.dump_outputs, gpu.outputs())
    launches = nrd.launch_count() - l0
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    if world > 1:
        gpu.synchronize()  # raises if an inter-GPU barrier timed out
    value = W * H * K / (ms_total * 1e-3) / 1e6

    # ---- N > 1: the strips of the last timed frame against the one-GPU result of the same sequence.  Rank 0 runs the whole
    # sequence through a one-GPU context on the strip build of the kernels (the build the strips run), so the comparison is bitwise.
    check = None
    if world > 1:
        def digest(t):
            v = t.contiguous().view(torch.int16).to(torch.int64).reshape(-1)
            w = (torch.arange(v.numel(), device=v.device, dtype=torch.int64) % 8191) + 1
            return torch.stack([v.sum(), (v * w).sum()])
        mine = torch.stack([digest(t) for _, t in sorted(gpu.read_outputs(stream=stream).items())])
        torch.cuda.synchronize(dev)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        if rank == 0:
            os.environ["NRD_B200_FORCE_STRIP_KERNELS"] = "1"
            try:
                ref = harness.GpuDenoiser(den, W, H, device=local_rank)
                for i in range(Wm + K):
                    ref.set_inputs(full_frames[i])
                    ref.denoise(harness.make_common_settings(full_frames[i], W, H, i))
                torch.cuda.synchronize(dev)
                outs = sorted(ref.outputs().items())
                rows = base["config"]["strips"]
                same = [bool(torch.equal(torch.stack([digest(t[a:b]) for _, t in outs]), every[r].to(dev))) for r, (a, b) in enumerate(rows)]
                check = {"against": "one-GPU run of the same %d frames (strip build of the kernels), position-weighted checksums per strip and output" % (Wm + K),
                         "strips_bit_identical": same, "ok": all(same)}
                ref.destroy()
                del ref, full_frames
                torch.cuda.empty_cache()
            finally:
                del os.environ["NRD_B200_FORCE_STRIP_KERNELS"]
        dist.barrier()

    # ---- per-pass breakdown with CUDA events around every dispatch (separate run, not part of `value`)
    per_pass = {}
    pipelines = gpu.instance.get_instance_desc()["pipelines"]
    import ctypes as C
    reps = min(K, 8)
    for i in range(Wm + K - reps, Wm + K):
        bind(frames[i])
        gpu.instance.set_common_settings(harness.make_common_settings(frames[i], W, H, i + K))
        r, raw, n = gpu.instance.get_compute_dispatches_raw([gpu.identifier])
        gpu.ctx.barrier(stream.cuda_stream)
        evs = []
        for j in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            gpu.ctx.execute_raw(C.byref(raw[j]), stream.cuda_stream)  # N > 1: includes the wait for the slowest peer
            b.record(stream)
            evs.append((raw[j].name.decode().split(" - ")[-1], a, b))
        torch.cuda.synchronize(dev)
        for name, a, b in evs:
            per_pass.setdefault(name, []).append(a.elapsed_time(b))
    pass_ms = {k: sum(v) / len(v) for k, v in per_pass.items()}
    peak, peak_kind = measured_peaks()
    blur_ms = pass_ms.get("Blur", 0.0) + pass_ms.get("Post-blur", 0.0)
    algo_bytes = (ALGO_BYTES_PER_PIXEL["Blur"] + ALGO_BYTES_PER_PIXEL["Post-blur"]) * W * H
    achieved = algo_bytes / (blur_ms * 1e-3) / 1e9 if blur_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": "REBLUR Blur + PostBlur (2 launches)", "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                # dram__bytes_read.sum + dram__bytes_write.sum of one Blur + one PostBlur launch at 3840x2160, from the ncu --set full
                # capture summarised in profiles/r1_reblur_ncu_summary.txt (304.9 MB + 305.6 MB); below the algorithmic bytes
                # because sky tiles are skipped
                "frac": achieved / peak, "traffic": measured_traffic(W, H, world), "algorithmic_bytes_per_launch_pair": algo_bytes,
                "per_pass_ms": pass_ms,
                "per_pass_frac": {k: (ALGO_BYTES_PER_PIXEL[k] * W * H / (v * 1e-3) / 1e9 / peak) for k, v in pass_ms.items() if k in ALGO_BYTES_PER_PIXEL and v > 0}}

    # ---- end to end with host buffers: pinned host -> H2D -> denoise -> D2H of both outputs, every step (per rank: its strip)
    nhost = min(K + Wm, 8)
    host_frames = [{n: frames[i][n].cpu().pin_memory() for n in in_names} for i in range(nhost)]
    rows = y1 - y0
    host_out = {}
    for n in out_names:
        fmt, dtype, ch = harness.USER_FORMATS[n]
        host_out[n] = torch.empty((rows, W, ch) if ch > 1 else (rows, W), dtype=dtype).pin_memory()
    if world == 1:
        for n in in_names:  # back to the context's own input textures
            t = gpu.tex[n]
            gpu.ctx.set_user_texture(getattr(nrd.ResourceType, n), t.data_ptr(), t.stride(0) * t.element_size(), harness.USER_FORMATS[n][0])
    h2d = sum(t.numel() * t.element_size() for t in host_frames[0].values())
    d2h = sum(t.numel() * t.element_size() for t in host_out.values())
    if world > 1:
        t = torch.tensor([float(h2d), float(d2h)], device=dev)
        dist.all_reduce(t)
        h2d, d2h = int(t[0].item()), int(t[1].item())

    # Pipelined like an application would: three streams, double-buffered staging.  Step i: H2D of its inputs (copy-in stream)
    # -> denoise + device copy of the outputs to a staging buffer (compute stream) -> D2H (copy-out stream); the H2D of step
    # i+1 and the D2H of step i-1 overlap the denoising of step i.  Every step still moves its own inputs and results.
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    rows_shape = lambda n: ((rows, W, harness.USER_FORMATS[n][2]) if harness.USER_FORMATS[n][2] > 1 else (rows, W))
    dev_in = [{n: torch.empty(rows_shape(n), dtype=harness.USER_FORMATS[n][1], device=dev) for n in in_names} for _ in range(2)]
    dev_out = [{n: torch.empty(rows_shape(n), dtype=harness.USER_FORMATS[n][1], device=dev) for n in out_names} for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_comp = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]

    def e2e_step(i):
        b = i & 1
        hf = host_frames[i % nhost]
        cs = harness.make_common_settings(frames[i % len(frames)], W, H, i + 2 * K)
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_comp[b])  # the denoise of step i-2 no longer reads this staging set
            for n in in_names:
                dev_in[b][n].copy_(hf[n], non_blocking=True)
            ev_in[b].record(s_in)
        stream.wait_event(ev_in[b])
        stream.wait_event(ev_out[b])      # the D2H of step i-2 has drained this output staging set
        if world == 1:
            bind(dev_in[b])
            gpu.denoise(cs)
            for n, t in gpu.outputs().items():
                dev_out[b][n].copy_(t, non_blocking=True)
        else:
            gpu.set_input_strips(dev_in[b], stream)
            gpu.denoise(cs)
            gpu.read_outputs(out=dev_out[b], stream=stream)
        ev_comp[b].record(stream)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_comp[b])
            for n in out_names:
                host_out[n].copy_(dev_out[b][n], non_blocking=True)
            ev_out[b].record(s_out)

    def e2e_join():
        stream.wait_event(ev_out[0])
        stream.wait_event(ev_out[1])

    for i in range(4):
        e2e_step(i)
    e2e_join()
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for i in range(K):
        e2e_step(4 + i)
    e2e_join()
    e1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    ms_e2e = max(e0.elapsed_time(e1), wall * 1e3)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    clocks = sampler.stop() if sampler else None  # sampled over both timed regions (device-resident and end-to-end)
    e2e = {"value": W * H * K / (ms_e2e * 1e-3) / 1e6, "unit": "Mpixels/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}

    out = dict(base)
    out.update({"value": value, "ms_per_step": ms_total / K, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "e2e": e2e})
    if check is not None:
        out["output_check"] = check

    if rank == 0 and args.gpus == 1 and not args.no_cpu_baseline:
        sample_frames = 3
        mpx, ms, info = run_cpu_reference(W, H, frames[Wm:Wm + 4], sample_frames, 1)
        out["cpu_baseline"] = {"value": mpx, "unit": "Mpixels/s", "kind": "port",
                               "sample": "%d timed frames (+1 warm-up) of the same %dx%d sequence on the host cores" % (sample_frames, W, H)}
        out["cpu_baseline"].update(info)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
