#!/usr/bin/env python
"""bench.py — the headline benchmark of functracer_b200.

Metric (BASELINE.json): Mrays/s, primary + secondary (shadow + unique reflection rays), for one
frame of a bundled scene.  A "step" is one frame: generateRays -> shade -> blendPixels
(Program.fs:54-64).  Default workload = the config BASELINE.json names for the 1/2/4/8-GPU sweep:
repeat.scene at 7680x4320, 64 jittered spp (configs[4]; it fits one GPU).  The other eight
configs ride in the same JSON line under `per_config` (N = 1).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes, after the timed steps, the frames the last timed step of each timed path returned, as float32
DIR/<name>.npy: `frame` (the device-resident step's RGB frame), `frame_rgba8` (the RGBA8 frame the e2e step downloaded)
and `per_config_<workload>` (each per-config frame).  A frame of more than DUMP_PIXELS pixels is cut to a fixed, seeded
sample of DUMP_PIXELS pixels (rows of the [H*W, C] view, ascending), so that two builds run with the same arguments can
be compared output for output: every input (scene, assets, jitter pattern, RNG seed) is fixed by the arguments.

N > 1 is launched by torchrun (one rank per GPU, NCCL): the frame's 16x16 tiles are dealt
round-robin to the ranks, each rank renders its tiles from its own atomic tile queue and its kernel
stores the finished pixels straight into rank 0's memory over NVLink (CUDA IPC peer arena; NCCL
gather as the fallback), where the frame is assembled.  Total work is fixed as N grows =>
"scaling": "strong".

`value`  : inputs resident (scene on the GPU), device-to-device: tiles -> assembled frame on rank 0.
`e2e`    : the same frame through the host-buffer C-ABI path the reference-side caller uses, into an
           ordinary PAGEABLE host buffer (np.empty; what a P/Invoke caller passes), as RGBA8 = what
           Image.write keeps of a frame (Image.fs:35-44); H2D of the step's inputs (jitter table, frame
           constants) and D2H of the frame inside the timed region.  N = 1: ftb_render.  N > 1: every
           rank renders band after band (ftb_render_tiles_device with band_count), rank 0 assembles
           each finished band (ftb_assemble_rows_device) and downloads it behind the rendering of the
           next (ftb_host_copy_begin / _finish).  `e2e.f64` = the same with the 24 B/pixel f64 frame;
           `e2e_inprocess` (N > 1) = rank 0 alone calling ftb_render(n_gpus = N), the call the CLI makes.
`roofline`: the render kernel against the FP32 pipe (this path is not HBM- or tensor-bound:
           the scene is KBs and rays live in registers; see DESIGN.md).
`cpu_baseline`: the CPU oracle (a C++ port of the reference's algorithm; the F# original cannot
           run in this image) on all host cores, on a bounded sample of the same frame, made in ONE
           call (one thread pool, >= 64 chunks of 1000 rays per thread); the same sample gives `parity`.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DEFAULT_WORKLOAD = "cfg5-repeat"
ALL_WORKLOADS = ["cfg1-sample", "cfg2-hollow-sphere", "cfg3-house", "cfg3-night-house", "cfg4-bunny", "cfg4-bunny-d12", "cfg4-bunny-full-d14",
                 "cfg5-moon", "cfg5-repeat"]
METRIC = "Mrays/sec (primary+secondary)"
UNIT = "Mrays/s"
RNG_SEED = 1234
E2E_BANDS = 4
CPU_SAMPLE_PRIMARY = 40e6   # primary samples of the headline's CPU sample (~10-20 s on 16-32 cores)
REF_STEP_PRIMARY = 9e6      # primary samples per step of the reference arm (cfg1 / cfg2: the whole frame)
MINI_SAMPLE_PRIMARY = 2.5e6  # per_config parity samples
DUMP_PIXELS = 1 << 18       # --dump-outputs: pixels kept per frame (10 frames of <= 16 B / pixel: at most 31 MB in all)
DUMP_SEED = 2024
DUMP_MAX_BYTES = 64 << 20


def dump_rows(W, H):
    """The pixels --dump-outputs keeps of a W x H frame, as ascending row indices of its [H*W, C] view: None (all of them)
    up to DUMP_PIXELS pixels, else the same seeded sample of DUMP_PIXELS for every run at this size."""
    import numpy as np
    if W * H <= DUMP_PIXELS:
        return None
    return np.sort(np.random.default_rng(DUMP_SEED).choice(W * H, DUMP_PIXELS, replace=False))


def dump_frame(frame, rows):
    """float32 host copy of `frame` ([H, W, C], a torch tensor on the device or a numpy array), cut to `rows` (dump_rows)."""
    import numpy as np
    import torch
    if torch.is_tensor(frame):
        if rows is not None:
            frame = frame.reshape(-1, frame.shape[-1])[torch.from_numpy(rows).to(frame.device)]
        return frame.float().cpu().numpy()
    if rows is not None:
        frame = frame.reshape(-1, frame.shape[-1])[rows]
    return frame.astype(np.float32)


def write_dumps(directory, arrays):
    """--dump-outputs: every array as <directory>/<name>.npy."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, "dumped outputs would take %d bytes" % total
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


# per-ray intersection cost of the reference's brute-force algorithm on the bundled scenes (SURVEY.md 8(d), flop table)
_BRUTE_FORCE_FLOPS_PER_RAY = {"sample": 366, "hollow_sphere": 2972, "house": 610, "night_house": 1285, "repeat": 1214, "moon": 244,
                              "bunny": 960 * 45 + 33}


def _fp32_peak_tflops():
    """FP32 pipe peak.  Prefers the on-box FMA-saturation measurement committed under profiles/
    (tools/fp32_peak.cu); else 148 SM x 128 lanes x 2 x clocks.max.sm from MEASURED_PEAKS.json."""
    p = os.path.join(ROOT, "profiles", "fp32_peak.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["fp32_tflops"]), "measured FMA-saturation microbenchmark (profiles/fp32_peak.json)"
        except Exception:
            pass
    pk, how = _peaks()
    mhz = float(pk.get("sm_max_mhz", 1965.0))
    return 148 * 128 * 2 * mhz * 1e6 / 1e12, "derived 148 SM x 128 lanes x 2 x %g MHz (%s MEASURED_PEAKS.json sm_max_mhz)" % (mhz, how)


def _traffic_per_launch(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of the render kernel from the committed `ncu --set full` capture."""
    p = os.path.join(ROOT, "profiles", "render_kernel_dram.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            if workload in d.get("per_workload", {}):
                return float(d["per_workload"][workload]["dram_bytes_per_launch"])
            if d.get("workload", "cfg2-hollow-sphere") == workload:
                return float(d["dram_bytes_per_launch"])
        except Exception:
            pass
    return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _workload(name):
    from functracer_b200 import frontend, scenes
    cfg = scenes.CONFIGS[name]
    text = scenes.config_text(name)
    parsed = frontend.ParsedScene(text, scenes.asset_dir())
    jit = frontend.jitter_pattern(cfg["seed"], parsed.spp)
    return cfg, parsed, jit


def cpu_sample(parsed, jit, target_primary, debug=False, threads=0, margin=1):
    """The CPU oracle on a bounded sample of the frame: the whole frame when it is small enough, else evenly spaced
    full-height stripes - in ONE call (one thread pool over all the sample's 1000-ray chunks).
    Returns (result of oracle.render_windows, windows, margin, rays, cores, description)."""
    from oracle import ftb_oracle as orc
    from oracle import parity
    W, H, spp = parsed.width, parsed.height, parsed.spp
    windows, margin = parity.sample_windows(W, H, spp, target_primary, margin=margin)
    p = orc.make_params(W, H, spp, jit, seed=RNG_SEED)
    res = orc.render_windows(parsed, p, windows, threads=threads, debug=debug)
    st = res["stats"]
    rays = st.primary_rays + st.shadow_rays + st.reflection_rays
    cores = threads if threads > 0 else (os.cpu_count() or 1)
    npix = sum((x1 - x0) * (y1 - y0) for x0, y0, x1, y1 in windows)
    what = ("the whole %dx%d x %d spp frame" % (W, H, spp)) if len(windows) == 1 and npix == W * H else \
        "%d full-height stripes of %d px = %.2f%% of the %dx%d x %d spp frame" % (len(windows), windows[0][2] - windows[0][0], 100.0 * npix / (W * H), W, H, spp)
    what += ", one call, %d chunks of 1000 rays per thread" % (st.primary_rays // 1000 // max(1, cores))
    return res, windows, margin, rays, cores, what


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the F# binary cannot run in this image: no dotnet)
    on all host cores; each step = one call on a bounded sample of the same frame (the whole frame for cfg1 / cfg2)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, parsed, jit = _workload(args.workload)
    W, H = parsed.width, parsed.height
    for _ in range(args.warmup):
        cpu_sample(parsed, jit, REF_STEP_PRIMARY / 8, margin=0)
    rays = secs = 0
    for _ in range(args.steps):
        res, windows, margin, r, cores, what = cpu_sample(parsed, jit, REF_STEP_PRIMARY, margin=0)
        rays += r; secs += res["seconds"]
    v = rays / secs / 1e6
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": args.workload, "scene": cfg["build"].__name__, "width": W, "height": H, "spp": parsed.spp,
                                         "note": "CPU oracle (C++ port of the F# algorithm, -O2, all host threads); F# reference not runnable here (no dotnet)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": what + " per step"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


class Runner:
    """One workload on this rank's GPU: scene, ray accounting, buffers, the device-resident step."""

    def __init__(self, name, rank, world, dev, stream):
        import torch
        from functracer_b200 import abi, api
        self.torch, self.abi, self.api = torch, abi, api
        self.name, self.rank, self.world, self.dev, self.stream = name, rank, world, dev, stream
        self.cfg, self.parsed, self.jit = _workload(name)
        self.W, self.H, self.spp = self.parsed.width, self.parsed.height, self.parsed.spp
        t0 = time.perf_counter()
        self.scene = api.Scene(self.parsed)
        self.create_ms = 1e3 * (time.perf_counter() - t0)
        self.build = self.scene.build_info()  # mesh index: built on the device (PLOC) or on the host, and how long it took
        self.p_f32 = self.params(out_format=abi.OUT_RGB_F32)
        self.tiles = torch.empty(api.tile_buffer_bytes(self.p_f32), dtype=torch.uint8, device=dev)
        st = self.scene.render_tiles_device(self.params(out_format=abi.OUT_RGB_F32, collect_stats=1), self.tiles.data_ptr(), stream=stream, stats=True)
        self.local_flops = float(st.flops)
        self.counts = [float(st.primary_rays), float(st.shadow_rays), float(st.reflection_rays), float(st.flops)]
        self.frame = torch.empty((self.H, self.W, 3), dtype=torch.float32, device=dev) if rank == 0 else None

    def params(self, **kw):
        kw.setdefault("shard_index", self.rank if self.world > 1 else 0)
        kw.setdefault("shard_count", self.world)
        return self.api.make_params(self.W, self.H, self.spp, self.jit, seed=RNG_SEED, **kw)

    def close(self):
        self.scene.close()
        self.tiles = self.frame = None
        self.torch.cuda.empty_cache()


def time_device(run, step, barrier, steps, warmup, flush):
    """W warm-up steps, then K timed ones with the L2 flushed in between; returns (sum of step ms, sum of kernel ms)."""
    torch = run.torch
    for _ in range(warmup):
        step()
    barrier()
    step_ms, kern_ms = [], []
    for _ in range(steps):
        flush.zero_()  # evicts L2 (not timed)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        e0.record()
        step(kev)
        e1.record()
        barrier()
        step_ms.append(e0.elapsed_time(e1))
        kern_ms.append(kev[0].elapsed_time(kev[1]))
    return sum(step_ms), sum(kern_ms)


def gpu_parity(run, res, windows, margin):
    """The kernel's frame and primary primitive-id plane against the CPU sample `res` (oracle.render_windows)."""
    from oracle import parity
    torch = run.torch
    W, H, spp = run.W, run.H, run.spp
    p_one = run.api.make_params(W, H, spp, run.jit, seed=RNG_SEED, out_format=run.abi.OUT_RGB_F32)
    tiles = torch.empty(run.api.tile_buffer_bytes(p_one), dtype=torch.uint8, device=run.dev)
    prim = torch.full((H, W, spp), -2, dtype=torch.int32, device=run.dev)
    frame = torch.empty((H, W, 3), dtype=torch.float32, device=run.dev)
    run.scene.render_tiles_device(p_one, tiles.data_ptr(), stream=run.stream, d_dbg=(prim.data_ptr(), 0, 0))
    run.api.assemble_device(p_one, [tiles.data_ptr()], frame.data_ptr(), stream=run.stream)
    torch.cuda.synchronize()
    parts = []
    for w in res["windows"]:
        x0, y0, x1, y1 = w["rect"]
        parts.append(parity.compare_window(w["rgb"], w["prim"], frame[y0:y1, x0:x1].cpu().numpy(), prim[y0:y1, x0:x1].cpu().numpy(), margin))
    m = parity.merge(parts)
    del prim, frame, tiles
    return {"frac_within_1_255": m["frac_within_1_255"], "max_err": m["max_err"], "pixels": m["pixels"], "primary_samples": m["samples"],
            "prim_id_mismatches": m["prim_mismatch"], "prim_id_unexplained": m["prim_unexplained"], "prim_id_edge_leaks": m.get("prim_edge_leak", 0), "nonfinite_pixels": m["nonfinite"],
            "note": "FP32 kernel vs the f64 CPU oracle on the cpu_baseline sample; a prim-id mismatch is explained when the oracle's own id map shows the "
                    "kernel's answer within one pixel of the sample (silhouette / tie)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline and e2e arms (the f64, in-process and per-config arms time min(K, 5))")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-config", action="store_true")
    ap.add_argument("--no-inprocess", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frames of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU path's frames; --impl reference has none")
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from functracer_b200 import abi, api
    from functracer_b200 import dist as fdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: functracer_b200 has no CPU path")
    torch.cuda.set_device(local)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cpu_group = dist.new_group(backend="gloo")  # host-side barrier while rank 0 drives every GPU by itself (e2e_inprocess)
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream().cuda_stream

    run = Runner(args.workload, rank, world, dev, stream)
    W, H, spp, scene, jit = run.W, run.H, run.spp, run.scene, run.jit
    counts = torch.tensor(run.counts, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(counts)
    n_primary, n_shadow, n_refl, flops_total = [float(x) for x in counts.tolist()]
    rays_per_frame = n_primary + n_shadow + n_refl

    # gather buffers (rank 0) + assembled frame
    p_f32 = run.p_f32
    sizes = [api.tile_buffer_bytes(api.make_params(W, H, spp, jit, shard_index=k, shard_count=world, out_format=abi.OUT_RGB_F32)) for k in range(world)]
    max_bytes = max(sizes)
    arena = None
    tiles = run.tiles
    gather_list = None
    if world > 1:
        tiles = torch.empty(max_bytes, dtype=torch.uint8, device=dev)  # equal-sized for gather
        gather_list = [torch.empty(max_bytes, dtype=torch.uint8, device=dev) for _ in range(world)] if rank == 0 else None
        if not os.environ.get("FTB_NO_P2P"):
            try:  # the render kernel writes its tiles straight into rank 0's memory over NVLink (functracer_b200/dist.py)
                arena = fdist.PeerArena(max_bytes)
            except Exception as e:  # no IPC / peer access: NCCL gather
                arena = None
                if rank == 0:
                    print("peer arena unavailable (%s): falling back to the NCCL gather" % e, file=sys.stderr)
    sync_flag = torch.zeros(1, dtype=torch.int32, device=dev)
    frame = run.frame
    # L2 flush between timed iterations: 256 MB > the 126 MB L2
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    my_tiles = arena.ptr(rank) if arena else tiles.data_ptr()

    def sources():
        return [arena.ptr(k) for k in range(world)] if arena else ([g.data_ptr() for g in gather_list] if world > 1 else [tiles.data_ptr()])

    def device_step(ev=None):
        if ev:
            ev[0].record()
        scene.render_tiles_device(p_f32, my_tiles, stream=stream)
        if ev:
            ev[1].record()
        if world > 1 and arena:
            dist.all_reduce(sync_flag)  # the only collective: every rank's stores have landed before rank 0 assembles
        elif world > 1:
            fdist.gather_tiles(tiles, max_bytes, gather_list)
        if rank == 0:
            api.assemble_device(p_f32, sources(), frame.data_ptr(), stream=stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident ------------------------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        device_step()
    barrier()
    if sampler:
        sampler.start()
    total_ms, kern_total_ms = time_device(run, device_step, barrier, args.steps, 0, flush)
    dumps = {}
    if args.dump_outputs and rank == 0:
        dump_sel = dump_rows(W, H)
        dumps["frame"] = dump_frame(frame, dump_sel)
    t = torch.tensor([total_ms, kern_total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kern_total_ms = [float(x) for x in t.tolist()]
    ms_per_step = total_ms / args.steps
    value = rays_per_frame / (ms_per_step * 1e-3) / 1e6

    # ---- e2e: pageable host buffer through the C ABI, RGBA8 (what Image.write keeps) ------------------------------------
    out_u8 = np.empty((H, W, 4), dtype=np.uint8) if rank == 0 else None  # ordinary pageable memory, as a P/Invoke caller passes
    p_host_u8 = api.make_params(W, H, spp, jit, seed=RNG_SEED, out_format=abi.OUT_RGBA8)
    p_host_f64 = api.make_params(W, H, spp, jit, seed=RNG_SEED, out_format=abi.OUT_RGB_F64)
    frame_u8 = torch.empty((H, W, 4), dtype=torch.uint8, device=dev) if (rank == 0 and world > 1) else None
    frame_f64 = None
    copy_stream = torch.cuda.Stream(device=dev, priority=-1) if (rank == 0 and world > 1) else None
    bands = E2E_BANDS if (world > 1 and arena and H >= 128) else 1
    p_band = [run.params(out_format=abi.OUT_RGB_F32, band_index=c, band_count=bands) for c in range(bands)]
    p_all_u8 = run.params(out_format=abi.OUT_RGBA8)
    p_all_f64 = run.params(out_format=abi.OUT_RGB_F64)
    rows = [api.band_rows(p_all_u8, c, bands) for c in range(bands)]

    def e2e_step(fmt="u8", host=None):
        if world == 1:
            scene.render_params(p_host_u8 if fmt == "u8" else p_host_f64, out=host)  # H2D (jitter, frame constants) + kernels + banded D2H, synchronous
            return
        bpp = 4 if fmt == "u8" else 24
        dst = frame_u8 if fmt == "u8" else frame_f64
        evs = []
        for c in range(bands):  # all rendering / assembly is queued first, the downloads follow in band order
            scene.render_tiles_device(p_band[c], my_tiles, stream=stream)
            if arena:
                dist.all_reduce(sync_flag)
            else:
                fdist.gather_tiles(tiles, max_bytes, gather_list)
            if rank == 0:
                y0, y1 = rows[c]
                api.assemble_rows_device(p_all_u8 if fmt == "u8" else p_all_f64, sources(), dst.data_ptr(), y0, y1, stream=stream)
                e = torch.cuda.Event()
                e.record()
                evs.append(e)
        if rank == 0:
            for c in range(bands):
                y0, y1 = rows[c]
                copy_stream.wait_event(evs[c])
                scene.host_copy_begin(dst.data_ptr() + y0 * W * bpp, host, stream=copy_stream.cuda_stream, offset=y0 * W * bpp, nbytes=(y1 - y0) * W * bpp)
            scene.host_copy_finish()
        torch.cuda.synchronize()

    def time_e2e(fmt, host, steps):
        for _ in range(min(args.warmup, 3)):
            e2e_step(fmt, host)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_step(fmt, host)
        barrier()
        s = time.perf_counter() - t0
        tt = torch.tensor([s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    e2e_s = time_e2e("u8", out_u8, args.steps)
    if args.dump_outputs and rank == 0:
        dumps["frame_rgba8"] = dump_frame(out_u8, dump_sel)
    e2e_value = rays_per_frame * args.steps / e2e_s / 1e6
    clocks = sampler.stop() if sampler else None  # sampled over both timed regions
    # the same with the f64 frame (24 B / pixel: Bitmap.pixels, Image.fs:30), a few steps
    f64_steps = max(1, min(args.steps, 5))
    out_f64 = np.empty((H, W, 3), dtype=np.float64) if rank == 0 else None
    if rank == 0 and world > 1:
        frame_f64 = torch.empty((H, W, 3), dtype=torch.float64, device=dev)
    e2e_f64_s = time_e2e("f64", out_f64, f64_steps)
    out_f64 = frame_f64 = None

    # ---- checks outside every timed region ------------------------------------------------------------------------
    frame_check = None
    inproc = None
    if world > 1:  # the sharded, peer-written frame equals rank 0's own unsharded render, bit for bit
        device_step()
        barrier()
        if rank == 0:
            p_one = api.make_params(W, H, spp, jit, seed=RNG_SEED, out_format=abi.OUT_RGB_F32)
            t1 = torch.empty(api.tile_buffer_bytes(p_one), dtype=torch.uint8, device=dev)
            f1 = torch.empty_like(frame)
            scene.render_tiles_device(p_one, t1.data_ptr(), stream=stream)
            api.assemble_device(p_one, [t1.data_ptr()], f1.data_ptr(), stream=stream)
            u1 = torch.empty((H, W, 4), dtype=torch.uint8, device=dev)
            api.assemble_device(api.make_params(W, H, spp, jit, seed=RNG_SEED, out_format=abi.OUT_RGBA8), [t1.data_ptr()], u1.data_ptr(), stream=stream)
            torch.cuda.synchronize()
            ok = bool((f1 == frame).all()) and bool((u1.cpu().numpy() == out_u8).all())
            frame_check = "bit-exact vs the 1-GPU render (device frame and downloaded RGBA8 frame)" if ok else "MISMATCH vs the 1-GPU render"
            del t1, f1, u1
        barrier()
        # rank 0 alone drives all N GPUs through ftb_render(n_gpus = N): the call the CLI / the F# shim makes
        if not args.no_inprocess and torch.cuda.device_count() >= world and api.device_count() >= world:
            dist.barrier(group=cpu_group)
            if rank == 0:
                p_in = api.make_params(W, H, spp, jit, seed=RNG_SEED, out_format=abi.OUT_RGBA8, n_gpus=world)
                host_in = np.empty((H, W, 4), dtype=np.uint8)
                try:
                    for _ in range(2):
                        scene.render_params(p_in, out=host_in)
                    k_in = max(1, min(args.steps, 5))
                    t0 = time.perf_counter()
                    for _ in range(k_in):
                        scene.render_params(p_in, out=host_in)
                    s_in = (time.perf_counter() - t0) / k_in
                    inproc = {"value": rays_per_frame / s_in / 1e6, "unit": UNIT, "ms_per_step": 1e3 * s_in, "n_gpus": world, "steps": k_in,
                              "call": "ftb_render(n_gpus=%d) from one process, pageable RGBA8 frame out" % world,
                              "frame_check": "bit-exact vs the multi-process frame" if bool((host_in == out_u8).all()) else "MISMATCH vs the multi-process frame"}
                except api.FtbError as e:
                    inproc = {"unavailable": str(e)}
            dist.barrier(group=cpu_group)

    line = None
    if rank == 0:
        peak, peak_how = _fp32_peak_tflops()
        kern_avg_ms = kern_total_ms / args.steps
        flops_launch = run.local_flops if world == 1 else flops_total / world
        achieved = flops_launch / (kern_avg_ms * 1e-3) / 1e12
        pk, pk_how = _peaks()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "scene": run.cfg["build"].__name__, "width": W, "height": H, "spp": spp,
                       "recursion_limit": 8, "rays_per_frame": {"primary": n_primary, "shadow": n_shadow, "reflection": n_refl},
                       "tile": "16x16 round-robin over ranks", "l2": "flushed between timed iterations (256 MB write)",
                       "parallelism": "tiles%d" % world, "gather": ("p2p-stores" if arena else "nccl-gather") if world > 1 else "none"},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": 1e3 * e2e_s / args.steps,
                    "h2d_bytes_per_step": int(16 * spp + 512), "d2h_bytes_per_step": int(W * H * 4),
                    "host_buffer": "pageable (np.empty)", "out_format": "RGBA8 (Image.write's quantisation, Image.fs:35-44, applied on the device)",
                    "call": "ftb_render" if world == 1 else (("%d bands: ftb_render_tiles_device (tiles stored into rank 0's memory over NVLink) + barrier + ftb_assemble_rows_device + ftb_host_copy_begin/finish" % bands) if arena
                                                           else "ftb_render_tiles_device + NCCL gather + ftb_assemble_device + ftb_host_copy_begin/finish"),
                    "f64": {"value": rays_per_frame * f64_steps / e2e_f64_s / 1e6, "ms_per_step": 1e3 * e2e_f64_s / f64_steps, "d2h_bytes_per_step": int(W * H * 24), "steps": f64_steps},
                    "scene_create_ms": run.create_ms, "mesh_index": run.build},
            "gpu_launches": int(args.steps * 2),
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": _traffic_per_launch(args.workload) if world == 1 else None,
                         "kernel": "ftb::render_kernel<float, FEAT, false> (the scene's feature-specialised variant)", "kernel_ms": kern_avg_ms,
                         "algorithmic_flops_per_launch": flops_launch, "peak_source": peak_how,
                         "hbm_note": "scene is KBs and rays never leave registers; algorithmic HBM bytes = framebuffer only (%d B/launch) vs %s %.0f GB/s"
                                     % (W * H * 12 // world, pk_how, pk.get("hbm_gbs", 0.0))},
            "clocks": clocks,
        }
        # What the same rays cost with the reference's own algorithm (every leaf tested for every ray, SURVEY.md 8(d)):
        # not the roofline figure -- that counts the tests this kernel performs -- but the size of the algorithmic win.
        brute = _BRUTE_FORCE_FLOPS_PER_RAY.get(run.cfg["build"].__name__) if not run.cfg.get("kw") else None
        if brute and world == 1:
            line["roofline"]["reference_algorithm"] = {
                "intersection_flops_per_ray": brute, "source": "SURVEY.md 8(d): every leaf tested per ray, no culling",
                "equivalent_tflops": rays_per_frame * brute / (kern_avg_ms * 1e-3) / 1e12}
        if frame_check:
            line["frame_check"] = frame_check
        if inproc:
            line["e2e_inprocess"] = inproc
        if not args.no_cpu_baseline and world == 1:
            res, windows, margin, rays, cores, what = cpu_sample(run.parsed, jit, CPU_SAMPLE_PRIMARY, debug=True)
            line["cpu_baseline"] = {"value": rays / res["seconds"] / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "%s, %.1f s of wall time" % (what, res["seconds"])}
            line["parity"] = gpu_parity(run, res, windows, margin)
            del res
    # ---- the other configs of BASELINE.json, one GPU, same method (fewer steps) ----------------------------------------------
    if world == 1 and not args.no_per_config:
        del frame, tiles
        run.close()
        per = {}
        peak, _ = _fp32_peak_tflops()
        for name in ALL_WORKLOADS:
            if name == args.workload:
                per[name] = {"see": "headline"}
                continue
            r = Runner(name, 0, 1, dev, stream)
            rays = sum(r.counts[:3])

            def step(ev=None, r=r):
                if ev:
                    ev[0].record()
                r.scene.render_tiles_device(r.p_f32, r.tiles.data_ptr(), stream=stream)
                if ev:
                    ev[1].record()
                api.assemble_device(r.p_f32, [r.tiles.data_ptr()], r.frame.data_ptr(), stream=stream)

            k = min(args.steps, 5)
            tot, kern = time_device(r, step, torch.cuda.synchronize, k, 3, flush)
            if args.dump_outputs:
                dumps["per_config_" + name] = dump_frame(r.frame, dump_rows(r.W, r.H))
            host = np.empty((r.H, r.W, 4), dtype=np.uint8)
            pu8 = api.make_params(r.W, r.H, r.spp, r.jit, seed=RNG_SEED, out_format=abi.OUT_RGBA8)
            for _ in range(2):
                r.scene.render_params(pu8, out=host)
            t0 = time.perf_counter()
            for _ in range(k):
                r.scene.render_params(pu8, out=host)
            e2e_ms = 1e3 * (time.perf_counter() - t0) / k
            ent = {"width": r.W, "height": r.H, "spp": r.spp, "ms_per_step": tot / k, "kernel_ms": kern / k, "value": rays / (tot / k * 1e-3) / 1e6,
                   "e2e_ms_per_step": e2e_ms, "e2e_value": rays / (e2e_ms * 1e-3) / 1e6, "rays_per_frame": rays,
                   "roofline_frac": r.local_flops / (kern / k * 1e-3) / 1e12 / peak, "scene_create_ms": r.create_ms, "mesh_index": r.build, "steps": k}
            if not args.no_cpu_baseline:
                res, windows, margin, crays, cores, what = cpu_sample(r.parsed, r.jit, MINI_SAMPLE_PRIMARY, debug=True)
                ent["cpu_value"] = crays / res["seconds"] / 1e6
                par = gpu_parity(r, res, windows, margin)
                par.pop("note", None)
                par["sample"] = what
                ent["parity"] = par
            per[name] = ent
            r.close()
        line["per_config"] = per
    if rank == 0:
        if args.dump_outputs:
            write_dumps(args.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1 or args.no_per_config:
        scene.close()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        if arena:
            arena.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
