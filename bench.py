#!/usr/bin/env python
"""bench.py -- headline benchmark of the forward splat path (BASELINE.json metric).

metric : rendered Msplats/sec @1080p, 6M-gaussian cloud  (= gaussians in the cloud x views / s)
config : C3 of BASELINE.json -- 6 M synthetic random_gaussians, f16 planar (128 B/gaussian),
         1920x1080, "Mip-NeRF-360-scale" = the generator's cloud with global_scale 0.02
         (SURVEY.md §8d); one camera view per GPU, cloud replicated, frames gathered on rank 0.
A step = one frame of every view: key-gen -> depth radix sort -> projection + SH colour -> tile
binning -> tile blend (+ the NCCL frame gather when N > 1).

  python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, through the C ABI)
  python bench.py --impl reference --steps K --warmup W    # the reference's path on the host CPU
                                                           # (oracle port: the reference cannot be built here)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's frames to DIR/*.npy
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

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

METRIC = "rendered Msplats/sec @1080p, 6M-gaussian cloud"
N_GAUSSIANS = 6_000_000
WIDTH, HEIGHT = 1920, 1080
GLOBAL_SCALE = 0.02
FRAMES_IN_FLIGHT = int(os.environ.get("BGS_FRAMES_IN_FLIGHT", "3"))   # contexts sharing the cloud (tuning knob)
WORKLOAD = ("C3: 6M random_gaussians (seed 0), f16 planar 128 B/gaussian, 1920x1080, global_scale=0.02 "
            "(Mip-NeRF-360-scale), headless camera (0,1.5,5) / one orbit view per GPU")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class NvmlClockSampler:
    """SM clock + throttle reasons sampled in-process through NVML every ~2 ms DURING the timed region (the timed
    region of the default run lasts ~35 ms: a 100 ms nvidia-smi loop cannot see it)."""

    def __init__(self, gpu_index: int):
        import pynvml

        self.nv = pynvml
        pynvml.nvmlInit()
        self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        self.sm, self.reasons, self.stop_flag, self.th = [], 0, False, None
        self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.reasons |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th is not None:
            self.th.join()
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, bit in names.items() if self.reasons & bit)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm, "reasons": reasons,
                "samples": len(self.sm), "source": "nvml, 2 ms period, inside the timed region"}


def make_clock_sampler(gpu_index: int):
    try:
        return NvmlClockSampler(gpu_index)
    except Exception:
        return ClockSampler(gpu_index)


class ClockSampler:
    """Fallback: nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 9 for i in range(4) if r[5 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_cloud(n: int):
    import bevy_gaussian_splatting_b200 as B

    return B.random_gaussians_3d_seeded(n, 0)


def read_device(ptr: int, nbytes: int) -> np.ndarray:
    """Device memory -> host bytes through the driver API (synchronous; the caller has synchronised the producers)."""
    import ctypes as C

    got = np.empty(nbytes, np.uint8)
    cu = C.CDLL("libcuda.so.1")
    cu.cuMemcpyDtoH_v2.argtypes = [C.c_void_p, C.c_uint64, C.c_size_t]
    assert cu.cuMemcpyDtoH_v2(got.ctypes.data_as(C.c_void_p), C.c_uint64(ptr), got.size) == 0
    return got


DUMP_LIMIT_BYTES = 64 << 20


def dump_frames(out_dir: str, frames: np.ndarray) -> None:
    """--dump-outputs: the (views, H, W, 4) RGBA8 frames of the last timed step as float32 .npy files, so that two builds
    can be compared output for output.  Frames larger than DUMP_LIMIT_BYTES in float32 (more than two 1080p views) are
    replaced by the same seeded sample of pixel positions in every view: frames_sample.npy (views, P, 4) and
    frames_sample_pixel.npy (P,), the row-major pixel indices as float64."""
    os.makedirs(out_dir, exist_ok=True)
    v, h, w, c = frames.shape
    if frames.size * 4 <= DUMP_LIMIT_BYTES:
        np.save(os.path.join(out_dir, "frames.npy"), frames.astype(np.float32))
        return
    p = (DUMP_LIMIT_BYTES - 4096) // (4 * v * c + 8)        # (4 KB for the two .npy headers)
    pix = np.sort(np.random.default_rng(0).choice(h * w, p, replace=False))
    np.save(os.path.join(out_dir, "frames_sample.npy"), frames.reshape(v, h * w, c)[:, pix].astype(np.float32))
    np.save(os.path.join(out_dir, "frames_sample_pixel.npy"), pix.astype(np.float64))


# ------------------------------------------------------------------------------------------------
def host_cores() -> int:
    """Cores the CPU arm may use: the process's affinity mask, NOT OMP_NUM_THREADS (torchrun exports 1)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def bench_config(views: int, world: int, extra: dict | None = None) -> dict:
    """The config dict both arms print (same keys, so the driver's same_config check compares like with like)."""
    cfg = {"workload": WORKLOAD, "n_gaussians": N_GAUSSIANS, "layout": "f16 planar (128 B/gaussian)", "width": WIDTH, "height": HEIGHT,
           "global_scale": GLOBAL_SCALE, "views": views, "frame_format": "rgba8_srgb",
           "parallelism": f"view-parallel x{world}, replicated cloud"}
    if extra:
        cfg.update(extra)
    return cfg


def cpu_reference_run(steps: int, warmup: int, budget_s: float, cloud=None, keep_image: bool = False):
    """The reference's path on the host CPU: oracle ref_mode (back-to-front instanced quads, exactly
    the reference's blending semantics), OpenMP over all host cores.  kind = "port": the Rust/WGSL
    reference cannot be built or run in this image (SURVEY.md §8c).  Best-of-`steps` (the box is shared)."""
    import bevy_gaussian_splatting_b200 as B
    from oracle import oracle as O

    if cloud is None:
        cloud = make_cloud(N_GAUSSIANS)
    cloud = cloud.rounded_to_f16()          # the f16 layout's behaviour: f32 maths on f16-rounded inputs
    view = B.headless_view(WIDTH, HEIGHT)
    s = B.CloudSettings(global_scale=GLOBAL_SCALE)
    u = B.GaussianSplattingPlugin.cloud_uniform(s)
    cores = host_cores()
    # size the sample from one probe frame on a 1/6 prefix
    n_probe = min(len(cloud), 1_000_000)
    t0 = time.perf_counter()
    O.render_ref(cloud.subset(n_probe), view.to_abi(), u, s.to_abi(), threads=cores)
    t_probe = time.perf_counter() - t0
    est_full = t_probe * max(1.0, len(cloud) / n_probe) * 0.6 + 0.2
    frames = steps + warmup
    n_s = len(cloud)
    if est_full * frames > budget_s:
        n_s = int(max(250_000, min(len(cloud), len(cloud) * budget_s / (est_full * frames))))
    sample = cloud.subset(n_s)
    img = None
    for _ in range(warmup):
        img = O.render_ref(sample, view.to_abi(), u, s.to_abi(), threads=cores)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        img = O.render_ref(sample, view.to_abi(), u, s.to_abi(), threads=cores)
        times.append(time.perf_counter() - t0)
    ms = 1000.0 * float(np.min(times))
    value = n_s / (ms / 1000.0) / 1e6
    desc = (f"first {n_s} of the {len(cloud)} gaussians of the same cloud, full 1920x1080 frame, oracle ref_mode "
            f"(key-gen + stable sort + back-to-front quad blending), best of {steps} frames after {warmup} warm-up, {cores} threads")
    return value, ms, cores, desc, n_s, (img if keep_image and n_s == len(cloud) else None)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    value, ms, cores, desc, n_s, _ = cpu_reference_run(args.steps, min(args.warmup, 2), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "Msplats/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 (f16-packed inputs)", "data": "synthetic",
        "config": bench_config(1, world, {"note": "CPU arm: ONE view on rank 0's host cores (the reference has no multi-GPU path); "
                                                  f"sample_gaussians={n_s}"}),
        "cpu_baseline": {"value": round(value, 3), "unit": "Msplats/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": round(value, 3), "unit": "Msplats/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
def parity_block(plugin, handle, settings, view, cloud, ref_img):
    """CUDA vs the oracle on the BENCHMARKED frame, outside any timed region: sorted (key, index) entries and tile
    ranges bit-exact, pixels vs the oracle's ref_mode (the reference's back-to-front semantics) and tile_mode."""
    from oracle import oracle as O

    oc = cloud.rounded_to_f16()
    u = plugin.cloud_uniform(settings, None, handle.aabb)
    img = plugin.render_view(handle, settings, view, fmt="rgba32f")
    got = plugin.sorted_entries()
    rng = plugin.tile_ranges()
    keys = O.keygen(oc.position_visibility, view.to_abi(), u, 32)
    sk, si = O.radix_sort(keys, 32)
    til = O.render_tiles(oc, view.to_abi(), u, settings.to_abi())
    if ref_img is None:
        ref_img = O.render_ref(oc, view.to_abi(), u, settings.to_abi(), threads=host_cores())
    return {"config": "the benchmarked C3 frame (6M f16, 1920x1080), rgba32f accumulators",
            "sorted_bit_exact": bool(np.array_equal(got[:, 0], sk) and np.array_equal(got[:, 1], si)),
            "ranges_bit_exact": bool(np.array_equal(rng, til["tile_ranges"])),
            "tile_slices_bit_exact": bool(np.array_equal(plugin.tile_entries(), til["tile_entries"])),
            "linf_vs_ref_mode": float(np.abs(img - ref_img).max()), "linf_vs_tile_mode": float(np.abs(img - til["image"]).max()),
            "tolerance": 1e-3}


def bind_to_gpu_numa_node(gpu_index: int):
    """Multi-GPU runs: keep this rank's threads (and so its pinned frame buffers: first touch) on the NUMA node its GPU
    hangs off, so eight ranks' device->host frame copies do not cross the socket interconnect.  Best effort."""
    try:
        import pynvml

        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(gpu_index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                   # "00000000:1b:00.0" -> "0000:1b:00.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def run_cuda(args):
    import torch

    import bevy_gaussian_splatting_b200 as B
    from bevy_gaussian_splatting_b200 import abi
    from bevy_gaussian_splatting_b200.multiview import MultiViewSession

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # FRAMES_IN_FLIGHT contexts on this GPU share the cloud; consecutive frames alternate between them, so one
    # frame's latency-bound front (key-gen, sorts, binning) overlaps the previous frame's raster.  Each context
    # has its own streams + scratch (bgs.h: "distinct contexts may be used concurrently"); a rank's contexts share
    # ONE NCCL communicator.
    frames_in_flight = FRAMES_IN_FLIGHT
    plugins = [B.GaussianSplattingPlugin(local_rank) for _ in range(frames_in_flight)]
    plugin = plugins[0]
    cloud = make_cloud(N_GAUSSIANS)
    handle = plugin.add_cloud(cloud, f16=True)
    settings = B.CloudSettings(global_scale=GLOBAL_SCALE)
    sessions = []
    for i, p in enumerate(plugins):
        share = os.environ.get("BGS_SHARED_COMM", "1") != "0"        # (tuning knob: one communicator per context instead)
        sessions.append(MultiViewSession(rank, world, 0, plugin=p if world > 1 else None,
                                         share_comm_of=sessions[0] if (world > 1 and i > 0 and share) else None))
    sess = sessions[0]
    view = sess.view(WIDTH, HEIGHT) if world > 1 else B.headless_view(WIDTH, HEIGHT)
    frame_bytes = WIDTH * HEIGHT * 4
    dev = torch.device("cuda", local_rank)
    streams = [torch.cuda.ExternalStream(p.stream_ptr, device=dev) for p in plugins]
    copy_streams = [torch.cuda.ExternalStream(p.copy_stream_ptr, device=dev) for p in plugins]
    all_frames = [torch.empty(world * frame_bytes, dtype=torch.uint8, device="cuda") if (world > 1 and rank == 0) else None
                  for _ in plugins]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def sync_all():
        ok = True
        for p in plugins:
            ok = p.sync() and ok
        return ok

    def step(i, out=None):
        # frames are only ENQUEUED (BGS_FLAG_ASYNC), as the reference submits command buffers without reading
        # anything back; sync_all() closes the timed region
        k = i % frames_in_flight
        p = plugins[k]
        p.render_view(handle, settings, view, fmt="rgba8_srgb", to_host=out is not None, out=out, asynchronous=True)
        if world > 1:
            sessions[k].gather_device(p.frame_device_ptr, all_frames[k].data_ptr() if all_frames[k] is not None else 0, frame_bytes)

    # ---- device-resident throughput ("value"): inputs (768 MB cloud >> 126 MB L2) already in HBM
    for p in plugins:
        p.render_view(handle, settings, view, fmt="rgba8_srgb", to_host=False)   # sizes every buffer
    # set-up, not warm-up: every context queues frames (and gathers) once so that lazily created state -- the second
    # device frame, the copy/comm stream's first use, NCCL's peer connections -- exists before the W warm-up steps
    for i in range(2 * frames_in_flight):
        step(i)
    assert sync_all()
    barrier()
    for i in range(args.warmup):
        step(i)
    assert sync_all()
    barrier()
    clocks = make_clock_sampler(local_rank)
    if rank == 0:
        clocks.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = [torch.cuda.Event(enable_timing=True) for _ in range(2 * len(plugins))]
    e0.record(streams[0])
    for i in range(args.steps):
        step(i)
    # the window ends when the LAST work of every stream has finished: render streams and copy/comm streams
    # (async frames are gathered over NCCL on the copy/comm stream)
    for ev, st_ in zip(e1, streams + copy_streams):
        ev.record(st_)
    assert sync_all(), "pair buffer overflowed inside the timed region"
    barrier()
    ms_total = max(e0.elapsed_time(ev) for ev in e1)     # device time from the first frame's start to the last frame's / gather's end
    clk = clocks.stop() if rank == 0 else None
    k_last = (args.steps - 1) % frames_in_flight
    # the last timed step's frame, read before anything renders into that context again
    dumped = None
    if args.dump_outputs and world == 1:
        dumped = read_device(plugins[k_last].frame_device_ptr, frame_bytes).reshape(1, HEIGHT, WIDTH, 4)
    # ---- multi-GPU correctness on hardware: rank 0 re-renders every rank's view locally and compares it with the
    #      gathered frames, byte for byte (outside the timed region)
    gather_ok = None
    if world > 1 and rank == 0:
        gather_ok = True
        gathered = all_frames[k_last].cpu().numpy().reshape(world, HEIGHT, WIDTH, 4)
        if args.dump_outputs:
            dumped = gathered
        for r in range(world):
            local = plugin.render_view(handle, settings, MultiViewSession(r, world, 0).view(WIDTH, HEIGHT), fmt="rgba8_srgb")
            gather_ok = gather_ok and bool(np.array_equal(local, gathered[r]))
    # ---- the same window with the frames moved by the GPUs themselves instead of NCCL kernels (CUDA IPC mapping of the
    #      root's frame stack + per-slot completion words awaited on the root's stream):
    #      "copy_engine": every rank pushes its finished frame with a peer-to-peer cudaMemcpyAsync (copy engines, no SM);
    #      "direct":      every rank RENDERS into its slot of the root's stack: the blend kernel's own pixel stores cross
    #                     NVLink, only the completion word follows.
    #      All transports are measured in the same run on the same box and verified frame by frame; the line's `value` is
    #      the fastest verified one (config.gather names it), the others stay beside it.
    gather_ce = gather_direct = None
    peer_ready = False
    if world > 1:
        def agree(ok: bool) -> bool:
            t_ = torch.tensor([1 if ok else 0], device="cuda", dtype=torch.int32)
            dist.all_reduce(t_, op=dist.ReduceOp.MIN)
            return bool(t_.item())

        try:
            for k in range(frames_in_flight):
                sessions[k].setup_peer_frames(local_rank, frame_bytes)
            peer_ready = True
        except Exception as e:          # (no peer access between the GPUs: NCCL stays the only transport)
            print(f"bench.py: rank {rank}: peer frame stack unavailable: {e}", file=sys.stderr)
        peer_ready = agree(peer_ready)

        def peer_leg(direct: bool):
            use_signal = [True]

            def step_p(i):
                k = i % frames_in_flight
                p = plugins[k]
                if direct:
                    slot = sessions[k].peer_slot_ptr(frame_bytes)
                    p.render_view_to_device(handle, settings, view, slot, fmt="rgba8_srgb", asynchronous=True)
                    sessions[k].push_device(slot, frame_bytes, signal=use_signal[0])     # (the word only: no copy)
                    return
                p.render_view(handle, settings, view, fmt="rgba8_srgb", to_host=False, asynchronous=True)
                if use_signal[0]:
                    try:
                        sessions[k].push_device(p.frame_device_ptr, frame_bytes, signal=True)
                        return
                    except abi.BgsError:
                        use_signal[0] = False
                sessions[k].push_device(p.frame_device_ptr, frame_bytes)

            # completion words are proven on the warm-up frames first (every rank's words must have reached the expected
            # sequence), before any stream is made to wait on them; else the host barrier stands in
            ok = True
            try:
                for i in range(2 * frames_in_flight + args.warmup):
                    step_p(i)
            except Exception as e:
                print(f"bench.py: rank {rank}: {'direct' if direct else 'copy-engine'} gather failed: {e}", file=sys.stderr)
                ok = False
            ok = sync_all() and ok
            barrier()
            if not agree(ok):
                return None
            sig_ok = use_signal[0]
            if rank == 0 and sig_ok:
                for k in range(frames_in_flight):
                    words = read_device(sessions[k].peer_flags_ptr(), 4 * world).view(np.uint32)
                    sig_ok = sig_ok and bool(np.all(words == np.uint32(sessions[k]._peer_seq & 0xFFFFFFFF)))
            use_signal[0] = agree(sig_ok)
            barrier()
            leg_clocks = make_clock_sampler(local_rank)
            if rank == 0:
                leg_clocks.start()
            c0 = torch.cuda.Event(enable_timing=True)
            c1 = [torch.cuda.Event(enable_timing=True) for _ in range(2 * len(plugins))]
            c0.record(streams[0])
            for i in range(args.steps):
                step_p(i)
            if rank == 0 and use_signal[0]:
                # the root's copy/comm streams resume when EVERY rank's last frame of that context has landed
                for k in range(frames_in_flight):
                    sessions[k].wait_frames(plugins[k].copy_stream_ptr, sessions[k]._peer_seq)
            for ev, st_ in zip(c1, streams + copy_streams):
                ev.record(st_)
            assert sync_all()
            leg_clk = leg_clocks.stop() if rank == 0 else None
            k_last = (args.steps - 1) % frames_in_flight
            got = None
            if rank == 0 and use_signal[0]:
                # read BEFORE any host barrier: the device-side wait alone has established that all frames are there
                got = read_device(sessions[k_last]._peer_ptr.value, world * frame_bytes)
            barrier()
            leg_ms = max(c0.elapsed_time(ev) for ev in c1) / args.steps
            t_ = torch.tensor([leg_ms], device="cuda")
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            leg_ms = float(t_.item())
            leg_ok = None
            if rank == 0:
                if got is None:
                    got = read_device(sessions[k_last]._peer_ptr.value, world * frame_bytes)
                got = got.reshape(world, HEIGHT, WIDTH, 4)
                leg_ok = True
                for r in range(world):
                    local = plugin.render_view(handle, settings, MultiViewSession(r, world, 0).view(WIDTH, HEIGHT), fmt="rgba8_srgb")
                    leg_ok = leg_ok and bool(np.array_equal(local, got[r]))
            barrier()
            return {"transport": ("bgs_render straight into the root's frame stack (CUDA IPC mapping): the blend kernel's pixel stores cross NVLink, no copy"
                                  if direct else "CUDA IPC + cudaMemcpyAsync peer pushes on each rank's copy stream (copy engines, no SM)"),
                    "value": round(N_GAUSSIANS * world / (leg_ms / 1000.0) / 1e6, 1), "unit": "Msplats/s", "ms_per_step": round(leg_ms, 4),
                    "frames_verified": leg_ok, "clocks": leg_clk, "device_signalling": bool(use_signal[0]),
                    "signalling": ("device: one 32-bit sequence word per slot stored after the frame, cuStreamWaitValue32 on the root's stream "
                                   "(frames read back before any host barrier)") if use_signal[0] else "host barrier"}

        if peer_ready:
            gather_ce = peer_leg(False)
            gather_direct = peer_leg(True)
    # per-frame / per-stage times (live CUDA events inside the library), one frame at a time on an idle GPU
    frame_us, stage_rows = [], []
    for _ in range(min(args.steps, 100)):
        plugin.render_view(handle, settings, view, fmt="rgba8_srgb", to_host=False)
        st = plugin.stage_times_us()
        frame_us.append(float(st[5])); stage_rows.append(st)
    ms_step = ms_total / args.steps
    if dist is not None:
        t = torch.tensor([ms_step], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item())
    # the line's transport: the fastest one whose gathered frames were verified (rank 0 decides, everybody follows)
    choice = 0
    if world > 1:
        if rank == 0:
            cands = [(ms_step, 0)] if gather_ok else []
            for code, leg in ((1, gather_ce), (2, gather_direct)):
                if leg and leg["frames_verified"]:
                    cands.append((leg["ms_per_step"], code))
            choice = min(cands)[1] if cands else 0
        t = torch.tensor([choice], device="cuda", dtype=torch.int32)
        dist.broadcast(t, src=0)
        choice = int(t.item())
    launches_per_frame = plugin.last_launch_count
    fs = plugin.frame_stats()
    stage_med = np.median(np.array(stage_rows), axis=0)

    # ---- end to end through the C ABI with HOST buffers: per step the view/uniform/settings structs go
    #      host->device as kernel arguments and the finished RGBA8 frame comes back into pinned host memory.
    # K frames in, K frames out: each frame's D2H copy (copy stream) overlaps later frames' kernels; pinned host
    # buffers alternate; sync_all() (every frame delivered to host memory) closes the timed region.
    # At N > 1 every rank's frame lands in its own host buffer AND in the root's frame stack, over the line's transport
    # (the copy-engine push when a peer transport was chosen: the frame is rendered into library memory for the D2H copy).
    host_frames = [torch.empty((HEIGHT, WIDTH, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2 * frames_in_flight)]
    e2e_push = world > 1 and choice != 0
    e2e_signal = bool(e2e_push and gather_ce and gather_ce["device_signalling"])

    def step_e2e(i):
        if not e2e_push:
            return step(i, out=host_frames[i % (2 * frames_in_flight)])
        k = i % frames_in_flight
        p = plugins[k]
        p.render_view(handle, settings, view, fmt="rgba8_srgb", to_host=True, out=host_frames[i % (2 * frames_in_flight)], asynchronous=True)
        sessions[k].push_device(p.frame_device_ptr, frame_bytes, signal=e2e_signal)

    def close_e2e():
        if e2e_signal and rank == 0:
            for k in range(frames_in_flight):
                sessions[k].wait_frames(plugins[k].copy_stream_ptr, sessions[k]._peer_seq)
        return sync_all()

    for i in range(2 * frames_in_flight):
        step_e2e(i)
    assert close_e2e()
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(i)
    assert close_e2e()
    barrier()
    e2e_ms = 1000.0 * (time.perf_counter() - t0) / args.steps
    if dist is not None:
        t = torch.tensor([e2e_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    h2d = sum(__import__("ctypes").sizeof(c) for c in (abi.bgs_view, abi.bgs_cloud_uniform, abi.bgs_settings))
    if peer_ready:
        barrier()
        for root_turn in (False, True):          # the ranks that opened the root's allocation close it before the root frees it
            if (rank == 0) == root_turn:
                for k in range(frames_in_flight):
                    sessions[k].release_peer_frames()
            barrier()

    if rank != 0:
        for se in sessions:
            se.destroy()
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- roofline (HBM): algorithmic bytes per launch / live CUDA-event duration of that launch
    peak, peak_src = peaks()
    n, nv, I = fs.n, fs.n_visible, int(fs.n_pairs)
    depth_passes = 4
    alg = {
        "keygen": 16 * n + 4 * (n // 32) * 2 + (16 + 12) * nv,            # positions in, mask bits out + in, visible re-read + (key,id,slot) out
        "depth_sort": depth_passes * 16 * nv,                             # P x (8 in + 8 out)  (histograms come from key-gen)
        "project": 4 * nv + (16 + 112) * nv + 48 * nv,                    # ids + f16 attrs (pos 16 + 16 + 96) + record
        "bin": 2 * 12 * nv + 8 * I + (4 * I + 2 * 16 * I) + 8 * fs.tiles_x * fs.tiles_y,   # 2 x (perm + bbox) + pairs out + hist read + 2 passes
        "raster": 4 * I + 48 * I + 4 * WIDTH * HEIGHT,
    }
    names = ["keygen", "depth_sort", "project", "bin", "raster"]
    stages = []
    for i, nm in enumerate(names):
        us = float(stage_med[i])
        gbs = alg[nm] / (us * 1e-6) / 1e9 if us > 0 else 0.0
        stages.append({"stage": nm, "us": round(us, 1), "alg_bytes": int(alg[nm]), "gbs": round(gbs, 1), "frac": round(gbs / peak, 4)})
    # north_star's "projection + sort stages": key-gen -> (depth sort || projection), as ONE segment of the frame
    front_us = float(stage_med[5] - stage_med[3] - stage_med[4])
    front_bytes = alg["keygen"] + alg["depth_sort"] + alg["project"]
    proj_sort = {"what": "key-gen + depth sort + projection (sort and projection overlap on two streams)", "us": round(front_us, 1),
                 "alg_bytes": int(front_bytes), "gbs": round(front_bytes / (front_us * 1e-6) / 1e9, 1),
                 "frac": round(front_bytes / (front_us * 1e-6) / 1e9 / peak, 4), "target": 0.70}
    dom = max(stages, key=lambda s: s["us"])
    traffic_path = os.path.join(ROOT, "profiles", "traffic.json")
    traffic = None
    if os.path.exists(traffic_path):
        traffic = json.load(open(traffic_path)).get(dom["stage"])
    roofline = {"kernel": dom["stage"], "bound": "hbm", "achieved": dom["gbs"], "peak": peak, "unit": "GB/s",
                "frac": dom["frac"], "traffic": traffic, "traffic_source": "static: ncu dram__bytes of the committed capture under profiles/ (not measured in this run)",
                "peak_source": peak_src,
                "note": "dominant kernel by time; raster is bound by instruction issue, not by HBM -- see roofline.issue and stages[]"}
    # the dominant kernel's OWN roofline: warp-instructions it executes per launch (ncu, profiles/traffic.json) against
    # the SMs' issue rate (4 warp-instructions per SM cycle) at the SM clock sampled during the timed region
    if traffic_path and os.path.exists(traffic_path):
        wi = json.load(open(traffic_path)).get("warp_inst", {}).get(dom["stage"])
        if wi:
            sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
            mhz = float((clk or {}).get("sm_mhz") or 1965.0)
            peak_gi = sms * 4 * mhz * 1e6 / 1e9
            ach_gi = wi / (dom["us"] * 1e-6) / 1e9
            roofline["issue"] = {"warp_inst_per_launch": int(wi), "achieved": round(ach_gi, 1), "peak": round(peak_gi, 1),
                                 "unit": "G warp-inst/s", "frac": round(ach_gi / peak_gi, 4),
                                 "source": "ncu smsp__inst_executed.sum of the committed capture (profiles/), live CUDA-event time"}

    # ---- CPU baseline beside it + parity of the benchmarked frame (rank 0, N=1 only; outside the timed regions)
    cpu, parity = None, None
    if world == 1 and not args.no_cpu_baseline:
        v, ms, cores, desc, _, ref_img = cpu_reference_run(steps=3, warmup=1, budget_s=25.0, cloud=cloud, keep_image=True)
        cpu = {"value": round(v, 3), "unit": "Msplats/s", "cores": cores, "kind": "port", "sample": desc}
        parity = parity_block(plugin, handle, settings, view, cloud, ref_img)
    # ---- the raw generator scale (global_scale 1.0, SURVEY.md §8d "also report 1.0 if it completes"): informational
    raw = None
    if world == 1 and not args.no_cpu_baseline:
        s_raw = B.CloudSettings(global_scale=1.0)
        rows = []
        for _ in range(12):
            plugin.render_view(handle, s_raw, view, fmt="rgba8_srgb", to_host=False)
            rows.append(plugin.stage_times_us())
        med = np.median(np.array(rows[4:]), axis=0)
        fr = plugin.frame_stats()
        raw = {"config": "same cloud and camera, global_scale 1.0 (raw generator), one frame at a time", "frame_ms_p50": round(float(med[5]) / 1000.0, 4),
               "Msplats_per_s": round(N_GAUSSIANS / float(med[5]), 1), "rounds": int(fr.rounds), "n_pairs_emitted": int(fr.n_pairs),
               "stage_us": [round(float(x), 1) for x in med[:5]]}

    views = world
    gather_nccl = None
    gather_name = None
    if world > 1:
        gather_nccl = {"transport": "bgs_gather_frames: NCCL send/recv on each rank's copy/comm stream (north_star's gather)",
                       "value": round(N_GAUSSIANS * views / (ms_step / 1000.0) / 1e6, 1), "unit": "Msplats/s",
                       "ms_per_step": round(ms_step, 4), "frames_verified": gather_ok, "clocks": clk}
        chosen = {0: gather_nccl, 1: gather_ce, 2: gather_direct}[choice]
        gather_name = {0: "nccl", 1: "copy_engine", 2: "direct"}[choice]
        ms_step, gather_ok, clk = chosen["ms_per_step"], chosen["frames_verified"], chosen["clocks"]
    value = N_GAUSSIANS * views / (ms_step / 1000.0) / 1e6
    line = {
        "impl": "cuda", "metric": METRIC, "value": round(value, 1), "unit": "Msplats/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (f16-packed inputs)", "data": "synthetic",
        "config": bench_config(views, world, {"n_visible": nv, "n_pairs": I, "l2": "inputs larger than L2 (768 MB cloud vs 126 MB)",
                                              "frames_in_flight": frames_in_flight, "rank0_numa_node": numa_node,
                                              "gather": None if world == 1 else
                                              f"{gather_name}: the fastest verified transport of this run (gather_nccl / gather_ce / gather_direct hold all three)",
                                              "timing": "value: 3 frames in flight, CUDA events over render + copy/comm streams; "
                                                        "stages[] / frame_ms_*: one frame at a time on an idle GPU"}),
        "frame_ms_p50": round(float(np.percentile(frame_us, 50)) / 1000.0, 4),
        "frame_ms_p95": round(float(np.percentile(frame_us, 95)) / 1000.0, 4),
        "secondary_metric": {"name": "frame-time p50 ms (one frame at a time)", "value": round(float(np.percentile(frame_us, 50)) / 1000.0, 4),
                             "fps": round(1e6 / float(np.percentile(frame_us, 50)), 1), "target_fps": 500},
        "fps_per_gpu": round(1000.0 / ms_step, 1),
        "e2e": {"value": round(N_GAUSSIANS * views / (e2e_ms / 1000.0) / 1e6, 1), "unit": "Msplats/s",
                "ms_per_step": round(e2e_ms, 4), "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": frame_bytes},
        "gpu_launches": int(launches_per_frame * args.steps),
        "roofline": roofline, "proj_sort_roofline": proj_sort, "stages": stages, "cpu_baseline": cpu, "parity": parity,
        "gathered_frames_verified": gather_ok, "gather_nccl": gather_nccl, "gather_ce": gather_ce, "gather_direct": gather_direct,
        "raw_scale_1": raw, "clocks": clk,
    }
    if dumped is not None:
        dump_frames(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)
    for se in sessions:
        se.destroy()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the frames of the last timed step to DIR/*.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm renders a sample of the cloud sized from its own timing, "
                 "so its output is not comparable from run to run")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())
