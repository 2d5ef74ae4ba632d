#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 raylib path tracer.

  python bench.py --gpus N --steps K --warmup W            # this repository's GPU path
  python bench.py --impl reference --gpus N ...            # the reference's own CPU renderer (oracle/_ref)

A "step" is one full frame of the workload rendered through the raylib API.  Default workload is
BASELINE.json configs[3]: the ~10M-triangle instance scatter at 3840x2160, 256 spp, depth 8 -- the
configuration the north star quotes its multi-GPU target on.  For N > 1 (torchrun, one process per GPU)
the frame is split into interleaved 16x16 tiles, every rank renders its tiles from a replicated scene and
stores the final pixels of its tiles straight into rank 0's frame over NVLink (CUDA IPC mapping; `--gather nccl`
selects shard buffers + one NCCL gather instead).  Strong scaling: total work fixed.

Prints ONE JSON line (rank 0).  Metric: Mrays/s = scene-level ray queries (camera + scattered + sun-shadow)
per second over the whole job; spp/s (pixel-samples per second) rides along as `spp_per_s`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "software-raytracing_b200"))

WORKLOADS = {
    # name: (demo config id, size param, description)
    "random_spheres_640x360_16spp_d5": (1, 0, "built-in random-spheres demo scene, 640x360, 16 spp, depth 5"),
    "cornell_1920x1080_64spp_d8": (2, 0, "procedural Cornell box (42 tris), 1920x1080, 64 spp, depth 8"),
    "grid1M_1920x1080_16spp_d2": (3, 0, "1,002,528-triangle displaced grid, 1920x1080, primary + AO (16 spp, depth 2)"),
    "scatter10M_3840x2160_256spp_d8": (4, 0, "9,999,362-triangle instance scatter (7812 meshes), 3840x2160, 256 spp, depth 8"),
    "textured2M_1920x1080_64spp_d8": (5, 0, "~2M-triangle textured microfacet room, 1920x1080, 64 spp, depth 8"),
}
DEFAULT_WORKLOAD = "scatter10M_3840x2160_256spp_d8"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("BENCH_WORKLOAD", DEFAULT_WORKLOAD), choices=sorted(WORKLOADS))
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (development only; flagged in config)")
    ap.add_argument("--size", type=int, default=0, help="override scene size parameter (development only; flagged in config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inprocess", action="store_true",
                    help="N GPUs inside ONE process through the plain reference entry points: RaylibB200_SetDevices(N), then "
                         "Raylib_Render spreads every frame over the N devices itself (no torchrun, no torch.distributed)")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: 'peer' = every rank stores its final pixels straight into rank 0's frame over NVLink (CUDA IPC "
                         "mapping, the gather is fused into the last accumulate kernel); 'nccl' = shard buffers + one NCCL gather + de-interleave")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frame of the last one to DIR as .npy (a fixed, seeded sample of its "
                         "pixels when the whole frame exceeds 64 MB), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the frame of the GPU path; the reference arm has none")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, frame, counts):
    """frame: the H x W x 4 float32 frame of the last timed step (what a caller of RaylibB200_RenderShardToFrame receives);
    counts: that frame's ray queries and pixel samples, summed over all ranks.  Frames above DUMP_LIMIT_BYTES are written
    as the pixels at fixed indices drawn from a seeded generator (frame_pixel_index.npy, row-major pixel numbers, float64
    holds them exactly)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    pixels = frame.reshape(-1, frame.shape[-1])
    if frame.nbytes <= DUMP_LIMIT_BYTES:
        np.save(os.path.join(directory, "frame.npy"), frame.astype(np.float32))
    else:
        k = DUMP_LIMIT_BYTES // 2 // (pixels.shape[1] * 4 + 8)
        idx = np.sort(np.random.default_rng(1337).choice(len(pixels), size=k, replace=False))
        np.save(os.path.join(directory, "frame_pixels.npy"), pixels[idx].astype(np.float32))
        np.save(os.path.join(directory, "frame_pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(directory, "ray_queries_pixel_samples.npy"), np.asarray(counts, dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.device_index = device_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s, MEASURED_PEAKS.json absent)"


def workload_settings(rl, info, args):
    s = info.settings
    if args.spp > 0:
        s = s.copy(samplesPerPixel=args.spp)
    return s


def config_dict(args, name, info, settings):
    """The workload, spelled identically by both arms (the driver compares `config` of the two lines).  Everything that
    describes one arm only -- device tree, scene bytes, the CPU arm's bounded sample -- goes to other keys."""
    cfg = {
        "workload": name, "description": WORKLOADS[name][2],
        "width": settings.viewportWidth, "height": settings.viewportHeight, "spp": settings.samplesPerPixel,
        "max_path_length": settings.maxPathLength, "triangles": int(info.numTriangles), "spheres": int(info.numSpheres),
        "meshes": int(info.numMeshes), "frame_seed": 1337,
        "l2": "scene + path-state arenas exceed the 126 MB L2 (no flush needed)",
    }
    if args.spp > 0 or args.size > 0:
        cfg["development_override"] = {"spp": args.spp, "size": args.size}
    return cfg


# ------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU renderer on a bounded sample of the same workload

CPU_SAMPLE_TARGET_S = 12.0      # CPU seconds one bounded sample should take


def cpu_sample_settings(settings, probe_samples_per_s):
    """Bounded sample of the workload for the CPU arm: same scene, camera and depth; the viewport is halved
    (quartered if still too slow) and spp chosen so one render costs about CPU_SAMPLE_TARGET_S seconds."""
    budget = max(1.0, probe_samples_per_s * CPU_SAMPLE_TARGET_S)
    for div in (1, 2, 4, 8):
        w = max(16, settings.viewportWidth // div)
        h = max(16, settings.viewportHeight // div)
        spp = int(budget // (w * h))
        if spp >= 1 or div == 8:
            return w, h, max(1, min(settings.samplesPerPixel, spp))


def run_cpu_reference(rl, name, args, native, steps=1, warmup=0, with_scene=None):
    """Times oracle/_ref (the compiled reference) on the host cores. Returns (dict, scene info, nominal settings)."""
    from oracle import bindings as ob      # the oracle: only this leg of bench.py touches it
    ref = ob.Reference()
    cfg_id, size, _ = WORKLOADS[name]
    t0 = time.time()
    info = ref.create_demo(cfg_id, args.size or size)
    build_s = time.time() - t0
    settings = workload_settings(rl, info, args)
    nominal = settings.copy()
    # probe: 1/8 viewport, 1 spp -> pixel-samples per second of this host on this scene
    pw, ph = max(16, settings.viewportWidth // 8), max(16, settings.viewportHeight // 8)
    ref.set_viewport(info, pw, ph)
    probe = info.settings.copy(samplesPerPixel=1, maxPathLength=nominal.maxPathLength, rayTMin=nominal.rayTMin)
    _, pst = ref.render_deterministic(probe, info.scene, info.camera)
    rate = pw * ph / max(pst.seconds, 1e-6)
    for _ in range(3):
        w, h, spp = cpu_sample_settings(nominal, rate)
        ref.set_viewport(info, w, h)
        s = info.settings.copy(samplesPerPixel=spp, maxPathLength=nominal.maxPathLength, rayTMin=nominal.rayTMin)
        # deterministic driver: counts ray queries (and is the parity oracle); same thread count as the native pool
        _, st = ref.render_deterministic(s, info.scene, info.camera)
        if st.seconds >= 0.5 * CPU_SAMPLE_TARGET_S or (w, h, spp) == (nominal.viewportWidth, nominal.viewportHeight, nominal.samplesPerPixel):
            break
        rate = w * h * spp / max(st.seconds, 1e-6)       # the small probe under-estimates (cold caches, thread start)
    rays_per_sample = st.rayQueries / float(w * h * spp)
    threads = int(ref.lib.oracle_hardware_threads())
    if native:
        secs = []
        for i in range(warmup + steps):
            _, sec = ref.render_native(s, info.scene, info.camera)
            if i >= warmup:
                secs.append(sec)
        sec = sum(secs) / len(secs)
        kind_note = "reference Renderer::RenderScene (own thread pool; wall time includes its 100 ms completion poll)"
    else:
        sec = st.seconds
        kind_note = "reference TraceScene/Camera/BVH driven by the deterministic oracle pixel loop"
    samples = w * h * spp
    out = {
        "value": samples * rays_per_sample / sec / 1e6, "unit": "Mrays/s", "spp_per_s": samples / sec,
        "cores": threads, "kind": "reference",
        "sample": "%dx%d, %d spp, depth %d of the same scene/camera (%s); rays/pixel-sample %.3f from the deterministic run"
                  % (w, h, spp, s.maxPathLength, kind_note, rays_per_sample),
        "seconds": sec, "scene_build_s": build_s,
    }
    if with_scene is not None:
        ref.set_viewport(info, nominal.viewportWidth, nominal.viewportHeight)
        out["parity"] = with_scene(ref, info, nominal)
    ref.destroy_demo(info)
    return out, info, nominal


def parity_check(rl, prod, pinfo, ref, rinfo, nominal):
    """Oracle as CHECKER inside the cpu_baseline leg: primary hit ids / t of the whole frame and the radiance of a centred
    crop at matched spp and seed, product (GPU, through the C ABI) against the compiled reference (CPU)."""
    import numpy as np
    W, H = nominal.viewportWidth, nominal.viewportHeight
    grank, gt = prod.primary_hits(nominal, pinfo.scene, pinfo.camera)
    rrank, rt_, _, _ = ref.primary_hits(nominal, rinfo.scene, rinfo.camera)
    same = grank == rrank
    both = same & (grank >= 0)
    spp = max(1, min(4, nominal.samplesPerPixel))
    cw, ch = min(W, 256), min(H, 256)
    x0, y0 = (W - cw) // 2, (H - ch) // 2
    s = nominal.copy(samplesPerPixel=spp)
    gimg = prod.render(s, pinfo.scene, pinfo.camera)[y0:y0 + ch, x0:x0 + cw]
    rimg, _ = ref.render_deterministic(s, rinfo.scene, rinfo.camera, region=(x0, y0, x0 + cw, y0 + ch))
    rimg = rimg[y0:y0 + ch, x0:x0 + cw]
    gb, rb = np.ascontiguousarray(gimg).view(np.uint32), np.ascontiguousarray(rimg).view(np.uint32)
    denom = np.maximum(np.abs(rimg), 1e-3)
    return {
        "primary_rays": int(W * H), "id_mismatch_rate": float(1.0 - same.mean()),
        "t_bit_match": float((gt[both].view(np.uint32) == rt_[both].view(np.uint32)).mean()) if both.any() else 1.0,
        "radiance_crop": "%dx%d centred, %d spp, depth %d, seed 1337" % (cw, ch, spp, nominal.maxPathLength),
        "psnr_db": float(rl.psnr(gimg, rimg)), "bit_identical": float((gb == rb).all(axis=-1).mean()),
        "rel_err_gt_1e-3": float((np.abs(gimg - rimg) / denom > 1e-3).any(axis=-1).mean()),
        "oracle": "oracle/_ref (compiled reference + counter-RNG shim), product through Raylib_Render / RaylibB200_PrimaryHits",
    }


def main_reference(args):
    import pyraylib as rl
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name = args.workload
    base, info, settings = run_cpu_reference(rl, name, args, native=True, steps=max(1, args.steps), warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": base["value"], "unit": "Mrays/s", "spp_per_s": base["spp_per_s"],
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["seconds"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, name, info, settings),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------------
# B200 arm

def main_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import pyraylib as rl
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a CUDA device (there is no CPU path)")
    torch.cuda.set_device(local_rank)
    if distributed:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    prod = rl.Product()
    prod.require_gpu()
    inprocess_gpus = 1
    if args.inprocess and not distributed:
        inprocess_gpus = int(prod.lib.RaylibB200_SetDevices(args.gpus))     # Raylib_Render spreads frames over these itself
        if inprocess_gpus != args.gpus:
            raise RuntimeError("--inprocess --gpus %d: only %d CUDA devices usable" % (args.gpus, inprocess_gpus))
    else:
        prod.lib.RaylibB200_SetDevice(local_rank)
    prod.lib.Raylib_Initialize()
    name = args.workload
    cfg_id, size, _ = WORKLOADS[name]
    t0 = time.time()
    info = prod.create_demo(cfg_id, args.size or size)
    scene_build_s = time.time() - t0
    settings = workload_settings(rl, info, args)
    W, H = settings.viewportWidth, settings.viewportHeight
    t0 = time.time()
    scene_bytes = int(prod.lib.RaylibB200_SceneDeviceBytes(info.scene))      # flatten + upload (outside the timed region)
    upload_s = time.time() - t0
    counts8 = (C.c_uint64 * 8)()
    prod.lib.RaylibB200_SceneCounts(info.scene, C.byref(counts8))

    stream = torch.cuda.current_stream().cuda_stream
    host_image = torch.empty((H, W, 4), dtype=torch.float32).pin_memory() if rank == 0 else None

    # ---- where the frame lives ----------------------------------------------------------------------
    # peer (default): rank 0 owns ONE row-major frame; the other ranks map it through a CUDA IPC handle and their last
    #   k_accumulate stores the final pixels of their tiles straight into it over NVLink -- no shard buffers, no
    #   collective on the data path, no de-interleave pass; a barrier orders "all ranks done" before the frame is read.
    # nccl: tile-major shard buffer per rank -> dist.gather to rank 0 -> k_assemble.
    gather = args.gather if distributed else "none"
    frame, frame_owned, peer_error = None, False, ""
    if gather == "peer":
        handle = torch.zeros(64, dtype=torch.uint8, device="cuda")
        if rank == 0:
            hbuf = (C.c_ubyte * 64)()
            frame = prod.lib.RaylibB200_FrameCreate(W, H, hbuf)
            if frame:
                frame_owned = True
                handle.copy_(torch.frombuffer(bytearray(bytes(hbuf)), dtype=torch.uint8))
            else:
                peer_error = prod.last_error()
        dist.broadcast(handle, src=0)
        if rank != 0:
            hbuf = (C.c_ubyte * 64).from_buffer_copy(bytes(handle.cpu().numpy().tobytes()))
            frame = prod.lib.RaylibB200_FrameOpen(hbuf)
            if not frame:
                peer_error = prod.last_error()
        ok = torch.tensor([1 if frame else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:          # e.g. no peer access between two devices: say so and use the collective
            sys.stderr.write("bench: rank %d: shared frame unavailable (%s); using the NCCL gather\n" % (rank, peer_error))
            if frame and frame_owned:
                prod.lib.RaylibB200_FrameDestroy(frame)
            elif frame:
                prod.lib.RaylibB200_FrameClose(frame)
            frame, frame_owned, gather = None, False, "nccl"
    if gather == "none":
        image = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
        frame = image.data_ptr()
    if gather == "nccl":
        cap = int(prod.lib.RaylibB200_ShardPixelCapacity(W, H, world))
        shard = torch.empty((cap, 4), dtype=torch.float32, device="cuda")
        gathered = torch.empty((world * cap, 4), dtype=torch.float32, device="cuda") if rank == 0 else None
        image = torch.empty((H, W, 4), dtype=torch.float32, device="cuda") if rank == 0 else None
        frame = image.data_ptr() if rank == 0 else None
    done_flag = torch.zeros(1, dtype=torch.int32, device="cuda")

    def step_device():
        """One frame, result left in HBM on rank 0 (row-major W x H float4). Returns this rank's stats."""
        if gather == "nccl":
            ok = prod.lib.RaylibB200_RenderShard(C.byref(settings), info.scene, info.camera, rank, world, shard.data_ptr(), stream)
        else:
            ok = prod.lib.RaylibB200_RenderShardToFrame(C.byref(settings), info.scene, info.camera, rank, world, frame, stream)
        if not ok:
            raise RuntimeError("RaylibB200_RenderShard* failed: " + prod.last_error())
        st = prod.last_stats()
        if gather == "peer":
            dist.all_reduce(done_flag)           # barrier: every rank's stores into rank 0's frame have completed
        elif gather == "nccl":
            dist.gather(shard, list(gathered.chunk(world)) if rank == 0 else None, dst=0)
            if rank == 0:
                if not prod.lib.RaylibB200_AssembleShards(gathered.data_ptr(), world, W, H, image.data_ptr(), stream):
                    raise RuntimeError("RaylibB200_AssembleShards failed: " + prod.last_error())
        return st

    def timed(fn, steps):
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        stats = [fn() for _ in range(steps)]
        ev1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
        if distributed:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), stats

    # ---- warm-up, then the timed device-resident region ------------------------------------------
    for _ in range(max(args.warmup, 0)):
        step_device()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total_ms, stats = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        last_counts = torch.tensor([stats[-1].rayQueries, stats[-1].pixelSamples], dtype=torch.float64, device="cuda")
        if distributed:
            dist.all_reduce(last_counts, op=dist.ReduceOp.SUM)
    if args.dump_outputs and rank == 0:
        if gather == "peer":
            if not prod.lib.RaylibB200_FrameRead(frame, W, H, host_image.data_ptr(), stream):
                raise RuntimeError("RaylibB200_FrameRead failed: " + prod.last_error())
            torch.cuda.synchronize()
            last_frame = host_image.numpy()
        else:
            last_frame = image.cpu().numpy()
        dump_outputs(args.dump_outputs, last_frame, last_counts.tolist())

    counts = torch.tensor([sum(s.rayQueries for s in stats), sum(s.pixelSamples for s in stats),
                           sum(s.kernelLaunches for s in stats) + (args.steps if (rank == 0 and gather == "nccl") else 0)],
                          dtype=torch.float64, device="cuda")
    if distributed:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    rays, samples, launches = [float(x) for x in counts.tolist()]
    sec = total_ms / 1e3
    value = rays / sec / 1e6

    # ---- end to end through the public API with HOST buffers ----------------------------------------
    if not distributed:
        img_handle = prod.lib.Raylib_CreateImage(W, H)

        def step_e2e():
            prod.lib.Raylib_Render(C.byref(settings), info.scene, info.camera, img_handle)   # kernels + D2H into the Image2D
            err = prod.last_error()
            if err:
                raise RuntimeError("Raylib_Render failed: " + err)
            return prod.last_stats()
        step_e2e()
        e2e_ms, e2e_stats = timed(step_e2e, args.steps)
        e2e_rays = sum(s.rayQueries for s in e2e_stats)
        e2e = {"value": e2e_rays / (e2e_ms / 1e3) / 1e6, "unit": "Mrays/s",
               "h2d_bytes_per_step": int(e2e_stats[-1].h2dBytes), "d2h_bytes_per_step": int(e2e_stats[-1].d2hBytes),
               "ms_per_step": e2e_ms / args.steps, "api": "Raylib_Render(settings, scene, camera, image) into a host Image2D"}
        prod.lib.Raylib_DestroyImage(img_handle)
    else:
        def step_e2e():
            st = step_device()
            if rank == 0:                                       # D2H of the finished frame into pinned host memory
                if not prod.lib.RaylibB200_FrameRead(frame, W, H, host_image.data_ptr(), stream):
                    raise RuntimeError("RaylibB200_FrameRead failed: " + prod.last_error())
            if gather == "peer":
                dist.all_reduce(done_flag)       # frame consumed: the next frame's stores may start
            return st
        step_e2e()
        e2e_ms, e2e_stats = timed(step_e2e, args.steps)
        c2 = torch.tensor([sum(s.rayQueries for s in e2e_stats)], dtype=torch.float64, device="cuda")
        dist.all_reduce(c2, op=dist.ReduceOp.SUM)
        e2e = {"value": float(c2.item()) / (e2e_ms / 1e3) / 1e6, "unit": "Mrays/s",
               "h2d_bytes_per_step": int(e2e_stats[-1].h2dBytes), "d2h_bytes_per_step": int(W * H * 16),
               "ms_per_step": e2e_ms / args.steps,
               "api": ("RaylibB200_RenderShardToFrame per rank into rank 0's frame (CUDA IPC over NVLink) + barrier + D2H of the frame on rank 0"
                       if gather == "peer" else
                       "RaylibB200_RenderShard per rank + NCCL gather + RaylibB200_AssembleShards + D2H of the frame on rank 0")}

    # ---- roofline of the dominant kernel (k_extend) --------------------------------------------------------------
    # The product overlaps two passes on two streams, so inside the region timed above a k_extend launch shares the SMs
    # with stage kernels of the other pass and its event-to-event duration is not the kernel's own.  The per-launch
    # durations are therefore taken on the same frames rendered with ONE pass in flight (kernels run back to back, as
    # under ncu), timed with CUDA events on the launching stream: `args.steps` extra frames of the same workload.
    roofline = None
    prod.lib.RaylibB200_SetPipes(1)
    prod.lib.RaylibB200_SetTimeStages(1)
    step_device()
    single_ms, single_stats = timed(step_device, args.steps)
    prod.lib.RaylibB200_SetTimeStages(0)
    prod.lib.RaylibB200_SetPipes(0)
    if rank == 0:
        extend_ms = sum(s.extendMs for s in single_stats)
        extend_launches = sum(s.extendLaunches for s in single_stats)
        stats_rays = sum(s.rayQueries for s in single_stats)
        prod.lib.RaylibB200_SetCollectStats(1)
        stat_settings = settings.copy(samplesPerPixel=1)
        shard1 = torch.empty((int(prod.lib.RaylibB200_ShardPixelCapacity(W, H, 1)), 4), dtype=torch.float32, device="cuda")
        prod.lib.RaylibB200_RenderShard(C.byref(stat_settings), info.scene, info.camera, 0, 1, shard1.data_ptr(), stream)
        ss = prod.last_stats()
        prod.lib.RaylibB200_SetCollectStats(0)
        del shard1
        n = max(1, ss.statRays)
        n_box, n_tri, n_sph = ss.refBoxTests / n, ss.refTriTests / n, ss.refSphereTests / n
        # (1) SURVEY 8(d): bytes the REFERENCE's exhaustive traversal of the reference tree touches for these rays
        b_ray_reference = 32.0 * n_box + 48.0 * n_tri + 16.0 * n_sph + 64.0
        # (2) bytes the DEVICE traversal has to fetch for the same rays on the tree it walks (record sizes of
        # include/rt_scene_format.h): 64 B per quantized 4-wide node visited, 64 B per triangle tested (RtTriHot),
        # 16 B per sphere, 48 B per cube, 32 B per exact gate box of an accepted hit, 64 B ray in + hit out
        d_node, d_tri, d_sph = ss.nodeVisits / n, ss.triTests / n, ss.sphereTests / n
        d_cube, d_gate = ss.cubeTests / n, ss.gateTests / n
        b_ray_device = 64.0 * d_node + 64.0 * d_tri + 16.0 * d_sph + 48.0 * d_cube + 32.0 * d_gate + 64.0
        # closest-hit rays handled by this rank's k_extend launches in the timed region
        extend_rays = stats_rays * (ss.statRays / max(1, ss.rayQueries))
        peak, peak_src = measured_peak_gbs()
        sec_extend = extend_ms / 1e3
        achieved = (extend_rays * b_ray_device) / sec_extend / 1e9 if extend_ms > 0 else None
        achieved_ref_tree = (extend_rays * b_ray_reference) / sec_extend / 1e9 if extend_ms > 0 else None
        # measured DRAM bytes: ncu dram__bytes_read+write per closest-hit ray (profiles/traffic.json, written by
        # tools/ncu_traffic.py from a capture of this same command) -- only trusted when it was captured on THIS build
        traffic, traffic_src, dram_frac, dram_per_ray, l2_per_ray = None, None, None, None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[name]
            if tj.get("device_source_hash") == rl.device_source_hash():
                dram_per_ray, l2_per_ray = tj["dram_bytes_per_ray"], tj["l2_bytes_per_ray"]
                traffic = dram_per_ray * extend_rays / max(1, extend_launches)
                traffic_src = tj["source"]
                dram_frac = (dram_per_ray * extend_rays) / sec_extend / 1e9 / peak if extend_ms > 0 else None
            else:
                traffic_src = "profiles/traffic.json was captured on another build (device_source_hash %s != %s): not used" % (
                    tj.get("device_source_hash"), rl.device_source_hash())
        except Exception:
            traffic_src = "profiles/traffic.json has no entry for this workload"
        roofline = {
            "bound": "hbm", "kernel": "k_extend (closest-hit BVH traversal)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
            "traffic": traffic, "traffic_source": traffic_src, "dram_frac": dram_frac,
            "dram_bytes_per_ray": dram_per_ray, "l2_bytes_per_ray": l2_per_ray, "peak_source": peak_src,
            "algorithmic_bytes_per_ray": b_ray_device,
            "frac_reference_tree": (achieved_ref_tree / peak) if achieved_ref_tree else None,
            "algorithmic_bytes_per_ray_reference_tree": b_ray_reference, "stat_rays_1spp": int(ss.statRays),
            "reference_tests_per_ray": {"box": n_box, "triangle": n_tri, "sphere": n_sph},
            "device_tests_per_ray": {"box": ss.boxTests / n, "triangle": d_tri, "sphere": d_sph, "cube": d_cube, "gate": d_gate, "nodes": d_node},
            "simd_lanes": {"node_phase_stepping": 32.0 * ss.nodeStep / max(1, ss.nodeIters), "node_phase_owning_a_ray": 32.0 * ss.nodeAlive / max(1, ss.nodeIters),
                           "leaf_phase_testing": 32.0 * ss.leafBusy / max(1, ss.leafIters), "node_iterations_per_ray": ss.nodeIters / 32.0 / n,
                           "leaf_iterations_per_ray": ss.leafIters / 32.0 / n},
            "extend_launches": int(extend_launches), "extend_ms_per_launch": extend_ms / max(1, extend_launches),
            "extend_share_of_step": extend_ms / single_ms if single_ms > 0 else None,
            "single_pipe_ms_per_step": single_ms / args.steps, "pipes_in_timed_region": 2,
            "note": "frac = (closest-hit rays x B_ray_device) / sum of k_extend CUDA-event durations on rank 0 / peak, measured on frames "
                    "with one pass in flight (the headline value overlaps two passes on two streams); B_ray_device = 64*nodes + 64*tris + "
                    "16*spheres + 48*cubes + 32*gates + 64 from the device's own counters on a 1-spp statistics frame: the bytes the "
                    "kernel must FETCH (from L1/L2/HBM); dram_frac = the same with DRAM bytes measured by ncu on this build "
                    "(null when profiles/traffic.json is stale); frac_reference_tree = SURVEY 8(d)'s definition on the reference's "
                    "exhaustive test counts (32*N_box + 48*N_tri + 16*N_sph + 64), a work ratio, not a utilisation",
        }

    # ---- CPU baseline on the host cores (rank 0, N = 1 only) ------------------------------------------------
    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and inprocess_gpus == 1 and not args.no_cpu_baseline and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libraylib_ref.so")):
        try:
            base, _, _ = run_cpu_reference(rl, name, args, native=False,
                                           with_scene=lambda ref, rinfo, nominal: parity_check(rl, prod, info, ref, rinfo, nominal))
            cpu_baseline = {k: base[k] for k in ("value", "unit", "spp_per_s", "cores", "kind", "sample", "seconds")}
            parity = base.get("parity")
        except Exception as exc:    # the baseline is reported, never required
            cpu_baseline = {"unavailable": repr(exc)}

    if rank == 0:
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "spp_per_s": samples / sec,
            "n_gpus": world * inprocess_gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, name, info, settings),
            "build": {
                "parallelism": ("tiles%d in one process (Raylib_Render over all devices)" % inprocess_gpus) if inprocess_gpus > 1 else "tiles%d" % world, "tile": "16x16 interleaved", "collective": {"peer": "none on the data path: final pixels stored straight into rank 0's frame over NVLink (CUDA IPC), then a barrier",
                               "nccl": "nccl gather of shard buffers + de-interleave",
                               "none": "none" if inprocess_gpus == 1 else "none: every device stores its tiles' final pixels straight into the frame on device 0 (peer access over NVLink)"}[gather],
                "scene_device_bytes": scene_bytes, "scene_build_s": scene_build_s, "flatten_upload_s": upload_s,
                "bvh_nodes": int(counts8[0]), "flattened_triangles": int(counts8[1]), "flattened_spheres": int(counts8[2]), "bvh_node_depth": int(counts8[6])},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity,
        }
        emit(line)

    if gather == "peer":
        dist.barrier()
        if frame_owned:
            prod.lib.RaylibB200_FrameDestroy(frame)
        else:
            prod.lib.RaylibB200_FrameClose(frame)
    prod.destroy_demo(info)
    prod.lib.Raylib_Terminate()
    if distributed:
        dist.destroy_process_group()
    return 0


def emit(line):
    """The one JSON line goes to the real stdout; everything else (library log, [STAT] lines) to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    a = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                    # C-level stdout of the libraries (raylib LOG) -> stderr
    sys.exit(main_reference(a) if a.impl == "reference" else main_b200(a))
