"""Cost of rendering a frame in installments (RaylibB200_RenderAccumulate) against one Raylib_Render of the same samples.

    python tools/progressive_bench.py [--quick] [--out FILE]

Cases, on the first visible GPU:
  * scatter10M (BASELINE config 4) at 3840x2160, 256 spp: one shot, then installments of 64, 16, 4 and 1 spp; every
    installment case must resolve to the one-shot frame's bits (checked here, reported as "bit_identical");
  * Cornell box (config 2) at 1920x1080 in 1-spp installments: preview latency per installment;
  * the resolve of a 4K accumulator (into device memory and into an Image2D on the host).
Device time is the sum of the CUDA-event times the library reports per call (GetLastStats.deviceMs); wall time is the
host clock around the calls, which all return after their device work (one shot: render + read-back into an Image2D;
wall_overhead sets the installments plus one resolve into an Image2D against that).  One JSON object per line on
stdout (and in --out); the first line names the GPU and its power limit (nvidia-smi, read-only query).  --quick shrinks
every case (a rehearsal of the script, not a measurement).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "software-raytracing_b200"))
import pyraylib as rl  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip()
    except OSError as e:
        out = "nvidia-smi unavailable: %s" % e
    return out.splitlines()[0] if out else ""


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


class Bench:
    def __init__(self, out):
        self.prod = rl.Product()
        self.prod.require_gpu()
        self.prod.lib.Raylib_Initialize()
        self.out = out

    def emit(self, record):
        line = json.dumps(record, sort_keys=True)
        print(line, flush=True)
        if self.out:
            self.out.write(line + "\n")
            self.out.flush()

    def one_shot(self, info, spp):
        t0 = time.perf_counter()
        img = self.prod.render(info.settings.copy(samplesPerPixel=spp), info.scene, info.camera)
        wall = (time.perf_counter() - t0) * 1e3
        st = self.prod.last_stats()
        return img, st, wall

    def installments(self, info, width, height, spp, chunk):
        """Renders spp samples in installments of `chunk`; -> (accumulator, per-installment device ms, wall ms, rays)."""
        lib = self.prod.lib
        acc = lib.RaylibB200_AccumulatorCreate(width, height)
        if not acc:
            raise RuntimeError("AccumulatorCreate failed: " + self.prod.last_error())
        device_ms, rays = [], 0
        t0 = time.perf_counter()
        for _ in range(spp // chunk):
            self.prod.accumulate(info.settings, info.scene, info.camera, acc, chunk)
            st = self.prod.last_stats()
            device_ms.append(st.deviceMs)
            rays += st.rayQueries
        wall = (time.perf_counter() - t0) * 1e3
        return acc, device_ms, wall, rays

    def scatter(self, quick):
        width, height, spp = (960, 540, 16) if quick else (3840, 2160, 256)
        chunks = (4, 1) if quick else (64, 16, 4, 1)
        info = self.prod.create_demo(4, 0)
        try:
            self.prod.set_viewport(info, width, height)
            self.one_shot(info, 1)                                  # scene upload, arenas, module load
            one, st, one_wall = self.one_shot(info, spp)
            base = {"case": "scatter10M", "width": width, "height": height, "spp": spp}
            self.emit(dict(base, mode="one_shot", device_ms=st.deviceMs, wall_ms=one_wall, ray_queries=st.rayQueries,
                           mrays_per_s=st.rayQueries / st.deviceMs * 1e-3, passes=st.passes))
            for chunk in chunks:
                acc, device_ms, wall, rays = self.installments(info, width, height, spp, chunk)
                try:
                    t0 = time.perf_counter()
                    img = self.prod.resolve(acc, width, height)
                    resolve_ms = (time.perf_counter() - t0) * 1e3
                    dev = sum(device_ms)
                    self.emit(dict(base, mode="installments", chunk=chunk, installments=len(device_ms), device_ms=dev,
                                   wall_ms=wall, ray_queries=rays, mrays_per_s=rays / dev * 1e-3,
                                   device_overhead=dev / st.deviceMs - 1.0, wall_overhead=(wall + resolve_ms) / one_wall - 1.0,
                                   per_installment_device_ms=float(np.median(device_ms)), resolve_to_host_ms=resolve_ms,
                                   bit_identical=bool(np.array_equal(bits(img), bits(one)))))
                finally:
                    self.prod.lib.RaylibB200_AccumulatorDestroy(acc)
        finally:
            self.prod.destroy_demo(info)

    def cornell_preview(self, quick):
        width, height, count = (480, 270, 8) if quick else (1920, 1080, 64)
        info = self.prod.create_demo(2, 0)
        try:
            self.prod.set_viewport(info, width, height)
            self.one_shot(info, 1)
            acc, device_ms, wall, rays = self.installments(info, width, height, count, 1)
            try:
                t0 = time.perf_counter()
                img = self.prod.resolve(acc, width, height)
                resolve_ms = (time.perf_counter() - t0) * 1e3
                one, st, _ = self.one_shot(info, count)
                self.emit({"case": "cornell_preview", "width": width, "height": height, "chunk": 1, "installments": count,
                           "first_installment_device_ms": device_ms[0], "median_installment_device_ms": float(np.median(device_ms)),
                           "median_installment_wall_ms": wall / count, "resolve_to_host_ms": resolve_ms,
                           "one_shot_device_ms": st.deviceMs, "installments_device_ms": sum(device_ms),
                           "bit_identical": bool(np.array_equal(bits(img), bits(one)))})
            finally:
                self.prod.lib.RaylibB200_AccumulatorDestroy(acc)
        finally:
            self.prod.destroy_demo(info)

    def resolve_4k(self, quick):
        width, height, reps = (960, 540, 5) if quick else (3840, 2160, 20)
        lib = self.prod.lib
        info = self.prod.create_demo(2, 0)
        acc = lib.RaylibB200_AccumulatorCreate(width, height)
        frame = lib.RaylibB200_FrameCreate(width, height, None)
        img = lib.Raylib_CreateImage(width, height)
        try:
            self.prod.set_viewport(info, width, height)
            self.prod.accumulate(info.settings, info.scene, info.camera, acc, 2)
            times = {"device": [], "host": [], "noise": []}
            mean = C.c_double()
            for _ in range(reps + 2):
                t0 = time.perf_counter()
                assert lib.RaylibB200_AccumulatorResolveDevice(acc, frame, None), self.prod.last_error()
                t1 = time.perf_counter()
                assert lib.RaylibB200_AccumulatorResolve(acc, img), self.prod.last_error()
                t2 = time.perf_counter()
                assert lib.RaylibB200_AccumulatorNoise(acc, None, C.byref(mean)), self.prod.last_error()
                t3 = time.perf_counter()
                for k, v in (("device", t1 - t0), ("host", t2 - t1), ("noise", t3 - t2)):
                    times[k].append(v * 1e3)
            med = {k: float(np.median(v[2:])) for k, v in times.items()}
            self.emit({"case": "resolve", "width": width, "height": height, "reps": reps,
                       "resolve_device_wall_ms": med["device"], "resolve_to_host_wall_ms": med["host"],
                       "noise_mean_wall_ms": med["noise"],
                       "resolve_device_gb_per_s": width * height * 32 / (med["device"] * 1e-3) / 1e9})
        finally:
            lib.Raylib_DestroyImage(img)
            lib.RaylibB200_FrameDestroy(frame)
            lib.RaylibB200_AccumulatorDestroy(acc)
            self.prod.destroy_demo(info)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="small sizes: rehearse the script")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--cases", default="scatter,cornell,resolve")
    args = ap.parse_args()
    out = open(args.out, "a") if args.out else None
    bench = Bench(out)
    bench.emit({"gpu": gpu_info(), "quick": args.quick})
    cases = args.cases.split(",")
    if "scatter" in cases:
        bench.scatter(args.quick)
    if "cornell" in cases:
        bench.cornell_preview(args.quick)
    if "resolve" in cases:
        bench.resolve_4k(args.quick)
    bench.prod.lib.Raylib_Terminate()


if __name__ == "__main__":
    main()
