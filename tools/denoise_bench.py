"""Time and quality of the denoiser (RaylibB200_DenoiseDevice, RaylibB200_Denoise, RaylibB200_AccumulatorDenoise).

    python tools/denoise_bench.py [--quick] [--out FILE]

Time: device-resident Cornell-box inputs (BASELINE config 2: a 16-spp render plus RaylibB200_RenderAux's albedo and normal
views) at 1920x1080 and 3840x2160.  RaylibB200_DenoiseDevice is called warm and bracketed by CUDA events on the stream it
runs on; the median of the timed calls is reported with the algorithmic bytes of one call (from the record sizes: the
prepare kernel reads colour, albedo and normal and writes two records, each a-trous iteration reads two records and writes
one, the last reads the albedo and writes the output) and the bytes per second that gives.  The taps' repeated reads of
the same records are not counted.

Quality: relative MSE, mean of (x - ref)^2 / (ref^2 + 0.01) over pixels and channels, against a 1024-spp render at another
frame seed, of the raw image and of the denoised one (image form and accumulator form), at 4 / 16 / 64 spp, 320x180, on
configs 2, 5 (size 40) and 4 (size 24).

The GPU's name and power limit are read in the same run (nvidia-smi, read-only query).  Writes one JSON document to --out
(default profiles/denoise_bench.json) and prints it.  --quick shrinks every case (a rehearsal, not a measurement).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "software-raytracing_b200"))
import pyraylib as rl  # noqa: E402

REFERENCE_SEED = 99991
FRAME_SEED = 1337
ITERATIONS = 5


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip()
    except OSError as e:
        out = "nvidia-smi unavailable: %s" % e
    return out.splitlines()[0] if out else ""


def algorithmic_bytes(width, height):
    px = width * height
    prepare = px * (3 * 16 + 2 * 16)
    middle = px * (2 * 16 + 16)
    last = px * (2 * 16 + 16 + 16)
    return prepare + (ITERATIONS - 1) * middle + last


def rel_mse(x, ref):
    x, ref = x.astype(np.float64), ref.astype(np.float64)
    return float(np.mean((x - ref) ** 2 / (ref ** 2 + 1e-2)))


def aux(prod, info, width, height):
    lib = prod.lib
    ah, nh = lib.Raylib_CreateImage(1, 1), lib.Raylib_CreateImage(1, 1)
    try:
        if not lib.RaylibB200_RenderAux(C.byref(info.settings), info.scene, info.camera, ah, nh):
            raise RuntimeError("RaylibB200_RenderAux failed: " + prod.last_error())
        return prod.dump_image(ah, width, height), prod.dump_image(nh, width, height)
    finally:
        lib.Raylib_DestroyImage(ah)
        lib.Raylib_DestroyImage(nh)


def demo(prod, cfg, size, width, height):
    info = prod.create_demo(cfg, size)
    prod.set_viewport(info, width, height)
    return info


def timing(prod, width, height, calls, warmup):
    import torch
    info = demo(prod, 2, 0, width, height)
    try:
        color = prod.render(info.settings.copy(samplesPerPixel=16), info.scene, info.camera)
        albedo, normal = aux(prod, info, width, height)
    finally:
        prod.destroy_demo(info)
    dev = lambda a: torch.from_numpy(np.concatenate([a, np.ones(a.shape[:2] + (1,), np.float32)], axis=2)).cuda()
    c, a, n = dev(color), dev(albedo), dev(normal)
    out = torch.empty_like(c)
    stream = torch.cuda.current_stream()
    ptr = lambda t: C.c_void_p(t.data_ptr())
    times, reported = [], []
    for k in range(warmup + calls):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        if not prod.lib.RaylibB200_DenoiseDevice(ptr(c), ptr(a), ptr(n), width, height, ptr(out), C.c_void_p(stream.cuda_stream)):
            raise RuntimeError("RaylibB200_DenoiseDevice failed: " + prod.last_error())
        t1.record(stream)
        t1.synchronize()
        if k >= warmup:
            times.append(t0.elapsed_time(t1))
            reported.append(prod.last_stats().deviceMs)
    ms = float(np.median(times))
    nbytes = algorithmic_bytes(width, height)
    return {"case": "time", "width": width, "height": height, "calls": calls, "warmup": warmup,
            "median_ms": ms, "min_ms": float(np.min(times)), "max_ms": float(np.max(times)),
            "median_stats_device_ms": float(np.median(reported)),
            "algorithmic_bytes": nbytes, "algorithmic_GB_per_s": nbytes / (ms * 1e-3) / 1e9,
            "inputs": "Cornell box (config 2), 16 spp + RenderAux, device-resident RGBA float4; working set %d MB "
                      "(three inputs, three scratch records, the output: 112 B per pixel), larger than the 126 MB L2" % (
                width * height * 112 // (1 << 20))}


def quality(prod, cfg, size, width, height, spps, ref_spp):
    info = demo(prod, cfg, size, width, height)
    rows = []
    try:
        prod.lib.RaylibB200_SetFrameSeed(REFERENCE_SEED)
        ref = prod.render(info.settings.copy(samplesPerPixel=ref_spp), info.scene, info.camera)
        prod.lib.RaylibB200_SetFrameSeed(FRAME_SEED)
        albedo, normal = aux(prod, info, width, height)
        for spp in spps:
            raw = prod.render(info.settings.copy(samplesPerPixel=spp), info.scene, info.camera)
            image = prod.denoise(raw, albedo, normal)
            acc = prod.lib.RaylibB200_AccumulatorCreate(width, height)
            try:
                prod.accumulate(info.settings, info.scene, info.camera, acc, spp)
                accum = prod.accumulator_denoise(acc, width, height, albedo, normal)
            finally:
                prod.lib.RaylibB200_AccumulatorDestroy(acc)
            e_raw, e_img, e_acc = rel_mse(raw, ref), rel_mse(image, ref), rel_mse(accum, ref)
            rows.append({"case": "quality", "config": cfg, "size": size, "width": width, "height": height, "spp": spp,
                         "reference_spp": ref_spp, "relmse_raw": e_raw, "relmse_denoised_image": e_img,
                         "relmse_denoised_accumulator": e_acc, "factor_image": e_raw / e_img, "factor_accumulator": e_raw / e_acc})
    finally:
        prod.lib.RaylibB200_SetFrameSeed(FRAME_SEED)
        prod.destroy_demo(info)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "denoise_bench.json"))
    args = ap.parse_args()
    prod = rl.Product()
    prod.require_gpu()
    prod.lib.Raylib_Initialize()
    doc = {"gpu": gpu_info(), "quick": args.quick, "results": []}
    sizes = [(320, 180)] if args.quick else [(1920, 1080), (3840, 2160)]
    for w, h in sizes:
        doc["results"].append(timing(prod, w, h, calls=3 if args.quick else 25, warmup=1 if args.quick else 5))
        print(json.dumps(doc["results"][-1]), flush=True)
    for cfg, size in ((2, 0), (5, 40), (4, 24)):
        for row in quality(prod, cfg, size, 320, 180, (4,) if args.quick else (4, 16, 64), 64 if args.quick else 1024):
            doc["results"].append(row)
            print(json.dumps(row), flush=True)
    prod.lib.Raylib_Terminate()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
