"""The denoiser (RaylibB200_Denoise, RaylibB200_DenoiseDevice, RaylibB200_AccumulatorDenoise of include/raylib_b200.h).

The GPU output is held bit for bit to tests/native/denoise_restatement.cc, the filter of DESIGN.md section 14 in plain
C++.  The CPU tests check the restatement's properties (a noise-free image is kept, no weight crosses an orthogonal or
surface/miss edge, a null guide equals its default image) and what the library decides without a device.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NO_DEVICE = "no CUDA device is available"
SIZES = [(1, 1), (3, 2), (17, 9), (200, 120), (333, 77)]       # 333 x 77: wider than the reach of the 16-step taps
GUIDES = ["both", "no-albedo", "no-normal", "none"]
QUALITY = [(2, 0), (5, 40), (4, 24)]


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def rgba(a):
    a = np.asarray(a, dtype=np.float32)
    out = np.ones(a.shape[:2] + (4,), dtype=np.float32)
    out[:, :, :a.shape[2]] = a
    return out


class Restatement:
    def __init__(self, path):
        self.lib = C.CDLL(path)
        f = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
        self.lib.denoise_restated.argtypes = [f, C.c_void_p, C.c_void_p, C.c_int, C.c_int, f]
        self.lib.denoise_sums_restated.argtypes = [f, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int, C.c_int, f]

    @staticmethod
    def _ptr(a):
        return None if a is None else a.ctypes.data

    def denoise(self, color, albedo=None, normal=None):
        """H x W x 3 of the filter on H x W x 3/4 inputs (guides None = null)."""
        color, albedo, normal = [None if a is None else rgba(a) for a in (color, albedo, normal)]
        out = np.empty_like(color)
        self.lib.denoise_restated(color, self._ptr(albedo), self._ptr(normal), color.shape[1], color.shape[0], out)
        return out[:, :, :3]

    def denoise_sums(self, sums, n, albedo=None, normal=None):
        sums = np.ascontiguousarray(sums, dtype=np.float32)
        albedo, normal = [None if a is None else rgba(a) for a in (albedo, normal)]
        out = np.empty_like(sums)
        self.lib.denoise_sums_restated(sums, n, self._ptr(albedo), self._ptr(normal), sums.shape[1], sums.shape[0], out)
        return out[:, :, :3]


@pytest.fixture(scope="module")
def restated(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("denoise") / "libdenoise_restatement.so")
    build = subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "include"),
                            os.path.join(HERE, "native", "denoise_restatement.cc"), "-o", path],
                           capture_output=True, text=True, timeout=300)
    assert build.returncode == 0, build.stderr[-2000:]
    return Restatement(path)


def encode(n):
    n = np.asarray(n, dtype=np.float32)
    return (0.5 + 0.5 * n).astype(np.float32)


def synthetic(seed, width, height):
    """Colour, albedo and encoded normals with misses, zero-albedo channels, fireflies and piecewise-smooth surfaces."""
    rng = np.random.default_rng(seed)
    color = rng.gamma(1.5, 0.4, (height, width, 3)).astype(np.float32)
    color[rng.random((height, width)) < 0.01] *= 50.0
    albedo = rng.uniform(0.0, 1.0, (height, width, 3)).astype(np.float32)
    albedo[rng.random((height, width, 3)) < 0.1] = 0.0
    planes = np.array([[0, 0, 1], [0, 1, 0], [1, 0, 0], [0.6, 0.0, 0.8]], dtype=np.float32)
    region = ((np.arange(width)[None, :] // 7 + np.arange(height)[:, None] // 5) % 4)
    n = planes[region] + rng.normal(0.0, 0.02, (height, width, 3)).astype(np.float32)
    n /= np.linalg.norm(n, axis=2, keepdims=True)
    normal = encode(n)
    normal[rng.random((height, width)) < 0.15] = 0.0
    return color, albedo, normal


def ulps(a, b):
    ia = bits(a).astype(np.int64)
    ib = bits(b).astype(np.int64)
    return np.abs(ia - ib)


# ---- CPU: the restatement ------------------------------------------------------------------------------------------

# Noise-free input c = a * k.  Powers of two k are exact (demodulation gives k, every weighted mean of equal values with
# power-of-two scaling rounds to k, remodulation gives c).  Other k: the standard error bounds of a 25-term weighted mean
# allow ~50 u of relative error per iteration (u = 2^-24), about 254 ulp after demodulation, five iterations and
# remodulation.  The bar below is empirical, not a bound: this seeded sweep of 24 constants measures at most 9 ulp, a wider
# one of 60 constants at most 11 (DESIGN.md §14).
NOISE_FREE_ULPS = 16


def test_noise_free_image_is_kept(restated):
    rng = np.random.default_rng(2024)
    for trial in range(24):
        seed = int(rng.integers(1 << 30))
        k = np.exp(rng.uniform(np.log(0.05), np.log(10.0), 3)).astype(np.float32)
        _, _, normal = synthetic(seed, 61, 37)
        albedo = np.random.default_rng(seed + 1).uniform(0.01, 1.0, normal.shape).astype(np.float32)
        for const, bar in ((k, NOISE_FREE_ULPS), (np.float32(2.0) ** np.round(np.log2(k)), 0)):
            color = (albedo * const).astype(np.float32)
            for guide in (normal, None):
                assert ulps(restated.denoise(color, albedo, guide), color).max() <= bar, (trial, const, guide is None)


@pytest.mark.parametrize("left", ["orthogonal", "miss"])
def test_no_weight_crosses_an_edge(restated, left):
    """Left half facing +x (or missing), right half facing +y: w_n = 0 across the edge, so every output is a weighted
    mean of its own side's inputs and lies in their range."""
    width, height = 48, 30
    rng = np.random.default_rng(11)
    color = np.empty((height, width, 3), dtype=np.float32)
    color[:, :width // 2] = rng.uniform(0.0, 1.0, (height, width // 2, 3))
    color[:, width // 2:] = rng.uniform(5.0, 9.0, (height, width - width // 2, 3))
    normal = np.empty((height, width, 3), dtype=np.float32)
    normal[:, :width // 2] = encode([1, 0, 0]) if left == "orthogonal" else 0.0
    normal[:, width // 2:] = encode([0, 1, 0])
    out = restated.denoise(color, None, normal)
    for side in (np.s_[:, :width // 2], np.s_[:, width // 2:]):
        for c in range(3):
            lo, hi = color[side][:, :, c].min(), color[side][:, :, c].max()
            assert lo <= out[side][:, :, c].min() and out[side][:, :, c].max() <= hi, (side, c)


def test_null_guides_equal_their_defaults(restated):
    color, albedo, normal = synthetic(5, 45, 28)
    ones = np.ones_like(albedo)
    up = np.broadcast_to(encode([0, 0, 1]), normal.shape)
    assert np.array_equal(bits(restated.denoise(color, None, normal)), bits(restated.denoise(color, ones, normal)))
    assert np.array_equal(bits(restated.denoise(color, albedo, None)), bits(restated.denoise(color, albedo, up)))
    sums = np.concatenate([color * 9.0, (color[:, :, :1] ** 2) * 20.0], axis=2).astype(np.float32)
    assert np.array_equal(bits(restated.denoise_sums(sums, 9, None, normal)), bits(restated.denoise_sums(sums, 9, ones, normal)))
    assert np.array_equal(bits(restated.denoise_sums(sums, 9, albedo, None)), bits(restated.denoise_sums(sums, 9, albedo, up)))


# ---- CPU: argument checks of the library -----------------------------------------------------------------------------

def test_argument_errors_are_refused(prod):
    lib = prod.lib
    main = prod.image_from_array(np.ones((6, 8, 3)))
    short = prod.image_from_array(np.ones((5, 8, 3)))
    empty = lib.Raylib_CreateImage(0, 0)
    out = lib.Raylib_CreateImage(1, 1)
    dev = C.c_void_p(0x1000)         # never dereferenced: the checks refuse first
    try:
        cases = [
            (lambda: lib.RaylibB200_Denoise(0, 0, 0, out), "null main or output image"),
            (lambda: lib.RaylibB200_Denoise(main, 0, 0, 0), "null main or output image"),
            (lambda: lib.RaylibB200_Denoise(empty, 0, 0, out), "non-empty"),
            (lambda: lib.RaylibB200_Denoise(main, short, 0, out), "the albedo image is 8x5, the main image is 8x6"),
            (lambda: lib.RaylibB200_Denoise(main, main, short, out), "the normal image is 8x5, the main image is 8x6"),
            (lambda: lib.RaylibB200_DenoiseDevice(None, None, None, 8, 6, dev, None), "null colour or output image"),
            (lambda: lib.RaylibB200_DenoiseDevice(dev, None, None, 8, 6, None, None), "null colour or output image"),
            (lambda: lib.RaylibB200_DenoiseDevice(dev, None, None, 0, 6, dev, None), "non-empty"),
            (lambda: lib.RaylibB200_DenoiseDevice(dev, None, None, 1 << 16, 1 << 15, dev, None), "below 2^31 pixels"),
            (lambda: lib.RaylibB200_DenoiseDevice(C.c_void_p(0x1004), None, None, 8, 6, dev, None), "16-byte aligned"),
            (lambda: lib.RaylibB200_DenoiseDevice(dev, C.c_void_p(0x1008), None, 8, 6, dev, None), "16-byte aligned"),
            (lambda: lib.RaylibB200_DenoiseDevice(dev, None, C.c_void_p(0x1001), 8, 6, dev, None), "16-byte aligned"),
            (lambda: lib.RaylibB200_DenoiseDevice(dev, None, None, 8, 6, C.c_void_p(0x100c), None), "16-byte aligned"),
            (lambda: lib.RaylibB200_AccumulatorDenoise(None, 0, 0, out), "null accumulator or output image"),
        ]
        for call, why in cases:
            assert call() == 0, why
            assert why in prod.last_error(), (why, prod.last_error())
        assert lib.Raylib_Denoise(main, 0, main, main, out) == 0 and lib.Raylib_IsDenoiserSupported() == 0
    finally:
        for h in (main, short, empty, out):
            lib.Raylib_DestroyImage(h)


def test_valid_call_without_a_device(prod):
    """Valid arguments pass every check, then the call fails with the no-device message and leaves `out` as it was."""
    if prod.device_count() > 0:
        pytest.skip("a GPU is visible here")
    lib = prod.lib
    color, albedo, normal = synthetic(1, 8, 6)
    handles = [prod.image_from_array(a) for a in (color, albedo, normal)]
    before = np.arange(3 * 2 * 4, dtype=np.float32).reshape(2, 3, 4)
    out = prod.image_from_array(before)
    dev = C.c_void_p(0x1000)
    try:
        assert lib.RaylibB200_Denoise(*handles, out) == 0 and NO_DEVICE in prod.last_error()
        assert lib.RaylibB200_Denoise(handles[0], 0, 0, out) == 0 and NO_DEVICE in prod.last_error()
        assert lib.RaylibB200_DenoiseDevice(dev, dev, None, 8, 6, dev, None) == 0 and NO_DEVICE in prod.last_error()
        after = np.empty_like(before)
        assert lib.RaylibB200_ImageGetRGBA(out, after) == 1
        assert np.array_equal(bits(after), bits(before))
    finally:
        for h in handles + [out]:
            lib.Raylib_DestroyImage(h)


# ---- GPU ---------------------------------------------------------------------------------------------------------

def guides_of(kind, albedo, normal):
    return (None if kind in ("no-albedo", "none") else albedo, None if kind in ("no-normal", "none") else normal)


@pytest.mark.gpu
@pytest.mark.parametrize("width,height", SIZES)
@pytest.mark.parametrize("guides", GUIDES)
def test_gpu_equals_restatement(gpu, restated, width, height, guides):
    """Device and image forms give the restatement's bits, twice; GetLastStats reports the call."""
    import torch
    color, albedo, normal = synthetic(width * 1000 + height, width, height)
    a, n = guides_of(guides, albedo, normal)
    want = restated.denoise(color, a, n)
    cuda = lambda x: None if x is None else torch.from_numpy(rgba(x)).cuda()
    for _ in range(2):
        got = gpu.denoise_device(cuda(color), cuda(a), cuda(n))
        assert np.array_equal(bits(got), bits(want))
        st = gpu.last_stats()
        assert st.kernelLaunches == 6 and st.rayQueries == 0 and st.h2dBytes == 0 and st.d2hBytes == 0 and st.deviceMs > 0
        got = gpu.denoise(color, a, n)
        assert np.array_equal(bits(got), bits(want))
        st = gpu.last_stats()
        uploads = 1 + (a is not None) + (n is not None)
        assert st.kernelLaunches == 6 and st.rayQueries == 0 and st.pixelSamples == 0
        assert st.h2dBytes == uploads * width * height * 16 and st.d2hBytes == width * height * 16
        assert st.totalMs >= st.deviceMs > 0


def aux(gpu, info, width, height):
    """(albedo, encoded normal) of RaylibB200_RenderAux, H x W x 3."""
    lib = gpu.lib
    ah, nh = lib.Raylib_CreateImage(1, 1), lib.Raylib_CreateImage(1, 1)
    try:
        assert lib.RaylibB200_RenderAux(C.byref(info.settings), info.scene, info.camera, ah, nh) == 1, gpu.last_error()
        return gpu.dump_image(ah, width, height), gpu.dump_image(nh, width, height)
    finally:
        lib.Raylib_DestroyImage(ah)
        lib.Raylib_DestroyImage(nh)


@pytest.mark.gpu
def test_accumulator_form_equals_restatement(gpu, restated):
    """After 2 / 16 / 37 samples: the restatement fed AccumulatorRead's sums, bit for bit; sums and n stay as they were, and
    later installments still resolve to Raylib_Render's bits."""
    from test_progressive import Accumulator, demo
    width, height = 96, 64
    info = demo(gpu, 6, 0, width, height)
    try:
        albedo, normal = aux(gpu, info, width, height)
        with Accumulator.create(gpu, width, height) as acc:
            for guides in ("both", "none"):
                for bad in (0, 1):       # n < 2 is refused
                    if acc.samples < bad:
                        gpu.accumulate(info.settings, info.scene, info.camera, acc.handle, bad - acc.samples)
                    out = gpu.lib.Raylib_CreateImage(1, 1)
                    assert gpu.lib.RaylibB200_AccumulatorDenoise(acc.handle, 0, 0, out) == 0
                    gpu.lib.Raylib_DestroyImage(out)
                    assert "at least 2 samples" in gpu.last_error()
                gpu.lib.RaylibB200_AccumulatorReset(acc.handle)
                for n in (2, 16, 37):
                    gpu.accumulate(info.settings, info.scene, info.camera, acc.handle, n - acc.samples)
                    sums = gpu.accumulator_sums(acc.handle, width, height)
                    a, nrm = guides_of(guides, albedo, normal)
                    got = gpu.accumulator_denoise(acc.handle, width, height, a, nrm)
                    assert np.array_equal(bits(got), bits(restated.denoise_sums(sums, n, a, nrm))), (guides, n)
                    assert gpu.last_stats().kernelLaunches == 6
                    assert acc.samples == n
                    assert np.array_equal(bits(gpu.accumulator_sums(acc.handle, width, height)), bits(sums))
                gpu.accumulate(info.settings, info.scene, info.camera, acc.handle, 3)
                one = gpu.render(info.settings.copy(samplesPerPixel=40), info.scene, info.camera)
                assert np.array_equal(bits(gpu.resolve(acc.handle, width, height)), bits(one))
                gpu.lib.RaylibB200_AccumulatorReset(acc.handle)
            short = gpu.image_from_array(np.ones((height - 1, width, 3)))
            out = gpu.lib.Raylib_CreateImage(1, 1)
            gpu.accumulate(info.settings, info.scene, info.camera, acc.handle, 2)
            assert gpu.lib.RaylibB200_AccumulatorDenoise(acc.handle, 0, short, out) == 0
            assert "the normal image is %dx%d, the accumulator is %dx%d" % (width, height - 1, width, height) in gpu.last_error()
            gpu.lib.Raylib_DestroyImage(short)
            gpu.lib.Raylib_DestroyImage(out)
    finally:
        gpu.destroy_demo(info)


def rel_mse(x, ref):
    x, ref = x.astype(np.float64), ref.astype(np.float64)
    return float(np.mean((x - ref) ** 2 / (ref ** 2 + 1e-2)))


# Measured on a B200 (tools/denoise_bench.py, profiles/denoise_bench.json): the filter's fixed constants miss the bar on
# the textured room, where one firefly dominates the 16-spp error, and on scatter10M, where the image form's spatial
# variance counts real detail as noise and blurs it (a bias that stays at 64 spp).  Strict: a change that meets the bar
# there has to update this list.
QUALITY_MISSES = {
    (5, 40, "image"): "relMSE x1.03 at 16 spp",
    (5, 40, "accumulator"): "relMSE x2.00 (1.9998) at 16 spp",
    (4, 24, "image"): "relMSE x0.12 at 16 spp: over-blurred",
    (4, 24, "accumulator"): "relMSE x1.42 at 16 spp",
}


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,size,form", [
    pytest.param(c, s, f, marks=pytest.mark.xfail(strict=True, reason=QUALITY_MISSES[(c, s, f)]) if (c, s, f) in QUALITY_MISSES else ())
    for c, s in QUALITY for f in ("image", "accumulator")])
def test_denoised_error_is_at_most_half_the_raw(gpu, cfg, size, form):
    """320 x 180 at 16 spp, guides from RenderAux, against 1024 spp at another frame seed: the relative MSE of the denoised
    image is at most half that of the raw one."""
    from test_progressive import Accumulator, demo
    width, height = 320, 180
    info = demo(gpu, cfg, size, width, height)
    try:
        gpu.lib.RaylibB200_SetFrameSeed(99991)
        ref = gpu.render(info.settings.copy(samplesPerPixel=1024), info.scene, info.camera)
        gpu.lib.RaylibB200_SetFrameSeed(1337)
        raw = gpu.render(info.settings.copy(samplesPerPixel=16), info.scene, info.camera)
        albedo, normal = aux(gpu, info, width, height)
        if form == "image":
            denoised = gpu.denoise(raw, albedo, normal)
        else:
            with Accumulator.create(gpu, width, height) as acc:
                gpu.accumulate(info.settings, info.scene, info.camera, acc.handle, 16)
                assert np.array_equal(bits(gpu.resolve(acc.handle, width, height)), bits(raw))
                denoised = gpu.accumulator_denoise(acc.handle, width, height, albedo, normal)
        e_raw, e_den = rel_mse(raw, ref), rel_mse(denoised, ref)
        print("config %d/%d, %s form: relMSE raw %.5f, denoised %.5f (x%.2f)" % (cfg, size, form, e_raw, e_den, e_raw / e_den))
        assert e_den <= 0.5 * e_raw, (e_raw, e_den)
    finally:
        gpu.lib.RaylibB200_SetFrameSeed(1337)
        gpu.destroy_demo(info)
