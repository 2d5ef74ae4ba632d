"""Progressive rendering (RaylibB200_RenderAccumulate and the RaylibB200_Accumulator* calls of include/raylib_b200.h).

A frame rendered in installments resolves to the bits of ONE Raylib_Render at the accumulated sample count: the random
stream of a sample depends only on (seed, pixel, sample index), and the running sums continue the per-pixel float
additions in sample order.  The CPU tests check what the library decides without a device: exports and the
validation of checkpoint files.

Run as a script, this file is the second process of the checkpoint round trip:
    python test_progressive.py resume <checkpoint> <out.npy> <W> <H> <samples> [<flattened-scene file>]
"""
import ctypes as C
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

W, H = 200, 120
SPLITS = [(13,), (1, 12), (5, 8), (1,) * 13, (4, 4, 4, 1)]
NO_DEVICE = "no CUDA device is available"
MASK64 = (1 << 64) - 1


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


class Accumulator:
    """Owns one accumulator handle of `prod` for a with-block."""

    def __init__(self, prod, handle):
        assert handle, prod.last_error()
        self.prod, self.handle = prod, handle

    @classmethod
    def create(cls, prod, width=W, height=H):
        return cls(prod, prod.lib.RaylibB200_AccumulatorCreate(width, height))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.prod.lib.RaylibB200_AccumulatorDestroy(self.handle)

    @property
    def samples(self):
        return int(self.prod.lib.RaylibB200_AccumulatorSamples(self.handle))


def demo(gpu, cfg, size=0, width=W, height=H):
    info = gpu.create_demo(cfg, size)
    gpu.set_viewport(info, width, height)
    return info


def render_in_installments(gpu, info, acc, splits, settings=None):
    """Adds the installments to `acc`; returns their statistics."""
    s = settings or info.settings
    stats = []
    for k in splits:
        gpu.accumulate(s, info.scene, info.camera, acc.handle, k)
        stats.append(gpu.last_stats())
    return stats


# ---- checkpoint files restated (the format of gpu_state.cc: header, binding record, sums, checksum) ----------------

def rt_checksum(h, data):
    """RtChecksum::Add (csrc/host/rt_checksum.h): 8-byte words, zero-padded tail, then the length."""
    def mix(h, w):
        h ^= w
        h = (h * 0xD6E8FEB86659FD93) & MASK64
        return h ^ (h >> 32)
    n = len(data)
    full = n - n % 8
    for w in np.frombuffer(data[:full], dtype="<u8").tolist():
        h = mix(h, w)
    if full < n:
        h = mix(h, int.from_bytes(data[full:] + bytes(8 - (n - full)), "little"))
    return mix(h, n)


def checkpoint_bytes(width, height, samples, sums):
    binding = struct.pack("<IIif Q", width, height, 6, 1e-3, 1337) + bytes(96) + struct.pack("<6f Q", *([0.0] * 6), 0x1234)
    assert len(binding) == 152
    payload = np.ascontiguousarray(sums, dtype=np.float32).tobytes()
    header = lambda checksum: b"RTACCUM1" + struct.pack("<IIIIII Q", 40, 152, width, height, samples, 1, checksum)
    h = 0x9E3779B97F4A7C15
    for part in (header(0), binding, payload):
        h = rt_checksum(h, part)
    return header(h) + binding + payload


def load(prod, path):
    return prod.lib.RaylibB200_AccumulatorLoad(str(path).encode())


# ---- CPU ---------------------------------------------------------------------------------------------------------

def test_damaged_checkpoint_files_are_refused(prod, tmp_path):
    """Empty, garbage, foreign-magic, truncated and bit-flipped files are refused before any device is touched, and the
    message names the file and what is wrong with it."""
    sums = np.arange(4 * 3 * 4, dtype=np.float32).reshape(3, 4, 4)
    good = checkpoint_bytes(4, 3, 3, sums)
    flipped = bytearray(good)
    flipped[40 + 152 + 17] ^= 0x10                      # one bit of the sums
    cases = {
        "empty": (b"", "not an accumulator checkpoint file"),
        "garbage": (os.urandom(4096), "not an accumulator checkpoint file"),
        "magic": (b"RTFLAT01" + good[8:], "not an accumulator checkpoint file"),
        "truncated": (good[:-5], "truncated"),
        "trailing": (good + b"\0", "trailing bytes"),
        "flipped": (bytes(flipped), "corrupt"),
    }
    for name, (data, why) in cases.items():
        path = tmp_path / (name + ".acc")
        path.write_bytes(data)
        assert not load(prod, path), name
        err = prod.last_error()
        assert str(path) in err and why in err, (name, err)
    assert not load(prod, tmp_path / "missing.acc") and "cannot open" in prod.last_error()


def test_valid_checkpoint_needs_a_device_only_after_validation(prod, tmp_path):
    """A valid file passes every check; on a host without a GPU the load then fails with the usual no-device message, on
    a GPU host it yields an accumulator with the stored count and sums."""
    sums = np.random.default_rng(7).random((3, 4, 4), dtype=np.float32)
    path = tmp_path / "ok.acc"
    path.write_bytes(checkpoint_bytes(4, 3, 3, sums))
    handle = load(prod, path)
    if prod.device_count() <= 0:
        assert not handle and NO_DEVICE in prod.last_error()
        return
    with Accumulator(prod, handle) as acc:
        assert acc.samples == 3
        assert np.array_equal(bits(prod.accumulator_sums(acc.handle, 4, 3)), bits(sums))


def test_accumulator_without_a_device(prod):
    if prod.device_count() > 0:
        pytest.skip("a GPU is visible here")
    assert not prod.lib.RaylibB200_AccumulatorCreate(16, 16)
    assert NO_DEVICE in prod.last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("cfg,size", [(6, 0), (2, 0), (5, 40), (7, 0)])
def test_installments_equal_one_shot(gpu, cfg, size):
    """Every split of 13 samples resolves to Raylib_Render at 13 spp, and the raw RGB sums agree bit for bit."""
    info = demo(gpu, cfg, size)
    try:
        s = info.settings.copy(samplesPerPixel=13)
        one = gpu.render(s, info.scene, info.camera)
        first_sums = None
        for splits in SPLITS:
            with Accumulator.create(gpu) as acc:
                stats = render_in_installments(gpu, info, acc, splits)
                assert acc.samples == 13
                assert [st.pixelSamples for st in stats] == [W * H * k for k in splits]
                assert np.array_equal(bits(gpu.resolve(acc.handle, W, H)), bits(one)), (cfg, splits)
                sums = gpu.accumulator_sums(acc.handle, W, H)
                if first_sums is None:
                    first_sums = sums
                assert np.array_equal(bits(sums[:, :, :3]), bits(first_sums[:, :, :3])), (cfg, splits)
    finally:
        gpu.destroy_demo(info)


@pytest.mark.gpu
def test_every_intermediate_resolve_is_exact(gpu):
    info = demo(gpu, 6)
    try:
        with Accumulator.create(gpu) as acc:
            for k in (1, 2, 3, 4, 3):
                render_in_installments(gpu, info, acc, (k,))
                n = acc.samples
                one = gpu.render(info.settings.copy(samplesPerPixel=n), info.scene, info.camera)
                assert np.array_equal(bits(gpu.resolve(acc.handle, W, H)), bits(one)), n
    finally:
        gpu.destroy_demo(info)


@pytest.mark.gpu
def test_scheduling_does_not_change_the_bits(gpu):
    """Pipes, ragged passes (SetSamplesPerPass) and the fused one-launch pass split the installments differently: same
    bits, and the installments' ray queries add up to the one-shot frame's."""
    info = demo(gpu, 6)
    try:
        one = gpu.render(info.settings.copy(samplesPerPixel=13), info.scene, info.camera)
        rays = gpu.last_stats().rayQueries
        for fused, pipes, per_pass in ((1, 1, 0), (1, 2, 0), (1, 4, 0), (1, 1, 3), (1, 2, 3), (1, 4, 3), (2, 1, 0)):
            gpu.lib.RaylibB200_SetFusedPass(fused)
            gpu.lib.RaylibB200_SetPipes(pipes)
            gpu.lib.RaylibB200_SetSamplesPerPass(per_pass)
            with Accumulator.create(gpu) as acc:
                stats = render_in_installments(gpu, info, acc, (5, 8))
                assert sum(st.rayQueries for st in stats) == rays, (fused, pipes, per_pass)
                if fused == 2:
                    assert [st.kernelLaunches for st in stats] == [1, 1]
                else:
                    assert all(st.kernelLaunches > 4 for st in stats)
                if per_pass == 3:
                    assert [st.passes for st in stats] == [2, 3]
                assert np.array_equal(bits(gpu.resolve(acc.handle, W, H)), bits(one)), (fused, pipes, per_pass)
    finally:
        gpu.lib.RaylibB200_SetFusedPass(0)
        gpu.lib.RaylibB200_SetPipes(0)
        gpu.lib.RaylibB200_SetSamplesPerPass(0)
        gpu.destroy_demo(info)


@pytest.mark.gpu
def test_large_frame_in_two_installments(gpu):
    """scatter10M at 1920x1080: each 8-spp installment runs the kernel-per-stage path with two pipes."""
    info = demo(gpu, 4, 0, 1920, 1080)
    try:
        s = info.settings.copy(samplesPerPixel=16)
        one = gpu.render(s, info.scene, info.camera)
        with Accumulator.create(gpu, 1920, 1080) as acc:
            stats = render_in_installments(gpu, info, acc, (8, 8), s)
            assert all(st.passes >= 2 and st.kernelLaunches > 4 for st in stats), [(st.passes, st.kernelLaunches) for st in stats]
            assert np.array_equal(bits(gpu.resolve(acc.handle, 1920, 1080)), bits(one))
    finally:
        gpu.destroy_demo(info)


@pytest.mark.gpu
def test_binding_is_enforced(gpu):
    """An installment that would mix two images is refused, names the differing field and leaves sums and count alone."""
    lib = gpu.lib
    info = demo(gpu, 6)
    other = demo(gpu, 2)
    moved = lib.Raylib_CreateCamera()
    sky = lib.Raylib_CreateImage(8, 4)
    try:
        lib.Raylib_CameraCopy(info.camera, moved)
        lib.Raylib_CameraSetPosition(moved, 0.1, 0.6, 3.2)
        with Accumulator.create(gpu) as acc:
            render_in_installments(gpu, info, acc, (2,))
            before = gpu.accumulator_sums(acc.handle, W, H)

            def refused(field, settings=None, scene=None, camera=None):
                ok = lib.RaylibB200_RenderAccumulate(C.byref(settings or info.settings), scene or info.scene,
                                                     camera or info.camera, acc.handle, 3)
                assert not ok, field
                err = gpu.last_error()
                assert field in err, (field, err)
                assert acc.samples == 2
                assert np.array_equal(bits(gpu.accumulator_sums(acc.handle, W, H)), bits(before)), field
                return err

            refused("camera", camera=moved)
            lib.RaylibB200_SetFrameSeed(1338)
            try:
                refused("frame seed")
            finally:
                lib.RaylibB200_SetFrameSeed(1337)
            refused("maxPathLength", info.settings.copy(maxPathLength=5))
            refused("rayTMin", info.settings.copy(rayTMin=info.settings.rayTMin * 2.0))
            lib.Raylib_SetSunIlluminance(info.scene, 3.0, 3.0, 2.0)
            try:
                refused("sun")
            finally:
                lib.Raylib_SetSunIlluminance(info.scene, 3.0, 3.0, 2.5)
            refused("viewport", info.settings.copy(viewportWidth=W + 16))
            refused("renderMode", info.settings.copy(renderMode=2))
            assert "sun" in refused("scene", scene=other.scene)        # the Cornell box has no sun: both fields are named
            # the binding still accepts the image it was made for
            render_in_installments(gpu, info, acc, (1,))
            assert acc.samples == 3
            before = gpu.accumulator_sums(acc.handle, W, H)
            rgba = np.random.default_rng(3).random((4, 8, 4), dtype=np.float32)
            assert lib.RaylibB200_ImageSetRGBA(sky, 8, 4, rgba)
            lib.Raylib_SetSkyPanorama(info.scene, sky)
            refused_sky = not lib.RaylibB200_RenderAccumulate(C.byref(info.settings), info.scene, info.camera, acc.handle, 3)
            assert refused_sky and "scene" in gpu.last_error(), gpu.last_error()
            assert acc.samples == 3 and np.array_equal(bits(gpu.accumulator_sums(acc.handle, W, H)), bits(before))
            # Reset starts a new image, bound to what the next installment renders
            assert lib.RaylibB200_AccumulatorReset(acc.handle)
            assert acc.samples == 0 and not gpu.accumulator_sums(acc.handle, W, H).any()
            render_in_installments(gpu, info, acc, (1, 2))
            one = gpu.render(info.settings.copy(samplesPerPixel=3), info.scene, info.camera)
            assert np.array_equal(bits(gpu.resolve(acc.handle, W, H)), bits(one))
    finally:
        lib.Raylib_DestroyCamera(moved)
        gpu.destroy_demo(other)
        gpu.destroy_demo(info)
        lib.Raylib_DestroyImage(sky)


def _resume_in_second_process(checkpoint, out, samples, flat=None):
    cmd = [sys.executable, os.path.abspath(__file__), "resume", str(checkpoint), str(out), str(W), str(H), str(samples)]
    if flat:
        cmd.append(str(flat))
    done = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert done.returncode == 0, done.stdout
    return np.load(out)


@pytest.mark.gpu
def test_checkpoint_round_trip(gpu, tmp_path):
    """Save after 5 samples; a second process loads the file, renders 8 more and resolves: the 13-spp frame.  The same
    with the scene read back from its flattened-scene file.  A flipped payload bit and a truncation are refused."""
    info = demo(gpu, 6)
    try:
        one = gpu.render(info.settings.copy(samplesPerPixel=13), info.scene, info.camera)
        ckpt = tmp_path / "five.acc"
        with Accumulator.create(gpu) as acc:
            render_in_installments(gpu, info, acc, (2, 3))
            assert gpu.lib.RaylibB200_AccumulatorSave(acc.handle, str(ckpt).encode()), gpu.last_error()
        flat = tmp_path / "scene6.rtflat"
        assert gpu.lib.RaylibB200_SaveFlattenedScene(info.scene, str(flat).encode()), gpu.last_error()
        for scene_file in (None, flat):
            got = _resume_in_second_process(ckpt, tmp_path / "resumed.npy", 8, scene_file)
            assert np.array_equal(bits(got), bits(one)), scene_file
        data = ckpt.read_bytes()
        flipped = bytearray(data)
        flipped[len(data) // 2] ^= 0x04
        (tmp_path / "flipped.acc").write_bytes(bytes(flipped))
        (tmp_path / "short.acc").write_bytes(data[:-16])
        for name, why in (("flipped.acc", "corrupt"), ("short.acc", "truncated")):
            assert not load(gpu, tmp_path / name)
            assert why in gpu.last_error(), gpu.last_error()
        with Accumulator(gpu, load(gpu, ckpt)) as acc:      # the original still loads here, too
            assert acc.samples == 5
    finally:
        gpu.destroy_demo(info)


def noise_restated(sums, n):
    """The per-pixel figure of RaylibB200_AccumulatorNoise in float32, operation by operation."""
    f = np.float32
    s = sums.astype(np.float32)
    n = f(n)
    lum = (s[..., 0] * f(0.2126) + s[..., 1] * f(0.7152)) + s[..., 2] * f(0.0722)
    m = lum / n
    var = np.maximum(f(0.0), (s[..., 3] - n * m * m) / (n - f(1.0)))
    return np.sqrt(var / n) / np.maximum(m, f(1e-4))


@pytest.mark.gpu
def test_noise_figure(gpu):
    info = demo(gpu, 6)
    try:
        with Accumulator.create(gpu) as acc:
            means = {}
            for k in (16, 48):
                render_in_installments(gpu, info, acc, (k,))
                per_pixel, mean = gpu.noise(acc.handle, W, H)
                expect = noise_restated(gpu.accumulator_sums(acc.handle, W, H), acc.samples)
                np.testing.assert_allclose(per_pixel, expect, rtol=1e-5, atol=1e-7)
                assert mean == pytest.approx(float(np.mean(expect, dtype=np.float64)), rel=1e-6)
                assert gpu.noise(acc.handle, W, H)[1] == mean          # a fixed reduction order: the same double
                means[acc.samples] = mean
            ratio = means[64] / means[16]
            assert 0.35 < ratio < 0.65, means                              # ~ 1 / sqrt(4)
        with Accumulator.create(gpu) as acc:
            render_in_installments(gpu, info, acc, (7, 9))
            _, again = gpu.noise(acc.handle, W, H)
            assert again == means[16]
            gpu.lib.RaylibB200_AccumulatorReset(acc.handle)
            render_in_installments(gpu, info, acc, (1,))
            assert not gpu.lib.RaylibB200_AccumulatorNoise(acc.handle, None, None)
            assert "2 samples" in gpu.last_error()
    finally:
        gpu.destroy_demo(info)


@pytest.mark.gpu
def test_installments_over_several_devices(gpu):
    """12-spp installments on 1, 2 and all GPUs in turn: the bits of the one-device one-shot frame."""
    n = gpu.device_count()
    if n < 2:
        pytest.skip("one CUDA device visible")
    info = demo(gpu, 4, 40, 640, 360)
    try:
        s = info.settings.copy(samplesPerPixel=36, maxPathLength=4)      # 2.76 M pixel-samples per installment
        assert gpu.lib.RaylibB200_SetDevices(1) == 1
        one = gpu.render(s, info.scene, info.camera)
        with Accumulator.create(gpu, 640, 360) as acc:
            for k in (1, 2, n):
                assert gpu.lib.RaylibB200_SetDevices(k) == k
                st = render_in_installments(gpu, info, acc, (12,), s)[0]
                assert st.devicesUsed == k, gpu.last_error()
            assert np.array_equal(bits(gpu.resolve(acc.handle, 640, 360)), bits(one))
    finally:
        gpu.lib.RaylibB200_SetDevice(0)
        gpu.destroy_demo(info)


def _resume(checkpoint, out, width, height, samples, flat=None):
    sys.path.insert(0, os.path.join(ROOT, "software-raytracing_b200"))
    import pyraylib as rl
    prod = rl.Product()
    prod.require_gpu()
    prod.lib.Raylib_Initialize()
    info = prod.create_demo(6)
    prod.set_viewport(info, int(width), int(height))
    scene = info.scene
    if flat:
        scene = prod.lib.RaylibB200_LoadFlattenedScene(flat.encode())
        assert scene, prod.last_error()
    acc = prod.lib.RaylibB200_AccumulatorLoad(checkpoint.encode())
    assert acc, prod.last_error()
    prod.accumulate(info.settings, scene, info.camera, acc, int(samples))
    np.save(out, prod.resolve(acc, int(width), int(height)))
    prod.lib.RaylibB200_AccumulatorDestroy(acc)
    if flat:
        prod.lib.Raylib_DestroyScene(scene)
    prod.destroy_demo(info)
    prod.lib.Raylib_Terminate()
    return 0


if __name__ == "__main__":
    if len(sys.argv) >= 7 and sys.argv[1] == "resume":
        sys.exit(_resume(*sys.argv[2:]))
    sys.exit("usage: test_progressive.py resume <checkpoint> <out.npy> <W> <H> <samples> [<flattened-scene file>]")
