"""GPU parity tests: every call goes through the C ABI of libraylib_b200.so (pyraylib is a ctypes shim).

Oracle = tests/golden (vectors generated from the compiled reference), the C restatement (oracle/rt_oracle.c, pinned to
those vectors) for primary hits and traced rays, and tests/golden/recorded for the outputs the compiled reference is no
longer at hand to produce (see conftest.RecordedOutputs).

Bars (north star):
  * primary rays: hit primitive ids identical to the reference; t bit-identical when the lens is a pinhole
    (aperture 0).  With a finite aperture the lens offset goes through cosf/sinf, which differ from glibc by
    <= 2 ulp on the device, so t may differ in the last bits there: ids must still match for >= 99.9 % of pixels.
  * radiance at matched spp and seed: BIT-IDENTICAL pixels.  Round 1 allowed PSNR >= 40 dB because the device's
    sinf/cosf/powf/... differed from glibc's by 1-2 ulp, which specular chains amplify; since round 2 the shaders call
    include/rt_libm.h, glibc's algorithms restated bit for bit, and every comparison below comes out 100 % identical on
    the GPU box (profiles/r02c_tests.log).  The asserted floor is 99.9 % of the pixels (EXACT_FLOOR): glibc picks its
    non-FMA build on a host CPU without FMA, whose results differ from the restated FMA build about once in 5e8 calls.
  * debug views: bit-identical (pinhole cameras); finite apertures move a handful of silhouette pixels.
"""
import ctypes as C
import numpy as np
import pytest
from conftest import load_golden, bits

pytestmark = pytest.mark.gpu
CONFIGS = [1, 2, 3, 4, 5, 6]
PINHOLE = {2, 3, 4, 5}          # configs whose camera has aperture 0


EXACT_FLOOR = 0.999       # fraction of bit-identical radiance pixels asserted against the compiled reference / golden vectors


def rel_outliers(img, ref, rel=1e-3, absolute=1e-3):
    d = np.abs(img.astype(np.float64) - ref.astype(np.float64))
    return float((d > rel * np.abs(ref) + absolute).any(axis=2).mean())


@pytest.mark.parametrize("cfg", CONFIGS)
def test_primary_hits_match_golden(gpu, rl, cfg):
    g = load_golden(cfg)
    w, h = [int(x) for x in g["primary_wh"]]
    info = gpu.create_demo(cfg, int(g["size"]))
    try:
        gpu.set_viewport(info, w, h)
        rank, t = gpu.primary_hits(info.settings, info.scene, info.camera)           # device ray generation
        id_match = float((rank == g["rank"]).mean())
        t_match = float((bits(t) == bits(g["t"])).mean())
        print("config%d primary: id match %.6f, t bit match %.6f" % (cfg, id_match, t_match))
        if cfg in PINHOLE:
            assert id_match == 1.0 and t_match == 1.0
        else:
            assert id_match >= 0.999
            # the r=1000 ground sphere amplifies a 1-ulp lens offset through b*b - a*c; ids are the contract here
            assert np.allclose(t[rank == g["rank"]], g["t"][rank == g["rank"]], rtol=5e-3, atol=1e-4)
        # the reference's own rays through the device traversal: exact, whatever the lens
        rank2, t2 = gpu.trace_rays(info.scene, g["rays"], info.settings.rayTMin)
        assert np.array_equal(rank2, g["rank"]), "mismatch rate %.2e" % float((rank2 != g["rank"]).mean())
        assert np.array_equal(bits(t2), bits(g["t"]))
    finally:
        gpu.destroy_demo(info)


@pytest.mark.parametrize("cfg", CONFIGS)
def test_radiance_matches_golden(gpu, rl, cfg):
    g = load_golden(cfg)
    rw, rh, spp = [int(x) for x in g["radiance_whs"]]
    info = gpu.create_demo(cfg, int(g["size"]))
    try:
        gpu.set_viewport(info, rw, rh)
        img = gpu.render(info.settings.copy(samplesPerPixel=spp), info.scene, info.camera)
        st = gpu.last_stats()
        refimg = g["radiance"]
        psnr = rl.psnr(img, refimg)
        out = rel_outliers(img, refimg)
        exact = float((bits(img) == bits(refimg)).all(axis=2).mean())
        print("config%d radiance: PSNR %.2f dB, outliers %.4f, bit-identical pixels %.4f, rays %d vs %d"
              % (cfg, psnr, out, exact, st.rayQueries, int(g["ray_queries"])))
        assert np.isfinite(img).all() == np.isfinite(refimg).all()
        assert psnr >= 40.0
        assert out <= 0.02
        assert exact >= EXACT_FLOOR, "radiance is no longer bit-identical to the reference (config%d: %.6f)" % (cfg, exact)
        assert abs(int(st.rayQueries) - int(g["ray_queries"])) <= 0.002 * int(g["ray_queries"]) + 8
        if cfg in (2, 3):
            assert exact >= 0.95
    finally:
        gpu.destroy_demo(info)


@pytest.mark.parametrize("cfg", CONFIGS)
def test_debug_views_match_golden(gpu, cfg):
    g = load_golden(cfg)
    rw, rh, _ = [int(x) for x in g["radiance_whs"]]
    info = gpu.create_demo(cfg, int(g["size"]))
    try:
        gpu.set_viewport(info, rw, rh)
        for mode in (1, 2, 4, 5):
            img = gpu.render(info.settings.copy(renderMode=mode), info.scene, info.camera)
            want = g["mode%d" % mode]
            exact = float((bits(img) == bits(want)).all(axis=2).mean())
            if cfg in PINHOLE and mode != 4:
                assert exact == 1.0, "mode %d: %.6f" % (mode, exact)
            else:
                # finite aperture: a 1-ulp lens difference moves a handful of silhouette pixels onto another primitive;
                # sphere UVs go through atanf/acosf; Cube::Hit leaves paramU/V uninitialised in the reference (cube.cc:25-39)
                close = np.isclose(img, want, rtol=1e-4, atol=2e-3).all(axis=2).mean()
                assert exact >= 0.85 and close >= 0.98, "mode %d: exact %.6f close %.6f" % (mode, exact, close)
    finally:
        gpu.destroy_demo(info)


def restated_primary(gpu, restate, info, seed=1337, scene=None):
    """Primary hits (rank, t) and camera rays of the C restatement (oracle/rt_oracle.c) for a demo scene's camera.  On the
    golden inputs its rays, ids and t are the compiled reference's bit for bit (tests/test_cpu_oracle.py); on other
    inputs it is an independent exhaustive implementation, and the device must trace the same rays to the same hits."""
    s = info.settings
    rank, t, _, rays = restate.primary(gpu.flat_desc(scene or info.scene), gpu.camera_block(info.camera), s.viewportWidth,
                                       s.viewportHeight, s.rayTMin, seed=seed, want_rays=True)
    return rank, t, rays


def test_against_compiled_reference_fresh_inputs(gpu, recorded, restate, rl):
    """Sizes/seeds that are NOT in the golden set: camera rays through the device traversal against the C restatement,
    radiance against the stored outputs (conftest.RecordedOutputs)."""
    for cfg, size, (w, h), spp, seed in [(3, 96, (200, 120), 3, 99), (4, 40, (128, 128), 2, 7), (6, 0, (111, 77), 5, 2024)]:
        pinfo = gpu.create_demo(cfg, size)
        key = "config%d_" % cfg
        try:
            gpu.set_viewport(pinfo, w, h)
            gpu.lib.RaylibB200_SetFrameSeed(seed)
            rr, rt, rays = restated_primary(gpu, restate, pinfo, seed)
            gr, gt = gpu.trace_rays(pinfo.scene, rays, pinfo.settings.rayTMin)
            assert np.array_equal(gr, rr) and np.array_equal(bits(gt), bits(rt))
            gimg = gpu.render(pinfo.settings.copy(samplesPerPixel=spp), pinfo.scene, pinfo.camera)
            g, r, _ = recorded.compare(key + "radiance", gimg)
            assert rl.psnr(g, r) >= 40.0 and rel_outliers(g, r) <= 0.02
            assert float((bits(g) == bits(r)).all(axis=2).mean()) >= EXACT_FLOOR
        finally:
            gpu.lib.RaylibB200_SetFrameSeed(1337)
            gpu.destroy_demo(pinfo)


def test_incoherent_rays_against_restatement(gpu, restate):
    """Random rays inside the 30k-triangle scatter: device traversal (pruned, near-first) vs the exhaustive C restatement."""
    info = gpu.create_demo(4, 24)
    try:
        rng = np.random.default_rng(5)
        n = 200000
        rays = np.zeros((n, 8), dtype=np.float32)
        rays[:, 0:3] = rng.uniform([-4, 0.01, -4], [4, 2.0, 4], size=(n, 3))
        v = rng.normal(size=(n, 3)); rays[:, 4:7] = v / np.linalg.norm(v, axis=1, keepdims=True)
        rays[:64, 4:7] = [0.0, -1.0, 0.0]
        grank, gt = gpu.trace_rays(info.scene, rays, 1e-4)
        crank, ct, _ = restate.trace(gpu.flat_desc(info.scene), rays, 1e-4)
        mismatch = float((grank != crank).mean())
        print("incoherent rays: id mismatch rate %.3e" % mismatch)
        assert mismatch <= 1e-5, "epsilon-tie budget exceeded"
        same = grank == crank
        assert np.array_equal(bits(gt[same]), bits(ct[same]))
    finally:
        gpu.destroy_demo(info)


def test_reference_work_counters_match_oracle(gpu):
    """The statistics build's 'reference work' counters (roofline accounting) equal the oracle's exhaustive counts."""
    for cfg in (1, 3, 4, 6):
        g = load_golden(cfg)
        info = gpu.create_demo(cfg, int(g["size"]))
        try:
            # plain uploads leave the reference topology on the host: without statistics the counters stay zero ...
            gpu.lib.RaylibB200_SetDevice(-1)                # a refused call leaves a message; a successful query clears it
            gpu.trace_rays(info.scene, g["rays"], info.settings.rayTMin)
            assert gpu.last_stats().refBoxTests == 0 and gpu.last_error() == ""
            # ... and asking for statistics uploads the scene again, with it
            gpu.lib.RaylibB200_SetCollectStats(1)
            gpu.trace_rays(info.scene, g["rays"], info.settings.rayTMin)
            gpu.lib.RaylibB200_SetCollectStats(0)
            st = gpu.last_stats()
            box, tri, sph, rays = [int(x) for x in g["ref_tests"]]
            assert (st.refBoxTests, st.refTriTests, st.refSphereTests, st.statRays) == (box, tri, sph, rays)
            assert st.boxTests <= 2 * box and st.triTests <= tri       # the device traversal prunes
        finally:
            gpu.destroy_demo(info)


def test_full_size_properties(gpu):
    """BASELINE-size frames: determinism, shard-count independence, energy bounds, ray accounting."""
    import torch
    info = gpu.create_demo(3, 0)            # 1,002,528 triangles, 1920x1080
    try:
        s = info.settings.copy(samplesPerPixel=2)
        a = gpu.render(s, info.scene, info.camera)
        st = gpu.last_stats()
        b = gpu.render(s, info.scene, info.camera)
        assert np.array_equal(bits(a), bits(b)), "same seed must give the same bits"
        assert np.isfinite(a).all() and a.min() >= 0.0 and a.max() <= 1.0 + 1e-6     # white sky, albedo 1, AO in [0,1]
        W, H = s.viewportWidth, s.viewportHeight
        assert st.pixelSamples == W * H * 2
        assert W * H * 2 <= st.rayQueries <= W * H * 2 * 2                          # depth 2: at most one bounce ray per sample
        # 1 shard vs 3 shards vs 8 shards: bit-identical frames (RNG is keyed on global pixel coordinates)
        for shards in (3, 8):
            cap = int(gpu.lib.RaylibB200_ShardPixelCapacity(W, H, shards))
            slabs = torch.zeros((shards * cap, 4), dtype=torch.float32, device="cuda")
            for r in range(shards):
                view = slabs[r * cap:(r + 1) * cap]
                assert gpu.lib.RaylibB200_RenderShard(C.byref(s), info.scene, info.camera, r, shards, view.data_ptr(), None), gpu.last_error()
            image = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
            assert gpu.lib.RaylibB200_AssembleShards(slabs.data_ptr(), shards, W, H, image.data_ptr(), None)
            assert np.array_equal(bits(image.cpu().numpy()[:, :, :3]), bits(a)), "%d shards differ from 1" % shards
        # primary visibility at full size: SurfaceNormal view has unit-length decoded normals wherever something was hit
        n = gpu.render(info.settings.copy(renderMode=2), info.scene, info.camera)
        hit = (n != 0).any(axis=2)
        ln = np.linalg.norm(2.0 * n[hit] - 1.0, axis=1)
        assert hit.mean() > 0.3 and np.allclose(ln, 1.0, atol=1e-5)
    finally:
        gpu.destroy_demo(info)


def test_edge_cases(gpu):
    info = gpu.create_demo(6)
    try:
        base = info.settings
        # spp <= 0 renders one sample (renderer.cc:224), depth 0 renders black (renderer.cc:120-123)
        gpu.set_viewport(info, 33, 17)        # not a multiple of the 16x16 tile
        one = gpu.render(base.copy(samplesPerPixel=1), info.scene, info.camera)
        zero = gpu.render(base.copy(samplesPerPixel=0), info.scene, info.camera)
        neg = gpu.render(base.copy(samplesPerPixel=-3), info.scene, info.camera)
        assert np.array_equal(bits(one), bits(zero)) and np.array_equal(bits(one), bits(neg))
        black = gpu.render(base.copy(maxPathLength=0), info.scene, info.camera)
        assert (black == 0).all()
        gpu.set_viewport(info, 1, 1)
        px = gpu.render(base, info.scene, info.camera)
        assert px.shape == (1, 1, 3) and np.isfinite(px).all()
        # image handle of the wrong size is resized (renderer.cc:292-296)
        gpu.set_viewport(info, 40, 24)
        img = gpu.lib.Raylib_CreateImage(3, 3)
        gpu.lib.Raylib_Render(C.byref(info.settings), info.scene, info.camera, img)
        assert gpu.last_error() == ""
        assert gpu.dump_image(img, 40, 24).shape == (24, 40, 3)
        gpu.lib.Raylib_DestroyImage(img)
        # many samples per pass vs one sample per pass: same bits (ordered accumulation)
        gpu.lib.RaylibB200_SetSamplesPerPass(1)
        a = gpu.render(base.copy(samplesPerPixel=7), info.scene, info.camera)
        gpu.lib.RaylibB200_SetSamplesPerPass(3)
        b = gpu.render(base.copy(samplesPerPixel=7), info.scene, info.camera)
        gpu.lib.RaylibB200_SetSamplesPerPass(0)
        c = gpu.render(base.copy(samplesPerPixel=7), info.scene, info.camera)
        assert np.array_equal(bits(a), bits(b)) and np.array_equal(bits(a), bits(c))
    finally:
        gpu.destroy_demo(info)


def test_errors_do_not_crash(gpu):
    lib = gpu.lib
    scene = lib.Raylib_CreateScene()
    cam = lib.Raylib_CreateCamera()
    img = lib.Raylib_CreateImage(8, 8)
    s = gpu.create_demo(6)
    try:
        lib.Raylib_Render(C.byref(s.settings), scene, cam, img)        # not finalized
        assert "not finalized" in gpu.last_error()
        lib.Raylib_FinalizeScene(scene)
        lib.Raylib_Render(C.byref(s.settings), scene, cam, img)        # finalized but empty
        assert "no elements" in gpu.last_error()
    finally:
        gpu.destroy_demo(s)
        lib.Raylib_DestroyImage(img); lib.Raylib_DestroyCamera(cam); lib.Raylib_DestroyScene(scene)


def test_aux_buffers_one_pass_equals_two_renders(gpu):
    """SURVEY 8(f) rank 2: Albedo + MicrosurfaceNormal from one primary-hit pass == the two separate debug renders."""
    for cfg in (5, 6):
        info = gpu.create_demo(cfg, 40 if cfg == 5 else 0)
        try:
            gpu.set_viewport(info, 320, 180)
            albedo = gpu.render(info.settings.copy(renderMode=1), info.scene, info.camera)
            normal = gpu.render(info.settings.copy(renderMode=3), info.scene, info.camera)
            rays_separate = 0
            a_img = gpu.lib.Raylib_CreateImage(8, 8)          # wrong size on purpose: the call resizes
            n_img = gpu.lib.Raylib_CreateImage(8, 8)
            try:
                assert gpu.lib.RaylibB200_RenderAux(C.byref(info.settings), info.scene, info.camera, a_img, n_img), gpu.last_error()
                st = gpu.last_stats()
                a2 = gpu.dump_image(a_img, 320, 180)
                n2 = gpu.dump_image(n_img, 320, 180)
            finally:
                gpu.lib.Raylib_DestroyImage(a_img); gpu.lib.Raylib_DestroyImage(n_img)
            assert np.array_equal(bits(a2), bits(albedo)), "config%d: fused albedo differs" % cfg
            assert np.array_equal(bits(n2), bits(normal)), "config%d: fused normal differs" % cfg
            assert st.rayQueries >= 320 * 180 and st.kernelLaunches >= 1
        finally:
            gpu.destroy_demo(info)


def test_gpu_postprocess_matches_host_postprocess(gpu):
    """SURVEY 8(f) rank 3: Image2D::PostProcess as CUDA kernels vs the host implementation (image.cc:44-103)."""
    import torch
    info = gpu.create_demo(2, 0)            # Cornell box: the light (15) is far above white
    try:
        gpu.set_viewport(info, 320, 180)
        s = info.settings.copy(samplesPerPixel=4)
        W, H = 320, 180
        host_img = gpu.lib.Raylib_CreateImage(W, H)
        gpu_img = gpu.lib.Raylib_CreateImage(W, H)
        try:
            gpu.lib.Raylib_Render(C.byref(s), info.scene, info.camera, host_img)
            gpu.lib.Raylib_Render(C.byref(s), info.scene, info.camera, gpu_img)
            raw = gpu.dump_image(host_img, W, H)
            gpu.lib.Raylib_PostProcess(host_img)
            assert gpu.lib.RaylibB200_PostProcessGPU(gpu_img), gpu.last_error()
            ref = gpu.dump_image(host_img, W, H)
            out = gpu.dump_image(gpu_img, W, H)
        finally:
            gpu.lib.Raylib_DestroyImage(host_img); gpu.lib.Raylib_DestroyImage(gpu_img)
        assert raw.max() > 1.0, "the test frame must exercise the max-white reduction"
        assert 0.0 <= out.min() and out.max() <= 1.0
        # identical arithmetic except powf (device libm vs glibc, <= 2 ulp)
        assert np.allclose(out, ref, rtol=2e-6, atol=1e-7), float(np.abs(out - ref).max())
        # device-resident form with the packed 8-bit output
        dev = torch.ones((H, W, 4), dtype=torch.float32, device="cuda")
        dev[:, :, :3] = torch.from_numpy(raw).cuda()
        packed = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        mw = C.c_float(0.0)
        assert gpu.lib.RaylibB200_PostProcessDevice(dev.data_ptr(), W, H, packed.data_ptr(), C.byref(mw), None), gpu.last_error()
        lum = raw[..., 0] * np.float32(0.2126) + raw[..., 1] * np.float32(0.7152) + raw[..., 2] * np.float32(0.0722)
        assert abs(mw.value - max(1.0, float(lum.max()))) <= 1e-5 * mw.value
        d = dev.cpu().numpy()
        assert np.allclose(d[:, :, :3], ref, rtol=2e-6, atol=1e-7)
        p = packed.cpu().numpy().view(np.uint32)
        expect = ((np.uint32(255) << 24) | ((d[..., 0] * 255.0).astype(np.uint32) << 16) | ((d[..., 1] * 255.0).astype(np.uint32) << 8)
                  | (d[..., 2] * 255.0).astype(np.uint32))
        assert np.array_equal(p, expect)
    finally:
        gpu.destroy_demo(info)


def test_obj_model_renders(gpu, rl, tmp_path):
    """Raylib_LoadOBJModel -> scene -> Raylib_Render through the reference C ABI only (src/main.cc:597-640 style)."""
    from test_cpu_host import OBJ_TEXT, MTL_TEXT, _write_png
    (tmp_path / "scene.obj").write_text(OBJ_TEXT)
    (tmp_path / "scene.mtl").write_text(MTL_TEXT)
    _write_png(str(tmp_path / "tiles.png"), np.full((4, 4, 4), 200, dtype=np.uint8))
    lib = gpu.lib
    model = lib.Raylib_LoadOBJModel(str(tmp_path / "scene.obj").encode())
    assert model
    lib.Raylib_FinalizeOBJModel(model)
    scene = lib.Raylib_CreateScene()
    lib.Raylib_AddOBJModelToScene(scene, model)
    lib.Raylib_SetSunIlluminance(scene, 5.0, 5.0, 5.0)
    lib.Raylib_SetSunDirection(scene, 0.0, -1.0, -0.3)
    lib.Raylib_FinalizeScene(scene)
    cam = lib.Raylib_CreateCamera()
    lib.Raylib_CameraSetPosition(cam, 0.0, 1.5, 3.0)
    lib.Raylib_CameraSetLookAt(cam, 0.0, 0.2, 0.0)
    lib.Raylib_CameraSetPerspective(cam, 60.0, 160.0 / 90.0)
    lib.Raylib_CameraSetLens(cam, 0.0, 3.0)
    lib.Raylib_CameraSetMotion(cam, 0.0, 0.0)
    s = rl.RendererSettings(160, 90, 8, 4, 1e-4, 0)
    img = gpu.render(s, scene, cam)
    normal = gpu.render(s.copy(renderMode=2), scene, cam)
    assert np.isfinite(img).all() and img.max() > 0.0
    hit = (normal != 0).any(axis=2)
    assert 0.03 < hit.mean() < 0.95, "the floor quad fills part of the view"
    up = normal[hit]
    assert np.allclose(up[up[:, 1] > 0.99][:, [0, 2]], 0.5, atol=1e-6), "floor normal (0,1,0) -> (0.5, 1, 0.5)"
    assert lib.Raylib_DestroyCamera(cam) == 1 and lib.Raylib_DestroyScene(scene) == 1 and lib.Raylib_UnloadOBJModel(model) == 1


@pytest.mark.parametrize("cfg,size", [(2, 0), (4, 24), (6, 0), (1, 0)])
def test_adversarial_rays_against_restatement(gpu, restate, cfg, size):
    """Rays chosen to stress the CONSERVATIVE inner-node test (quantized boxes, ray-space slabs, clamped 1/d): axis-parallel
    and nearly axis-parallel directions (zero, denormal and 1e-20 components), origins lying exactly on box / wall planes,
    origins very far from the scene.  The device must still return what the exhaustive restatement returns."""
    info = gpu.create_demo(cfg, size)
    try:
        desc = gpu.flat_desc(info.scene)
        lo = np.array(desc.contents.rootMin[:], dtype=np.float64); hi = np.array(desc.contents.rootMax[:], dtype=np.float64)
        lo = np.maximum(lo, -50.0); hi = np.minimum(hi, 50.0)            # config 1/6 hold a r=1000 ground sphere
        rng = np.random.default_rng(11)
        n = 60000
        o = rng.uniform(lo - 0.5, hi + 0.5, size=(n, 3))
        v = rng.normal(size=(n, 3)); d = v / np.linalg.norm(v, axis=1, keepdims=True)
        k = n // 6
        # 1. exactly axis-parallel (one or two zero components, both signs of zero)
        axis = rng.integers(0, 3, size=k); d[:k] = 0.0; d[np.arange(k), axis] = rng.choice([-1.0, 1.0], size=k)
        d[:k // 2][d[:k // 2] == 0.0] = -0.0
        z = rng.integers(0, 3, size=k); d[np.arange(k, 2 * k), z] = 0.0
        # 2. nearly parallel: denormal and tiny components (1/d overflows or is astronomically large)
        t = rng.integers(0, 3, size=k); d[np.arange(2 * k, 3 * k), t] = rng.choice([1e-42, -1e-42, 1e-20, -1e-20, 3e-39], size=k)
        # 3. origins exactly on the root-box planes and on round coordinates (walls / grid lines of the procedural scenes)
        a = rng.integers(0, 3, size=k); o[np.arange(3 * k, 4 * k), a] = np.where(rng.random(k) < 0.5, lo[a], hi[a])
        o[4 * k:5 * k] = np.round(o[4 * k:5 * k] * 2.0) / 2.0
        # 4. far away, aimed at the scene
        c = 0.5 * (lo + hi); far = rng.normal(size=(n - 5 * k, 3)); far /= np.linalg.norm(far, axis=1, keepdims=True)
        dist = 10.0 ** rng.uniform(3, 6, size=(n - 5 * k, 1))
        target = rng.uniform(lo, hi, size=(n - 5 * k, 3))
        o[5 * k:] = c + far * dist
        dd = target - o[5 * k:]; d[5 * k:] = dd / np.linalg.norm(dd, axis=1, keepdims=True)
        rays = np.zeros((n, 8), dtype=np.float32)
        rays[:, 0:3] = o; rays[:, 4:7] = d
        grank, gt = gpu.trace_rays(info.scene, rays, 1e-4)
        crank, ct, _ = restate.trace(desc, rays, 1e-4)
        missed = int(((grank < 0) & (crank >= 0)).sum())
        mismatch = float((grank != crank).mean())
        print("config%d adversarial rays: hit fraction %.3f, id mismatch rate %.3e, missed hits %d" % (cfg, float((crank >= 0).mean()), mismatch, missed))
        for i in np.nonzero(grank != crank)[0][:5]:
            print("  ray %d o=%r d=%r device (rank %d, t %r) oracle (rank %d, t %r)" % (i, rays[i, 0:3].tolist(), rays[i, 4:7].tolist(),
                  grank[i], float(gt[i]), crank[i], float(ct[i])))
        assert missed == 0, "a conservative culling test must never lose a hit the reference finds"
        assert mismatch <= 1e-5
        same = grank == crank
        assert np.array_equal(bits(gt[same]), bits(ct[same]))
    finally:
        gpu.destroy_demo(info)


def test_full_size_scatter10M_against_compiled_reference(gpu, recorded, restate, rl):
    """The headline workload at FULL scene size (9,999,362 triangles, 7812 meshes, two-level BVH, 8 materials, sun + sky):
    primary-hit ids / t and the camera rays through the device traversal against the C restatement, radiance at matched
    spp and seed against the stored outputs (conftest.RecordedOutputs), and shard-count independence of the device frame."""
    import torch
    pinfo = gpu.create_demo(4, 0)
    try:
        W, H = 640, 360
        gpu.set_viewport(pinfo, W, H)
        gr, gt = gpu.primary_hits(pinfo.settings, pinfo.scene, pinfo.camera)
        rr, rt, rays = restated_primary(gpu, restate, pinfo)
        print("scatter10M primary: id match %.6f, t bit match %.6f, hit fraction %.3f"
              % (float((gr == rr).mean()), float((bits(gt) == bits(rt)).mean()), float((rr >= 0).mean())))
        assert np.array_equal(gr, rr) and np.array_equal(bits(gt), bits(rt))          # pinhole camera: exact
        gr2, gt2 = gpu.trace_rays(pinfo.scene, rays, pinfo.settings.rayTMin)
        assert np.array_equal(gr2, rr) and np.array_equal(bits(gt2), bits(rt))
        # radiance, 2 spp, depth 8
        s = pinfo.settings.copy(samplesPerPixel=2)
        gimg = gpu.render(s, pinfo.scene, pinfo.camera)
        st = gpu.last_stats()
        g, r, _ = recorded.compare("radiance", gimg)
        rays = int(recorded.value("radiance_rays"))
        psnr, out = rl.psnr(g, r), rel_outliers(g, r)
        exact = float((bits(g) == bits(r)).all(axis=2).mean())
        print("scatter10M radiance (sample): PSNR %.2f dB, outliers %.4f, bit-identical pixels %.4f, rays %d vs %d" % (psnr, out, exact, st.rayQueries, rays))
        assert psnr >= 40.0 and out <= 0.02 and exact >= EXACT_FLOOR
        assert abs(int(st.rayQueries) - rays) <= 0.002 * rays + 8
        # 1 shard vs 8 shards, bit-identical
        cap = int(gpu.lib.RaylibB200_ShardPixelCapacity(W, H, 8))
        slabs = torch.zeros((8 * cap, 4), dtype=torch.float32, device="cuda")
        for r in range(8):
            assert gpu.lib.RaylibB200_RenderShard(C.byref(s), pinfo.scene, pinfo.camera, r, 8, slabs[r * cap:(r + 1) * cap].data_ptr(), None), gpu.last_error()
        image = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
        assert gpu.lib.RaylibB200_AssembleShards(slabs.data_ptr(), 8, W, H, image.data_ptr(), None)
        assert np.array_equal(bits(image.cpu().numpy()[:, :, :3]), bits(gimg))
    finally:
        gpu.destroy_demo(pinfo)


def test_pipes_do_not_change_the_image(gpu):
    """1, 2 or 4 passes in flight (streams + arenas): same bits -- the per-pixel sums stay in sample order."""
    info = gpu.create_demo(6)
    try:
        gpu.set_viewport(info, 200, 120)
        s = info.settings.copy(samplesPerPixel=13)          # odd: the last pass is ragged
        frames = []
        for pipes, spp_per_pass in ((1, 0), (2, 0), (4, 0), (2, 3), (3, 1)):
            gpu.lib.RaylibB200_SetPipes(pipes)
            gpu.lib.RaylibB200_SetSamplesPerPass(spp_per_pass)
            frames.append(gpu.render(s, info.scene, info.camera))
            st = gpu.last_stats()
            assert st.pixelSamples == 200 * 120 * 13
        for f in frames[1:]:
            assert np.array_equal(bits(f), bits(frames[0]))
    finally:
        gpu.lib.RaylibB200_SetPipes(0)
        gpu.lib.RaylibB200_SetSamplesPerPass(0)
        gpu.destroy_demo(info)


def test_fused_pass_is_the_same_image(gpu):
    """Small frames run as ONE cooperative launch (k_pass_fused: the stage functions of the separate kernels between grid-wide
    barriers).  Same bits as the kernel-per-stage path, on the mixed scene (all materials, sun: the sun-visibility stage
    shares a phase with the next bounce's extend), on a scene without sun, at depth 1 and with every path ending early."""
    try:
        for cfg, w, h, spp, depth in ((6, 200, 120, 5, 8), (6, 64, 48, 1, 1), (1, 160, 90, 3, 5), (2, 96, 96, 4, 50), (7, 120, 80, 2, 4)):
            info = gpu.create_demo(cfg)
            try:
                gpu.set_viewport(info, w, h)
                s = info.settings.copy(samplesPerPixel=spp, maxPathLength=depth)
                frames, launches = [], []
                for mode in (1, 2):
                    gpu.lib.RaylibB200_SetFusedPass(mode)
                    frames.append(gpu.render(s, info.scene, info.camera))
                    st = gpu.last_stats()
                    launches.append(st.kernelLaunches)
                    assert st.pixelSamples == w * h * spp
                    rays = st.rayQueries if mode == 1 else rays
                    assert st.rayQueries == rays
                assert launches[1] == 1 and launches[0] > 4, launches
                assert np.array_equal(bits(frames[0]), bits(frames[1])), "config %d" % cfg
            finally:
                gpu.destroy_demo(info)
        # automatic mode: one launch up to 1 Mi paths (width x height x samples), the kernel-per-stage path above
        gpu.lib.RaylibB200_SetFusedPass(0)
        info = gpu.create_demo(6)
        try:
            gpu.set_viewport(info, 256, 128)
            for spp, one_launch in ((16, True), (48, False)):          # 0.5 Mi and 1.5 Mi paths
                gpu.render(info.settings.copy(samplesPerPixel=spp), info.scene, info.camera)
                assert (gpu.last_stats().kernelLaunches == 1) == one_launch, (spp, gpu.last_stats().kernelLaunches)
        finally:
            gpu.destroy_demo(info)
    finally:
        gpu.lib.RaylibB200_SetFusedPass(0)


def test_shared_frame_is_the_gather(gpu, tmp_path):
    """RenderShardToFrame: ranks store their final pixels straight into one row-major frame.  (a) three shards into a local
    frame, (b) two PROCESSES -- the second maps this process' frame through a CUDA IPC handle, as the one-process-per-GPU
    launch does over NVLink -- both give the bits of the whole-frame render."""
    import subprocess, sys, os
    info = gpu.create_demo(6)
    try:
        W, H = 203, 117                     # ragged tiles on both edges
        gpu.set_viewport(info, W, H)
        s = info.settings.copy(samplesPerPixel=5)
        whole = gpu.render(s, info.scene, info.camera)
        handle = (C.c_ubyte * 64)()
        frame = gpu.lib.RaylibB200_FrameCreate(W, H, handle)
        assert frame, gpu.last_error()
        host = np.full((H, W, 4), -1.0, dtype=np.float32)
        try:
            for r in range(3):
                assert gpu.lib.RaylibB200_RenderShardToFrame(C.byref(s), info.scene, info.camera, r, 3, frame, None), gpu.last_error()
            assert gpu.lib.RaylibB200_FrameRead(frame, W, H, host.ctypes.data, None), gpu.last_error()
            assert np.array_equal(bits(host[:, :, :3]), bits(whole)) and (host[:, :, 3] == 1.0).all()
            # (b) shard 0 here, shard 1 in a second process through the IPC mapping
            host[:] = -1.0
            worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "frame_worker.py")
            child = subprocess.Popen([sys.executable, worker, bytes(handle).hex(), str(W), str(H), "5", "1", "2"],
                                     stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            assert gpu.lib.RaylibB200_RenderShardToFrame(C.byref(s), info.scene, info.camera, 0, 2, frame, None), gpu.last_error()
            out, _ = child.communicate(timeout=600)
            assert child.returncode == 0, out
            assert gpu.lib.RaylibB200_FrameRead(frame, W, H, host.ctypes.data, None), gpu.last_error()
            assert np.array_equal(bits(host[:, :, :3]), bits(whole)), "two processes into one frame differ from one process"
        finally:
            gpu.lib.RaylibB200_FrameDestroy(frame)
    finally:
        gpu.destroy_demo(info)


def test_flattened_scene_cache_renders_identically(gpu, tmp_path):
    """A scene read back from its flattened-scene file (no object graph, no BVH builds) renders the same bits, answers
    the same ray queries and shards like the scene it was saved from."""
    for cfg, size in ((6, 0), (5, 64)):
        info = gpu.create_demo(cfg, size)
        try:
            gpu.set_viewport(info, 160, 90)
            s = info.settings.copy(samplesPerPixel=3)
            path = str(tmp_path / ("scene%d.rtflat" % cfg)).encode()
            assert gpu.lib.RaylibB200_SaveFlattenedScene(info.scene, path) == 1, gpu.last_error()
            loaded = gpu.lib.RaylibB200_LoadFlattenedScene(path)
            assert loaded, gpu.last_error()
            a = gpu.render(s, info.scene, info.camera)
            b = gpu.render(s, loaded, info.camera)
            assert np.array_equal(bits(a), bits(b))
            ra, ta = gpu.primary_hits(s, info.scene, info.camera)
            rb, tb = gpu.primary_hits(s, loaded, info.camera)
            assert np.array_equal(ra, rb) and np.array_equal(bits(ta), bits(tb))
            n = gpu.render(s.copy(renderMode=2), loaded, info.camera)
            assert np.array_equal(bits(n), bits(gpu.render(s.copy(renderMode=2), info.scene, info.camera)))
            assert gpu.lib.Raylib_DestroyScene(loaded) == 1
        finally:
            gpu.destroy_demo(info)


@pytest.mark.parametrize("cfg,name,psnr_floor", [(3, "grid1M", 60.0), (5, "textured2M", 40.0)])
def test_full_size_scenes_against_compiled_reference(gpu, recorded, restate, rl, cfg, name, psnr_floor):
    """BASELINE configurations 3 (1,002,528-triangle displaced grid, primary + AO) and 5 (~2 M textured microfacet
    triangles with alpha cut-outs, mirror / dielectric / metal objects) at FULL scene size: primary-hit ids and t against
    the C restatement; the SurfaceNormal view (README "VertexNormal") and radiance at matched spp and seed against the
    stored outputs (conftest.RecordedOutputs)."""
    pinfo = gpu.create_demo(cfg, 0)
    try:
        W, H = 480, 270
        gpu.set_viewport(pinfo, W, H)
        gr, gt = gpu.primary_hits(pinfo.settings, pinfo.scene, pinfo.camera)
        rr, rt, rays = restated_primary(gpu, restate, pinfo)
        idm, tm = float((gr == rr).mean()), float((bits(gt) == bits(rt)).mean())
        print("%s primary: id match %.6f, t bit match %.6f, hit fraction %.3f" % (name, idm, tm, float((rr >= 0).mean())))
        assert np.array_equal(gr, rr) and np.array_equal(bits(gt), bits(rt))          # pinhole cameras: exact
        gr2, gt2 = gpu.trace_rays(pinfo.scene, rays, pinfo.settings.rayTMin)
        assert np.array_equal(gr2, rr) and np.array_equal(bits(gt2), bits(rt))
        # SurfaceNormal debug view: bit-identical (triangles only, no transcendental on the way)
        gn = gpu.render(pinfo.settings.copy(renderMode=2), pinfo.scene, pinfo.camera)
        assert recorded.compare("normal_view", gn)[2]
        # radiance, 2 spp at the configuration's own depth
        s = pinfo.settings.copy(samplesPerPixel=2)
        gimg = gpu.render(s, pinfo.scene, pinfo.camera)
        st = gpu.last_stats()
        g, r, _ = recorded.compare("radiance", gimg)
        rays = int(recorded.value("radiance_rays"))
        psnr, out = rl.psnr(g, r), rel_outliers(g, r)
        exact = float((bits(g) == bits(r)).all(axis=2).mean())
        print("%s radiance (sample): PSNR %.2f dB, outliers %.4f, bit-identical pixels %.4f, rays %d vs %d" % (name, psnr, out, exact, st.rayQueries, rays))
        assert psnr >= psnr_floor and out <= 0.02 and exact >= EXACT_FLOOR
        assert abs(int(st.rayQueries) - rays) <= 0.002 * rays + 8
    finally:
        gpu.destroy_demo(pinfo)


# ---- round 2: comparisons that used to be self-comparisons, now against the compiled reference ---------------------

def test_gpu_postprocess_vs_compiled_reference(gpu, recorded):
    """SURVEY 8(f) rank 3 against the ORACLE: the same HDR frame through the reference's own Raylib_PostProcess
    (render/image.cc:44-103, compiled unmodified; its output is stored, see conftest.RecordedOutputs) and through
    RaylibB200_PostProcessGPU / _PostProcessDevice."""
    import torch
    info = gpu.create_demo(2, 0)            # Cornell box: the light (15) is far above white
    try:
        W, H = 320, 180
        gpu.set_viewport(info, W, H)
        s = info.settings.copy(samplesPerPixel=4)
        img = gpu.lib.Raylib_CreateImage(W, H)
        try:
            gpu.lib.Raylib_Render(C.byref(s), info.scene, info.camera, img)
            raw = np.empty((H, W, 4), dtype=np.float32)
            assert gpu.lib.RaylibB200_ImageGetRGBA(img, raw) == 1
            assert gpu.lib.RaylibB200_PostProcessGPU(img), gpu.last_error()
            out = np.empty_like(raw)
            assert gpu.lib.RaylibB200_ImageGetRGBA(img, out) == 1
        finally:
            gpu.lib.Raylib_DestroyImage(img)
        assert raw[..., :3].max() > 1.0, "the test frame must exercise the max-white reduction"
        assert recorded.compare("input", raw)[2], "the rendered input frame is not the one the reference post-processed"
        out, want, _ = recorded.compare("postprocess", out)
        # identical arithmetic except powf (device libm vs glibc): report how many pixels are bit-identical
        exact = float((bits(out) == bits(want)).all(axis=2).mean())
        print("GPU post-process vs reference (sample): bit-identical pixels %.4f, max abs diff %.3g" % (exact, float(np.abs(out - want).max())))
        assert np.allclose(out, want, rtol=2e-6, atol=1e-7)
        assert exact >= EXACT_FLOOR
        # device-resident form with the packed 8-bit output (Pixel::ToUint32, image.h:57-64)
        dev = torch.from_numpy(raw).cuda()
        packed = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        mw = C.c_float(0.0)
        assert gpu.lib.RaylibB200_PostProcessDevice(dev.data_ptr(), W, H, packed.data_ptr(), C.byref(mw), None), gpu.last_error()
        assert np.allclose(recorded.sample("postprocess", dev.cpu().numpy()), want, rtol=2e-6, atol=1e-7)
        p = recorded.sample("postprocess", packed.cpu().numpy()[..., None])[..., 0].view(np.uint32)
        w8 = (want * 255.0).astype(np.uint32) & 0xff
        expect = (w8[..., 3] << 24) | (w8[..., 0] << 16) | (w8[..., 1] << 8) | w8[..., 2]
        assert (p == expect).mean() >= 0.99 and np.abs(((p >> 8) & 0xff).astype(np.int32) - w8[..., 1].astype(np.int32)).max() <= 1
    finally:
        gpu.destroy_demo(info)


@pytest.mark.parametrize("cfg,size", [(5, 40), (6, 0), (2, 0)])
def test_microsurface_normal_and_reflectance_views_vs_compiled_reference(gpu, recorded, cfg, size):
    """Render modes 3 (MicrosurfaceNormal) and 6 (Reflectance) -- deterministic in the reference after all: the debug path
    never builds the tangent frame, but a default-constructed HitResult holds ZERO tangent / bitangent (vec3() = 0,
    core/vec3.h:16), so mode 3 shows N.z * n and mode 6 scatters on the zero frame.  Also the normal half of
    RaylibB200_RenderAux (SURVEY 8f rank 2), which is the same pass.  Views compared with the stored outputs (conftest.RecordedOutputs)."""
    pinfo = gpu.create_demo(cfg, size)
    try:
        W, H = 240, 136
        gpu.set_viewport(pinfo, W, H)
        for mode in (3, 6):
            gimg = gpu.render(pinfo.settings.copy(renderMode=mode), pinfo.scene, pinfo.camera)
            g, r, same = recorded.compare("mode%d" % mode, gimg)
            exact = float((bits(g) == bits(r)).all(axis=2).mean())
            close = float(np.isclose(g, r, rtol=1e-4, atol=2e-3).all(axis=2).mean())
            print("config%d mode %d vs reference (sample): bit-identical %.4f, close %.4f" % (cfg, mode, exact, close))
            if cfg in PINHOLE:
                assert same if mode == 3 else exact >= EXACT_FLOOR
            else:
                assert exact >= 0.98 and close >= 0.98      # a finite aperture can move a silhouette pixel onto another primitive
        a_img, n_img = gpu.lib.Raylib_CreateImage(W, H), gpu.lib.Raylib_CreateImage(W, H)
        try:
            assert gpu.lib.RaylibB200_RenderAux(C.byref(pinfo.settings), pinfo.scene, pinfo.camera, a_img, n_img), gpu.last_error()
            aux_a, aux_n = gpu.dump_image(a_img, W, H), gpu.dump_image(n_img, W, H)
        finally:
            gpu.lib.Raylib_DestroyImage(a_img); gpu.lib.Raylib_DestroyImage(n_img)
        if cfg in PINHOLE:
            assert recorded.compare("mode1", aux_a)[2] and recorded.compare("mode3", aux_n)[2]
        else:
            g, r, _ = recorded.compare("mode3", aux_n)
            assert (bits(g) == bits(r)).all(axis=2).mean() >= 0.85
    finally:
        gpu.destroy_demo(pinfo)


@pytest.mark.parametrize("cfg,size", [(5, 40), (6, 0), (4, 24)])
def test_shallow_paths_vs_compiled_reference(gpu, recorded, rl, cfg, size):
    """Where does the radiance start to differ?  maxPathLength 1 (emission + sky + sun visibility of the camera ray; no
    scattered direction is ever used) must be bit-identical on (nearly) every pixel; maxPathLength 2 adds ONE scattered ray
    whose direction went through sinf/cosf/powf on the device instead of glibc -- values agree to float rounding.  Deeper
    paths only amplify those last-bit differences (specular chains), which is what the 40 dB bar of the full-depth tests
    absorbs; a first-bounce disagreement would show up here.  Frames compared with the stored outputs (conftest.RecordedOutputs)."""
    pinfo = gpu.create_demo(cfg, size)
    try:
        W, H = 256, 144
        gpu.set_viewport(pinfo, W, H)
        for depth, spp in ((1, 4), (2, 4)):
            s = pinfo.settings.copy(samplesPerPixel=spp, maxPathLength=depth)
            gimg = gpu.render(s, pinfo.scene, pinfo.camera)
            grays = gpu.last_stats().rayQueries
            g, r, _ = recorded.compare("depth%d" % depth, gimg)
            rays = int(recorded.value("depth%d_rays" % depth))
            exact = float((bits(g) == bits(r)).all(axis=2).mean())
            off = rel_outliers(g, r, rel=1e-4, absolute=1e-5)
            print("config%d depth %d (sample): bit-identical pixels %.4f, pixels off by > 1e-4 rel: %.4f, PSNR %.1f dB, rays %d vs %d"
                  % (cfg, depth, exact, off, rl.psnr(g, r), grays, rays))
            assert exact >= EXACT_FLOOR and off <= 0.001
            assert abs(int(grays) - rays) <= 4
    finally:
        gpu.destroy_demo(pinfo)


def test_lighting_is_read_at_every_render(gpu, recorded, rl):
    """The reference reads Scene::GetSun and the sky panorama live on every miss (renderer.cc:160-191): a client may change
    them between frames of a finalized scene.  The uploaded copy must follow (the sun travels per frame, a changed sky
    re-uploads).  The frames after each change are compared with the stored outputs (conftest.RecordedOutputs)."""
    pinfo = gpu.create_demo(4, 16)
    try:
        W, H = 160, 90
        gpu.set_viewport(pinfo, W, H)
        s = pinfo.settings.copy(samplesPerPixel=2, maxPathLength=3)
        first = gpu.render(s, pinfo.scene, pinfo.camera)
        gpu.lib.Raylib_SetSunIlluminance(pinfo.scene, 1.5, 9.0, 0.25)
        gpu.lib.Raylib_SetSunDirection(pinfo.scene, 0.6, -1.0, 0.2)
        second = gpu.render(s, pinfo.scene, pinfo.camera)
        assert not np.array_equal(first, second), "the new sun was ignored"
        g, r, _ = recorded.compare("new_sun", second)
        assert rl.psnr(g, r) >= 40.0 and rel_outliers(g, r) <= 0.02
        # sun off (renderer.cc:191: no visibility rays at all), then a different sky image
        gpu.lib.Raylib_SetSunIlluminance(pinfo.scene, 0.0, 0.0, 0.0)
        third = gpu.render(s, pinfo.scene, pinfo.camera)
        rays3 = gpu.last_stats().rayQueries
        g, r, _ = recorded.compare("sun_off", third)
        want_rays3 = int(recorded.value("sun_off_rays"))
        assert rl.psnr(g, r) >= 40.0 and abs(int(rays3) - want_rays3) <= 0.002 * want_rays3 + 8
        sky = np.zeros((8, 16, 4), dtype=np.float32); sky[..., 0] = 2.0; sky[..., 3] = 1.0      # a red sky
        g_sky = gpu.lib.Raylib_CreateImage(16, 8)
        try:
            assert gpu.lib.RaylibB200_ImageSetRGBA(g_sky, 16, 8, sky) == 1
            gpu.lib.Raylib_SetSkyPanorama(pinfo.scene, g_sky)
            fourth = gpu.render(s, pinfo.scene, pinfo.camera)
            assert fourth[..., 0].mean() > 4.0 * fourth[..., 2].mean(), "the new sky was ignored"
            g, r, _ = recorded.compare("red_sky", fourth)
            assert rl.psnr(g, r) >= 40.0 and rel_outliers(g, r) <= 0.02
        finally:
            gpu.lib.Raylib_SetSkyPanorama(pinfo.scene, 0)
            gpu.lib.Raylib_DestroyImage(g_sky)
    finally:
        gpu.destroy_demo(pinfo)


@pytest.mark.parametrize("cfg,size", [(6, 0), (5, 40), (1, 0)])
def test_cross_abi_client_renders_like_the_native_client(gpu, rl, cfg, size):
    """A client compiled against the REFERENCE's headers (oracle/_ref/libscenes_xabi.so) and one compiled against this
    repository's headers build the same scene through the same library: frames must be bit-identical."""
    import os
    from oracle import bindings as ob
    if not os.path.exists(ob.XABI_SCENES):
        pytest.skip("oracle/_ref/libscenes_xabi.so not built (needs /root/reference)")
    xprod = rl.Product(scenes_path=ob.XABI_SCENES)
    a, b = gpu.create_demo(cfg, size), xprod.create_demo(cfg, size)
    try:
        gpu.set_viewport(a, 200, 112); xprod.set_viewport(b, 200, 112)
        s = a.settings.copy(samplesPerPixel=3)
        img_a = gpu.render(s, a.scene, a.camera)
        img_b = xprod.render(s, b.scene, b.camera)
        assert np.array_equal(bits(img_a), bits(img_b))
        for mode in (1, 2, 4):
            assert np.array_equal(bits(gpu.render(s.copy(renderMode=mode), a.scene, a.camera)),
                                  bits(xprod.render(s.copy(renderMode=mode), b.scene, b.camera)))
    finally:
        gpu.destroy_demo(a); xprod.destroy_demo(b)


def test_all_devices_behind_plain_raylib_render(gpu, rl):
    """Raylib_Render spreads a frame over every active GPU inside one process (raylib/render/renderer.cc:286-334 uses every
    core): the image must not depend on how many devices took part."""
    n = gpu.device_count()
    if n < 2:
        pytest.skip("one CUDA device visible; run with gpurun --gpus 2")
    import ctypes
    libc = ctypes.CDLL(None)
    info = gpu.create_demo(4, 40)
    try:
        gpu.set_viewport(info, 640, 360)
        s = info.settings.copy(samplesPerPixel=12, maxPathLength=4)        # 2.76 M pixel-samples: above the multi-device floor
        assert gpu.lib.RaylibB200_SetDevices(1) == 1
        one = gpu.render(s, info.scene, info.camera)
        st1 = gpu.last_stats()
        assert st1.devicesUsed == 1
        for k in sorted({2, n}):
            assert gpu.lib.RaylibB200_SetDevices(k) == k
            many = gpu.render(s, info.scene, info.camera)
            st = gpu.last_stats()
            assert st.devicesUsed == k, gpu.last_error()
            assert np.array_equal(bits(one), bits(many)), "%d devices: image differs from one device" % k
            assert st.rayQueries == st1.rayQueries and st.pixelSamples == st1.pixelSamples
    finally:
        gpu.lib.RaylibB200_SetDevice(0)
        gpu.destroy_demo(info)


def test_raw_hitable_list_element_on_the_device(gpu, recorded, restate, rl):
    """SURVEY 8a row a13 on the GPU: config 7 (a raw HitableList scene element with duplicated members) -- primary ids and t
    against the C restatement (pinhole camera: exact), then radiance at matched spp and seed against the stored outputs
    (conftest.RecordedOutputs)."""
    pinfo = gpu.create_demo(7)
    try:
        gr, gt = gpu.primary_hits(pinfo.settings, pinfo.scene, pinfo.camera)
        rr, rt, rays = restated_primary(gpu, restate, pinfo)
        assert np.array_equal(gr, rr) and np.array_equal(bits(gt), bits(rt))
        gr2, gt2 = gpu.trace_rays(pinfo.scene, rays, pinfo.settings.rayTMin)
        assert np.array_equal(gr2, rr) and np.array_equal(bits(gt2), bits(rt))
        gimg = gpu.render(pinfo.settings, pinfo.scene, pinfo.camera)
        rays = int(recorded.value("radiance_rays"))
        g, r, _ = recorded.compare("radiance", gimg)
        print("config7 radiance (sample): PSNR %.2f dB, bit-identical pixels %.4f" % (rl.psnr(g, r), float((bits(g) == bits(r)).all(axis=2).mean())))
        assert rl.psnr(g, r) >= 40.0 and rel_outliers(g, r) <= 0.02
        assert float((bits(g) == bits(r)).all(axis=2).mean()) >= EXACT_FLOOR
        assert abs(int(gpu.last_stats().rayQueries) - rays) <= 0.002 * rays + 8
    finally:
        gpu.destroy_demo(pinfo)


def test_device_transcendentals_equal_the_host_c_library(gpu):
    """include/rt_libm.h on the DEVICE against the host C library the compiled reference calls (glibc: sinf, cosf, tanf,
    asinf, acosf, atanf, expf, logf, powf, atan2f): bit for bit on 2 M arguments per function -- the ranges the shaders
    use, the whole float range, and the special values.  (The same header is checked against glibc over all 2^32 arguments on
    the host by oracle/libm_check.cc, tests/test_cpu_oracle.py.)"""
    import ctypes.util
    libm = C.CDLL(ctypes.util.find_library("m") or "libm.so.6")
    rng = np.random.default_rng(2025)
    n = 1 << 21
    wide = rng.integers(0, 1 << 32, size=n // 2, dtype=np.uint64).astype(np.uint32).view(np.float32)
    special = np.array([0.0, -0.0, 1.0, -1.0, 0.5, -0.5, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1.17549435e-38, 3.4028235e38, 88.7, -103.9, 120.0, 1e9,
                        0.78539816, 0.975, 0.4375, 2.4375, 0.6744], dtype=np.float32)
    names = ["sinf", "cosf", "tanf", "asinf", "acosf", "atanf", "expf", "logf", "powf", "atan2f"]
    ranges = {"sinf": (-8.0, 8.0), "cosf": (-8.0, 8.0), "tanf": (-1.6, 1.6), "asinf": (-1.0, 1.0), "acosf": (-1.0, 1.0), "atanf": (-50.0, 50.0),
              "expf": (-30.0, 5.0), "logf": (1e-9, 4.0), "powf": (0.0, 2.0), "atan2f": (-3.0, 3.0)}
    for fn, name in enumerate(names):
        lo, hi = ranges[name]
        x = np.concatenate([rng.uniform(lo, hi, size=n - len(wide) - len(special)).astype(np.float32), wide, special])
        two = name in ("powf", "atan2f")
        y = None
        if two:
            y = np.concatenate([rng.choice(np.array([2.2, 1.0 / 2.2, 5.0, 0.4265, 1.3], dtype=np.float32), size=n // 2),
                                rng.uniform(-4.0, 4.0, size=n - n // 2).astype(np.float32)]) if name == "powf" else rng.uniform(-3.0, 3.0, size=n).astype(np.float32)
        out = np.empty(n, dtype=np.float32)
        assert gpu.lib.RaylibB200_LibmEval(fn, x, y.ctypes.data if two else None, out, n) == 1, gpu.last_error()
        f = getattr(libm, name)
        f.restype = C.c_float
        f.argtypes = [C.c_float, C.c_float] if two else [C.c_float]
        idx = rng.choice(n, size=60000, replace=False)
        idx = np.concatenate([idx, np.arange(n - len(special), n)])          # a sample through ctypes (slow), incl. all special values
        want = np.array([f(float(x[i]), float(y[i])) if two else f(float(x[i])) for i in idx], dtype=np.float32)
        got = out[idx]
        same = (bits(got) == bits(want)) | (np.isnan(got) & np.isnan(want))
        assert same.all(), "%s: %d of %d differ, first at x=%r" % (name, int((~same).sum()), len(idx), x[idx[np.argmin(same)]])


def test_obj_import_renders_like_the_reference_conversion(gpu, recorded, restate, rl, tmp_path):
    """Raylib_LoadOBJModel -> Raylib_AddOBJModelToScene -> Raylib_Render on the GPU against the compiled reference rendering
    the same file imported through the object API with the reference's conversion rules (scene client config 8; its
    frames are stored, see conftest.RecordedOutputs): primary ids and t exact against the C restatement (pinhole camera),
    radiance at matched spp and seed, debug views, and bit-identical to the product's own object path."""
    import ctypes, os
    from test_cpu_oracle import write_test_obj, load_obj_scene
    libc = ctypes.CDLL(None)
    path = write_test_obj(str(tmp_path))
    os.environ["DEMO_OBJ_PATH"] = path; libc.setenv(b"DEMO_OBJ_PATH", path.encode(), 1)
    try:
        pinfo = gpu.create_demo(8)
        model, scene = load_obj_scene(gpu.lib, path)
        try:
            s = pinfo.settings
            gr, gt = gpu.primary_hits(s, scene, pinfo.camera)
            rr, rt, _ = restated_primary(gpu, restate, pinfo, scene=scene)
            assert np.array_equal(gr, rr) and np.array_equal(bits(gt), bits(rt))
            img_import = gpu.render(s, scene, pinfo.camera)
            img_objects = gpu.render(s, pinfo.scene, pinfo.camera)
            assert np.array_equal(bits(img_import), bits(img_objects)), "importer and object path differ"
            g, r, _ = recorded.compare("radiance", img_import)
            exact = float((bits(g) == bits(r)).all(axis=2).mean())
            print("OBJ scene radiance vs reference (sample): PSNR %.2f dB, bit-identical pixels %.4f" % (rl.psnr(g, r), exact))
            assert rl.psnr(g, r) >= 40.0 and rel_outliers(g, r) <= 0.02 and exact >= EXACT_FLOOR
            for mode in (1, 2, 4, 5):
                g = gpu.render(s.copy(renderMode=mode), scene, pinfo.camera)
                assert recorded.compare("mode%d" % mode, g)[2], "debug view %d" % mode
        finally:
            gpu.lib.Raylib_DestroyScene(scene); gpu.lib.Raylib_UnloadOBJModel(model)
            gpu.destroy_demo(pinfo)
    finally:
        os.environ.pop("DEMO_OBJ_PATH", None); libc.unsetenv(b"DEMO_OBJ_PATH")
