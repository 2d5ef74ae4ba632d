"""CPU-only: pins the oracle.

1. the plain-C restatement (oracle/rt_oracle.c) run on the PRODUCT's flattened scene must reproduce the
   golden vectors generated from the compiled reference (tests/golden, tools/make_golden.py) bit for bit --
   this covers the host BVH build, the flattener and the traversal semantics without a GPU;
2. where oracle/_ref exists, the compiled reference itself must still reproduce the golden vectors; the restatement
   must give the answers stored for random rays (tests/golden/recorded, see conftest.RecordedOutputs);
3. analytic known-answer tests (the reference has no tests of its own, SURVEY.md section 4).
"""
import numpy as np
import pytest
from conftest import load_golden, bits

CONFIGS = [1, 2, 3, 4, 5, 6]


@pytest.mark.parametrize("cfg", CONFIGS)
def test_restatement_matches_golden_primary_hits(prod, restate, cfg):
    g = load_golden(cfg)
    w, h = [int(x) for x in g["primary_wh"]]
    info = prod.create_demo(cfg, int(g["size"]))
    try:
        prod.set_viewport(info, w, h)
        desc = prod.flat_desc(info.scene)
        cam = prod.camera_block(info.camera)
        rank, t, counts, rays = restate.primary(desc, cam, w, h, info.settings.rayTMin, seed=int(g["seed"]), want_rays=True)
        assert np.array_equal(bits(rays), bits(g["rays"])), "camera rays differ from the compiled reference's"
        assert g["rank"].max() < desc.contents.numLeaves
        assert np.array_equal(rank, g["rank"]), "primitive ids differ from the compiled reference"
        assert np.array_equal(bits(t), bits(g["t"])), "hit distances differ from the compiled reference (bit compare)"
        # the restatement merges StaticMesh bounds + root box into one test; everything else is counted alike
        ref_box, ref_tri, ref_sph, ref_rays = [int(x) for x in g["ref_tests"]]
        assert counts[1] == ref_tri and counts[2] == ref_sph
        assert counts[0] <= ref_box
        # the same rays, fed back as explicit rays
        rank2, t2, _ = restate.trace(desc, g["rays"], info.settings.rayTMin)
        assert np.array_equal(rank2, g["rank"]) and np.array_equal(bits(t2), bits(g["t"]))
        # the device's traversal tree (SAH over the reference's leaf groups) must select the same candidates
        assert desc.contents.treeKind == 1
        restate.select_tree(True)
        try:
            rank3, t3, counts3 = restate.trace(desc, g["rays"], info.settings.rayTMin)
        finally:
            restate.select_tree(False)
        assert np.array_equal(rank3, g["rank"]) and np.array_equal(bits(t3), bits(g["t"]))
        assert counts3[1] <= ref_tri and counts3[2] == ref_sph, "tight triangle boxes cull more, spheres keep their gates"
        # ... and so must its 4-wide collapse, which is what the kernels walk
        assert desc.contents.numWideNodes > 0 or desc.contents.numNodes == 0
        restate.select_tree(2)
        try:
            rank4, t4, counts4 = restate.trace(desc, g["rays"], info.settings.rayTMin)
        finally:
            restate.select_tree(0)
        assert np.array_equal(rank4, g["rank"]) and np.array_equal(bits(t4), bits(g["t"]))
        assert counts4[1] == counts3[1] and counts4[2] == counts3[2], "same leaves reached through either tree"
        # ... and the 64-byte quantized nodes the kernels fetch: every decoded box contains the exact one
        assert restate.check_quantization(desc) == 0
        restate.select_tree(3)
        try:
            rank5, t5, counts5 = restate.trace(desc, g["rays"], info.settings.rayTMin)
        finally:
            restate.select_tree(0)
        assert np.array_equal(rank5, g["rank"]) and np.array_equal(bits(t5), bits(g["t"]))
        assert counts5[1] >= counts4[1], "looser boxes can only reach more leaves"
        print("config%d box tests/ray: exact wide %.1f, quantized %.1f" % (cfg, counts4[0] / len(rank4), counts5[0] / len(rank5)))
    finally:
        prod.destroy_demo(info)


@pytest.mark.parametrize("cfg", CONFIGS)
def test_compiled_reference_reproduces_golden(ref, cfg):
    g = load_golden(cfg)
    w, h = [int(x) for x in g["primary_wh"]]
    info = ref.create_demo(cfg, int(g["size"]))
    try:
        ref.set_viewport(info, w, h)
        rank, t, _, st = ref.primary_hits(info.settings, info.scene, info.camera, seed=int(g["seed"]))
        assert st.walkVsHitMismatches == 0, "labelling walk disagrees with the reference's own BVHNode::Hit"
        assert np.array_equal(rank, g["rank"]) and np.array_equal(bits(t), bits(g["t"]))
        rw, rh, spp = [int(x) for x in g["radiance_whs"]]
        ref.set_viewport(info, rw, rh)
        img, st2 = ref.render_deterministic(info.settings.copy(samplesPerPixel=spp), info.scene, info.camera, threads=3)
        assert np.array_equal(bits(img), bits(g["radiance"])), "reference radiance is not reproducible (thread count / run)"
        assert int(st2.rayQueries) == int(g["ray_queries"])
        assert st2.debugbreaks == 0
    finally:
        ref.destroy_demo(info)


@pytest.mark.parametrize("cfg", [1, 4, 6])
def test_restatement_vs_reference_random_rays(prod, recorded, restate, cfg):
    """Incoherent rays (random origins inside the scene bounds, random directions): the restatement against the stored
    answers (conftest.RecordedOutputs)."""
    g = load_golden(cfg)
    size = int(g["size"])
    pinfo = prod.create_demo(cfg, size)
    try:
        rng = np.random.default_rng(1234 + cfg)
        n = 20000
        d = prod.flat_desc(pinfo.scene).contents
        lo, hi = np.array(d.rootMin[:]), np.array(d.rootMax[:])
        lo, hi = np.maximum(lo, -60.0), np.minimum(hi, 60.0)
        rays = np.zeros((n, 8), dtype=np.float32)
        rays[:, 0:3] = rng.uniform(lo, hi, size=(n, 3))
        rays[:, 3] = rng.uniform(0.0, 2.0, size=n)
        v = rng.normal(size=(n, 3))
        rays[:, 4:7] = v / np.linalg.norm(v, axis=1, keepdims=True)
        # axis-aligned directions exercise 1/0 = inf in the slab test (aabb.h:43)
        rays[:50, 4:7] = np.array([0.0, -1.0, 0.0]); rays[50:100, 4:7] = np.array([1.0, 0.0, 0.0])
        c_rank, c_t, _ = restate.trace(prod.flat_desc(pinfo.scene), rays, 1e-4)
        assert recorded.compare("rank", c_rank)[2]
        assert recorded.compare("t", c_t)[2]
    finally:
        prod.destroy_demo(pinfo)


def test_known_answers_on_mixed_scene(prod, restate):
    """Config 6 holds a sphere of radius 0.5 at (0,0,-1), a mirror wall in the plane z=-2.5 and a cube."""
    info = prod.create_demo(6)
    try:
        desc = prod.flat_desc(info.scene)
        rays = np.array([
            [0, 0, 3, 0,   0, 0, -1, 0],       # straight at the sphere: t = 3.5 exactly (near root)
            [0, 0, -1, 0,  0, 0, -1, 0],       # from the sphere centre: near root negative -> far root t = 0.5
            [0, 0, 3, 0,   0, 0, 1, 0],        # looking away: miss
            [0, 1.0, -2.0, 0, 1, 0, 0, 0],     # parallel to the wall plane z=-2.5 (d.n = 0): t = inf/NaN -> rejected
            [0, 0.75, 3, 0, 0, 0, -1, 0],      # above the sphere: passes it, hits the wall at z=-2.5 -> t = 5.5
            [0, 0, 0.4999, 0, 0, 0, -2, 0],    # non-unit direction: t scales (sphere at distance 0.9999 -> t = 0.49995)
        ], dtype=np.float32)
        rank, t, _ = restate.trace(desc, rays, 1e-4)
        assert rank[0] >= 0 and t[0] == np.float32(3.5)
        assert rank[1] == rank[0] and t[1] == np.float32(0.5)
        assert rank[2] == -1
        assert rank[3] == -1
        assert rank[4] >= 0 and rank[4] != rank[0] and abs(t[4] - 5.5) < 1e-5
        assert rank[5] == rank[0] and abs(t[5] - 0.49995) < 1e-5
    finally:
        prod.destroy_demo(info)


def test_host_postprocess_equals_the_reference(prod, recorded):
    """Image2D::PostProcess of the product's HOST object model (what Raylib_PostProcess runs) against the reference's own
    Raylib_PostProcess (render/image.cc:44-103; its output is stored, conftest.RecordedOutputs) on the same synthetic HDR frame: all
    four channels bit for bit (both run glibc's powf).  The GPU form is compared with the same oracle in
    tests/test_gpu_parity.py."""
    rng = np.random.default_rng(11)
    h, w = 37, 53
    rgba = np.ones((h, w, 4), dtype=np.float32)
    rgba[..., :3] = rng.gamma(0.6, 1.5, size=(h, w, 3)).astype(np.float32)      # plenty of values above white
    rgba[0, :5, :3] = 0.0                                                          # luminance <= 1e-4 -> black
    rgba[1, :5, :3] = 2.0e-5
    rgba[2, 0, :3] = [40.0, 55.0, 3.0]                                             # sets the max-white luminance
    img = prod.lib.Raylib_CreateImage(w, h)
    try:
        assert prod.lib.RaylibB200_ImageSetRGBA(img, w, h, rgba) == 1
        prod.lib.Raylib_PostProcess(img)
        got = np.empty_like(rgba)
        assert prod.lib.RaylibB200_ImageGetRGBA(img, got) == 1
    finally:
        prod.lib.Raylib_DestroyImage(img)
    got_s, want_s, same = recorded.compare("postprocess", got)
    assert same, float(np.abs(got_s - want_s).max())
    assert got.max() <= 1.0 and (got[0, :5, :3] == 0).all()


@pytest.mark.parametrize("cfg", CONFIGS)
def test_cross_abi_client_flattens_to_the_golden_hits(rl, restate, cfg):
    """The drop-in boundary, proven with a client compiled against the REFERENCE's headers (oracle/_ref/libscenes_xabi.so:
    scenes/scenes.cc with -I/root/reference/raylib, linked against libraylib_b200.so with --no-undefined): the objects it
    lays out -- Sphere, Cube, Triangle, StaticMesh, six materials, textures, Image2D, Camera -- are read by the product
    library and flatten to a scene whose primary hits are the golden ones, bit for bit."""
    import os
    from oracle import bindings as ob
    if not os.path.exists(ob.XABI_SCENES):
        pytest.skip("oracle/_ref/libscenes_xabi.so not built (needs /root/reference)")
    xprod = rl.Product(scenes_path=ob.XABI_SCENES)
    g = load_golden(cfg)
    w, h = [int(x) for x in g["primary_wh"]]
    info = xprod.create_demo(cfg, int(g["size"]))
    try:
        xprod.set_viewport(info, w, h)
        desc = xprod.flat_desc(info.scene)
        cam = xprod.camera_block(info.camera)
        rank, t, _ = restate.primary(desc, cam, w, h, info.settings.rayTMin, seed=int(g["seed"]))
        assert np.array_equal(rank, g["rank"]) and np.array_equal(bits(t), bits(g["t"]))
        restate.select_tree(3)
        try:
            rank3, t3, _ = restate.trace(desc, g["rays"], info.settings.rayTMin)
        finally:
            restate.select_tree(0)
        assert np.array_equal(rank3, g["rank"]) and np.array_equal(bits(t3), bits(g["t"]))
    finally:
        xprod.destroy_demo(info)


def test_both_clients_report_the_same_scene_size(prod, recorded):
    """DemoSceneInfo.numTriangles counts mesh triangles (bench.py prints it in `config` of both arms); the reference
    client's counts are stored (conftest.RecordedOutputs)."""
    for cfg, size in ((2, 0), (4, 12), (6, 0)):
        a = prod.create_demo(cfg, size)
        try:
            got = (a.numTriangles, a.numSpheres, a.numMeshes)
            assert tuple(recorded.value("config%d_size%d" % (cfg, size))) == got
            assert a.numTriangles == prod.flat_desc(a.scene).contents.numTris
        finally:
            prod.destroy_demo(a)


def test_raw_hitable_list_element(prod, recorded, restate):
    """SURVEY 8a row a13, HitableList::Hit (geom/hit.cc:34-50) as a scene element: config 7 holds a raw list of spheres, cubes
    and triangles with duplicated members.  The flattened scene (restatement: reference topology and the quantized tree the
    device walks) must select what the compiled reference selects (stored, conftest.RecordedOutputs) -- ids by the labelling of
    oracle_driver.cc (spheres in reverse list order, then the other members in list order) -- including the equal-t ties
    between duplicates."""
    pinfo = prod.create_demo(7)
    try:
        w, h = 160, 90
        prod.set_viewport(pinfo, w, h)
        desc = prod.flat_desc(pinfo.scene)
        _, _, _, rays = restate.primary(desc, prod.camera_block(pinfo.camera), w, h, pinfo.settings.rayTMin, want_rays=True)
        assert desc.contents.numLeaves == 12
        for tree in (0, 3):
            restate.select_tree(tree)
            try:
                cr, ct, _ = restate.trace(desc, rays, pinfo.settings.rayTMin)
            finally:
                restate.select_tree(0)
            assert recorded.compare("primary_rank", cr)[2], "tree %d: ids differ" % tree
            assert recorded.compare("primary_t", ct)[2], "tree %d: t differs" % tree
        hit_members = set(int(x) for x in np.unique(cr))
        assert len(hit_members - {-1}) >= 6, hit_members             # duplicates never win: 9 of the 12 leaves can be seen at most
        # incoherent rays through the list's neighbourhood
        rng = np.random.default_rng(77)
        n = 20000
        rnd = np.zeros((n, 8), dtype=np.float32)
        rnd[:, 0:3] = rng.uniform([-2, -0.5, -2], [2, 2, 3], size=(n, 3))
        v = rng.normal(size=(n, 3)); rnd[:, 4:7] = v / np.linalg.norm(v, axis=1, keepdims=True)
        restate.select_tree(3)
        try:
            c_rank, c_t, _ = restate.trace(desc, rnd, 1e-4)
        finally:
            restate.select_tree(0)
        assert recorded.compare("random_rank", c_rank)[2] and recorded.compare("random_t", c_t)[2]
    finally:
        prod.destroy_demo(pinfo)


@pytest.mark.parametrize("name,stride", [("sinf", 53), ("cosf", 59), ("tanf", 61), ("asinf", 67), ("acosf", 71), ("atanf", 73), ("expf", 79), ("logf", 83),
                                         ("powf", 911), ("atan2f", 613)])
def test_restated_transcendentals_equal_the_host_c_library(name, stride):
    """include/rt_libm.h (what the device's shaders call) against the host C library (what the compiled reference calls):
    every `stride`-th float of the whole 2^32 range for the one-argument functions -- oracle/libm_check.cc with stride 1
    is the exhaustive run, a few minutes per function --, every stride-th x against twelve exponents plus random pairs for
    powf / atan2f.  Bit for bit; both sides run the library's FMA build on AVX2 hosts."""
    import os, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "oracle", "lib", "libm_check")
    if not os.path.exists(exe):
        subprocess.run(["g++", "-O2", "-mfma", "-ffp-contract=off", "-pthread", os.path.join(root, "oracle", "libm_check.cc"), "-o", exe, "-lm"], check=True)
    if "fma" not in open("/proc/cpuinfo").read():
        pytest.skip("this host has no FMA unit: glibc resolves its non-FMA build here, rt_libm.h restates the FMA build")
    out = subprocess.run([exe, name, str(stride)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and " 0 mismatches" in out.stdout, out.stdout + out.stderr


def write_test_obj(directory, grid=24):
    """A small OBJ + MTL that exercises the reference's conversion rules (loader/obj_loader.cc:113-245, :294-400): several
    shapes, faces with and without normals / texcoords, negative (relative) indices, Microfacet / Dielectric / Mirror /
    emissive materials and a shape without material (Lambertian 0.5 fallback)."""
    import os
    lines = ["mtllib parity.mtl"]
    nv = nvt = nvn = 0

    def v(x, y, z):
        nonlocal nv
        lines.append("v %.9g %.9g %.9g" % (x, y, z)); nv += 1; return nv

    def vt(a, b):
        nonlocal nvt
        lines.append("vt %.9g %.9g" % (a, b)); nvt += 1; return nvt

    def vn(x, y, z):
        nonlocal nvn
        lines.append("vn %.9g %.9g %.9g" % (x, y, z)); nvn += 1; return nvn

    # floor: displaced grid with normals and texcoords
    lines += ["g floor", "usemtl clay"]
    up = vn(0.0, 1.0, 0.0)
    idx = {}
    for j in range(grid + 1):
        for i in range(grid + 1):
            x, z = -2.0 + 4.0 * i / grid, -2.0 + 4.0 * j / grid
            idx[i, j] = (v(x, 0.05 * np.sin(3.0 * x) * np.cos(2.0 * z), z), vt(i / grid, j / grid))
    for j in range(grid):
        for i in range(grid):
            a, b, c, d = idx[i, j], idx[i + 1, j], idx[i + 1, j + 1], idx[i, j + 1]
            lines.append("f %d/%d/%d %d/%d/%d %d/%d/%d" % (a[0], a[1], up, c[0], c[1], up, b[0], b[1], up))
            lines.append("f %d/%d/%d %d/%d/%d %d/%d/%d" % (a[0], a[1], up, d[0], d[1], up, c[0], c[1], up))
    # a glass tetrahedron without normals (face normals are derived), relative indices
    lines += ["g gem", "usemtl glass"]
    for p in ((-0.6, 0.1, 0.2), (0.0, 0.1, 0.6), (0.1, 0.1, -0.1), (-0.2, 0.9, 0.2)):
        v(*p)
    lines += ["f -4 -3 -2", "f -4 -1 -3", "f -3 -1 -2", "f -2 -1 -4"]
    # a chrome box: positions + normals, no texcoords
    lines += ["g box", "usemtl chrome"]
    c0 = nv
    for p in [(0.5, 0.0, -0.6), (1.2, 0.0, -0.6), (1.2, 0.0, 0.1), (0.5, 0.0, 0.1), (0.5, 0.7, -0.6), (1.2, 0.7, -0.6), (1.2, 0.7, 0.1), (0.5, 0.7, 0.1)]:
        v(*p)
    faces = [((0, 1, 5, 4), (0, 0, -1)), ((1, 2, 6, 5), (1, 0, 0)), ((2, 3, 7, 6), (0, 0, 1)), ((3, 0, 4, 7), (-1, 0, 0)), ((4, 5, 6, 7), (0, 1, 0))]
    for quad, nrm in faces:
        n = vn(*nrm)
        q = [c0 + 1 + k for k in quad]
        lines.append("f %d//%d %d//%d %d//%d" % (q[0], n, q[1], n, q[2], n))
        lines.append("f %d//%d %d//%d %d//%d" % (q[0], n, q[2], n, q[3], n))
    # an emissive panel and a shape with no material at all
    lines += ["g lamp", "usemtl glow"]
    l = [v(-0.5, 2.2, -0.5), v(0.5, 2.2, -0.5), v(0.5, 2.2, 0.5), v(-0.5, 2.2, 0.5)]
    lines += ["f %d %d %d" % (l[0], l[1], l[2]), "f %d %d %d" % (l[0], l[2], l[3])]
    lines += ["g plain"]
    s = [v(-1.6, 0.0, -1.2), v(-1.0, 0.0, -1.2), v(-1.3, 0.8, -1.2)]
    lines.append("usemtl does_not_exist")
    lines.append("f %d %d %d" % tuple(s))
    open(os.path.join(directory, "parity.obj"), "w").write("\n".join(lines) + "\n")
    open(os.path.join(directory, "parity.mtl"), "w").write(
        "newmtl clay\nKd 0.7 0.45 0.3\nKs 0.2 0.2 0.2\nNs 40\nillum 2\n"
        "newmtl glass\nKd 0 0 0\nTf 0.9 0.95 1.0\nNi 1.45\nillum 4\n"
        "newmtl chrome\nKd 0.8 0.8 0.85\nillum 3\n"
        "newmtl glow\nKd 0.2 0.2 0.2\nKe 6 5 4\nPr 0.6\nPm 0.1\nillum 2\n")
    return os.path.join(directory, "parity.obj")


def load_obj_scene(lib, path):
    model = lib.Raylib_LoadOBJModel(path.encode())
    assert model
    lib.Raylib_FinalizeOBJModel(model)
    scene = lib.Raylib_CreateScene()
    lib.Raylib_AddOBJModelToScene(scene, model)
    lib.Raylib_SetSunIlluminance(scene, 5.0, 5.0, 5.0)
    lib.Raylib_SetSunDirection(scene, 0.2, -1.0, -0.3)
    lib.Raylib_FinalizeScene(scene)
    return model, scene


def test_obj_import_against_the_reference_conversion(prod, recorded, restate, tmp_path):
    """Raylib_LoadOBJModel -> Raylib_AddOBJModelToScene (SURVEY 8f row 4) against an oracle: config 8 of the scene client
    imports the same file through the CLIENT OBJECT API with the reference's conversion rules.  The product's importer
    must flatten to the very arrays its own object path produces, and the primary hits of that scene must be the compiled
    reference's (stored, conftest.RecordedOutputs), ids and t bit for bit."""
    import ctypes, os
    libc = ctypes.CDLL(None)
    path = write_test_obj(str(tmp_path))
    os.environ["DEMO_OBJ_PATH"] = path; libc.setenv(b"DEMO_OBJ_PATH", path.encode(), 1)
    try:
        pinfo = prod.create_demo(8)
        model, scene = load_obj_scene(prod.lib, path)
        try:
            a, b = prod.flat_desc(scene).contents, prod.flat_desc(pinfo.scene).contents
            assert a.numTris == b.numTris == pinfo.numTriangles == 2 * 24 * 24 + 4 + 10 + 2 + 1
            assert int(recorded.value("triangles")) == pinfo.numTriangles
            assert a.materialTypeMask == b.materialTypeMask == (1 << 5) | (1 << 2) | (1 << 3) | (1 << 0)
            for count, fields in (("numTris", [("triHot", 64), ("triCold", 64), ("triRank", 4), ("triGate", 4)]), ("numGates", [("gateBoxes", 32)]),
                                  ("numRefNodes", [("refNodes", 64)]), ("numWideNodes", [("quantNodes", 64)])):
                n = getattr(a, count)
                assert n == getattr(b, count), count
                for name, size in fields:
                    x = np.ctypeslib.as_array(ctypes.cast(getattr(a, name), ctypes.POINTER(ctypes.c_uint8)), shape=(n * size,))
                    y = np.ctypeslib.as_array(ctypes.cast(getattr(b, name), ctypes.POINTER(ctypes.c_uint8)), shape=(n * size,))
                    if name in ("triHot", "triCold"):
                        # material INDICES may be numbered differently (importer: .mtl order; object path: first use)
                        x, y = x.reshape(n, size).copy(), y.reshape(n, size).copy()
                        word = 13 * 4 if name == "triHot" else 60
                        x[:, word:word + 4] = 0; y[:, word:word + 4] = 0
                    assert np.array_equal(x, y), name
            w, h = pinfo.settings.viewportWidth, pinfo.settings.viewportHeight
            _, _, _, rays = restate.primary(prod.flat_desc(pinfo.scene), prod.camera_block(pinfo.camera), w, h,
                                            pinfo.settings.rayTMin, want_rays=True)
            for tree in (0, 3):
                restate.select_tree(tree)
                try:
                    cr, ct, _ = restate.trace(prod.flat_desc(scene), rays, pinfo.settings.rayTMin)
                finally:
                    restate.select_tree(0)
                assert (cr >= 0).mean() > 0.3
                assert recorded.compare("primary_rank", cr)[2] and recorded.compare("primary_t", ct)[2], "tree %d" % tree
        finally:
            prod.lib.RaylibB200_ReleaseInspection(scene)
            prod.lib.Raylib_DestroyScene(scene); prod.lib.Raylib_UnloadOBJModel(model)
            prod.destroy_demo(pinfo)
    finally:
        os.environ.pop("DEMO_OBJ_PATH", None); libc.unsetenv(b"DEMO_OBJ_PATH")
