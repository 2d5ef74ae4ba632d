"""Ray-level parity of the traversal kernels a render runs, through RaylibB200_TraceRaysStaged.

RaylibB200_TraceRays runs k_trace_rays (one ray per thread, no refill) and RaylibB200_PrimaryHits runs k_debug_view; almost
every ray of a frame goes through other code: k_extend (per-lane refill under the refill / walk thresholds, hit records
written as hits are accepted, a push to the material queue of the hit), the opt-in k_extend_pool, and k_shadow, the only
any-hit walk.  Here those kernels trace seeded ray sets -- incoherent rays, the adversarial families of
test_cpu_host._adversarial_rays, rays aimed at every kind of primitive, secondary-like rays leaving the restatement's own hit points, shutter times across moving
cubes -- under many schedules (grids of 1 and 2 CTAs refill every warp thousands of times), queue orders and thresholds.
Every answer is held to the exhaustive C restatement (oracle/rt_oracle.c) and, for closest hits, bit for bit to k_trace_rays.

Bars:
  * closest hit vs k_trace_rays: rank and t bits equal on every ray (the kernels share trav_step / trav_leaf: scheduling
    must not change an answer);
  * closest hit vs the restatement: no lost hits, rank mismatch <= 1e-5 (exact-tie budget of
    test_gpu_parity.test_incoherent_rays_against_restatement), t and the hit record's bu / bv (triangle barycentrics, cube
    face) bit-identical wherever the ranks agree;
  * queues: every ray in exactly one queue; a hit in the queue of its primitive's material type, a miss in the miss queue;
  * any hit: occluded exactly where the restatement finds any hit -- no lost occluder, no hit that no exact test accepts.
Failing rays are printed with origin, direction, time and both answers.
"""
import ctypes as C
import numpy as np
import pytest
from conftest import bits
from test_cpu_host import _adversarial_rays

SCENES = [(2, 0), (4, 24), (6, 0), (1, 0), (5, 40), (7, 0)]
QUEUE_MISS = 6
F32_EPS = float(np.finfo(np.float32).eps)


# ---- scene tables (host copy of the flattened scene: what the device uploads) ------------------------------------------

def _words(ptr, count, dtype):
    if not ptr or count == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array((C.c_uint32 * count).from_address(ptr)).view(dtype).copy()


class Tables:
    """Rank and material type of every primitive of a flattened scene, and the triangle / cube geometry."""

    def __init__(self, desc):
        d = desc.contents
        self.tri_hot = _words(d.triHot, 16 * d.numTris, np.float32).reshape(-1, 16)
        tri_cold = _words(d.triCold, 16 * d.numTris, np.uint32).reshape(-1, 16)
        self.cubes = _words(d.cubes, 12 * d.numCubes, np.float32).reshape(-1, 12)
        self.spheres = _words(d.spheres, 4 * d.numSpheres, np.float32).reshape(-1, 4)
        mat_type = _words(d.materials, 16 * d.numMaterials, np.uint32).reshape(-1, 16)[:, 0].astype(np.int32)
        self.rank = {1: _words(d.triRank, d.numTris, np.uint32), 3: _words(d.sphereRank, d.numSpheres, np.uint32),
                     5: _words(d.cubeRank, d.numCubes, np.uint32)}
        self.mat = {1: mat_type[tri_cold[:, 15]] if d.numTris else np.zeros(0, np.int32),
                    3: mat_type[_words(d.sphereMaterial, d.numSpheres, np.uint32)],
                    5: mat_type[self.cubes.view(np.uint32)[:, 7]] if d.numCubes else np.zeros(0, np.int32)}
        # rank -> (kind, index)
        self.by_rank = {}
        for kind, ranks in self.rank.items():
            for i, r in enumerate(ranks):
                self.by_rank[int(r)] = (kind, i)

    def decode(self, ref_bits):
        """Device primitive references -> (rank, material type, kind); -1 where the reference names no primitive."""
        ref_bits = np.asarray(ref_bits, dtype=np.uint32)
        kind = (ref_bits >> 28).astype(np.int64)
        idx = (ref_bits & 0x0FFFFFFF).astype(np.int64)
        rank = np.full(len(ref_bits), -1, dtype=np.int64)
        mat = np.full(len(ref_bits), -1, dtype=np.int32)
        for k in (1, 3, 5):
            sel = (kind == k) & (idx < len(self.rank[k]))
            rank[sel] = self.rank[k][idx[sel]]
            mat[sel] = self.mat[k][idx[sel]]
        return rank, mat, kind


def scene_box(desc):
    d = desc.contents
    lo = np.array(d.rootMin[:], dtype=np.float64); hi = np.array(d.rootMax[:], dtype=np.float64)
    return np.maximum(lo, -50.0), np.minimum(hi, 50.0)        # configs 1 and 6 hold a ground sphere of radius 100-1000


# ---- ray sets (seeded, float32) ----------------------------------------------------------------------------------------

def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def incoherent_rays(lo, hi, n, seed):
    """Origins uniform in the scene box, directions uniform on the sphere, shutter times in [0, 2)."""
    rng = np.random.default_rng(seed)
    rays = np.zeros((n, 8), dtype=np.float32)
    rays[:, 0:3] = rng.uniform(lo, hi, size=(n, 3))
    rays[:, 3] = rng.uniform(0.0, 2.0, size=n)
    rays[:, 4:7] = _unit(rng, n)
    return rays


def secondary_rays(restate, desc, lo, hi, n, seed):
    """Origins at the restatement's own hit points (o + t d, rounded to float32 as a shade stage does), random directions:
    tMin decides whether a ray finds the surface it starts on."""
    src = incoherent_rays(lo, hi, 3 * n, seed)
    rank, t, _ = restate.trace(desc, src, 1e-4)
    src, t = src[rank >= 0][:n], t[rank >= 0][:n]
    rng = np.random.default_rng(seed + 1)
    rays = np.zeros((len(src), 8), dtype=np.float32)
    rays[:, 0:3] = src[:, 0:3] + t[:, None] * src[:, 4:7]
    rays[:, 3] = src[:, 3]
    rays[:, 4:7] = _unit(rng, len(src))
    return rays


def shutter_rays(tables, lo, hi, n, seed):
    """Config 6: rays aimed into each cube's box swept over its motion, at shutter times before, at and after the start of
    the motion."""
    rng = np.random.default_rng(seed)
    rays = np.zeros((n, 8), dtype=np.float32)
    rays[:, 0:3] = rng.uniform(lo, hi, size=(n, 3))
    cube = tables.cubes[rng.integers(0, len(tables.cubes), size=n)]
    start = cube[:, 3].astype(np.float64)
    time = start + rng.uniform(-1.0, 3.0, size=n)
    time[: n // 8] = start[: n // 8]                                  # exactly at the start of the motion
    move = cube[:, 8:11] * np.maximum(0.0, time - start)[:, None]
    target = rng.uniform(cube[:, 0:3] + move, cube[:, 4:7] + move)
    d = target - rays[:, 0:3]
    rays[:, 3] = time
    rays[:, 4:7] = d / np.linalg.norm(d, axis=1, keepdims=True)
    return rays


def aimed_rays(tables, lo, hi, n, seed):
    """Rays from origins in the scene box aimed at a point of a primitive drawn uniformly from all of them: small primitives
    next to a large ground sphere are hit often, and so are the duplicated members of config 7's hitable list, whose equal t
    only the tie rule decides."""
    rng = np.random.default_rng(seed)
    rays = np.zeros((n, 8), dtype=np.float32)
    rays[:, 0:3] = rng.uniform(lo, hi, size=(n, 3))
    rays[:, 3] = rng.uniform(0.0, 2.0, size=n)
    nt, ns, nc = len(tables.tri_hot), len(tables.spheres), len(tables.cubes)
    pick = rng.integers(0, nt + ns + nc, size=n)
    target = np.zeros((n, 3))
    tri, sph, cub = pick < nt, (pick >= nt) & (pick < nt + ns), pick >= nt + ns
    if tri.any():
        q = tables.tri_hot[pick[tri]].astype(np.float64)
        u = rng.random(tri.sum()); v = rng.random(tri.sum()); flip = u + v > 1.0
        u[flip], v[flip] = 1.0 - u[flip], 1.0 - v[flip]
        target[tri] = q[:, 0:3] + u[:, None] * q[:, 6:9] + v[:, None] * q[:, 9:12]
    if sph.any():
        s = tables.spheres[pick[sph] - nt].astype(np.float64)
        target[sph] = s[:, 0:3] + 0.9 * s[:, 3:4] * _unit(rng, sph.sum()) * rng.random((sph.sum(), 1))
    if cub.any():
        c = tables.cubes[pick[cub] - nt - ns].astype(np.float64)
        target[cub] = rng.uniform(c[:, 0:3], c[:, 4:7])
    d = target - rays[:, 0:3]
    rays[:, 4:7] = d / np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-30)
    return rays


def camera_hit_points(gpu, restate, info, desc, width=128, height=72):
    """Where real sun rays start: the restatement's hit points of the scene's camera rays (with their shutter times)."""
    gpu.set_viewport(info, width, height)
    rank, t, _, rays = restate.primary(desc, gpu.camera_block(info.camera), width, height, info.settings.rayTMin, want_rays=True)
    rays, t = rays[rank >= 0], t[rank >= 0]
    out = rays.copy()
    out[:, 0:3] = rays[:, 0:3] + t[:, None] * rays[:, 4:7]
    return out


def cell_order(rays, lo, hi, cells=16):
    """Queue order of a binned bounce: rays sorted by the cell of their origin in the scene box."""
    c = np.clip(((rays[:, 0:3] - lo) / np.maximum(hi - lo, 1e-30) * cells).astype(np.int64), 0, cells - 1)
    return np.argsort((c[:, 0] * cells + c[:, 1]) * cells + c[:, 2], kind="stable").astype(np.uint32)


def tmin_values(info):
    return sorted({0.0, float(np.float32(1e-4)), float(np.float32(info.settings.rayTMin))})      # {0, 1e-4, the scene's own}


# ---- comparisons -------------------------------------------------------------------------------------------------------

def _ray_text(rays, i):
    return "ray %d o=%r d=%r time=%r" % (i, rays[i, 0:3].tolist(), rays[i, 4:7].tolist(), float(rays[i, 3]))


class Reference:
    """The restatement's answer (with hit-record fields) and k_trace_rays' answer for one ray set."""

    def __init__(self, gpu, restate, scene, desc, rays, tmin):
        self.rank, self.t, uv, face, self.mat, _ = restate.trace_hits(desc, rays, tmin)
        hit = self.rank >= 0
        # the record a device path holds: triangle barycentrics, the face of a cube, zeros for a sphere
        self.bu = np.where(face >= 0, face.astype(np.float32), uv[:, 0]).astype(np.float32)
        self.bv = np.where(face >= 0, np.float32(0.0), uv[:, 1]).astype(np.float32)
        self.bu[~hit] = 0.0; self.bv[~hit] = 0.0
        self.trank, self.tt = gpu.trace_rays(scene, rays, tmin)


def check_closest(label, rays, ref, tables, queue, record, counts):
    """Bars of a closest-hit stage launch; returns the printed summary line.  Raises with the failing rays on a violation."""
    n = len(rays)
    problems = []
    if int(counts.astype(np.int64).sum()) != n:
        problems.append("queue counters sum to %d for %d rays" % (int(counts.astype(np.int64).sum()), n))
    bad_queue = np.nonzero((queue < 0) | (queue > QUEUE_MISS))[0]
    if len(bad_queue):
        problems.append("%d rays in no queue or in several (first %r)" % (len(bad_queue), bad_queue[:5].tolist()))
    t, bu, bv = record[:, 0], record[:, 1], record[:, 2]
    rank, mat, _ = tables.decode(record[:, 3].view(np.uint32))
    hit = queue != QUEUE_MISS
    rank = np.where(hit, rank, -1)
    # the queue is the material type of the primitive the record names
    wrong_queue = np.nonzero(hit & (queue != mat))[0]
    # against k_trace_rays: every ray, zero tolerance
    vs_trace = np.nonzero((rank != ref.trank) | (hit & (bits(t) != bits(ref.tt))))[0]
    # against the restatement
    lost = np.nonzero((rank < 0) & (ref.rank >= 0))[0]
    differ = np.nonzero(rank != ref.rank)[0]
    same = (rank == ref.rank) & (rank >= 0)
    record_differs = np.nonzero(same & ((bits(t) != bits(ref.t)) | (bits(bu) != bits(ref.bu)) | (bits(bv) != bits(ref.bv))))[0]
    queue_vs_restatement = np.nonzero(same & (queue != ref.mat))[0]
    line = ("%s: rays %d, hit fraction %.3f, rank mismatches %d, lost hits %d, vs k_trace_rays %d, record mismatches %d, "
            "wrong queues %d" % (label, n, float((ref.rank >= 0).mean()), len(differ), len(lost), len(vs_trace),
                                 len(record_differs), len(wrong_queue) + len(queue_vs_restatement)))
    for what, idx in (("differs from k_trace_rays", vs_trace), ("lost hit", lost), ("rank differs from the restatement", differ),
                      ("hit record differs", record_differs), ("queue is not the hit's material type", wrong_queue),
                      ("queue is not the restatement's material type", queue_vs_restatement)):
        if len(idx) and (what != "rank differs from the restatement" or len(differ) > 1e-5 * n):
            problems.append("%d rays: %s" % (len(idx), what))
        for i in idx[:4]:
            print("  %s: %s\n    stage: queue %d rank %d t %r bu %r bv %r | k_trace_rays: rank %d t %r | restatement: rank %d "
                  "t %r bu %r bv %r material %d" % (what, _ray_text(rays, i), queue[i], rank[i], float(t[i]), float(bu[i]),
                                                    float(bv[i]), ref.trank[i], float(ref.tt[i]), ref.rank[i], float(ref.t[i]),
                                                    float(ref.bu[i]), float(ref.bv[i]), ref.mat[i]))
    print(line)
    assert not problems, label + ": " + "; ".join(problems)
    return line


def closest_variants(rays, lo, hi, seed):
    """(label, keyword arguments of trace_rays_staged): grids, thresholds, queue orders, the pooled kernel."""
    n = len(rays)
    rng = np.random.default_rng(seed)
    v = [("k_extend persistent grid", {}), ("k_extend 1 CTA", dict(grid_ctas=1)), ("k_extend 2 CTAs", dict(grid_ctas=2))]
    for refill in (1, 20, 32):
        for walk in (1, 20, 32):
            v.append(("k_extend 2 CTAs refill %d walk %d" % (refill, walk), dict(grid_ctas=2, refill=refill, walk=walk)))
    orders = {"reversed": np.arange(n, dtype=np.uint32)[::-1].copy(), "random": rng.permutation(n).astype(np.uint32),
              "origin cell": cell_order(rays, lo, hi)}
    for name, order in orders.items():
        v.append(("k_extend persistent grid, %s order" % name, dict(order=order)))
        v.append(("k_extend 3 CTAs, %s order" % name, dict(order=order, grid_ctas=3)))
    v += [("k_extend_pool persistent grid", dict(mode="extend_pool")),
          ("k_extend_pool 1 CTA node 1 refill 64", dict(mode="extend_pool", grid_ctas=1, pool_node=1, pool_refill=64)),
          ("k_extend_pool 2 CTAs node 32 refill 1", dict(mode="extend_pool", grid_ctas=2, pool_node=32, pool_refill=1)),
          ("k_extend_pool 1 CTA node 32 refill 32, random order", dict(mode="extend_pool", grid_ctas=1, pool_node=32,
                                                                       pool_refill=32, order=orders["random"]))]
    return v


def closest_ray_sets(gpu, restate, info, desc, tables, cfg, n):
    """(name, rays, tMin) of the closest-hit cases of a scene."""
    lo, hi = scene_box(desc)
    d = desc.contents
    sets = [("incoherent", incoherent_rays(lo, hi, n, 100 + cfg), 1e-4),
            ("adversarial", _adversarial_rays(np.array(d.rootMin[:], np.float64), np.array(d.rootMax[:], np.float64), n, 11 + cfg), 1e-4),
            ("aimed", aimed_rays(tables, lo, hi, n, 150 + cfg), 1e-4)]
    sec = secondary_rays(restate, desc, lo, hi, n, 200 + cfg)
    sets += [("secondary", sec, tmin) for tmin in tmin_values(info)]
    if cfg == 6:
        sets.append(("shutter", shutter_rays(tables, lo, hi, n, 300 + cfg), 1e-4))
    return sets


# ---- GPU tests ---------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("cfg,size", SCENES)
def test_closest_hit_stages_against_restatement(gpu, restate, cfg, size):
    """k_extend and k_extend_pool under every schedule and queue order give k_trace_rays' answer on every ray, the
    restatement's within its bars, and push every ray to the queue of its hit's material."""
    info = gpu.create_demo(cfg, size)
    try:
        desc = gpu.flat_desc(info.scene)
        tables = Tables(desc)
        lo, hi = scene_box(desc)
        for name, rays, tmin in closest_ray_sets(gpu, restate, info, desc, tables, cfg, 24000):
            ref = Reference(gpu, restate, info.scene, desc, rays, tmin)
            for label, kw in closest_variants(rays, lo, hi, 400 + cfg):
                queue, record, counts = gpu.trace_rays_staged(info.scene, rays, tmin, **kw)
                check_closest("config%d %s tMin %g, %s" % (cfg, name, tmin, label), rays, ref, tables, queue, record, counts)
    finally:
        gpu.destroy_demo(info)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,size", SCENES)
def test_extend_statistics_build(gpu, restate, cfg, size):
    """k_extend<true>: the answers of k_extend, statRays = n, and the reference-work counters that k_trace_rays<true> reports
    for the same rays."""
    info = gpu.create_demo(cfg, size)
    gpu.lib.RaylibB200_SetCollectStats(1)          # uploads the scene again, with the reference topology the counters walk
    try:
        desc = gpu.flat_desc(info.scene)
        tables = Tables(desc)
        lo, hi = scene_box(desc)
        rays = np.concatenate([incoherent_rays(lo, hi, 12000, 500 + cfg),
                               _adversarial_rays(np.array(desc.contents.rootMin[:], np.float64),
                                                 np.array(desc.contents.rootMax[:], np.float64), 12000, 600 + cfg)])
        ref = Reference(gpu, restate, info.scene, desc, rays, 1e-4)
        want = gpu.last_stats()
        assert want.statRays == len(rays) and want.refBoxTests > 0
        for label, kw in (("persistent grid", {}), ("1 CTA", dict(grid_ctas=1)), ("2 CTAs refill 32 walk 1", dict(grid_ctas=2, refill=32, walk=1))):
            queue, record, counts = gpu.trace_rays_staged(info.scene, rays, 1e-4, mode="extend_stats", **kw)
            st = gpu.last_stats()
            check_closest("config%d k_extend<true> %s" % (cfg, label), rays, ref, tables, queue, record, counts)
            got = (st.statRays, st.refBoxTests, st.refTriTests, st.refSphereTests)
            print("  counters: statRays %d, reference box / triangle / sphere tests %d / %d / %d (k_trace_rays<true>: %d / %d / %d)"
                  % (got + (want.refBoxTests, want.refTriTests, want.refSphereTests)))
            assert got == (len(rays), want.refBoxTests, want.refTriTests, want.refSphereTests)
            assert st.extendLaunches == 1 and st.rayQueries == len(rays)
    finally:
        gpu.lib.RaylibB200_SetCollectStats(0)
        gpu.destroy_demo(info)


def sun_directions(desc, seed):
    """The scene's own sun, the six axis directions with the other components +0.0 and -0.0, directions with denormal and
    tiny components, and random ones."""
    dirs = []
    sun = np.array(desc.contents.sunDirection[:], dtype=np.float32)
    if np.any(sun != 0.0):
        dirs.append(sun)
    for axis in range(3):
        for sign in (1.0, -1.0):
            for zero in (0.0, -0.0):
                d = np.full(3, zero, dtype=np.float32)
                d[axis] = sign
                dirs.append(d)
    dirs += [np.array(v, dtype=np.float32) for v in ((-1e-42, -1.0, 1e-42), (3e-39, -1.0, -0.0), (1.0, -1e-20, 1e-42),
                                                      (0.3, -0.9, -3e-39), (-1e-20, 1e-20, -1.0))]
    dirs += list(_unit(np.random.default_rng(seed), 12).astype(np.float32))
    return dirs


ANY_HIT_SCHEDULES = [{}, dict(grid_ctas=1), dict(grid_ctas=2, refill=1, walk=32), dict(grid_ctas=2, refill=32, walk=1),
                     dict(grid_ctas=3, refill=20, walk=20)]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,size", SCENES)
def test_any_hit_stage_against_restatement(gpu, restate, cfg, size):
    """k_shadow: a sun ray is occluded exactly where the exhaustive restatement finds any hit along it -- from camera hit
    points (where real sun rays start), incoherent, adversarial and secondary origins, toward the scene's sun, the axes
    (both signs of zero), directions with denormal components and random ones, under several schedules and queue orders."""
    info = gpu.create_demo(cfg, size)
    try:
        desc = gpu.flat_desc(info.scene)
        d = desc.contents
        lo, hi = scene_box(desc)
        rng = np.random.default_rng(700 + cfg)
        parts = [camera_hit_points(gpu, restate, info, desc), incoherent_rays(lo, hi, 4000, 710 + cfg),
                 _adversarial_rays(np.array(d.rootMin[:], np.float64), np.array(d.rootMax[:], np.float64), 4000, 720 + cfg),
                 secondary_rays(restate, desc, lo, hi, 4000, 730 + cfg)]
        origins = np.concatenate([p[rng.permutation(len(p))[:4000]] for p in parts])
        tmin = float(info.settings.rayTMin)
        total_lost = total_phantom = 0
        for j, sun in enumerate(sun_directions(desc, 740 + cfg)):
            rays = origins.copy()
            rays[:, 4:7] = -sun                     # k_shadow traces along -sunDirection
            crank, _, _ = restate.trace(desc, rays, tmin)
            n = len(rays)
            order = [None, np.arange(n, dtype=np.uint32)[::-1].copy(), rng.permutation(n).astype(np.uint32)][j % 3]
            schedule = ANY_HIT_SCHEDULES[j % len(ANY_HIT_SCHEDULES)]
            queue, radiance, _ = gpu.trace_rays_staged(info.scene, rays, tmin, mode="shadow", sun_direction=sun, order=order,
                                                       **schedule)
            assert (queue >= 0).all(), "%d paths end with a radiance that is neither the sun nor 0: %r" % (
                int((queue < 0).sum()), radiance[queue < 0][:3].tolist())
            occluded = queue == 1
            lost = np.nonzero(~occluded & (crank >= 0))[0]
            phantom = np.nonzero(occluded & (crank < 0))[0]
            print("config%d any hit, sun %r, schedule %r: rays %d, occluded fraction %.3f, lost occluders %d, phantom hits %d"
                  % (cfg, sun.tolist(), schedule, n, float(occluded.mean()), len(lost), len(phantom)))
            for what, idx in (("lost occluder", lost), ("phantom hit", phantom)):
                for i in idx[:4]:
                    print("  %s: %s | k_shadow: %s | restatement: rank %d" % (what, _ray_text(rays, i),
                          "occluded" if occluded[i] else "visible", crank[i]))
            total_lost += len(lost); total_phantom += len(phantom)
        assert total_lost == 0, "k_shadow let the sun through %d occluders the restatement finds" % total_lost
        assert total_phantom == 0, "k_shadow reported %d occlusions no exact test accepts" % total_phantom
    finally:
        gpu.destroy_demo(info)


@pytest.mark.gpu
def test_extend_at_full_width(gpu, restate):
    """4 Mi rays on the 30k-triangle scatter: the persistent grid (about 148 SMs x 9 CTAs x 128 lanes) refills every lane many
    times at full width, in a random order."""
    info = gpu.create_demo(4, 24)
    try:
        desc = gpu.flat_desc(info.scene)
        tables = Tables(desc)
        lo, hi = scene_box(desc)
        rays = incoherent_rays(lo, hi, 4 << 20, 800)
        ref = Reference(gpu, restate, info.scene, desc, rays, 1e-4)
        order = np.random.default_rng(801).permutation(len(rays)).astype(np.uint32)
        for label, kw in (("k_extend persistent grid, random order", dict(order=order)),
                          ("k_extend_pool persistent grid, random order", dict(mode="extend_pool", order=order))):
            queue, record, counts = gpu.trace_rays_staged(info.scene, rays, 1e-4, **kw)
            check_closest("config4 4 Mi rays, " + label, rays, ref, tables, queue, record, counts)
    finally:
        gpu.destroy_demo(info)


# ---- CPU tests ---------------------------------------------------------------------------------------------------------

def test_staged_trace_refuses_bad_arguments(prod):
    """Bad arguments are refused with a message before any device is touched; valid ones without a device get the no-device
    message."""
    info = prod.create_demo(6, 0)
    lib = prod.lib
    try:
        n = 8
        rays = np.zeros((n, 8), dtype=np.float32)
        rays[:, 6] = -1.0
        order = np.arange(n, dtype=np.uint32)
        queue = np.empty(n, dtype=np.int32)
        hit = np.empty((n, 4), dtype=np.float32)
        counts = np.empty(7, dtype=np.uint32)
        sun = np.array([0.0, -1.0, 0.0], dtype=np.float32)
        p = lambda a: None if a is None else a.ctypes.data

        def call(scene=info.scene, mode=0, rays=rays, order=order, count=n, sun=sun, schedule=(0, 0, 0, 0, 0), queue=queue, hit=hit):
            return lib.RaylibB200_TraceRaysStaged(scene, mode, p(rays), p(order), count, 1e-4, p(sun), *schedule,
                                                  p(queue), p(hit), p(counts))

        def refused(why, **kw):
            assert call(**kw) == 0
            msg = prod.last_error()
            assert msg.startswith("RaylibB200_TraceRaysStaged: ") and why in msg, msg

        refused("null scene", scene=0)
        refused("null ray, order or output buffer", rays=None)
        refused("null ray, order or output buffer", order=None)
        refused("null ray, order or output buffer", queue=None)
        refused("null ray, order or output buffer", hit=None)
        refused("ray count", count=0)
        refused("ray count", count=-5)
        refused("ray count", count=1 << 31)                   # refused before the order is read
        refused("unknown mode", mode=4)
        refused("unknown mode", mode=-1)
        refused("not a permutation", order=np.array([0, 1, 2, 3, 4, 5, 6, 6], dtype=np.uint32))
        refused("not a permutation", order=np.array([0, 1, 2, 3, 4, 5, 6, 8], dtype=np.uint32))
        for bad in ((0.0, 0.0, 0.0), (-0.0, 0.0, -0.0), (np.nan, -1.0, 0.0), (0.0, np.inf, 0.0), (0.0, -1.0, -np.inf)):
            refused("finite and non-zero", mode=3, sun=np.array(bad, dtype=np.float32))
        refused("needs a sun direction", mode=3, sun=None)
        for schedule in ((33, 0, 0, 0, 0), (0, 33, 0, 0, 0), (0, 0, 33, 0, 0), (0, 0, 0, 65, 0), (0, 0, 0, 0, 4097)):
            refused("scheduling out of range", schedule=schedule)
        # closest-hit modes do not read the sun direction
        for mode in range(4):
            ok = call(mode=mode, sun=sun if mode == 3 else None, schedule=(32, 1, 32, 64, 4096))
            if prod.device_count() <= 0:
                assert ok == 0 and "no CUDA device" in prod.last_error(), prod.last_error()
            else:
                assert ok == 1, prod.last_error()
    finally:
        prod.destroy_demo(info)


@pytest.mark.parametrize("cfg,size", SCENES)
def test_restatement_hits_agree_with_trace(prod, restate, cfg, size):
    """rt_oracle_trace_hits answers rt_oracle_trace's rank and t, with the same work counts, and its material type is the
    type of the ranked primitive's material."""
    info = prod.create_demo(cfg, size)
    try:
        desc = prod.flat_desc(info.scene)
        tables = Tables(desc)
        lo, hi = scene_box(desc)
        d = desc.contents
        rays = np.concatenate([incoherent_rays(lo, hi, 6000, 900 + cfg),
                               _adversarial_rays(np.array(d.rootMin[:], np.float64), np.array(d.rootMax[:], np.float64), 6000, 910 + cfg),
                               secondary_rays(restate, desc, lo, hi, 3000, 920 + cfg)])
        for tmin in (0.0, 1e-4):
            rank, t, counts = restate.trace(desc, rays, tmin)
            rank2, t2, uv, face, mat, counts2 = restate.trace_hits(desc, rays, tmin)
            assert (rank >= 0).mean() > 0.05
            assert np.array_equal(rank, rank2) and np.array_equal(bits(t), bits(t2)) and counts == counts2
            hit = rank >= 0
            kinds = np.array([tables.by_rank[int(r)][0] if r >= 0 else 0 for r in rank])
            want = np.array([tables.mat[k][i] for k, i in (tables.by_rank[int(r)] for r in rank[hit])], dtype=np.int32)
            assert np.array_equal(mat[hit], want) and (mat[~hit] == -1).all()
            assert ((face >= 0) == (kinds == 5)).all() and (face[kinds == 5] <= 5).all()
            assert (uv[kinds != 1] == 0.0).all()
    finally:
        prod.destroy_demo(info)


@pytest.mark.parametrize("cfg,size", SCENES)
def test_restatement_hit_details_rederive_the_hit_point(prod, restate, cfg, size):
    """The barycentrics of a triangle hit give back o + t d through v0 + u e1 + v e2, and a cube hit lies on the plane of
    the face it names (moved to the ray's time), within float rounding."""
    info = prod.create_demo(cfg, size)
    try:
        desc = prod.flat_desc(info.scene)
        tables = Tables(desc)
        lo, hi = scene_box(desc)
        rays = np.concatenate([incoherent_rays(lo, hi, 8000, 950 + cfg), secondary_rays(restate, desc, lo, hi, 4000, 960 + cfg)])
        if len(tables.cubes):
            rays = np.concatenate([rays, shutter_rays(tables, lo, hi, 4000, 970 + cfg)])
        rank, t, uv, face, _, _ = restate.trace_hits(desc, rays, 1e-4)
        o = rays[:, 0:3].astype(np.float64); dd = rays[:, 4:7].astype(np.float64)
        p = o + t.astype(np.float64)[:, None] * dd
        scale = np.abs(o).max(axis=1) + np.abs(t.astype(np.float64)) * np.abs(dd).max(axis=1) + 1.0
        tri_hits = cube_hits = 0
        for i in np.nonzero(rank >= 0)[0]:
            kind, idx = tables.by_rank[int(rank[i])]
            if kind == 1:
                q = tables.tri_hot[idx].astype(np.float64)
                u, v = float(uv[i, 0]), float(uv[i, 1])
                assert u >= 0.0 and v >= 0.0 and u + v <= 1.0, (i, u, v)
                pb = q[0:3] + u * q[6:9] + v * q[9:12]
                tol = 64.0 * F32_EPS * (scale[i] + np.abs(q[0:3]).max() + np.abs(q[6:9]).max() + np.abs(q[9:12]).max())
                assert np.abs(pb - p[i]).max() <= tol, (_ray_text(rays, i), pb.tolist(), p[i].tolist(), tol)
                tri_hits += 1
            elif kind == 5:
                c = tables.cubes[idx].astype(np.float64)
                move = c[8:11] * max(0.0, float(np.float32(rays[i, 3]) - np.float32(c[3])))
                axis, high = divmod(int(face[i]), 2)
                plane = (c[4 + axis] if high else c[axis]) + move[axis]
                tol = 16.0 * F32_EPS * (scale[i] + abs(plane))
                assert abs(p[i, axis] - plane) <= tol, (_ray_text(rays, i), int(face[i]), p[i].tolist(), plane)
                cube_hits += 1
        print("config%d: %d triangle hits and %d cube hits re-derived" % (cfg, tri_hits, cube_hits))
        assert tri_hits + cube_hits > 0 or cfg == 1
    finally:
        prod.destroy_demo(info)
