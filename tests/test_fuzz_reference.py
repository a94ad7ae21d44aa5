"""Adversarial batches (tests/tools/fuzz_ref.py): axis-aligned and coincident poses, touching surfaces, extreme
scales, symmetric hulls, degenerate meshes and random request fields, compared record by record between the
reference build (oracle/_ref, or its recorded answers where it is not built), the oracle and the device code --
compiled for the host here, the real kernels under `-m gpu`.  The rows on which the reference itself is undefined
(Project::ProjectResult read uninitialised for an exactly degenerate simplex, internal/intersect.h:58-70) are
recognised and excluded.
"""
import pytest

from tests.tools import fuzz_ref


@pytest.mark.parametrize("first", [1, 41, 81])
def test_fuzz_oracle_reference_and_device_code(first):
    for seed in range(first, first + 40):
        ok, tag = fuzz_ref.one_round(seed, 1500, True, True)
        assert ok, tag


@pytest.mark.parametrize("lanes,seeds", [(2, (3, 4, 5)), (8, (3, 4))])
def test_fuzz_device_code_through_lane_groups(lanes, seeds):
    """the rounds the GPU failed (seeds 3 and 4 at n = 4000, see below) with phase 1 run by lane groups of host
    threads (tests/emu lanesim): fails on the code of that GPU run ("the lanes of a group disagreed"), passes now"""
    from tests.common import EmuScene
    for seed in seeds:
        dev = EmuScene()
        dev.lanes = lanes
        ok, tag = fuzz_ref.one_round(seed, 4000, True, dev)
        assert ok, tag


def test_fuzz_every_contact_of_mesh_pairs():
    """the mesh collide cases of the rounds through batch_collide_contacts: numContacts() and contacts[1..]"""
    fuzz_ref.CONTACTS[0] = True
    try:
        for seed in range(200, 230):
            ok, tag = fuzz_ref.one_round(seed, 1500, True, True)
            assert ok, tag
    finally:
        fuzz_ref.CONTACTS[0] = False


def test_fuzz_plane_family():
    """the rounds with Halfspace / Plane geometries added (axis-aligned, tilted, parallel and mirrored planes against
    every shape, hull and each other): reference build, oracle and the host build of the device code.  (On the GPU the
    family is covered by tests/test_plane_halfspace.py; the GPU fuzz below keeps the rounds it was confirmed on.)"""
    fuzz_ref.PLANES[0] = True
    try:
        for seed in range(300, 340):
            ok, tag = fuzz_ref.one_round(seed, 1500, True, True)
            assert ok, tag
    finally:
        fuzz_ref.PLANES[0] = False


def test_fuzz_drifted_rotations():
    """the rounds with coaxial, nearly touching pairs under rotations that are orthonormal only to 1e-14 ... 1e-8
    (fuzz_ref --drift): reference build, oracle and the host build of the device code"""
    fuzz_ref.DRIFT[0] = True
    try:
        for seed in range(400, 425):
            ok, tag = fuzz_ref.one_round(seed, 1500, True, True)
            assert ok, tag
    finally:
        fuzz_ref.DRIFT[0] = False


def test_degenerate_sizes():
    """shapes with sizes that are exactly zero -- a point for a sphere, a segment for a capsule or a cylinder, a
    disc, a plate, a needle of a box: the reference takes them as they are (no size checks in the constructors), so
    does the arena; reference build, oracle and host build of the device code on 20 000 random pairs of them"""
    import numpy as np
    from tests.common import P, compare_distance, make_scenes, ref_agrees
    from hppfcl_b200 import workloads as W
    rng = np.random.default_rng(5)
    sc = make_scenes(ref=True)
    types, params = [], []
    for t in (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER, P.GEOM_CONE, P.GEOM_ELLIPSOID):
        for _ in range(12):
            p = rng.uniform(0.1, 0.6, 3)
            p[rng.random(3) < 0.4] = 0.0
            if t == P.GEOM_SPHERE:
                p[1:] = 0
            if t in (P.GEOM_CAPSULE, P.GEOM_CYLINDER, P.GEOM_CONE):
                p[2] = 0
            types.append(t)
            params.append(p)
    h = sc.register_shapes(P.make_shapes(types, params))
    sc.commit()
    n = 20000
    h1, h2 = h[rng.integers(0, len(h), n)], h[rng.integers(0, len(h), n)]
    t1 = W.random_transforms(rng, n, (-.5, -.5, -.5), (.5, .5, .5))
    t2 = W.random_transforms(rng, n, (-.5, -.5, -.5), (.5, .5, .5))
    for fn, req in (("batch_distance", P.DistanceRequestPOD()), ("batch_collide", P.CollisionRequestPOD()),
                    ("batch_collide", P.CollisionRequestPOD(enable_contact=0, security_margin=0.05)),
                    ("batch_distance", P.DistanceRequestPOD(gjk_variant=P.NesterovAcceleration))):
        ro = getattr(sc.b["oracle"], fn)(h1, t1, h2, t2, req, nthreads=0)
        compare_distance(ro, getattr(sc.b["emu"], fn)(h1, t1, h2, t2, req), what=fn + ", degenerate sizes")
        ref_agrees(sc, fn, ro, (h1, t1, h2, t2, req), fn + ", degenerate sizes")


def test_extreme_request_fields():
    """request fields at and beyond the ends of their ranges (no iterations at all, tolerances of 1 and of 1e-300,
    margins of +-DBL_MAX and infinity, a negative upper bound, negative and huge collision thresholds, ...): none of
    them is refused by the reference, all of them must give the same records in the reference build, the oracle and
    the host build of the device code"""
    import numpy as np
    from tests.common import P, compare_distance, make_scenes, ref_agrees
    from hppfcl_b200 import workloads as W
    rng = np.random.default_rng(6)
    sc = make_scenes(ref=True)
    h = sc.register_shapes(W.random_primitive_shapes(rng, 64, (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER,
                                                              P.GEOM_CONE, P.GEOM_ELLIPSOID)))
    pts, tris = W.icosahedron_from_ellipsoid((0.3, 0.4, 0.5))
    cid = sc.register_convex(pts, tris)
    h = np.concatenate([h, sc.register_shapes(P.make_shapes([P.GEOM_CONVEX], [[0, 0, 0]], data=[cid]))])
    sc.commit()
    n = 6000
    h1, h2 = h[rng.integers(0, len(h), n)], h[rng.integers(0, len(h), n)]
    t1 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
    t2 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
    cases = [("batch_distance", dict(gjk_max_iterations=0)), ("batch_distance", dict(epa_max_iterations=0)),
             ("batch_distance", dict(gjk_tolerance=1.0)), ("batch_distance", dict(epa_tolerance=1.0)),
             ("batch_distance", dict(gjk_tolerance=1e-300)), ("batch_distance", dict(gjk_max_iterations=1, epa_max_iterations=1)),
             ("batch_distance", dict(gjk_max_iterations=100000)), ("batch_distance", dict(enable_nearest_points=0)),
             ("batch_collide", dict(security_margin=P.DBL_MAX)), ("batch_collide", dict(security_margin=-P.DBL_MAX)),
             ("batch_collide", dict(security_margin=float("inf"))), ("batch_collide", dict(distance_upper_bound=-1.0)),
             ("batch_collide", dict(collision_distance_threshold=-1.0)), ("batch_collide", dict(collision_distance_threshold=10.0)),
             ("batch_collide", dict(num_max_contacts=1000)), ("batch_collide", dict(break_distance=-1.0)),
             ("batch_collide", dict(gjk_max_iterations=0, enable_contact=0))]
    for fn, kw in cases:
        req = (P.DistanceRequestPOD if fn == "batch_distance" else P.CollisionRequestPOD)(**kw)
        ro = getattr(sc.b["oracle"], fn)(h1, t1, h2, t2, req, nthreads=0)
        compare_distance(ro, getattr(sc.b["emu"], fn)(h1, t1, h2, t2, req), what="%s %s" % (fn, kw))
        ref_agrees(sc, fn, ro, (h1, t1, h2, t2, req), "%s %s" % (fn, kw))


def test_huge_translations():
    """scenes far from the origin: both operands displaced by 1e6 ... 1e100 (half of the pairs next to each other
    there, half far apart) -- cancellation everywhere, but the same operations in the same order: reference build,
    oracle and host build of the device code must still agree bit for bit, shape pairs and mesh walks.  (From 1e154
    on, where squares overflow, the mesh queries of oracle and reference build part ways -- the per-query box fit
    runs an eigen decomposition on infinities; nothing there means anything.)"""
    import numpy as np
    from tests.common import P, compare_distance, make_scenes, ref_agrees
    from hppfcl_b200 import workloads as W
    rng = np.random.default_rng(8)
    sc = make_scenes(ref=True)
    h = sc.register_shapes(W.random_primitive_shapes(rng, 64, (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER,
                                                              P.GEOM_CONE, P.GEOM_ELLIPSOID)))
    v, f = W.sphere_mesh(1.0, 12, 6, noise=0.05, rng=rng)
    bid, _ = sc.register_bvh(v, f)
    hm = sc.register_shapes(P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[bid]))
    sc.commit()
    n, m = 3000, 400
    for mag in (1e6, 1e9, 1e12, 1e15, 1e100):
        h1, h2 = h[rng.integers(0, len(h), n)], h[rng.integers(0, len(h), n)]
        off = rng.normal(size=(n, 3)) * mag
        t1 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
        t2 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
        t1["T"] += off
        t2["T"] += off * (1 + (rng.random((n, 1)) < 0.5) * rng.normal(size=(n, 1)))
        for fn, req in (("batch_distance", P.DistanceRequestPOD()), ("batch_collide", P.CollisionRequestPOD())):
            ro = getattr(sc.b["oracle"], fn)(h1, t1, h2, t2, req, nthreads=0)
            compare_distance(ro, getattr(sc.b["emu"], fn)(h1, t1, h2, t2, req), what="%s at %g" % (fn, mag))
            ref_agrees(sc, fn, ro, (h1, t1, h2, t2, req), "%s at %g" % (fn, mag))
        hq = np.full(m, hm[0], dtype=np.uint32)
        a = (hq, t1[:m], h2[:m], t2[:m], P.DistanceRequestPOD())
        ro = sc.b["oracle"].batch_distance(*a, nthreads=0)
        compare_distance(ro, sc.b["emu"].batch_distance(*a), what="mesh-shape at %g" % mag)
        ref_agrees(sc, "batch_distance", ro, a, "mesh-shape at %g" % mag, fields=("min_distance", "p1", "p2", "normal", "b1", "b2"))


def test_hulls_at_the_linear_scan_threshold():
    """hulls of 31 and 32 vertices: the last sizes the reference scans linearly (support_functions.cpp:429,
    num_vertices_large_convex_threshold = 32; above it climbs hills) -- here the device code's exhaustive argmax must
    be index-exact: status words, iteration counts, support hints' consequences, every double, three-way"""
    import numpy as np
    from tests.common import P, compare_distance, make_scenes, ref_agrees
    from hppfcl_b200 import workloads as W
    rng = np.random.default_rng(12)
    sc = make_scenes(ref=True)
    hs = []
    for nv in (31, 32, 32, 32):
        pts, tris = W.ellipsoid_hull(rng, nv)
        assert len(pts) == nv
        cid = sc.register_convex(pts, tris)
        hs.append(int(sc.register_shapes(P.make_shapes([P.GEOM_CONVEX], [[0, 0, 0]], data=[cid]))[0]))
    hp = sc.register_shapes(W.random_primitive_shapes(rng, 16, (P.GEOM_BOX, P.GEOM_CAPSULE, P.GEOM_SPHERE)))
    sc.commit()
    hs = np.array(hs, dtype=np.uint32)
    pool = np.concatenate([hs, hp])
    n = 8000
    h1, h2 = hs[rng.integers(0, 4, n)], pool[rng.integers(0, len(pool), n)]
    t1 = W.random_transforms(rng, n, (-.6, -.6, -.6), (.6, .6, .6))
    t2 = W.random_transforms(rng, n, (-.6, -.6, -.6), (.6, .6, .6))
    for fn, req in (("batch_distance", P.DistanceRequestPOD()),
                    ("batch_distance", P.DistanceRequestPOD(gjk_variant=P.NesterovAcceleration)),
                    ("batch_collide", P.CollisionRequestPOD())):
        ro = getattr(sc.b["oracle"], fn)(h1, t1, h2, t2, req, nthreads=0)
        compare_distance(ro, getattr(sc.b["emu"], fn)(h1, t1, h2, t2, req), what=fn + ", 32-vertex hulls")
        ref_agrees(sc, fn, ro, (h1, t1, h2, t2, req), fn + ", 32-vertex hulls")


@pytest.mark.timeout(300)
def test_non_finite_poses_terminate():
    """NaN and +-Inf in a translation or rotation entry of half of the pairs: nothing is refused (the reference does
    not look either); every loop of the device code is bounded, so the batch comes back, and status words, iteration
    counts, distances and collision flags are those of the oracle and of the reference build.  Witness points and
    normals of such rows are left out: the reference's closed forms leave them unset (uninitialised memory there,
    stale registers here)."""
    import numpy as np
    from tests.common import P, make_scenes
    from hppfcl_b200 import workloads as W
    rng = np.random.default_rng(9)
    sc = make_scenes(ref=True)
    h = sc.register_shapes(W.random_primitive_shapes(rng, 64, (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER,
                                                              P.GEOM_CONE, P.GEOM_ELLIPSOID)))
    pts, tris = W.icosahedron_from_ellipsoid((0.3, 0.4, 0.5))
    cid = sc.register_convex(pts, tris)
    h = np.concatenate([h, sc.register_shapes(P.make_shapes([P.GEOM_CONVEX], [[0, 0, 0]], data=[cid]))])
    v, f = W.sphere_mesh(1.0, 12, 6, noise=0.05, rng=rng)
    bid, _ = sc.register_bvh(v, f)
    hm = sc.register_shapes(P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[bid]))
    sc.commit()
    n = 2000
    h1, h2 = h[rng.integers(0, len(h), n)], h[rng.integers(0, len(h), n)]
    t1 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
    t2 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
    vals = rng.choice([np.nan, np.inf, -np.inf], n)
    which = rng.integers(0, 12, n)
    for i in np.nonzero(rng.random(n) < 0.5)[0]:
        tgt = t2 if rng.random() < 0.5 else t1
        if which[i] < 3:
            tgt["T"][i, which[i]] = vals[i]
        else:
            tgt["R"][i, which[i] - 3] = vals[i]

    def same(a, b, fields):
        for fld in fields:
            x, y = a[fld], b[fld]
            ok = (x == y) | (np.isnan(x) & np.isnan(y)) if x.dtype.kind == "f" else x == y
            assert np.all(ok), fld
    for fn, req, fields in (("batch_distance", P.DistanceRequestPOD(), ("status", "iterations", "min_distance")),
                            ("batch_collide", P.CollisionRequestPOD(), ("status", "iterations", "num_contacts", "distance_lower_bound"))):
        ro = getattr(sc.b["oracle"], fn)(h1, t1, h2, t2, req, nthreads=0)
        same(ro, getattr(sc.b["emu"], fn)(h1, t1, h2, t2, req), fields)
        if "ref" in sc.b:
            same(ro, getattr(sc.b["ref"], fn)(h1, t1, h2, t2, req, nthreads=0), fields)
    m = 300  # the mesh walks: oracle and device code (the reference's box fit runs its eigen solver on NaNs)
    hq = np.full(m, hm[0], dtype=np.uint32)
    for fn, req, fields in (("batch_distance", P.DistanceRequestPOD(), ("min_distance", "b1", "b2")),
                            ("batch_collide", P.CollisionRequestPOD(), ("num_contacts", "b1", "b2"))):
        ro = getattr(sc.b["oracle"], fn)(hq, t1[:m], h2[:m], t2[:m], req, nthreads=0)
        same(ro, getattr(sc.b["emu"], fn)(hq, t1[:m], h2[:m], t2[:m], req), fields)


# Seeds 1, 2, 5-10 were green on a B200 in round 1 (profiles/r01_summary.md).  3 and 4 exposed a defect of the
# lane-group support argmax: a NaN direction (GJK produces one from 0/0 in the projection of a degenerate simplex,
# and carries on -- so does the reference) left the lanes of a group with different vertices.  Fixed in
# hfb_shapes.cuh, reproduced and pinned on the host (test_fuzz_device_code_through_lane_groups above and
# tests/test_emu_parity.py::test_lane_group_argmax_... / test_phase1_through_lane_groups); the driver's GPU run at
# the end of round 1 passed every seed (GPUTEST_r01.json), so all of them are plain tests.
GPU_SEEDS = list(range(1, 25))


def _gpu_round(seed):
    import hppfcl_b200 as hf
    eng = hf.Engine(0)
    ok, tag = fuzz_ref.one_round(seed, 4000, True, eng)
    assert ok, tag
    assert eng.stats()["watchdog_trips"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("seed", GPU_SEEDS)
def test_fuzz_on_the_gpu(seed):
    _gpu_round(seed)
