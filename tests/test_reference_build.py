"""The oracle against THE REFERENCE ITSELF: oracle/_ref/libhppfcl_ref.so is hpp-fcl's source tree compiled in
place, unmodified (recipe: `make -C oracle ref`; Eigen/Boost stand-ins under oracle/ref_shim/).  The
oracle's restatement must reproduce the reference's own collide()/distance() bit for bit: status words,
iteration counts, distances, witness points, normals, contact ids, and the OBBRSS tree its builder makes.
The same answers are the yardstick for the CUDA path.  Where oracle/_ref is not built, the reference's recorded
answers to the same calls stand in for it (tests/recorded_reference.py).
"""
import numpy as np
import pytest

from tests.common import P, compare_distance
from hppfcl_b200 import workloads as W
from oracle import oracle_lib
from tests.recorded_reference import reference_scene

ALL = (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER, P.GEOM_CONE, P.GEOM_ELLIPSOID)


def scenes():
    return oracle_lib.OracleScene(P), reference_scene(P)


def cmp_collide(ref, got, what=""):
    """the reference has no `distance` for a pair without contact; the record of the oracle / the kernels
    carries the computed signed distance there"""
    ref, got = ref.copy(), got.copy()
    nc = ref["num_contacts"] == 0
    ref["distance"][nc] = 0
    got["distance"][nc] = 0
    compare_distance(ref, got, what=what)


def cmp_fields(a, b, fields):
    for f in fields:
        x, y = a[f], b[f]
        ok = (x == y) | (np.isnan(x) & np.isnan(y)) if x.dtype.kind == "f" else x == y
        assert np.all(ok), "field %s differs at rows %s" % (f, np.unique(np.nonzero(~ok)[0])[:8])


@pytest.mark.parametrize("kw", [dict(), dict(gjk_variant=P.NesterovAcceleration),
                                dict(gjk_variant=P.PolyakAcceleration, gjk_convergence_criterion=P.DualityGap),
                                dict(gjk_convergence_criterion=P.Hybrid, gjk_convergence_criterion_type=P.Absolute),
                                dict(enable_signed_distance=0), dict(gjk_max_iterations=4), dict(epa_max_iterations=3),
                                dict(epa_tolerance=1e-10)])
def test_primitives_distance(kw):
    n = 20000
    w = W.config2_mixed_primitives(n, pool=512, types=ALL, seed=3)
    orc, ref = scenes()
    h = orc.register_shapes(w["shapes"])
    assert np.array_equal(h, ref.register_shapes(w["shapes"]))
    req = P.DistanceRequestPOD(**kw)
    a = ref.batch_distance(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"], req, want_guess=True, nthreads=0)
    b = orc.batch_distance(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"], req, want_guess=True, nthreads=0)
    compare_distance(a[0], b[0], what="primitives %s" % kw)
    assert np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64)) and np.array_equal(a[2], b[2])  # cached guesses
    assert (a[0]["min_distance"] < 0).sum() > 100


@pytest.mark.parametrize("kw", [dict(), dict(security_margin=0.05), dict(security_margin=-0.02), dict(enable_contact=0),
                                dict(distance_upper_bound=0.3), dict(enable_contact=0, distance_upper_bound=0.0),
                                dict(gjk_variant=P.NesterovAcceleration, gjk_tolerance=1e-3, epa_tolerance=1e-3)])
def test_primitives_collide(kw):
    n = 20000
    w = W.config2_mixed_primitives(n, pool=512, types=ALL, seed=4)
    orc, ref = scenes()
    h = orc.register_shapes(w["shapes"])
    ref.register_shapes(w["shapes"])
    req = P.CollisionRequestPOD(**kw)
    cmp_collide(ref.batch_collide(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"], req, nthreads=0),
                orc.batch_collide(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"], req, nthreads=0), what="collide %s" % kw)


def test_swept_radii_guess_modes_and_request_fields():
    n = 20000
    w = W.config2_mixed_primitives(n, pool=512, types=ALL, seed=11)
    rng = np.random.default_rng(1)
    shapes = w["shapes"].copy()
    shapes["ssr"] = np.where(rng.random(len(shapes)) < 0.5, rng.random(len(shapes)) * 0.1, 0.0)  # swept-sphere radii
    orc, ref = scenes()
    h = orc.register_shapes(shapes)
    ref.register_shapes(shapes)
    h1, h2 = h[w["h1"]], h[w["h2"]]
    compare_distance(ref.batch_distance(h1, w["tf1"], h2, w["tf2"], nthreads=0), orc.batch_distance(h1, w["tf1"], h2, w["tf2"], nthreads=0))
    gg = rng.normal(size=(n, 3))
    gg[:100] = 0  # below the tolerance: the (-1,0,0) restart of gjk.cpp:208-213
    gh = np.zeros((n, 2), dtype=np.int32)
    for mode in (P.CachedGuess, P.BoundingVolumeGuess):
        dreq, creq = P.DistanceRequestPOD(gjk_initial_guess=mode), P.CollisionRequestPOD(gjk_initial_guess=mode)
        if mode == P.CachedGuess:
            for r in (dreq, creq):
                r.q.cached_gjk_guess = gg.ctypes.data
                r.q.cached_support_func_guess = gh.ctypes.data
        compare_distance(ref.batch_distance(h1, w["tf1"], h2, w["tf2"], dreq, nthreads=0),
                         orc.batch_distance(h1, w["tf1"], h2, w["tf2"], dreq, nthreads=0), what="guess mode %d" % mode)
        cmp_collide(ref.batch_collide(h1, w["tf1"], h2, w["tf2"], creq, nthreads=0),
                    orc.batch_collide(h1, w["tf1"], h2, w["tf2"], creq, nthreads=0), what="guess mode %d" % mode)
    for kw in (dict(distance_upper_bound=0.1, security_margin=0.3), dict(num_max_contacts=5), dict(break_distance=0.5),
               dict(gjk_variant=P.PolyakAcceleration), dict(gjk_tolerance=1e-9, epa_tolerance=1e-9)):
        creq = P.CollisionRequestPOD(**kw)
        cmp_collide(ref.batch_collide(h1, w["tf1"], h2, w["tf2"], creq, nthreads=0),
                    orc.batch_collide(h1, w["tf1"], h2, w["tf2"], creq, nthreads=0), what=str(kw))


def convex_scene(n=6000):
    c3 = W.config3_convex_pairs(n, pool=24, nv=64, seed=5)
    orc, ref = scenes()
    ids = []
    hulls = list(c3["hulls"]) + [W.icosahedron_from_ellipsoid(r) for r in ((0.2, 0.3, 0.25), (0.5, 0.1, 0.3))]
    for pts, tris in hulls:
        a, b = orc.register_convex(pts, tris), ref.register_convex(pts, tris)
        assert a == b
        ids.append(a)
    recs = P.make_shapes([P.GEOM_CONVEX] * len(ids), np.zeros((len(ids), 3)), data=ids)
    hc = orc.register_shapes(recs)
    ref.register_shapes(recs)
    prim = W.random_primitive_shapes(np.random.default_rng(1), 64, ALL)
    hp = orc.register_shapes(prim)
    ref.register_shapes(prim)
    # (TriangleP operands are not in the reference's public dispatch tables: they are exercised as mesh
    # leaves by test_mesh_queries, triangle-shape and triangle-triangle)
    rng = np.random.default_rng(2)
    allh = np.concatenate([hc, hc, hp])
    h1, h2 = allh[rng.integers(0, len(allh), n)], allh[rng.integers(0, len(allh), n)]
    return orc, ref, h1, c3["tf1"], h2, c3["tf2"]


@pytest.mark.parametrize("kw", [dict(), dict(gjk_variant=P.NesterovAcceleration)])
def test_convex_hill_climb_and_mixed(kw):
    """ConvexBase with 64 vertices takes the neighbour hill-climb with warm starts in the reference
    (support_functions.cpp:324-397): the oracle's faithful mode must follow it vertex for vertex"""
    orc, ref, h1, tf1, h2, tf2 = convex_scene()
    req = P.DistanceRequestPOD(**kw)
    a = ref.batch_distance(h1, tf1, h2, tf2, req, want_guess=True, nthreads=0)
    b = orc.batch_distance(h1, tf1, h2, tf2, req, want_guess=True, nthreads=0)
    compare_distance(a[0], b[0], what="convex %s" % kw)
    assert np.array_equal(a[2], b[2])  # support-function hints
    cmp_collide(ref.batch_collide(h1, tf1, h2, tf2, nthreads=0), orc.batch_collide(h1, tf1, h2, tf2, nthreads=0))


def mesh_scene():
    orc, ref = scenes()
    rng = np.random.default_rng(7)
    va, ta = W.sphere_mesh(1.0, 20, 10, noise=0.03, rng=rng)
    vb, tb = W.sphere_mesh(0.6, 12, 6, noise=0.05, rng=rng)
    (ia, na), (ib, nb) = orc.register_bvh(va, ta), orc.register_bvh(vb, tb)
    (ra, rna), (rb, rnb) = ref.register_bvh(va, ta), ref.register_bvh(vb, tb)
    rec = P.make_shapes([P.BV_OBBRSS] * 2, [[0, 0, 0]] * 2, data=[ia, ib])
    hm = orc.register_shapes(rec)
    ref.register_shapes(rec)
    prims = W.random_primitive_shapes(rng, 48, ALL)
    prims["p"] *= 0.3
    hp = orc.register_shapes(prims)
    ref.register_shapes(prims)
    return orc, ref, hm, hp, rng, (na, rna, nb, rnb), ((va, ta), (vb, tb))


def test_bvh_builders_agree():
    """BVHModel<OBBRSS>::endModel of the reference == the oracle's restatement == the product's host builder"""
    from hppfcl_b200.engine import build_bvh_obbrss
    orc, ref, hm, hp, rng, (na, rna, nb, rnb), meshes = mesh_scene()
    assert na.tobytes() == rna.tobytes() and nb.tobytes() == rnb.tobytes()
    for (v, t), want in zip(meshes, (rna, rnb)):
        assert build_bvh_obbrss(v, t).tobytes() == want.tobytes()
    v, t = W.sphere_mesh(1.0, 100, 50, noise=0.01, rng=np.random.default_rng(3))  # config 4's mesh size
    _, nodes = ref.register_bvh(v, t)
    assert len(nodes) == 19999 and build_bvh_obbrss(v, t).tobytes() == nodes.tobytes()


def test_mesh_queries():
    orc, ref, hm, hp, rng, _, _ = mesh_scene()
    m = 3000
    tf1 = W.random_transforms(rng, m, (-.2, -.2, -.2), (.2, .2, .2))
    tf2 = W.random_transforms(rng, m, (-1.8, -1.8, -1.8), (1.8, 1.8, 1.8))
    hq = hp[rng.integers(0, len(hp), m)]
    h1 = hm[rng.integers(0, 2, m)]
    h2 = hm[rng.integers(0, 2, m)]
    D = ("min_distance", "p1", "p2", "normal", "b1", "b2")
    Cf = ("p1", "p2", "normal", "pos", "distance_lower_bound", "b1", "b2", "num_contacts")
    for req in (P.DistanceRequestPOD(), P.DistanceRequestPOD(rel_err=0.05, abs_err=0.01)):
        cmp_fields(ref.batch_distance(h1, tf1, hq, tf2, req, nthreads=0), orc.batch_distance(h1, tf1, hq, tf2, req, nthreads=0), D)
    cmp_fields(ref.batch_distance(hq, tf2, h1, tf1, nthreads=0), orc.batch_distance(hq, tf2, h1, tf1, nthreads=0), D)
    for kw in (dict(), dict(security_margin=0.05), dict(num_max_contacts=4, enable_contact=0)):
        req = P.CollisionRequestPOD(**kw)
        cmp_fields(ref.batch_collide(h1, tf1, hq, tf2, req, nthreads=0), orc.batch_collide(h1, tf1, hq, tf2, req, nthreads=0), Cf)
        cmp_fields(ref.batch_collide(hq, tf2, h1, tf1, req, nthreads=0), orc.batch_collide(hq, tf2, h1, tf1, req, nthreads=0), Cf)
    # mesh-mesh (the reference never writes `normal` on the distance path)
    cmp_fields(ref.batch_distance(h1, tf1, h2, tf2, nthreads=0), orc.batch_distance(h1, tf1, h2, tf2, nthreads=0),
               ("min_distance", "p1", "p2", "b1", "b2"))
    for kw in (dict(), dict(security_margin=0.05), dict(security_margin=-0.01), dict(gjk_variant=P.NesterovAcceleration)):
        req = P.CollisionRequestPOD(**kw)
        cmp_fields(ref.batch_collide(h1, tf1, h2, tf2, req, nthreads=0), orc.batch_collide(h1, tf1, h2, tf2, req, nthreads=0), Cf)


@pytest.mark.gpu
def test_gpu_against_the_reference_build():
    """the CUDA path (C ABI) directly against the reference's own code on the same inputs"""
    import hppfcl_b200 as hf
    n = 200_000
    w = W.config2_mixed_primitives(n, pool=4096, types=ALL, seed=9)
    ref = reference_scene(P)
    eng = hf.Engine(0)
    h = eng.register_shapes(w["shapes"])
    ref.register_shapes(w["shapes"])
    eng.commit()
    for kw in (dict(), dict(gjk_variant=P.NesterovAcceleration)):
        req = P.DistanceRequestPOD(**kw)
        compare_distance(ref.batch_distance(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"], req, nthreads=0),
                         eng.batch_distance(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"], req), what="gpu vs reference %s" % kw)
    cmp_collide(ref.batch_collide(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"], nthreads=0),
                eng.batch_collide(h[w["h1"]], w["tf1"], h[w["h2"]], w["tf2"]))
    # mesh vs shapes and mesh vs mesh, tree built by the product's host builder
    rng = np.random.default_rng(5)
    eng2, ref2 = hf.Engine(0), reference_scene(P)
    va, ta = W.sphere_mesh(1.0, 30, 15, noise=0.02, rng=rng)
    bid = eng2.register_bvh_obbrss(None, va, ta)
    rbid, _ = ref2.register_bvh(va, ta)
    rec = P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[bid])
    hm = eng2.register_shapes(rec)
    ref2.register_shapes(P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[rbid]))
    prims = W.random_primitive_shapes(rng, 64, ALL)
    prims["p"] *= 0.3
    hp = eng2.register_shapes(prims)
    ref2.register_shapes(prims)
    eng2.commit()
    m = 20000
    tf1 = W.random_transforms(rng, m, (-.2, -.2, -.2), (.2, .2, .2))
    tf2 = W.random_transforms(rng, m, (-1.8, -1.8, -1.8), (1.8, 1.8, 1.8))
    hq = hp[rng.integers(0, len(hp), m)]
    hmm = np.full(m, hm[0], dtype=np.uint32)
    cmp_fields(ref2.batch_distance(hmm, tf1, hq, tf2, nthreads=0), eng2.batch_distance(hmm, tf1, hq, tf2),
               ("min_distance", "p1", "p2", "normal", "b1", "b2"))
    k = 2000
    cmp_fields(ref2.batch_distance(hmm[:k], tf1[:k], hmm[:k], tf2[:k], nthreads=0), eng2.batch_distance(hmm[:k], tf1[:k], hmm[:k], tf2[:k]),
               ("min_distance", "p1", "p2", "b1", "b2"))


def test_plain_obb_models():
    """BVHModel<OBB> (row X1): the reference's plain OBB tree of a mesh IS the OBB half of its OBBRSS tree, and collide()
    on it -- mesh-shape with computeBV<OBB, S>'s boxes, mesh-mesh -- is reproduced bit for bit by the oracle and by the
    host build of the device code.  distance() on a plain OBB model is not offered (unsupported records)."""
    from tests.common import EmuScene
    orc, ref, hm, hp, rng, (na, rna, nb, rnb), ((va, ta), (vb, tb)) = mesh_scene()
    assert ref.bvh_obb_is_obbrss_half(0) == 1 and ref.bvh_obb_is_obbrss_half(1) == 1
    emu = EmuScene()
    assert emu.register_bvh_obbrss(na, va, ta) == 0 and emu.register_bvh_obbrss(nb, vb, tb) == 1
    # the same two meshes once more, as plain OBB models (ids 2 and 3 in every backend)
    for sc in (orc, ref):
        assert sc.register_bvh(va, ta)[0] == 2 and sc.register_bvh(vb, tb)[0] == 3
    assert emu.register_bvh_obb(na, va, ta) == 2 and emu.register_bvh_obb(nb, vb, tb) == 3
    rec0 = P.make_shapes([P.BV_OBBRSS] * 2, [[0, 0, 0]] * 2, data=[0, 1])
    rec = P.make_shapes([P.BV_OBB] * 2, [[0, 0, 0]] * 2, data=[2, 3])
    ho = orc.register_shapes(rec)
    assert np.array_equal(ref.register_shapes(rec), ho)
    # the emu scene: same handle numbering as the other two (mesh_scene drew its primitives from its own generator
    # after the two meshes: the same draws again)
    assert np.array_equal(emu.register_shapes(rec0), hm)
    rng2 = np.random.default_rng(7)
    W.sphere_mesh(1.0, 20, 10, noise=0.03, rng=rng2)
    W.sphere_mesh(0.6, 12, 6, noise=0.05, rng=rng2)
    prims = W.random_primitive_shapes(rng2, 48, ALL)
    prims["p"] *= 0.3
    assert np.array_equal(emu.register_shapes(prims), hp)
    assert np.array_equal(emu.register_shapes(rec), ho)
    m = 2500
    tf1 = W.random_transforms(rng, m, (-.2, -.2, -.2), (.2, .2, .2))
    tf2 = W.random_transforms(rng, m, (-1.5, -1.5, -1.5), (1.5, 1.5, 1.5))
    hq = hp[rng.integers(0, len(hp), m)]
    h1 = ho[rng.integers(0, 2, m)]
    h2 = ho[rng.integers(0, 2, m)]
    Cf = ("p1", "p2", "normal", "pos", "distance_lower_bound", "b1", "b2", "num_contacts")
    for kw in (dict(), dict(security_margin=0.05), dict(num_max_contacts=4, enable_contact=0)):
        req = P.CollisionRequestPOD(**kw)
        for a1, t1, a2, t2 in ((h1, tf1, hq, tf2), (hq, tf2, h1, tf1), (h1, tf1, h2, tf2)):
            want = ref.batch_collide(a1, t1, a2, t2, req, nthreads=0)
            got = orc.batch_collide(a1, t1, a2, t2, req, nthreads=0)
            cmp_fields(want, got, Cf)
            dev = emu.batch_collide(a1, t1, a2, t2, req)
            cmp_fields(got, dev, Cf + ("iterations", "status"))
    assert want["num_contacts"].sum() > 20
    # mixed kinds and distance(): unsupported in the product and the oracle alike
    mix = orc.batch_collide(h1[:8], tf1[:8], hm[:1].repeat(8), tf2[:8], nthreads=0)
    assert np.all(P.status_path(mix["status"]) == P.PATH_UNSUPPORTED)
    assert np.all(P.status_path(emu.batch_collide(h1[:8], tf1[:8], hm[:1].repeat(8), tf2[:8])["status"]) == P.PATH_UNSUPPORTED)
    for sc in (orc, emu):
        d = sc.batch_distance(h1[:8], tf1[:8], hq[:8], tf2[:8], **({"nthreads": 0} if sc is orc else {}))
        assert np.all(P.status_path(d["status"]) == P.PATH_UNSUPPORTED)
        d = sc.batch_distance(h1[:8], tf1[:8], h2[:8], tf2[:8], **({"nthreads": 0} if sc is orc else {}))
        assert np.all(P.status_path(d["status"]) == P.PATH_UNSUPPORTED)
