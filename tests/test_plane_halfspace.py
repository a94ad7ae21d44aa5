"""Plane / Halfspace geometries (SURVEY 8 row a13, the closed forms of src/narrowphase/details.h:343-693 behind the
ShapeShapeDistance specialisations of src/distance/<shape>_halfspace.cpp and <shape>_plane.cpp): every partner
type, both operand orders, swept-sphere radii, axis-aligned and tilted normals, the plane-plane / halfspace-
halfspace / halfspace-plane pairs (parallel, anti-parallel, crossing), distance() and collide().

  reference (oracle/_ref, /root/reference compiled in place)  ==  oracle          (CPU, where _ref exists)
  host build of the device code (tests/emu)                   ==  oracle          (CPU)
  CUDA kernels through the C-ABI                              ==  oracle          (B200)
bit for bit (compare_distance(exact=True): status words, distances, witness points, normals).
"""
import numpy as np
import pytest

from tests.common import P, compare_distance, make_scenes, EmuScene
from hppfcl_b200 import workloads as W
from oracle import oracle_lib

PARTNERS = (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER, P.GEOM_CONE, P.GEOM_ELLIPSOID)


def plane_world(seed=7, n_planes=48, n_prims=96, n_pairs=6000):
    """geometry + pairs of one test scene, as plain arrays (registered backend by backend below)"""
    rng = np.random.default_rng(seed)
    nd = np.concatenate([rng.normal(size=(n_planes, 3)) * rng.uniform(0.2, 3.0, (n_planes, 1)),  # not unit: the library normalises
                         rng.uniform(-1.0, 1.0, (n_planes, 1))], axis=1)
    axes = np.array([[0, 0, 1, 0.0], [0, 0, -1, 0.25], [1, 0, 0, -0.5], [0, -2, 0, 0.5], [0, 1, 0, 0.0], [0, 0, 0, 1.0]])
    nd[:len(axes)] = axes  # floors, walls, and the degenerate normal (-> (1, 0, 0), 0)
    nd[len(axes)] = nd[len(axes) + 1] * 2.5  # the same plane twice, scaled: parallel pairs
    nd[len(axes) + 2, :3] = -nd[len(axes) + 1, :3]  # and its mirror image: anti-parallel pairs
    ssr = np.where(rng.random(n_planes) < 0.3, rng.uniform(0.01, 0.2, n_planes), 0.0)
    prims = W.random_primitive_shapes(rng, n_prims, PARTNERS)
    prims["ssr"] = np.where(rng.random(n_prims) < 0.3, rng.uniform(0.01, 0.1, n_prims), 0.0)
    hulls = [W.ellipsoid_hull(rng, 64), W.ellipsoid_hull(rng, 40), W.ellipsoid_hull(rng, 20),
             W.icosahedron_from_ellipsoid((0.2, 0.3, 0.25))]
    tris = [rng.normal(size=(3, 3)) * 0.4 for _ in range(6)]
    return dict(rng=rng, nd=nd, ssr=ssr, prims=prims, hulls=hulls, tris=tris, n_pairs=n_pairs)


def register(sc, w, backend):
    """-> handles of halfspaces, planes, partners (primitives, hulls, triangles)"""
    hs = sc.register_halfspaces(P.GEOM_HALFSPACE, w["nd"], w["ssr"])
    ps = sc.register_halfspaces(P.GEOM_PLANE, w["nd"], w["ssr"])
    pr = sc.register_shapes(w["prims"])
    cids = []
    for pts, tr in w["hulls"]:
        cids.append(sc.register_convex(pts, tr) if backend in ("oracle", "ref") else sc.register_convex(pts))
    tids = []
    for t in w["tris"]:
        if backend == "ref":
            tids.append(sc.register_points(t))
        elif backend == "oracle":
            tids.append(sc.register_convex(t, None))
        else:
            tids.append(sc.register_convex(t))
    hv = sc.register_shapes(P.make_shapes([P.GEOM_CONVEX] * len(cids), np.zeros((len(cids), 3)), data=cids,
                                          ssr=[0.0, 0.05, 0.0, 0.0]))
    tv = sc.register_shapes(P.make_shapes([P.GEOM_TRIANGLE] * len(tids), np.zeros((len(tids), 3)), data=tids,
                                          ssr=[0.0, 0.0, 0.03, 0.0, 0.0, 0.0]))
    if hasattr(sc, "commit"):
        sc.commit()
    return hs, ps, np.concatenate([pr, hv, tv])


def pairs(w, hs, ps, others):
    """plane-family handle on a random side, any partner on the other (a tenth of them another plane / halfspace);
    poses: random, with identity / pure-translation cases mixed in (the floor under a robot)"""
    rng = np.random.default_rng(99)
    n = w["n_pairs"]
    fam = np.concatenate([hs, ps])
    a = fam[rng.integers(0, len(fam), n)]
    b = np.where(rng.random(n) < 0.12, fam[rng.integers(0, len(fam), n)], others[rng.integers(0, len(others), n)])
    swap = rng.random(n) < 0.5
    h1, h2 = np.where(swap, b, a).astype(np.uint32), np.where(swap, a, b).astype(np.uint32)
    tf1 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
    tf2 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
    ident = W.identity_transforms(n)
    m = rng.random(n) < 0.3
    tf1["R"][m] = ident["R"][m]
    m2 = rng.random(n) < 0.2
    tf2["R"][m2] = ident["R"][m2]
    m3 = rng.random(n) < 0.05
    tf1["T"][m3] = 0
    # the parallel / anti-parallel plane pairs only stay so under the same rotation
    same = rng.random(n) < 0.3
    tf2["R"][same] = tf1["R"][same]
    return h1, tf1, h2, tf2


def run_both(sc, h1, tf1, h2, tf2, **kw):
    d = sc.batch_distance(h1, tf1, h2, tf2, **kw)
    out = [d]
    for ckw in (dict(), dict(security_margin=0.1), dict(security_margin=-0.05, enable_contact=0)):
        out.append(sc.batch_collide(h1, tf1, h2, tf2, P.CollisionRequestPOD(**ckw), **kw))
    return out


def check(ref_out, got_out, what):
    compare_distance(ref_out[0], got_out[0], what=what + " distance()")
    for k in range(1, len(ref_out)):
        r, g = ref_out[k].copy(), got_out[k].copy()
        nc = r["num_contacts"] == 0  # the reference leaves `distance` unset without a contact
        r["distance"][nc] = 0
        g["distance"][nc] = 0
        compare_distance(r, g, what=what + " collide() #%d" % k)


def test_oracle_equals_the_reference():
    from tests.recorded_reference import reference_scene
    w = plane_world()
    orc, ref = oracle_lib.OracleScene(P), reference_scene(P)
    ho = register(orc, w, "oracle")
    hr = register(ref, w, "ref")
    for x, y in zip(ho, hr):
        assert np.array_equal(x, y)
    h1, tf1, h2, tf2 = pairs(w, *ho)
    a = run_both(ref, h1, tf1, h2, tf2, nthreads=0)
    b = run_both(orc, h1, tf1, h2, tf2, nthreads=0)
    # TriangleP operands are in the reference's collision matrix only (collision_func_matrix.cpp:295-450; the distance
    # matrix has no TriangleP row or column): their distance() is checked against the oracle alone, below
    tri = np.isin(h1, ho[2][-len(w["tris"]):]) | np.isin(h2, ho[2][-len(w["tris"]):])
    assert np.all(P.status_path(a[0]["status"][tri]) == P.PATH_UNSUPPORTED) and tri.sum() > 100
    a[0], b[0] = a[0][~tri], b[0][~tri]
    check(a, b, "reference vs oracle")
    d = a[0]
    assert np.all(P.status_path(d["status"]) == P.PATH_CLOSED_FORM)
    assert (d["min_distance"] < 0).sum() > 500 and (d["min_distance"] > 0).sum() > 500
    assert (d["min_distance"] == -np.finfo(np.float64).max).sum() > 20  # crossing planes: infinite penetration
    assert a[1]["num_contacts"].sum() > 500


def test_host_build_of_the_device_code_equals_the_oracle():
    w = plane_world(seed=8)
    orc, emu = oracle_lib.OracleScene(P), EmuScene()
    ho = register(orc, w, "oracle")
    he = register(emu, w, "emu")
    for x, y in zip(ho, he):
        assert np.array_equal(x, y)
    h1, tf1, h2, tf2 = pairs(w, *ho)
    check(run_both(orc, h1, tf1, h2, tf2), run_both(emu, h1, tf1, h2, tf2), "oracle vs host build of the device code")


def test_mesh_partner_is_unsupported_and_records_are_refused():
    w = plane_world(n_pairs=10)
    orc, emu = oracle_lib.OracleScene(P), EmuScene()
    for sc, name in ((orc, "oracle"), (emu, "emu")):
        hs, ps, _ = register(sc, w, name)
    v, t = W.sphere_mesh(1.0, 8, 4)
    bid, nodes = orc.register_bvh(v, t)
    emu.register_bvh_obbrss(nodes, v, t)
    rec = P.make_shapes([P.BV_OBBRSS], np.zeros((1, 3)), data=[bid])
    hm_o, hm_e = orc.register_shapes(rec), emu.register_shapes(rec)
    assert np.array_equal(hm_o, hm_e)
    tf = W.identity_transforms(2)
    h1, h2 = np.array([hm_o[0], hs[0]], dtype=np.uint32), np.array([hs[0], hm_o[0]], dtype=np.uint32)
    for sc in (orc, emu):
        d = sc.batch_distance(h1, tf, h2, tf)
        assert np.all(P.status_path(d["status"]) == P.PATH_UNSUPPORTED)


@pytest.mark.gpu
def test_cuda_kernels_equal_the_oracle():
    import hppfcl_b200 as hf
    w = plane_world(seed=9, n_pairs=60000)
    orc, eng = oracle_lib.OracleScene(P), hf.Engine(0)
    ho = register(orc, w, "oracle")
    hg = register(eng, w, "gpu")
    for x, y in zip(ho, hg):
        assert np.array_equal(x, y)
    h1, tf1, h2, tf2 = pairs(w, *ho)
    check(run_both(orc, h1, tf1, h2, tf2, nthreads=0), run_both(eng, h1, tf1, h2, tf2), "oracle vs CUDA")
    # a scene without hulls or triangles takes the primitive-only kernels (the plane class of the closed-form kernel)
    eng2, orc2 = hf.Engine(0), oracle_lib.OracleScene(P)
    out = []
    for sc in (orc2, eng2):
        hs = sc.register_halfspaces(P.GEOM_HALFSPACE, w["nd"], w["ssr"])
        ps = sc.register_halfspaces(P.GEOM_PLANE, w["nd"], w["ssr"])
        pr = sc.register_shapes(w["prims"])
        if hasattr(sc, "commit"):
            sc.commit()
        q = pairs(w, hs, ps, pr)
        out.append(run_both(sc, *q))
    check(out[0], out[1], "oracle vs CUDA, primitives only")
    # the generic record call refuses the two types: a 40-byte record has no room for n and d
    with pytest.raises(hf.EngineError):
        eng2.register_shapes(P.make_shapes([P.GEOM_HALFSPACE], np.zeros((1, 3))))


@pytest.mark.gpu
def test_python_mirror_floor_under_a_box():
    """collide() / distance() of the host mirror with a Halfspace floor, against the oracle; a floor changed in place
    is registered anew"""
    import hppfcl_b200 as hf
    floor, box = hf.Halfspace([0, 0, 1], 0.0), hf.Box(1, 1, 1)
    tfb = hf.Transform3f.from_quat(0.9238795325112867, 0.3826834323650898, 0, 0, (0.1, 0.2, 0.9))
    res = hf.DistanceResult()
    d = hf.distance(floor, hf.Transform3f(), box, tfb, hf.DistanceRequest(), res)
    orc = oracle_lib.OracleScene(P)
    hh = orc.register_halfspaces(P.GEOM_HALFSPACE, [[0, 0, 1, 0.0]])
    hb = orc.register_shapes(P.make_shapes([P.GEOM_BOX], [[0.5, 0.5, 0.5]]))
    tf1, tf2 = W.identity_transforms(1), P.make_transforms(tfb.R[None], tfb.T[None])
    ref = orc.batch_distance(hh, tf1, hb, tf2)[0]
    assert d == ref["min_distance"] and np.array_equal(res.nearest_points[1], ref["p2"]) and np.array_equal(res.normal, ref["normal"])
    assert 0.19 < d < 0.2  # the lowest corner: 0.9 - sqrt(2) / 2
    cres = hf.CollisionResult()
    assert hf.collide(box, tfb, floor, hf.Transform3f(), hf.CollisionRequest(), cres) == 0
    floor.d = 0.25  # the floor rises: the box's corner is now 0.057 below it
    res2 = hf.DistanceResult()
    d2 = hf.distance(floor, hf.Transform3f(), box, tfb, hf.DistanceRequest(), res2)
    assert abs((d - d2) - 0.25) < 1e-15
    cres = hf.CollisionResult()
    assert hf.collide(box, tfb, floor, hf.Transform3f(), hf.CollisionRequest(), cres) == 1
    assert abs(cres.getContact(0).penetration_depth - d2) < 1e-15
