"""OBBRSS BVH vs shape (SURVEY rows a14/a15): oracle (reference builder, recursion) vs the emulated
device code (explicit-stack traversal, per-query shape BV, RSS/OBB tests) on CPU, and vs the CUDA
kernel on the GPU box.  The tree itself comes from the oracle's restatement of the reference builder
and reaches the product through hfb_geom_register_bvh_obbrss, like a binding would pass
BVHModel<OBBRSS>::bvs.  Bar: everything bit-identical, incl. witness triangle ids and the
BV-test / leaf-test counters (they pin the traversal order)."""
import numpy as np
import pytest

from tests.common import P, compare_distance, make_scenes
from hppfcl_b200 import workloads as W

SHAPES = (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER, P.GEOM_CONE, P.GEOM_ELLIPSOID)


def build_scene(gpu, emu, seg=24, ring=12, n=3000, seed=1):
    sc = make_scenes(gpu=gpu, emu=emu)
    rng = np.random.default_rng(seed)
    verts, tris = W.sphere_mesh(1.0, seg, ring, noise=0.02, rng=rng)
    bid, nodes = sc.register_bvh(verts, tris)
    hb = sc.register_shapes(P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[bid]))
    prims = W.random_primitive_shapes(rng, 96, SHAPES)
    prims["p"] *= 0.3
    hp = sc.register_shapes(prims)
    pts, ctris = W.icosahedron_from_ellipsoid((0.2, 0.3, 0.25))
    cid = sc.register_convex(pts, ctris)
    hc = sc.register_shapes(P.make_shapes([P.GEOM_CONVEX], [[0, 0, 0]], data=[cid]))
    sc.commit()
    allh = np.concatenate([hp, hc])
    hs = allh[rng.integers(0, len(allh), n)]
    tfm = W.random_transforms(rng, n, (-0.3, -0.3, -0.3), (0.3, 0.3, 0.3))
    tfs = W.random_transforms(rng, n, (-1.6, -1.6, -1.6), (1.6, 1.6, 1.6))
    hm = np.full(n, hb[0], dtype=np.uint32)
    return sc, nodes, hm, tfm, hs, tfs, (verts, tris)


def test_builder_invariants():
    sc, nodes, hm, tfm, hs, tfs, (verts, tris) = build_scene(False, False, n=10)
    assert len(nodes) == 2 * len(tris) - 1
    leaf = nodes["first_child"] < 0
    assert leaf.sum() == len(tris)
    assert sorted(-(nodes["first_child"][leaf] + 1)) == list(range(len(tris)))  # every triangle exactly once
    inner = nodes[~leaf]
    assert np.all(inner["first_child"] > np.nonzero(~leaf)[0])                   # children follow the parent
    # OBB axes orthonormal, extents >= 0, RSS contains the OBB centre roughly
    A = nodes["obb_axes"].reshape(-1, 3, 3)
    assert np.allclose(np.einsum("nij,nkj->nik", A, A), np.eye(3), atol=1e-9)
    assert np.all(nodes["obb_extent"] >= 0) and np.all(nodes["rss_radius"] >= 0)
    # root OBB contains every vertex
    R = nodes["obb_axes"][0].reshape(3, 3).T
    loc = (verts - nodes["obb_To"][0]) @ R
    assert np.all(np.abs(loc) <= nodes["obb_extent"][0] + 1e-9)


@pytest.mark.parametrize("seg,ring,noise", [(24, 12, 0.02), (100, 50, 0.02), (8, 5, 0.0), (3, 2, 0.0)])
def test_product_builder_matches_reference_builder(seg, ring, noise):
    """hfb_bvh_build_obbrss (host code of the product, no GPU) against the oracle's restatement of
    BVHModel<OBBRSS>::endModel: every node bit-identical (fit, split, numbering)."""
    from hppfcl_b200.engine import build_bvh_obbrss
    from oracle import oracle_lib
    verts, tris = W.sphere_mesh(1.0, seg, ring, noise=noise, rng=np.random.default_rng(seg))
    orc = oracle_lib.OracleScene(P)
    _, ref = orc.register_bvh(verts, tris)
    got = build_bvh_obbrss(verts, tris)
    assert ref.dtype == got.dtype and len(ref) == 2 * len(tris) - 1
    assert ref.tobytes() == got.tobytes()
    # degenerate / invalid input is refused, not built
    from hppfcl_b200.engine import EngineError
    with pytest.raises(EngineError):
        build_bvh_obbrss(verts, np.array([[0, 1, len(verts)]], dtype=np.uint32))


def _check(sc, backend, hm, tfm, hs, tfs):
    o, e = sc.b["oracle"], sc.b[backend]
    for req in (P.DistanceRequestPOD(), P.DistanceRequestPOD(enable_signed_distance=0),
                P.DistanceRequestPOD(gjk_variant=P.NesterovAcceleration), P.DistanceRequestPOD(rel_err=0.05, abs_err=0.01)):
        ro = o.batch_distance(hm, tfm, hs, tfs, req, nthreads=0)
        re = e.batch_distance(hm, tfm, hs, tfs, req)
        compare_distance(ro, re, what="bvh distance")
        assert np.all(P.status_path(ro["status"]) == P.PATH_BVH)
    assert (ro["min_distance"] < 0).sum() > 20 and (ro["b1"] >= 0).all()
    # (shape, mesh) operand order: results swapped back (distance.cpp:74-89)
    rs = o.batch_distance(hs, tfs, hm, tfm, nthreads=0)
    compare_distance(rs, e.batch_distance(hs, tfs, hm, tfm), what="bvh distance swapped")
    r0 = o.batch_distance(hm, tfm, hs, tfs, nthreads=0)
    m = ~np.isnan(r0["p1"][:, 0])
    assert np.array_equal(rs["p1"][m], r0["p2"][m]) and np.array_equal(rs["normal"][m], -r0["normal"][m])
    for creq in (P.CollisionRequestPOD(), P.CollisionRequestPOD(security_margin=0.05),
                 P.CollisionRequestPOD(num_max_contacts=4, enable_contact=0)):
        co = o.batch_collide(hm, tfm, hs, tfs, creq, nthreads=0)
        compare_distance(co, e.batch_collide(hm, tfm, hs, tfs, creq), what="bvh collide")
        cs = o.batch_collide(hs, tfs, hm, tfm, creq, nthreads=0)
        compare_distance(cs, e.batch_collide(hs, tfs, hm, tfm, creq), what="bvh collide swapped")
    assert co["num_contacts"].sum() > 20
    # negative margin is rejected for BVH models (collision_func_matrix.cpp:109-112)
    bad = e.batch_collide(hm[:4], tfm[:4], hs[:4], tfs[:4], P.CollisionRequestPOD(security_margin=-0.01))
    assert np.all(P.status_path(bad["status"]) == P.PATH_UNSUPPORTED)


def test_bvh_emulated_device_code_vs_oracle():
    sc, nodes, hm, tfm, hs, tfs, _ = build_scene(False, True)
    _check(sc, "emu", hm, tfm, hs, tfs)


@pytest.mark.parametrize("knobs", ["0,1,6,2,3,30", "0,2,1,1,1,0", "-1,3,5,0,2,0", "40,4,9,3,100,10", "0,5,32,1,4,1000000", "3,6,3,8,1,5"])
def test_bvh_task_system_walk_vs_oracle(knobs, monkeypatch):
    """hfb_bvhq.cuh (the walk of kernel k_bvhq) on the host: queries as state machines, their bounding-volume and
    leaf items executed one at a time in RANDOM order, subtrees speculated after `spec_after` items
    (knobs = spec_after, seed, slots in flight, treelet buffers, GJK iterations a leaf item runs before it parks its
    solver state and queues itself again -- EPA is an item of its own --, items more before subtrees of up to 128
    triangles are speculated instead of 32).  Bit-identical to the recursion, counters
    included."""
    monkeypatch.setenv("HFB_EMU_BVHQ", knobs)
    sc, nodes, hm, tfm, hs, tfs, _ = build_scene(False, True, n=1500, seed=int(knobs.split(",")[1]))
    o, e = sc.b["oracle"], sc.b["emu"]
    it0, sp0 = e.L.emu_q_items(), e.L.emu_q_spec_items()
    for req in (P.DistanceRequestPOD(), P.DistanceRequestPOD(enable_signed_distance=0),
                P.DistanceRequestPOD(rel_err=0.05, abs_err=0.01)):
        compare_distance(o.batch_distance(hm, tfm, hs, tfs, req, nthreads=0), e.batch_distance(hm, tfm, hs, tfs, req),
                         what="task-system walk")
    compare_distance(o.batch_distance(hs, tfs, hm, tfm, nthreads=0), e.batch_distance(hs, tfs, hm, tfm),
                     what="task-system walk, swapped operands")
    spec = e.L.emu_q_spec_items() - sp0
    assert e.L.emu_q_items() - it0 > 10000
    if knobs.startswith("-1") or knobs.split(",")[3] == "0":
        assert spec == 0
    else:
        assert spec > 1000  # the speculated path really ran
    # CachedGuess chains the solver's guess from leaf to leaf: such a request must never speculate
    n = 300
    req = P.DistanceRequestPOD(gjk_initial_guess=P.CachedGuess)
    g = np.tile(np.array([0.3, -0.2, 0.9]), (n, 1))
    hint = np.zeros((n, 2), dtype=np.int32)
    req.q.cached_gjk_guess = g.ctypes.data
    req.q.cached_support_func_guess = hint.ctypes.data
    sp1 = e.L.emu_q_spec_items()
    compare_distance(o.batch_distance(hm[:n], tfm[:n], hs[:n], tfs[:n], req, nthreads=0),
                     e.batch_distance(hm[:n], tfm[:n], hs[:n], tfs[:n], req), what="task-system walk, cached guess")
    assert e.L.emu_q_spec_items() == sp1


def test_bvh_distance_is_the_true_minimum():
    """differential check in the style of test/distance.cpp: traversal result == brute force over all triangles"""
    sc, nodes, hm, tfm, hs, tfs, (verts, tris) = build_scene(False, False, seg=12, ring=6, n=40)
    o = sc.b["oracle"]
    cids = [o.register_convex(verts[t], None) for t in tris]
    ht = o.register_shapes(P.make_shapes([P.GEOM_TRIANGLE] * len(tris), np.zeros((len(tris), 3)), data=cids))
    r = o.batch_distance(hm, tfm, hs, tfs)
    for q in range(len(hm)):
        nt = len(tris)
        rr = o.batch_distance(ht, np.repeat(tfm[q:q + 1], nt), np.full(nt, hs[q], dtype=np.uint32), np.repeat(tfs[q:q + 1], nt))
        assert rr["min_distance"][r[q]["b1"]] == r[q]["min_distance"]
        if rr["min_distance"].min() > 0:
            assert r[q]["min_distance"] == rr["min_distance"].min()
        else:  # once a penetrating triangle is found every BV lower bound (>= 0) prunes: any negative leaf
            assert r[q]["min_distance"] <= 0


# ---- mesh-mesh (BVHModel<OBBRSS> x BVHModel<OBBRSS>) --------------------------------------------
def build_mesh_pair_scene(gpu, emu, n=300, seed=5, seg=14, ring=8):
    sc = make_scenes(gpu=gpu, emu=emu)
    rng = np.random.default_rng(seed)
    va, ta = W.sphere_mesh(1.0, seg, ring, noise=0.03, rng=rng)
    vb, tb = W.sphere_mesh(0.6, seg - 4, ring - 2, noise=0.05, rng=rng)
    vb = vb * np.array([1.0, 0.6, 1.4])
    ia, _ = sc.register_bvh(va, ta)
    ib, _ = sc.register_bvh(vb, tb)
    h = sc.register_shapes(P.make_shapes([P.BV_OBBRSS, P.BV_OBBRSS], [[0, 0, 0]] * 2, data=[ia, ib]))
    sc.commit()
    which = rng.integers(0, 2, (n, 2))
    h1, h2 = h[which[:, 0]], h[which[:, 1]]
    tf1 = W.random_transforms(rng, n, (-0.2, -0.2, -0.2), (0.2, 0.2, 0.2))
    tf2 = W.random_transforms(rng, n, (-2.2, -2.2, -2.2), (2.2, 2.2, 2.2))
    return sc, h1, tf1, h2, tf2, ((va, ta), (vb, tb)), which


def _check_mesh_pairs(sc, backend, h1, tf1, h2, tf2):
    o, e = sc.b["oracle"], sc.b[backend]
    for req in (P.DistanceRequestPOD(), P.DistanceRequestPOD(rel_err=0.05, abs_err=0.01),
                P.DistanceRequestPOD(enable_nearest_points=0)):
        ro = o.batch_distance(h1, tf1, h2, tf2, req, nthreads=0)
        compare_distance(ro, e.batch_distance(h1, tf1, h2, tf2, req), what="mesh-mesh distance")
        assert np.all(P.status_path(ro["status"]) == P.PATH_BVH)
    ro = o.batch_distance(h1, tf1, h2, tf2, nthreads=0)
    assert (ro["min_distance"] == 0).sum() > 10 and (ro["min_distance"] > 0).sum() > 10
    assert np.all(ro["b1"] >= 0) and np.all(ro["b2"] >= 0) and np.all(np.isnan(ro["normal"]))
    sep = ro["min_distance"] > 0  # nearest points are world-frame and realise the distance
    assert np.allclose(np.linalg.norm(ro["p1"][sep] - ro["p2"][sep], axis=1), ro["min_distance"][sep], rtol=1e-9)
    for creq in (P.CollisionRequestPOD(), P.CollisionRequestPOD(security_margin=0.05),
                 P.CollisionRequestPOD(security_margin=-0.01), P.CollisionRequestPOD(num_max_contacts=3, enable_contact=0),
                 P.CollisionRequestPOD(gjk_variant=P.NesterovAcceleration)):
        co = o.batch_collide(h1, tf1, h2, tf2, creq, nthreads=0)
        compare_distance(co, e.batch_collide(h1, tf1, h2, tf2, creq), what="mesh-mesh collide")
    co = o.batch_collide(h1, tf1, h2, tf2, nthreads=0)
    assert co["num_contacts"].sum() > 10 and (co["num_contacts"] == 0).sum() > 10
    hit = co["num_contacts"] == 1
    assert np.all(co["b1"][hit] >= 0) and np.all(co["b2"][hit] >= 0)
    # collide and distance agree on which pairs touch
    assert np.array_equal(hit, ro["min_distance"] <= 1e-12)


def test_mesh_mesh_emulated_device_code_vs_oracle():
    sc, h1, tf1, h2, tf2, _, _ = build_mesh_pair_scene(False, True)
    _check_mesh_pairs(sc, "emu", h1, tf1, h2, tf2)


def test_mesh_mesh_distance_is_the_true_minimum():
    """differential check (test/distance.cpp style): BVTT walk + sqrTriDistance == brute force over all
    triangle pairs with the GJK triangle-triangle path"""
    sc, h1, tf1, h2, tf2, meshes, which = build_mesh_pair_scene(False, False, n=6, seg=8, ring=5)
    o = sc.b["oracle"]
    r = o.batch_distance(h1, tf1, h2, tf2)
    hts = []
    for (v, t) in meshes:
        cids = [o.register_convex(v[tri], None) for tri in t]
        hts.append(o.register_shapes(P.make_shapes([P.GEOM_TRIANGLE] * len(t), np.zeros((len(t), 3)), data=cids)))
    for q in range(len(h1)):
        ha, hb = hts[which[q, 0]], hts[which[q, 1]]
        ia, ib = np.meshgrid(np.arange(len(ha)), np.arange(len(hb)), indexing="ij")
        ia, ib = ia.ravel(), ib.ravel()
        rr = o.batch_distance(ha[ia], np.repeat(tf1[q:q + 1], len(ia)), hb[ib], np.repeat(tf2[q:q + 1], len(ia)),
                              nthreads=0)
        brute = max(rr["min_distance"].min(), 0.0)
        assert abs(r[q]["min_distance"] - brute) <= 1e-6 * max(1.0, brute)
        k = np.nonzero((ia == r[q]["b1"]) & (ib == r[q]["b2"]))[0][0]
        assert abs(max(rr["min_distance"][k], 0.0) - r[q]["min_distance"]) <= 1e-6


@pytest.mark.gpu
def test_mesh_mesh_gpu_vs_oracle():
    sc, h1, tf1, h2, tf2, _, _ = build_mesh_pair_scene(True, False, n=3000, seg=24, ring=12)
    _check_mesh_pairs(sc, "gpu", h1, tf1, h2, tf2)


@pytest.mark.gpu
def test_python_api_bvh_model():
    """the Python mirror of BVHModel<OBBRSS> + distance()/collide() against the batch path"""
    import hppfcl_b200 as hf
    verts, tris = W.sphere_mesh(1.0, 16, 8, noise=0.0, rng=np.random.default_rng(0))
    m = hf.BVHModelOBBRSS()
    with pytest.raises(ValueError):
        m.addVertex([0, 0, 0])
    m.beginModel()
    m.addSubModel(verts, tris)
    m.endModel()
    assert m.getNumBVs() == 2 * len(tris) - 1
    s = hf.Sphere(0.2)
    res = hf.DistanceResult()
    d = hf.distance(m, hf.Transform3f(), s, hf.Transform3f(T=[2.0, 0.1, 0.2]), hf.DistanceRequest(), res)
    r = np.linalg.norm([2.0, 0.1, 0.2])
    assert 0 <= d - (r - 1.0 - 0.2) < 8e-2 and res.b1 >= 0 and res.b2 == -1  # faceted sphere: inside the true one, within the facet sag
    cres = hf.CollisionResult()
    assert hf.collide(m, hf.Transform3f(), s, hf.Transform3f(T=[1.1, 0, 0]), hf.CollisionRequest(), cres) == 1
    cres.clear()
    assert hf.collide(m, hf.Transform3f(), m, hf.Transform3f(T=[2.5, 0, 0]), hf.CollisionRequest(), cres) == 0
    res.clear()
    d = hf.distance(m, hf.Transform3f(), m, hf.Transform3f(T=[2.5, 0, 0]), hf.DistanceRequest(), res)
    assert 0 <= d - 0.5 < 0.16 and res.b1 >= 0 and res.b2 >= 0
    # BVHModel<OBB>: collide() gives the OBBRSS model's contact (the plain OBB tree is its OBB half; for a primitive
    # partner the two models fit different boxes around it, but both are exact at the leaves); distance() is not offered
    mo = hf.BVHModelOBB()
    mo.beginModel()
    mo.addSubModel(verts, tris)
    mo.endModel()
    assert mo.getNodeType() == P.BV_OBB and mo.getNumBVs() == m.getNumBVs()
    box = hf.Box(0.4, 0.3, 0.5)
    tfb = hf.Transform3f.from_quat(0.9238795325112867, 0, 0.3826834323650898, 0, (1.05, 0.1, -0.2))
    ca, cb = hf.CollisionResult(), hf.CollisionResult()
    req = hf.CollisionRequest()
    req.num_max_contacts = 8
    na, nb = hf.collide(mo, hf.Transform3f(), box, tfb, req, ca), hf.collide(m, hf.Transform3f(), box, tfb, req, cb)
    assert na == nb and na >= 1
    assert sorted(c.b1 for c in ca.contacts) == sorted(c.b1 for c in cb.contacts)
    cm = hf.CollisionResult()
    assert hf.collide(mo, hf.Transform3f(), mo, hf.Transform3f(T=[1.9, 0, 0]), hf.CollisionRequest(), cm) == 1
    with pytest.raises(ValueError):
        hf.distance(mo, hf.Transform3f(), box, tfb, hf.DistanceRequest(), hf.DistanceResult())


@pytest.mark.gpu
def test_bvh_gpu_vs_oracle():
    sc, nodes, hm, tfm, hs, tfs, _ = build_scene(True, False, seg=40, ring=20, n=20000)
    _check(sc, "gpu", hm, tfm, hs, tfs)


@pytest.mark.gpu
def test_bvh_config4_shape():
    """config 4 geometry (10 000-triangle mesh vs capsules) on a 20k-query slice"""
    sc = make_scenes(gpu=True, emu=False)
    w = W.config4_mesh_vs_capsules(20000)
    bid, nodes = sc.register_bvh(w["verts"], w["tris"])
    assert len(w["tris"]) == 10000 and len(nodes) == 19999
    hb = sc.register_shapes(P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[bid]))
    hc = sc.register_shapes(w["capsules"])
    sc.commit()
    hm = np.full(len(w["hc"]), hb[0], dtype=np.uint32)
    ro = sc.b["oracle"].batch_distance(hm, w["tf_mesh"], hc[w["hc"]], w["tf_caps"], nthreads=0)
    rg = sc.b["gpu"].batch_distance(hm, w["tf_mesh"], hc[w["hc"]], w["tf_caps"])
    compare_distance(ro, rg, what="config4")


def _contacts_scene(backends):
    """two meshes and a pool of shapes registered identically in every backend given (name -> scene)"""
    rng = np.random.default_rng(5)
    ALL = (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER, P.GEOM_CONE, P.GEOM_ELLIPSOID)
    meshes = [W.sphere_mesh(1.0, 20, 10, noise=0.03, rng=rng), W.sphere_mesh(0.6, 12, 6, noise=0.05, rng=rng)]
    from oracle import oracle_lib
    from hppfcl_b200.engine import build_bvh_obbrss
    ids = []
    for v, t in meshes:
        got = set()
        for s in backends.values():
            if isinstance(s, oracle_lib.OracleScene):
                got.add(int(s.register_bvh(v, t)[0]))
            else:
                got.add(int(s.register_bvh_obbrss(build_bvh_obbrss(v, t), v, t)))
        assert len(got) == 1
        ids.append(got.pop())
    prims = W.random_primitive_shapes(rng, 32, ALL)
    prims["p"] *= 0.4
    rec = np.concatenate([P.make_shapes([P.BV_OBBRSS] * 2, [[0, 0, 0]] * 2, data=ids), prims])
    hs = [s.register_shapes(rec) for s in backends.values()]
    for s in backends.values():
        if hasattr(s, "commit"):
            s.commit()
    h = hs[0]
    n = 3000
    pool = np.concatenate([h[:2], h[:2], h])
    h1, h2 = pool[rng.integers(0, len(pool), n)], pool[rng.integers(0, len(pool), n)]
    tf1 = W.random_transforms(rng, n, (-.3, -.3, -.3), (.3, .3, .3))
    tf2 = W.random_transforms(rng, n, (-1.2, -1.2, -1.2), (1.2, 1.2, 1.2))
    return h1, tf1, h2, tf2


CONTACT_FIELDS = ("b1", "b2", "p1", "p2", "normal", "pos", "distance", "num_contacts")


def _same_fields(a, b, fields):
    for f in fields:
        x, y = a[f], b[f]
        ok = (x == y) | (np.isnan(x) & np.isnan(y)) if x.dtype.kind == "f" else x == y
        assert np.all(ok), "field %s differs" % f


def _check_contacts(backends, h1, tf1, h2, tf2, first, others):
    """hfb_batch_collide_contacts: every contact the reference keeps in CollisionResult::contacts (mesh-shape,
    shape-mesh with the operand swap, mesh-mesh), numContacts(), and contacts counted but not stored"""
    from oracle import oracle_lib
    total_extra = 0
    for kw, mx in ((dict(num_max_contacts=6), 3), (dict(num_max_contacts=3, security_margin=0.05), 5),
                   (dict(num_max_contacts=1), 2), (dict(num_max_contacts=50, enable_contact=0), 8)):
        req = P.CollisionRequestPOD(**kw)

        def run(s):
            kws = dict(nthreads=0) if isinstance(s, oracle_lib.OracleScene) else {}
            return s.batch_collide_contacts(h1, tf1, h2, tf2, req, mx, **kws)
        fo, fe, fc = run(backends[first])
        if isinstance(backends[first], oracle_lib.OracleScene) and not isinstance(backends[first], oracle_lib.RefScene):
            assert fo.tobytes() == backends[first].batch_collide(h1, tf1, h2, tf2, req, nthreads=0).tobytes()
        for name in others:
            o, e, c = run(backends[name])
            assert np.array_equal(fc, c), "numContacts differs (%s vs %s)" % (first, name)
            a, b_ = fo.copy(), o.copy()
            a["distance"][fc == 0] = 0  # the reference keeps no distance for a pair without a contact
            b_["distance"][fc == 0] = 0
            _same_fields(a, b_, CONTACT_FIELDS)
            for k in range(mx):
                m = fc > k + 1
                _same_fields(fe[m, k], e[m, k], CONTACT_FIELDS)
                total_extra += int(m.sum())
        assert fc.max() == min(kw["num_max_contacts"], fc.max())
    assert total_extra > 1000


def test_all_contacts_of_mesh_pairs():
    from oracle import oracle_lib
    from tests.common import EmuScene
    from tests.recorded_reference import reference_scene
    b = {"oracle": oracle_lib.OracleScene(P), "emu": EmuScene(), "ref": reference_scene(P)}
    h1, tf1, h2, tf2 = _contacts_scene(b)
    _check_contacts(b, h1, tf1, h2, tf2, "oracle", [k for k in b if k != "oracle"])


@pytest.mark.gpu
def test_plain_obb_models_gpu_vs_oracle():
    """BVHModel<OBB> (row X1): collide() of (OBB mesh, shape), (shape, OBB mesh) and (OBB mesh, OBB mesh) on the GPU
    against the oracle (which tests/test_reference_build.py::test_plain_obb_models pins to the reference build);
    distance() on a plain OBB model and mixed OBB / OBBRSS mesh pairs come back unsupported"""
    sc = make_scenes(gpu=True, emu=False)
    rng = np.random.default_rng(3)
    va, ta = W.sphere_mesh(1.0, 30, 15, noise=0.02, rng=rng)
    vb, tb = W.sphere_mesh(0.5, 12, 6, noise=0.04, rng=rng)
    b0, _ = sc.register_bvh(va, ta)
    b1, _ = sc.register_bvh_obb(va, ta)
    b2, _ = sc.register_bvh_obb(vb, tb)
    hm = sc.register_shapes(P.make_shapes([P.BV_OBBRSS, P.BV_OBB, P.BV_OBB], [[0, 0, 0]] * 3, data=[b0, b1, b2]))
    prims = W.random_primitive_shapes(rng, 64, SHAPES)
    prims["p"] *= 0.3
    hp = sc.register_shapes(prims)
    pts, ctris = W.icosahedron_from_ellipsoid((0.2, 0.3, 0.25))
    hc = sc.register_shapes(P.make_shapes([P.GEOM_CONVEX], [[0, 0, 0]], data=[sc.register_convex(pts, ctris)]))
    sc.commit()
    n = 20000
    tf1 = W.random_transforms(rng, n, (-.2, -.2, -.2), (.2, .2, .2))
    tf2 = W.random_transforms(rng, n, (-1.4, -1.4, -1.4), (1.4, 1.4, 1.4))
    hq = np.concatenate([hp, hc])[rng.integers(0, 65, n)]
    ho = hm[1:][rng.integers(0, 2, n)]
    ho2 = hm[1:][rng.integers(0, 2, n)]
    o, g = sc.b["oracle"], sc.b["gpu"]
    for req in (P.CollisionRequestPOD(), P.CollisionRequestPOD(security_margin=0.03, num_max_contacts=3)):
        for a1, t1, a2, t2 in ((ho, tf1, hq, tf2), (hq, tf2, ho, tf1), (ho[:4000], tf1[:4000], ho2[:4000], tf2[:4000])):
            want = o.batch_collide(a1, t1, a2, t2, req, nthreads=0)
            compare_distance(want, g.batch_collide(a1, t1, a2, t2, req), what="plain OBB collide")
    assert want["num_contacts"].sum() > 50
    for a2 in (hq[:64], ho2[:64], hm[:1].repeat(64)):
        d = g.batch_distance(ho[:64], tf1[:64], a2, tf2[:64])
        assert np.all(P.status_path(d["status"]) == P.PATH_UNSUPPORTED)
    c = g.batch_collide(ho[:64], tf1[:64], hm[:1].repeat(64), tf2[:64])
    assert np.all(P.status_path(c["status"]) == P.PATH_UNSUPPORTED)
