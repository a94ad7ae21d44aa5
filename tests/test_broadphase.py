"""Broadphase feed of the batched narrow phase (BASELINE config 5): scene boxes and overlapping pairs.
oracle/_ref cannot build hpp-fcl's broadphase managers (boost::function), so the checks are the definitions
themselves: CollisionObject::computeAABB restated in numpy (include/hpp/fcl/collision_object.h:258-278) and the
brute-force O(n^2) AABB::overlap test (BV/AABB.h:111-118) -- the set of pairs ANY of the reference's managers
reports to its collision callback."""
import numpy as np
import pytest

from tests.common import P, hf
from hppfcl_b200 import workloads as W


def brute_pairs(bb):
    n = len(bb)
    lo, hi = bb[:, None, :3], bb[:, None, 3:]
    ov = np.all((lo <= hi.transpose(1, 0, 2)) & (hi >= lo.transpose(1, 0, 2)), axis=2)
    i, j = np.nonzero(np.triu(ov, 1))
    return set(zip(i.tolist(), j.tolist()))


def ref_aabbs(local, tf):
    """computeAABB: the box around the rotated local box (rotation not the identity)"""
    R = tf["R"].reshape(-1, 3, 3).transpose(0, 2, 1)
    lo = R * local[None, None, :3]
    hi = R * local[None, None, 3:]
    mn = np.minimum(lo, hi)
    mx = np.maximum(lo, hi)
    out = np.empty((len(tf), 6))
    out[:, :3] = tf["T"] + ((mn[:, :, 0] + mn[:, :, 1]) + mn[:, :, 2])
    out[:, 3:] = tf["T"] + ((mx[:, :, 0] + mx[:, :, 1]) + mx[:, :, 2])
    return out


@pytest.mark.parametrize("n,scale", [(1, 10.0), (2, 1.0), (400, 40.0), (3000, 120.0), (3000, 30.0)])
def test_host_pair_finder_equals_brute_force(n, scale):
    rng = np.random.default_rng(n)
    c = scale * (2 * rng.random((n, 3)) - 1)
    e = 0.5 + 8 * rng.random((n, 3)) * (rng.random((n, 1)) < 0.9) + 60 * (rng.random((n, 1)) < 0.02)  # a few huge boxes
    bb = np.concatenate([c - e, c + e], axis=1)
    if n > 2:
        bb[1, :3] = bb[0, 3:]  # touching boxes overlap (closed intervals)
    f, s = hf.broadphase_pairs(bb)
    got = set(zip(f.tolist(), s.tolist()))
    assert len(got) == len(f) and all(a < b for a, b in got)
    assert got == brute_pairs(bb)
    # a capacity below the count: everything counted, `capacity` stored
    if len(f) > 5:
        f2, s2 = hf.broadphase_pairs(bb, capacity=5)
        assert len(f2) == 5 and set(zip(f2.tolist(), s2.tolist())) <= got


def test_unbounded_boxes_pair_with_everything_they_touch():
    """a Halfspace / Plane object has a box that is all of space on two or three axes: it stays out of the grid and is
    tested against every object (and against the other unbounded ones once)"""
    rng = np.random.default_rng(3)
    n = 1500
    c = 30 * (2 * rng.random((n, 3)) - 1)
    e = 0.5 + 3 * rng.random((n, 3))
    bb = np.concatenate([c - e, c + e], axis=1)
    big = np.finfo(np.float64).max
    bb[7] = [-big, -big, -big, big, big, 0.0]       # a floor: z <= 0
    bb[400] = [-np.inf, -np.inf, -np.inf, np.inf, np.inf, np.inf]   # a tilted halfspace: everything
    bb[1499] = [5.0, -big, -big, 5.0, big, big]     # a plane x = 5
    bb[3, :3], bb[3, 3:] = big, -big                 # an object without a box
    f, s = hf.broadphase_pairs(bb)
    got = set(zip(f.tolist(), s.tolist()))
    assert len(got) == len(f) and all(a < b for a, b in got)
    assert got == {p for p in brute_pairs(bb) if 3 not in p}  # (the boxless marker would "overlap" an infinite box)
    assert (7, 400) in got and (400, 1499) in got and (7, 1499) in got and not any(3 in p for p in got)
    assert sum(1 for p in got if 400 in p) == n - 2  # everything but itself and the boxless object


def test_scene_boxes_equal_the_reference():
    """aabb_local of every shape type (computeLocalAABB, Halfspace and Plane included) and CollisionObject::computeAABB,
    against the reference build itself: the host build of the product code (tests/emu) must give the same boxes bit for
    bit, poses with and without rotation"""
    from tests.common import EmuScene
    from tests.recorded_reference import reference_scene
    rng = np.random.default_rng(12)
    ref, emu = reference_scene(P), EmuScene()
    prims = W.random_primitive_shapes(rng, 48, (P.GEOM_BOX, P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_CYLINDER, P.GEOM_CONE,
                                                P.GEOM_ELLIPSOID))
    prims["ssr"] = np.where(rng.random(48) < 0.3, 0.05, 0.0)
    nd = np.concatenate([rng.normal(size=(12, 3)), rng.uniform(-2, 2, (12, 1))], axis=1)
    nd[:6] = [[0, 0, 1, 0.5], [0, 0, -3, 1.0], [2, 0, 0, -1.0], [0, -1, 0, 0.25], [0, 1, 0, 0], [-1, 0, 0, 2.0]]
    ssr = np.array([0.0, 0.1] * 6)
    pts, tris = W.ellipsoid_hull(rng, 24)
    hs = []
    for sc, name in ((ref, "ref"), (emu, "emu")):
        h = [sc.register_shapes(prims), sc.register_halfspaces(P.GEOM_HALFSPACE, nd, ssr),
             sc.register_halfspaces(P.GEOM_PLANE, nd, ssr)]
        cid = sc.register_convex(pts, tris) if name == "ref" else sc.register_convex(pts)
        h.append(sc.register_shapes(P.make_shapes([P.GEOM_CONVEX], [[0, 0, 0]], data=[cid])))
        hs.append(np.concatenate(h))
    assert np.array_equal(hs[0], hs[1])
    n = 4000
    oh = hs[0][rng.integers(0, len(hs[0]), n)]
    tf = W.random_transforms(rng, n, (-5, -5, -5), (5, 5, 5))
    tf[:1500] = W.identity_transforms(1500, T=tf["T"][:1500])
    a, b = ref.object_aabbs(oh, tf), emu.scene_aabbs(oh, tf)
    same = (a == b) | (np.isnan(a) & np.isnan(b))
    assert same.all(), "boxes differ at rows %s" % np.unique(np.nonzero(~same)[0])[:10]
    assert np.isinf(a).any() and (np.abs(a) == np.finfo(np.float64).max).any()  # rotated and unrotated halfspaces
    # and the pairs these boxes give are the brute-force set
    f, s = hf.broadphase_pairs(b[:800])
    assert set(zip(f.tolist(), s.tolist())) == brute_pairs(b[:800])


def test_config5_scene_has_the_intended_density():
    w = W.config5_moving_boxes(20_000, target_pairs=100_000)
    local = np.array([-2.5, -5, -10, 2.5, 5, 10.0])
    bb = ref_aabbs(local, w["obj_tf"])
    f, s = hf.broadphase_pairs(bb)
    assert 50_000 < len(f) < 200_000
    moved = w["step"](3)
    assert np.abs(moved["T"] - w["obj_tf"]["T"]).max() <= 1.0
    R = moved["R"].reshape(-1, 3, 3)
    assert np.allclose(R @ R.transpose(0, 2, 1), np.eye(3), atol=1e-12)


@pytest.mark.gpu
def test_scene_aabbs_and_device_broadphase():
    """scene boxes (host and device) against the numpy restatement; the device pair finder against the host one;
    and the whole feed: boxes -> pairs -> hfb_batch_collide_objects_device against the pair-row call"""
    import torch
    rng = np.random.default_rng(5)
    eng = hf.Engine(0)
    prims = W.random_primitive_shapes(rng, 64, (P.GEOM_BOX, P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_CYLINDER, P.GEOM_CONE,
                                                P.GEOM_ELLIPSOID))
    hp = eng.register_shapes(prims)
    pts, _ = W.ellipsoid_hull(rng, 24)
    hc = eng.register_shapes(P.make_shapes([P.GEOM_CONVEX], [[0, 0, 0]], data=[eng.register_convex(pts)]))
    eng.commit()
    n = 30_000
    oh = np.concatenate([hp, hc])[rng.integers(0, 65, n)].astype(np.uint32)
    tf = W.random_transforms(rng, n, (-14, -14, -14), (14, 14, 14))
    tf[:50] = W.identity_transforms(50, T=tf["T"][:50])  # the isIdentity() branch of computeAABB
    bb = eng.scene_aabbs(oh, tf)
    # numpy restatement for the box objects
    for h in hp[:8]:
        m = (oh == h) & (np.arange(n) >= 50)
        rec = prims[h - hp[0]]
        if rec["type"] != P.GEOM_BOX or not m.any():
            continue
        local = np.concatenate([-rec["p"], rec["p"]])
        assert np.array_equal(bb[m], ref_aabbs(local, tf[m]))
    box0 = prims["type"][oh[:50] - hp[0]] == P.GEOM_BOX if (oh[:50] < hc[0]).all() else None

    def dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()

    stream = torch.cuda.current_stream().cuda_stream
    d_h, d_tf = dev(oh), dev(tf)
    d_bb = torch.empty(n * 6, dtype=torch.float64, device="cuda")
    eng.scene_aabbs_device(n, d_h.data_ptr(), d_tf.data_ptr(), d_bb.data_ptr(), stream)
    torch.cuda.synchronize()
    assert np.array_equal(d_bb.cpu().numpy().reshape(n, 6), bb)
    f, s = hf.broadphase_pairs(bb)
    want = set(zip(f.tolist(), s.tolist()))
    assert len(want) > 20_000
    cap = len(want) + 1000
    d_f = torch.empty(cap, dtype=torch.int32, device="cuda")
    d_s = torch.empty(cap, dtype=torch.int32, device="cuda")
    d_n = torch.zeros(1, dtype=torch.int32, device="cuda")
    for _ in range(2):  # twice: the scratch is reused
        eng.broadphase_pairs_device(n, d_bb.data_ptr(), d_f.data_ptr(), d_s.data_ptr(), cap, d_n.data_ptr(), stream)
    torch.cuda.synchronize()
    k = int(d_n.item())
    gf, gs = d_f[:k].cpu().numpy().astype(np.uint32), d_s[:k].cpu().numpy().astype(np.uint32)
    assert k == len(want) and set(zip(gf.tolist(), gs.tolist())) == want
    # the feed end to end: device pairs -> collide of the object pairs == collide of the expanded rows
    d_out = torch.empty(k * P.contact_dtype.itemsize, dtype=torch.uint8, device="cuda")
    eng.batch_collide_objects_device(n, d_h.data_ptr(), d_tf.data_ptr(), k, d_f.data_ptr(), d_s.data_ptr(), d_out.data_ptr(),
                                     stream=stream)
    torch.cuda.synchronize()
    rows = eng.batch_collide(oh[gf], tf[gf], oh[gs], tf[gs])
    assert d_out.cpu().numpy().tobytes() == rows.tobytes()
    assert rows["num_contacts"].sum() > 1000
    # a capacity below the count: everything counted
    eng.broadphase_pairs_device(n, d_bb.data_ptr(), d_f.data_ptr(), d_s.data_ptr(), 100, d_n.data_ptr(), stream)
    torch.cuda.synchronize()
    assert int(d_n.item()) == len(want)
    # the scene cut in three ranges of objects (three GPUs): the union of the ranges' pairs is the whole set
    got = set()
    for lo, cnt in ((0, 10_000), (10_000, 7_777), (17_777, n)):
        eng.broadphase_pairs_device(n, d_bb.data_ptr(), d_f.data_ptr(), d_s.data_ptr(), cap, d_n.data_ptr(), stream,
                                    first_object=lo, num_first_objects=cnt)
        torch.cuda.synchronize()
        kk = int(d_n.item())
        part = set(zip(d_f[:kk].cpu().numpy().tolist(), d_s[:kk].cpu().numpy().tolist()))
        assert len(part) == kk and all(lo <= a < lo + cnt for a, _ in part) and not (part & got)
        got |= part
    assert got == want


@pytest.mark.gpu
def test_scene_with_a_floor_and_a_wall():
    """a Halfspace floor and a Plane wall among ten thousand shapes: boxes against the reference build, the device pair
    finder against the host one and brute force, hfb_scene_collide against the oracle on exactly those pairs"""
    from oracle import oracle_lib
    from tests.recorded_reference import reference_scene
    rng = np.random.default_rng(17)
    eng, orc = hf.Engine(0), oracle_lib.OracleScene(P)
    prims = W.random_primitive_shapes(rng, 32, (P.GEOM_BOX, P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_CYLINDER))
    nd_floor, nd_wall = [[0, 0, 1, 0.0]], [[1, 0, 0, 6.0]]
    hs = []
    for sc in (eng, orc):
        hs.append(np.concatenate([sc.register_shapes(prims), sc.register_halfspaces(P.GEOM_HALFSPACE, nd_floor),
                                  sc.register_halfspaces(P.GEOM_PLANE, nd_wall)]))
    eng.commit()
    assert np.array_equal(hs[0], hs[1])
    n = 10_000
    oh = hs[0][rng.integers(0, 32, n)].astype(np.uint32)
    tf = W.random_transforms(rng, n, (-10, -10, 0.2), (10, 10, 6))
    oh[0], oh[n - 1] = hs[0][32], hs[0][33]  # the floor first, the wall last
    tf[0] = W.identity_transforms(1)[0]
    tf[n - 1] = W.identity_transforms(1)[0]
    tf["T"][:400, 2] = rng.uniform(-0.3, 0.6, 400)  # four hundred objects on or in the floor
    tf["T"][0] = 0
    bb = eng.scene_aabbs(oh, tf)
    ref = reference_scene(P)
    assert np.array_equal(np.concatenate([ref.register_shapes(prims), ref.register_halfspaces(P.GEOM_HALFSPACE, nd_floor),
                                          ref.register_halfspaces(P.GEOM_PLANE, nd_wall)]), hs[0])
    assert np.array_equal(ref.object_aabbs(oh, tf), bb)
    f, s = hf.broadphase_pairs(bb)
    want = set(zip(f.tolist(), s.tolist()))
    assert sum(1 for a, b in want if a == 0) > 150 and sum(1 for a, b in want if b == n - 1) > 20
    assert want == brute_pairs(bb[:1500]) | {p for p in want if p[1] >= 1500}  # brute force on a prefix
    fo, so, rec, ncand, nhit = eng.scene_collide(oh, tf, capacity=len(want) + 100)
    assert set(zip(fo.tolist(), so.tolist())) <= want and ncand == len(want) and nhit == len(fo)
    ro = orc.batch_collide(oh[f], tf[f], oh[s], tf[s], nthreads=0)
    hit = {(int(a), int(b)) for a, b, c in zip(f, s, ro["num_contacts"]) if c}
    assert hit == set(zip(fo.tolist(), so.tolist())) and len(hit) > 100
    key = {p: k for k, p in enumerate(zip(f.tolist(), s.tolist()))}
    order = np.array([key[p] for p in zip(fo.tolist(), so.tolist())])
    assert rec.tobytes() == ro[order].tobytes()


@pytest.mark.gpu
def test_scene_collide_in_one_call():
    """hfb_scene_collide (boxes, broadphase, collide of the candidates, compaction -- all on the device) against the
    pieces: host pair finder + pair-row collide; whole scene and cut in two ranges of objects"""
    w = W.config5_moving_boxes(20_000, target_pairs=150_000)
    eng = hf.Engine(0)
    hb = eng.register_shapes(w["shapes"])
    eng.commit()
    oh = hb[w["obj_h"]]
    for k in (0, 1):
        tf = w["step"](k)
        f, s, rec, ncand, nhit = eng.scene_collide(oh, tf)
        pf, ps = hf.broadphase_pairs(eng.scene_aabbs(oh, tf))
        assert ncand == len(pf) and ncand > 50_000
        rows = eng.batch_collide(oh[pf], tf[pf], oh[ps], tf[ps])
        hit = rows["num_contacts"] > 0
        assert nhit == int(hit.sum()) == len(f) and nhit > 1000
        want = {(int(a), int(b)): rows[i].tobytes() for i, (a, b) in enumerate(zip(pf, ps)) if hit[i]}
        got = {(int(a), int(b)): rec[i].tobytes() for i, (a, b) in enumerate(zip(f, s))}
        assert got == want
    half = len(oh) // 2
    f1, s1, _, c1, h1 = eng.scene_collide(oh, tf, first_object=0, num_first_objects=half)
    f2, s2, _, c2, h2 = eng.scene_collide(oh, tf, first_object=half, num_first_objects=len(oh))
    assert c1 + c2 == ncand and h1 + h2 == nhit and (f1 < half).all() and (f2 >= half).all()
    # capacity below the number of colliding pairs: all counted
    f3, _, _, _, h3 = eng.scene_collide(oh, tf, capacity=50)
    assert h3 == nhit and len(f3) == 50


@pytest.mark.gpu
def test_python_manager_mirror():
    """DynamicAABBTreeCollisionManager / CollisionObject / CollisionCallBackCollect of the Python mirror: the pairs the
    callback sees are the brute-force set of overlapping boxes, collide_batch() agrees with collide() pair by pair, a
    floor Halfspace takes part, update() follows moved objects"""
    rng = np.random.default_rng(31)
    geoms = [hf.Box(*(0.2 + rng.random(3))) for _ in range(6)] + [hf.Sphere(0.3), hf.Capsule(0.2, 0.6), hf.Cylinder(0.25, 0.5)]
    objs = [hf.CollisionObject(geoms[rng.integers(0, len(geoms))],
                               hf.Transform3f.from_quat(*(lambda q: q / np.linalg.norm(q))(rng.normal(size=4)), rng.uniform(-3, 3, 3)))
            for _ in range(400)]
    floor = hf.CollisionObject(hf.Halfspace([0, 0, 1], -2.5))
    mgr = hf.DynamicAABBTreeCollisionManager()
    mgr.registerObjects(objs)
    mgr.registerObject(floor)
    mgr.setup()
    assert mgr.size() == 401 and not mgr.empty()
    bb = np.array([np.concatenate([o.getAABB().min_, o.getAABB().max_]) for o in mgr.getObjects()])
    cb = hf.CollisionCallBackCollect(100000)
    mgr.collide(cb)
    idx = {id(o): k for k, o in enumerate(mgr.getObjects())}
    got = {tuple(sorted((idx[id(a)], idx[id(b)]))) for a, b in cb.getCollisionPairs()}
    assert got == brute_pairs(bb) and len(got) == cb.numCollisionPairs() and any(400 in p for p in got)
    first, second, rec = mgr.collide_batch()
    assert {(int(a), int(b)) for a, b in zip(first, second)} == got
    req = hf.CollisionRequest()
    for k in rng.choice(len(first), 40, replace=False):
        a, b = mgr.getObjects()[first[k]], mgr.getObjects()[second[k]]
        res = hf.CollisionResult()
        assert hf.collide(a.geom, a.tf, b.geom, b.tf, req, res) == int(rec["num_contacts"][k])
    assert rec["num_contacts"].sum() > 10
    objs[0].setTransform(hf.Transform3f(T=[50.0, 50.0, 50.0]))  # far away from everything (and above the floor)
    mgr.update()
    f2, s2 = mgr.pairs()
    assert not np.any(f2 == 0) and not np.any(s2 == 0)
