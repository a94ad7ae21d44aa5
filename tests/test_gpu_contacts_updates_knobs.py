"""GPU tests of the entry points added late in round 1 (all contacts of a mesh pair, in-place geometry updates,
the scheduling knobs of the mesh-shape kernels).  They passed on the driver's GPU run of round 1 and are plain
tests since."""
import pytest

from tests.common import P, hf

@pytest.mark.gpu
def test_all_contacts_of_mesh_pairs_on_the_gpu():
    from oracle import oracle_lib
    from tests.recorded_reference import reference_scene
    from tests.test_bvh_parity import _check_contacts, _contacts_scene
    b = {"oracle": oracle_lib.OracleScene(P), "gpu": hf.Engine(0), "ref": reference_scene(P)}
    h1, tf1, h2, tf2 = _contacts_scene(b)
    _check_contacts(b, h1, tf1, h2, tf2, "oracle", [k for k in b if k != "oracle"])


@pytest.mark.gpu
def test_geometry_update_and_release_on_the_gpu():
    from tests.test_cabi_and_host import _update_scenario
    _update_scenario(hf.Engine(0), hf.Engine(0))


@pytest.mark.gpu
def test_python_collide_keeps_every_contact_of_a_mesh_pair():
    import numpy as np
    from hppfcl_b200 import workloads as W
    verts, tris = W.sphere_mesh(1.0, 16, 8, noise=0.0, rng=np.random.default_rng(0))
    m = hf.BVHModelOBBRSS()
    m.beginModel()
    m.addSubModel(verts, tris)
    m.endModel()
    box = hf.Box(0.6, 0.6, 0.6)
    req = hf.CollisionRequest(num_max_contacts=8)
    res = hf.CollisionResult()
    n = hf.collide(m, hf.Transform3f(), box, hf.Transform3f.from_quat(1, 0, 0, 0, (0.9, 0, 0)), req, res)
    assert n == res.numContacts() and 1 < n <= 8
    assert len({c.b1 for c in res.contacts}) == n  # distinct triangles
    one = hf.CollisionResult()
    hf.collide(m, hf.Transform3f(), box, hf.Transform3f.from_quat(1, 0, 0, 0, (0.9, 0, 0)), hf.CollisionRequest(), one)
    assert one.numContacts() == 1 and one.contacts[0].b1 == res.contacts[0].b1


@pytest.mark.gpu
@pytest.mark.parametrize("env", [dict(HFB_BVHQ="0", HFB_BVH_QUORUM="1"), dict(HFB_BVHQ="0", HFB_BVH_BPS="2"),
                                 dict(HFB_BVHQ="0", HFB_BVH_QUORUM="1", HFB_BVH_BPS="1"),
                                 dict(HFB_BVHQ="0", HFB_BVH_ORDER="1"),
                                 dict(HFB_BVHQ="0", HFB_BVH_ORDER="1", HFB_BVH_QUORUM="1", HFB_BVH_BPS="2"),
                                 dict(HFB_BVH_SPEC="-1"), dict(HFB_BVH_SPEC="0"), dict(HFB_BVH_SPEC="0", HFB_BVH_ORDER="1"),
                                 dict(HFB_BVH_SPEC="25"), dict(HFB_BVH_SPEC="200", HFB_BVH_ORDER="1")])
def test_bvh_scheduling_knobs_do_not_change_results(env, monkeypatch):
    """k_bvh's set-up quorum, grid size and hand-out order (HFB_BVHQ=0: the lane-per-query kernel), and the
    speculation threshold / hand-out order of the task-system walk k_bvhq only change which lane runs what when; the
    batch also holds mesh-mesh and plain shape pairs, whose slices of the class-sorted index list the reordering must
    leave alone"""
    import numpy as np
    from hppfcl_b200 import workloads as W
    from oracle import oracle_lib
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    w = W.config4_mesh_vs_capsules(6000, seg=30, ring=15)
    eng, orc = hf.Engine(0), oracle_lib.OracleScene(P)
    bid = eng.register_bvh_obbrss(None, w["verts"], w["tris"])
    obid, _ = orc.register_bvh(w["verts"], w["tris"])
    assert bid == obid
    rec = np.concatenate([P.make_shapes([P.BV_OBBRSS], [[0, 0, 0]], data=[bid]), w["capsules"]])
    h = eng.register_shapes(rec)
    assert np.array_equal(h, orc.register_shapes(rec))
    eng.commit()
    hm = np.full(len(w["hc"]), h[0], dtype=np.uint32)
    hq = h[1:][w["hc"]]
    hm, hq = hm.copy(), hq.copy()
    hq[::50] = h[0]          # mesh-mesh pairs
    hm[1::50] = h[1:][w["hc"]][1::50]  # shape-shape pairs
    hm[2::50], hq[2::50] = hq[2::50].copy(), hm[2::50].copy()  # (shape, mesh): swapped operands
    got = eng.batch_distance(hm, w["tf_mesh"], hq, w["tf_caps"])
    want = orc.batch_distance(hm, w["tf_mesh"], hq, w["tf_caps"], nthreads=0)
    mm = (hm == h[0]) & (hq == h[0])  # the reference never writes `normal` on the mesh-mesh distance path
    for f in ("min_distance", "p1", "p2", "normal", "b1", "iterations"):
        x, y = got[f].copy(), want[f].copy()
        if f == "normal":
            x[mm] = y[mm] = 0
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), f
    tf_near = w["tf_caps"].copy()
    tf_near["T"] *= 0.5
    cg = eng.batch_collide(hm, w["tf_mesh"], hq, tf_near)
    cw = orc.batch_collide(hm, w["tf_mesh"], hq, tf_near, nthreads=0)
    for f in ("num_contacts", "b1", "p1", "p2", "normal", "distance_lower_bound"):
        assert np.array_equal(cg[f], cw[f], equal_nan=cg[f].dtype.kind == "f"), f
    assert cw["num_contacts"].sum() > 50
    assert eng.stats()["watchdog_trips"] == 0
