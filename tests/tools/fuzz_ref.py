"""Three-way fuzz on the CPU: the reference build (oracle/_ref, hpp-fcl's sources compiled in place), the
oracle's restatement and the DEVICE code compiled for the host (tests/emu) on adversarial batches:
axis-aligned poses, coincident centres, touching surfaces, nested shapes, extreme scales, symmetric
hulls, degenerate meshes, random request fields.  Every record must agree bit for bit.

    python tests/tools/fuzz_ref.py --minutes 10 [--seed 1] [--n 4000]

Prints one line per round; stops at the first mismatch (exit 1) unless --keep-going; a failing round is
rebuilt from its seed with build_cases().
(Test infrastructure: the reference leg needs oracle/_ref (oracle/Makefile `ref`); without it only oracle vs emu run.)
"""
import argparse
import itertools
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from tests.common import P, EmuScene, compare_distance  # noqa: E402
from hppfcl_b200 import workloads as W  # noqa: E402
from oracle import oracle_lib  # noqa: E402
from tests.recorded_reference import reference_scene  # noqa: E402

ALL = (P.GEOM_SPHERE, P.GEOM_CAPSULE, P.GEOM_BOX, P.GEOM_CYLINDER, P.GEOM_CONE, P.GEOM_ELLIPSOID)


def signed_permutations():
    out = []
    for perm in itertools.permutations(range(3)):
        for sg in itertools.product((1.0, -1.0), repeat=3):
            R = np.zeros((3, 3))
            for r, (c, s) in enumerate(zip(perm, sg)):
                R[r, c] = s
            if np.linalg.det(R) > 0:
                out.append(R)
    return np.array(out)


AXIS_ROT = signed_permutations()


def adversarial_shapes(rng, n, scale):
    s = W.random_primitive_shapes(rng, n, ALL)
    k = rng.random(n)
    # round numbers (ties in the Voronoi tests), equal sides, thin shapes
    m = k < 0.25
    s["p"][m] = np.round(s["p"][m] * 4 + 0.5) / 4
    m = (k >= 0.25) & (k < 0.35)
    s["p"][m, 1] = s["p"][m, 0]
    s["p"][m, 2] = np.where(s["type"][m] == P.GEOM_BOX, s["p"][m, 0], s["p"][m, 2])
    m = (k >= 0.35) & (k < 0.45)
    s["p"][m, 0] *= 1e-3
    t = s["type"]
    s["p"][(t == P.GEOM_SPHERE), 1:] = 0
    s["p"][(t == P.GEOM_CAPSULE) | (t == P.GEOM_CYLINDER) | (t == P.GEOM_CONE), 2] = 0
    el = t == P.GEOM_ELLIPSOID
    s["p"][el] = np.maximum(s["p"][el], 1e-3)
    s["p"] *= scale
    if rng.random() < 0.3:
        s["ssr"] = np.where(rng.random(n) < 0.5, rng.random(n) * 0.1 * scale, 0.0)
    return s


def adversarial_poses(rng, n, scale, mode):
    if mode == "random":
        tf1 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
        tf2 = W.random_transforms(rng, n, (-2, -2, -2), (2, 2, 2))
    elif mode == "axis":
        R1 = AXIS_ROT[rng.integers(0, len(AXIS_ROT), n)]
        R2 = AXIS_ROT[rng.integers(0, len(AXIS_ROT), n)]
        T1 = np.round(rng.uniform(-1, 1, (n, 3)) * 4) / 4
        T2 = np.round(rng.uniform(-2, 2, (n, 3)) * 4) / 4
        tf1, tf2 = P.make_transforms(R1, T1), P.make_transforms(R2, T2)
    elif mode == "coincident":
        tf1 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
        tf2 = W.random_transforms(rng, n, (0, 0, 0), (0, 0, 0))
        tf2["T"] = tf1["T"]
        same = rng.random(n) < 0.5
        tf2["R"][same] = tf1["R"][same]
        tiny = rng.random(n) < 0.3
        tf2["T"][tiny] += rng.normal(size=(int(tiny.sum()), 3)) * 1e-9
    elif mode == "identity":
        tf1 = W.identity_transforms(n)
        tf2 = W.identity_transforms(n, rng.uniform(-2, 2, (n, 3)) * (rng.random((n, 3)) < 0.5))
    elif mode == "far":
        tf1 = W.random_transforms(rng, n, (-1, -1, -1), (1, 1, 1))
        tf2 = W.random_transforms(rng, n, (1e3, -1, -1), (1e4, 1, 1))
    else:
        raise ValueError(mode)
    tf1["T"] *= scale
    tf2["T"] *= scale
    return tf1, tf2


def touching(orc, h1, tf1, h2, tf2, rng):
    """slide operand 2 along the separating normal until the surfaces (almost) touch"""
    r = orc.batch_distance(h1, tf1, h2, tf2, nthreads=0)
    ok = np.isfinite(r["min_distance"]) & np.all(np.isfinite(r["normal"]), axis=1) & (np.abs(r["min_distance"]) < 1e30)
    eps = rng.choice([0.0, 1e-12, -1e-12, 1e-9, -1e-9, 1e-6, -1e-6, 1e-3, -1e-3], size=len(r))
    tf2 = tf2.copy()
    shift = r["normal"] * (r["min_distance"] * (1.0 + eps))[:, None]
    tf2["T"][ok] -= shift[ok]
    return tf2


def random_request(rng, kind):
    kw = {}
    if rng.random() < 0.6:
        kw["gjk_variant"] = int(rng.choice([P.DefaultGJK, P.PolyakAcceleration, P.NesterovAcceleration]))
    if rng.random() < 0.4:
        kw["gjk_convergence_criterion"] = int(rng.choice([P.Default, P.DualityGap, P.Hybrid]))
        kw["gjk_convergence_criterion_type"] = int(rng.choice([P.Relative, P.Absolute]))
    if rng.random() < 0.3:
        kw["gjk_tolerance"] = float(rng.choice([1e-3, 1e-8, 1e-10]))
    if rng.random() < 0.3:
        kw["epa_tolerance"] = float(rng.choice([1e-3, 1e-8, 1e-10]))
    if rng.random() < 0.2:
        kw["gjk_max_iterations"] = int(rng.choice([1, 2, 5, 20]))
    if rng.random() < 0.2:
        kw["epa_max_iterations"] = int(rng.choice([1, 2, 5, 20]))
    if rng.random() < 0.2:
        kw["gjk_initial_guess"] = P.BoundingVolumeGuess
    if kind == "distance":
        if rng.random() < 0.2:
            kw["enable_signed_distance"] = 0
        return P.DistanceRequestPOD(**kw), kw
    if rng.random() < 0.4:
        kw["security_margin"] = float(rng.choice([0.05, -0.02, 1e-9, 0.5]))
    if rng.random() < 0.2:
        kw["enable_contact"] = 0
    if rng.random() < 0.2:
        kw["distance_upper_bound"] = float(rng.choice([0.0, 0.3, 1e-9]))
    if rng.random() < 0.2:
        kw["num_max_contacts"] = int(rng.choice([2, 5]))
    if rng.random() < 0.1:
        kw["collision_distance_threshold"] = float(rng.choice([0.0, 1e-6]))
    return P.CollisionRequestPOD(**kw), kw


def small_hulls(rng, scale):
    hulls = [W.icosahedron_from_ellipsoid(rng.uniform(0.1, 1, 3)) for _ in range(3)]
    # cube and brick as ConvexBase (ties between vertices for axis-aligned directions)
    for half in ((0.5, 0.5, 0.5), (0.25, 0.5, 1.0)):
        pts = np.array(list(itertools.product((-1, 1), repeat=3)), dtype=np.float64) * half
        hulls.append((pts, hull_tris(pts)))
    tet = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float64) - 0.25
    hulls.append((tet, hull_tris(tet)))
    for nv in (6, 10, 20, 32):
        hulls.append(W.ellipsoid_hull(rng, nv))
    return [(p * scale, t) for p, t in hulls]


def big_hulls(rng, scale):
    """more than 32 vertices: the reference climbs over neighbours (support_functions.cpp:324-397); lattices and
    prisms give it plateaus and ties to walk through"""
    hulls = [W.ellipsoid_hull(rng, nv) for nv in (33, 48, 64, 100)]
    k = 12  # 2 x 3k-gon prism, regular: every side face is a rectangle (ties along edges)
    ang = 2 * np.pi * np.arange(3 * k) / (3 * k)
    ring = np.stack([np.cos(ang), np.sin(ang)], axis=1)
    prism = np.concatenate([np.c_[ring, np.full(3 * k, -0.5)], np.c_[ring, np.full(3 * k, 0.5)]])
    hulls.append((prism, hull_tris(prism)))
    g = np.array(list(itertools.product((-1.0, -1 / 3, 1 / 3, 1.0), repeat=3)))
    shell = g[np.abs(g).max(axis=1) == 1.0]  # 56 lattice points on the faces of a cube: coplanar quadruples
    shell = shell / np.linalg.norm(shell, axis=1, keepdims=True) * (1 + 0.05 * rng.random((len(shell), 1)))
    hulls.append((shell, hull_tris(shell)))
    return [(np.ascontiguousarray(p * scale), t) for p, t in hulls if len(np.unique(t)) == len(p)]


def hull_tris(pts):
    from scipy.spatial import ConvexHull
    h = ConvexHull(pts)
    tris = h.simplices.astype(np.uint32)
    c = pts.mean(axis=0)
    a, b, cc = pts[tris[:, 0]], pts[tris[:, 1]], pts[tris[:, 2]]
    flip = np.einsum("ij,ij->i", np.cross(b - a, cc - a), a - c) < 0
    tris[flip] = tris[flip][:, [0, 2, 1]]
    return tris


BIG_MESHES = [False]  # --big-meshes: deeper trees (1 600 and 640 triangles) and more mesh queries per round


def fuzz_meshes(rng, scale):
    out = []
    if BIG_MESHES[0]:
        out.append(W.sphere_mesh(1.0, 40, 20, noise=0.02, rng=rng))
        out.append(W.sphere_mesh(0.7, 32, 10, noise=0.0, rng=rng))
    out.append(W.sphere_mesh(1.0, 12, 6, noise=0.05, rng=rng))
    out.append(W.sphere_mesh(0.5, 8, 4, noise=0.0, rng=rng))  # symmetric: ties in the fit and the walk
    # flat grid (rank-deficient covariance), then a soup of random triangles
    g = 5
    xs, ys = np.meshgrid(np.arange(g + 1) / g - 0.5, np.arange(g + 1) / g - 0.5)
    v = np.stack([xs.ravel(), ys.ravel(), np.zeros(xs.size)], axis=1)
    t = []
    for i in range(g):
        for j in range(g):
            a = i * (g + 1) + j
            t += [[a, a + 1, a + g + 2], [a, a + g + 2, a + g + 1]]
    out.append((v, np.array(t, dtype=np.uint32)))
    sv = rng.uniform(-1, 1, (60, 3))
    out.append((sv, rng.integers(0, 60, (40, 3)).astype(np.uint32)))
    out.append((rng.uniform(-1, 1, (3, 3)), np.array([[0, 1, 2]], dtype=np.uint32)))  # one triangle: root is a leaf
    return [(np.ascontiguousarray(v * scale), t) for v, t in out]


class Backends:
    """`emu` is any scene with the product's registration interface: the host build of the device code
    (EmuScene) or, on a GPU box, hppfcl_b200.Engine"""

    def __init__(self, use_ref, use_emu):
        self.orc = oracle_lib.OracleScene(P)
        self.ref = reference_scene(P) if use_ref else None
        self.emu = (use_emu if not isinstance(use_emu, bool) else EmuScene()) if use_emu else None

    def register_shapes(self, s):
        h = self.orc.register_shapes(s)
        if self.ref:
            assert np.array_equal(h, self.ref.register_shapes(s))
        if self.emu:
            assert np.array_equal(h, self.emu.register_shapes(s))
        return h

    def register_convex(self, pts, tris):
        i = self.orc.register_convex(pts, tris)
        if self.ref:
            assert self.ref.register_convex(pts, tris) == i
        if self.emu:
            assert self.emu.register_convex(pts) == i
        return i

    def register_halfspaces(self, kind, nd, ssr):
        h = self.orc.register_halfspaces(kind, nd, ssr)
        if self.ref:
            assert np.array_equal(h, self.ref.register_halfspaces(kind, nd, ssr))
        if self.emu:
            assert np.array_equal(h, self.emu.register_halfspaces(kind, nd, ssr))
        return h

    def register_bvh(self, v, t):
        i, nodes = self.orc.register_bvh(v, t)
        if self.ref:
            j, rn = self.ref.register_bvh(v, t)
            assert i == j
            assert nodes.tobytes() == rn.tobytes(), "BVH builders differ"
        if self.emu:
            assert self.emu.register_bvh_obbrss(nodes, v, t) == i
        return i

    def commit(self):
        if self.emu:
            self.emu.commit()


D_MESH = ("min_distance", "p1", "p2", "b1", "b2")
C_MESH = ("p1", "p2", "normal", "pos", "distance_lower_bound", "b1", "b2", "num_contacts")


def cmp_fields(a, b, fields, what):
    for f in fields:
        x, y = a[f], b[f]
        ok = (x == y) | (np.isnan(x) & np.isnan(y)) if x.dtype.kind == "f" else x == y
        assert np.all(ok), "%s: field %s differs at rows %s" % (what, f, np.unique(np.nonzero(~ok)[0])[:8])


def cmp_collide(ref, got, what):
    ref, got = ref.copy(), got.copy()
    nc = ref["num_contacts"] == 0
    ref["distance"][nc] = 0
    got["distance"][nc] = 0
    compare_distance(ref, got, what=what)


def build_cases(seed, n, use_ref, use_emu):
    """-> (backends, tag, [(name, kind, h1, tf1, h2, tf2, request, request kwargs)])"""
    rng = np.random.default_rng(seed)
    scale = float(rng.choice([1.0, 1.0, 1.0, 1e-3, 1e3, 37.5]))
    B = Backends(use_ref, use_emu)
    prim = adversarial_shapes(rng, 256, scale)
    hp = B.register_shapes(prim)
    ids = [B.register_convex(p, t) for p, t in small_hulls(rng, scale)]
    hc = B.register_shapes(P.make_shapes([P.GEOM_CONVEX] * len(ids), np.zeros((len(ids), 3)), data=ids))
    big = big_hulls(rng, scale)
    bids = [B.register_convex(p, t) for p, t in big]
    hb = B.register_shapes(P.make_shapes([P.GEOM_CONVEX] * len(bids), np.zeros((len(bids), 3)), data=bids))
    mids = [B.register_bvh(v, t) for v, t in fuzz_meshes(rng, scale)]
    hm = B.register_shapes(P.make_shapes([P.BV_OBBRSS] * len(mids), np.zeros((len(mids), 3)), data=mids))
    # Plane / Halfspace geometries (--planes; their own generator, so that the other cases of a seed do not change):
    # axis-aligned and tilted normals of any length, the same plane twice and mirrored (parallel / anti-parallel pairs),
    # offsets at the scene's scale, some with a swept-sphere radius
    hh = hq = None
    if PLANES[0]:
        prng = np.random.default_rng([seed, 0x9E3779B9])
        npl = 24
        nd = np.concatenate([prng.normal(size=(npl, 3)) * prng.uniform(0.1, 10, (npl, 1)), prng.uniform(-1.5, 1.5, (npl, 1)) * scale], axis=1)
        for k, ax in enumerate(((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1), (0, 0, 1), (0, 0, 0))):
            nd[k, :3] = np.asarray(ax, dtype=np.float64) * prng.uniform(0.5, 2.0)  # (the last: the degenerate normal -> (1, 0, 0), 0)
        nd[8] = nd[9] * 3.0
        nd[10, :3] = -nd[9, :3]
        nd[11, 3] = 0.0
        pssr = np.where(prng.random(npl) < 0.3, prng.uniform(0.0, 0.2, npl) * scale, 0.0)
        hh = B.register_halfspaces(P.GEOM_HALFSPACE, nd, pssr)
        hq = B.register_halfspaces(P.GEOM_PLANE, nd, pssr)
    B.commit()
    mode = str(rng.choice(["random", "axis", "coincident", "identity", "far", "touch", "touch"]))
    base = "random" if mode == "touch" else mode
    tf1, tf2 = adversarial_poses(rng, n, scale, base)
    pool = np.concatenate([hp, hc, hc, hc])
    h1, h2 = pool[rng.integers(0, len(pool), n)], pool[rng.integers(0, len(pool), n)]
    if mode == "touch":
        tf2 = touching(B.orc, h1, tf1, h2, tf2, rng)
    dreq, dkw = random_request(rng, "distance")
    creq, ckw = random_request(rng, "collide")
    tag = "seed %d scale %g mode %s" % (seed, scale, mode)
    cases = [("shapes", "distance", h1, tf1, h2, tf2, dreq, dkw), ("shapes", "collide", h1, tf1, h2, tf2, creq, ckw)]
    # CachedGuess with arbitrary guesses (some below the tolerance: the (-1,0,0) restart of gjk.cpp:208-213)
    gg = rng.normal(size=(n, 3)) * scale
    gg[rng.random(n) < 0.1] = 0
    gh = np.zeros((n, 2), dtype=np.int32)
    for kind in ("distance", "collide"):
        req, kw = random_request(rng, kind)
        req.q.gjk_initial_guess = P.CachedGuess
        req.q.cached_gjk_guess = gg.ctypes.data
        req.q.cached_support_func_guess = gh.ctypes.data
        kw = dict(kw, gjk_initial_guess="cached")
        cases.append(("shapes", kind, h1, tf1, h2, tf2, req, kw, (gg, gh)))  # the arrays the request points into
    # the plane family against everything (and itself), either operand order
    if PLANES[0]:
        npf = max(200, n // 3)
        fam = np.concatenate([hh, hq])
        pa = fam[prng.integers(0, len(fam), npf)]
        pb = np.where(prng.random(npf) < 0.15, fam[prng.integers(0, len(fam), npf)], pool[prng.integers(0, len(pool), npf)])
        sw = prng.random(npf) < 0.5
        p1, p2 = np.where(sw, pb, pa).astype(np.uint32), np.where(sw, pa, pb).astype(np.uint32)
        pt1, pt2 = tf1[:npf].copy(), tf2[:npf].copy()
        same = prng.random(npf) < 0.3  # (parallel planes stay parallel under a common rotation)
        pt2["R"][same] = pt1["R"][same]
        for kind in ("distance", "collide"):
            req, kw = random_request(prng, kind)
            cases.append(("planes", kind, p1, pt1, p2, pt2, req, kw))
    # --drift: poses as they come out of files and long products -- quaternions rounded to 8 ... 14 digits and not
    # normalised again, or matrices with a relative error of 1e-14 ... 1e-9 --, the same rotation for both operands,
    # the second one on an axis of the first and slid until the surfaces (almost) touch: GJK then ends with the
    # origin on its last simplex up to rounding and the answers sit next to tolerance and threshold (found by the
    # reference's collide_conecylinder case, tests/test_shape_collide_known_answers.py)
    if DRIFT[0]:
        drng = np.random.default_rng([seed, 0x51ED270B])
        nd_ = max(200, n // 3)
        q = drng.normal(size=(nd_, 4))
        q /= np.linalg.norm(q, axis=1)[:, None]
        digits = drng.integers(8, 15, nd_)
        q = np.where((drng.random(nd_) < 0.7)[:, None], np.round(q * 10.0 ** digits[:, None]) / 10.0 ** digits[:, None], q)
        Rd = W.quat_to_rot(q[:, 0], q[:, 1], q[:, 2], q[:, 3])
        warp = drng.random(nd_) < 0.3
        Rd[warp] = Rd[warp] @ (np.eye(3) + drng.normal(size=(int(warp.sum()), 3, 3)) * 10.0 ** drng.uniform(-14, -9, (int(warp.sum()), 1, 1)))
        Td = drng.uniform(-1, 1, (nd_, 3)) * scale
        ax = drng.integers(0, 3, nd_)
        sign = drng.choice([-1.0, 1.0], nd_)
        axis_w = Rd[np.arange(nd_), :, ax] * sign[:, None]  # a body axis of operand 1 in the world
        dt1 = P.make_transforms(Rd, Td)
        dt2 = P.make_transforms(Rd, Td + axis_w * 4.0 * scale)
        d1, d2 = pool[drng.integers(0, len(pool), nd_)], pool[drng.integers(0, len(pool), nd_)]
        dt2 = touching(B.orc, d1, dt1, d2, dt2, drng)
        deep = drng.random(nd_) < 0.3  # a third of them overlapping by a visible amount
        dt2["T"][deep] -= axis_w[deep] * (drng.uniform(0.01, 0.2, (int(deep.sum()), 1)) * scale)
        for kind in ("distance", "collide", "collide"):
            req, kw = random_request(drng, kind)
            if kind == "collide" and drng.random() < 0.5:
                req.enable_contact = 0
                kw = dict(kw, enable_contact=0)
            cases.append(("drift", kind, d1, dt1, d2, dt2, req, kw))
    # hulls of more than 32 vertices: reference vs oracle only (the device code takes the exhaustive argmax)
    nb = max(200, n // 4)
    bpool = np.concatenate([hb, hb, hp])
    b1, b2 = bpool[rng.integers(0, len(bpool), nb)], bpool[rng.integers(0, len(bpool), nb)]
    for kind in ("distance", "collide"):
        req, kw = random_request(rng, kind)
        cases.append(("big-hulls", kind, b1, tf1[:nb], b2, tf2[:nb], req, kw))
    # meshes: against shapes (both operand orders) and against each other
    m = max(200, n // (2 if BIG_MESHES[0] else 8))
    mt1, mt2 = adversarial_poses(rng, m, scale, base if base != "far" else "random")
    g1 = hm[rng.integers(0, len(hm), m)]
    g2 = hm[rng.integers(0, len(hm), m)]
    q = pool[rng.integers(0, len(pool), m)]
    _, mdkw = random_request(rng, "distance")
    for k in ("gjk_max_iterations", "epa_max_iterations"):
        mdkw.pop(k, None)
    mreq = P.DistanceRequestPOD(**mdkw)
    _, mckw = random_request(rng, "collide")
    for k in ("gjk_max_iterations", "epa_max_iterations"):
        mckw.pop(k, None)
    mcreq = P.CollisionRequestPOD(**mckw)
    for name, a, b in (("mesh-shape", g1, q), ("shape-mesh", q, g1), ("mesh-mesh", g1, g2)):
        cases.append((name, "distance", a, mt1, b, mt2, mreq, mdkw))
        cases.append((name, "collide", a, mt1, b, mt2, mcreq, mckw))
    if DRIFT[0]:  # the mesh walks under drifted rotations (the BV tests multiply them like any other matrix)
        mrng = np.random.default_rng([seed, 0x51ED270C])
        md = max(100, m // 2)

        def drifted(k):
            qq = mrng.normal(size=(k, 4))
            qq /= np.linalg.norm(qq, axis=1)[:, None]
            dg = 10.0 ** mrng.integers(8, 15, (k, 1))
            qq = np.round(qq * dg) / dg
            return W.quat_to_rot(qq[:, 0], qq[:, 1], qq[:, 2], qq[:, 3])
        dm1 = P.make_transforms(drifted(md), mt1["T"][:md])
        dm2 = P.make_transforms(drifted(md), mt2["T"][:md])
        same = mrng.random(md) < 0.3
        dm2["R"][same] = dm1["R"][same]
        for name, a, b in (("mesh-shape", g1[:md], q[:md]), ("mesh-mesh", g1[:md], g2[:md])):
            cases.append((name, "distance", a, dm1, b, dm2, mreq, dict(mdkw, drift=1)))
            cases.append((name, "collide", a, dm1, b, dm2, mcreq, dict(mckw, drift=1)))
    return B, tag, cases


PLANES = [False]  # --planes: Plane / Halfspace geometries against everything (and each other)
DRIFT = [False]  # --drift: rotations that are orthonormal only to 1e-14 ... 1e-8, shared by coaxial, nearly touching shapes
CONTACTS = [False]  # --contacts: mesh collide cases go through batch_collide_contacts (every contact of a pair)
MAX_EXTRA = 4


def run_case(scene, case):
    name, kind, a, t1, b, t2, req = case[:7]
    kw = dict(nthreads=0) if isinstance(scene, oracle_lib.OracleScene) else {}
    if CONTACTS[0] and kind == "collide" and "mesh" in name:
        out, extra, counts = scene.batch_collide_contacts(a, t1, b, t2, req, MAX_EXTRA, **kw)
        # one structured array per pair: the first record, numContacts and the stored extra contacts
        # (unused slots zeroed so that whole rows compare)
        rec = np.zeros(len(out), dtype=[("first", out.dtype), ("count", "<u4"), ("extra", out.dtype, (MAX_EXTRA,))])
        rec["first"], rec["count"] = out, counts
        for k in range(MAX_EXTRA):
            m = counts > k + 1
            rec["extra"][m, k] = extra[m, k]
        return rec
    return (scene.batch_distance if kind == "distance" else scene.batch_collide)(a, t1, b, t2, req, **kw)


def compare_case(case, ref, got, what):
    name, kind = case[0], case[1]
    if ref.dtype.names and "first" in ref.dtype.names:
        assert np.array_equal(ref["count"], got["count"]), "%s: numContacts differs" % what
        cmp_fields(ref["first"], got["first"], C_MESH, what)
        for k in range(MAX_EXTRA):
            cmp_fields(ref["extra"][:, k], got["extra"][:, k], ("p1", "p2", "normal", "pos", "b1", "b2", "distance"),
                       what + " contacts[%d]" % (k + 1))
        return
    if name in ("shapes", "big-hulls", "planes", "drift"):
        if kind == "distance":
            compare_distance(ref, got, what=what)
        else:
            cmp_collide(ref, got, what)
    elif kind == "distance":
        cmp_fields(ref, got, D_MESH if name == "mesh-mesh" else D_MESH + ("normal",), what)
    else:
        cmp_fields(ref, got, C_MESH, what)


def rows_differing(case, ref, got):
    name, kind = case[0], case[1]
    if ref.dtype.names and "first" in ref.dtype.names:
        bad = ref["count"] != got["count"]
        for k in range(MAX_EXTRA):
            for f in ("p1", "p2", "normal", "pos", "b1", "b2", "distance"):
                x, y = ref["extra"][:, k][f], got["extra"][:, k][f]
                ne = ~((x == y) | (np.isnan(x) & np.isnan(y))) if x.dtype.kind == "f" else x != y
                bad |= ne.reshape(len(ref), -1).any(axis=1)
        return np.union1d(np.nonzero(bad)[0], rows_differing(case, ref["first"], got["first"]))
    if name in ("shapes", "big-hulls", "planes", "drift"):
        fields = ["status", "iterations", "b1", "b2", "p1", "p2", "normal"]
        fields += ["min_distance"] if kind == "distance" else ["distance", "pos", "distance_lower_bound", "num_contacts"]
    elif kind == "distance":
        fields = list(D_MESH if name == "mesh-mesh" else D_MESH + ("normal",))
    else:
        fields = list(C_MESH)
    bad = np.zeros(len(ref), dtype=bool)
    for f in fields:
        x, y = ref[f], got[f]
        if f == "distance":
            x, y = x.copy(), y.copy()
            x[ref["num_contacts"] == 0] = 0
            y[ref["num_contacts"] == 0] = 0
        ne = ~((x == y) | (np.isnan(x) & np.isnan(y))) if x.dtype.kind == "f" else x != y
        bad |= ne.reshape(len(ref), -1).any(axis=1)
    return np.nonzero(bad)[0]


def reference_undefined(B, case, rows):
    """True when, on every row given, the oracle went through a projection of an exactly degenerate simplex:
    the reference answers those from uninitialised memory (Project::ProjectResult, internal/intersect.h:58-70)"""
    import ctypes
    L = oracle_lib.lib()
    L.oracle_undefined_projections.restype = ctypes.c_ulonglong
    for r in rows:
        one = list(case)
        for k in (2, 3, 4, 5):
            one[k] = case[k][r:r + 1].copy()
        if len(case) > 8:  # per-pair cached guesses: point a copy of the request at this row's
            gg, gh = case[8][0][r:r + 1].copy(), case[8][1][r:r + 1].copy()
            one[6] = type(case[6]).from_buffer_copy(case[6])
            one[6].q.cached_gjk_guess = gg.ctypes.data
            one[6].q.cached_support_func_guess = gh.ctypes.data
            one[8] = (gg, gh)
        before = L.oracle_undefined_projections()
        run_case(B.orc, one)
        if L.oracle_undefined_projections() == before:
            return False
    return True


UNDEFINED_ROWS = [0]


def one_round(seed, n, use_ref, use_emu):
    B, tag, cases = build_cases(seed, n, use_ref, use_emu)
    try:
        for case in cases:
            what = "%s %s %s %s" % (case[0], case[1], tag, case[7])
            o = run_case(B.orc, case)
            if B.ref:
                r = run_case(B.ref, case)
                rows = rows_differing(case, r, o)
                if len(rows) and len(rows) <= 8 and reference_undefined(B, case, rows):
                    UNDEFINED_ROWS[0] += len(rows)
                    print("     %s: %d row(s) where the reference reads uninitialised memory" % (what, len(rows)))
                    # the comparison below must hold on every other row
                    keep = np.ones(len(r), dtype=bool)
                    keep[rows] = False
                    compare_case(case, r[keep], o[keep], "ref/oracle " + what)
                else:
                    compare_case(case, r, o, "ref/oracle " + what)
            if B.emu and case[0] != "big-hulls":
                compare_case(case, o, run_case(B.emu, case), "oracle/device code " + what)
    except AssertionError as e:
        print("MISMATCH", e, flush=True)
        return False, tag
    return True, tag


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--minutes", type=float, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--n", type=int, default=4000)
    ap.add_argument("--no-emu", action="store_true")
    ap.add_argument("--keep-going", action="store_true")
    ap.add_argument("--big-meshes", action="store_true")
    ap.add_argument("--contacts", action="store_true", help="mesh collide cases keep every contact (batch_collide_contacts)")
    ap.add_argument("--planes", action="store_true", help="add the Plane / Halfspace family to every round")
    ap.add_argument("--drift", action="store_true",
                    help="add coaxial, nearly touching pairs under rotations that are not quite orthonormal to every round")
    ap.add_argument("--gpu", action="store_true", help="the real kernels (hppfcl_b200.Engine) instead of the host build")
    ap.add_argument("--lanes", type=int, default=1, help="host build: lane groups of this many threads for phase 1")
    a = ap.parse_args()
    use_ref = False
    BIG_MESHES[0] = a.big_meshes
    CONTACTS[0] = a.contacts
    PLANES[0] = a.planes
    DRIFT[0] = a.drift
    oracle_lib.build_ref()
    use_ref = oracle_lib.ref_available()
    t0, seed, bad = time.time(), a.seed, 0
    while time.time() - t0 < a.minutes * 60:
        dev = not a.no_emu
        if dev and a.lanes > 1:
            dev = EmuScene()
            dev.lanes = a.lanes
        if a.gpu:
            import hppfcl_b200 as hf
            dev = hf.Engine(0)
        ok, tag = one_round(seed, a.n, use_ref, dev)
        print("%s %s (ref %s)" % ("ok  " if ok else "FAIL", tag, use_ref), flush=True)
        bad += not ok
        if not ok and not a.keep_going:
            sys.exit(1)
        seed += 1
    print("rounds %d failures %d; rows on which the reference is undefined: %d" % (seed - a.seed, bad, UNDEFINED_ROWS[0]))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
