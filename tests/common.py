"""Shared test helpers: the same geometry registered in the oracle (CPU
restatement of the reference), the CPU emulation of the device code (tests/emu)
and -- on a GPU box -- the CUDA engine; plus the parity comparison."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import hppfcl_b200 as hf  # noqa: E402
from hppfcl_b200 import _pod as P  # noqa: E402
from oracle import oracle_lib  # noqa: E402

EMU_DIR = os.path.join(ROOT, "tests", "emu")
_EMU = None


def emu_lib():
    global _EMU
    if _EMU is None:
        so = os.environ.get("HFB_EMU_SO") or os.path.join(EMU_DIR, "libemu.so")  # another build under test
        src = os.path.join(EMU_DIR, "emu.cpp")
        csrc = os.path.join(ROOT, "hpp-fcl_b200", "csrc")
        deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
        if "HFB_EMU_SO" not in os.environ and (
                not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps)):
            subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off",
                                   "-march=x86-64-v2", "-Wno-unknown-pragmas", "-pthread", "-shared", "-o", so, src])
        L = C.CDLL(so)
        L.emu_create.restype = C.c_void_p
        L.emu_destroy.argtypes = [C.c_void_p]
        L.emu_register_convex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.emu_register_shapes.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.emu_register_shapes.restype = C.c_int64
        L.emu_register_halfspaces.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t]
        L.emu_register_halfspaces.restype = C.c_int64
        for name in ("emu_batch_distance", "emu_batch_collide"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 7
        L.emu_batch_convex_support.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 4
        L.emu_register_bvh.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p,
                                       C.c_uint32]
        L.emu_register_bvh_obb.argtypes = L.emu_register_bvh.argtypes
        L.emu_update_shapes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.emu_update_convex.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
        _EMU = L
    return _EMU


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class EmuScene:
    def __init__(self):
        self.L = emu_lib()
        self.h = C.c_void_p(self.L.emu_create())

    def __del__(self):
        try:
            self.L.emu_destroy(self.h)
        except Exception:
            pass

    def register_convex(self, points):
        pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        return self.L.emu_register_convex(self.h, _ptr(pts), pts.shape[0])

    def register_bvh_obbrss(self, nodes, vertices, triangles):
        nodes = np.ascontiguousarray(nodes, dtype=P.bvh_node_dtype)
        v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, dtype=np.uint32).reshape(-1, 3)
        bid = self.L.emu_register_bvh(self.h, _ptr(nodes), nodes.shape[0], _ptr(v), v.shape[0], _ptr(t), t.shape[0])
        assert bid >= 0
        return bid

    def register_bvh_obb(self, nodes, vertices, triangles):
        nodes = np.ascontiguousarray(nodes, dtype=P.bvh_node_dtype)
        v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, dtype=np.uint32).reshape(-1, 3)
        bid = self.L.emu_register_bvh_obb(self.h, _ptr(nodes), nodes.shape[0], _ptr(v), v.shape[0], _ptr(t), t.shape[0])
        assert bid >= 0
        return bid

    def register_shapes(self, shapes):
        shapes = np.ascontiguousarray(shapes, dtype=P.shape_dtype)
        first = self.L.emu_register_shapes(self.h, _ptr(shapes), shapes.shape[0])
        assert first >= 0
        return np.arange(first, first + shapes.shape[0], dtype=np.uint32)

    def register_halfspaces(self, kind, n_d, ssr=None):
        nd = np.ascontiguousarray(n_d, dtype=np.float64).reshape(-1, 4)
        r = None if ssr is None else np.ascontiguousarray(ssr, dtype=np.float64).reshape(-1)
        first = self.L.emu_register_halfspaces(self.h, int(kind), _ptr(nd), None if r is None else _ptr(r), nd.shape[0])
        assert first >= 0
        return np.arange(first, first + nd.shape[0], dtype=np.uint32)

    def scene_aabbs(self, handles, tfs):
        h = np.ascontiguousarray(handles, dtype=np.uint32)
        tf = np.ascontiguousarray(tfs, dtype=P.transform_dtype)
        out = np.zeros((len(h), 6))
        self.L.emu_scene_aabbs.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
        assert self.L.emu_scene_aabbs(self.h, len(h), _ptr(h), _ptr(tf), _ptr(out)) == 0
        return out

    def commit(self):
        pass

    def update_shapes(self, handles, shapes):
        handles = np.ascontiguousarray(handles, dtype=np.uint32)
        shapes = np.ascontiguousarray(shapes, dtype=P.shape_dtype)
        rc = self.L.emu_update_shapes(self.h, _ptr(handles), _ptr(shapes), C.c_size_t(handles.shape[0]))
        if rc != 0:
            raise ValueError("emu error %d" % rc)

    def update_convex(self, convex_id, points):
        pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        rc = self.L.emu_update_convex(self.h, C.c_uint32(int(convex_id)), _ptr(pts), C.c_uint32(pts.shape[0]))
        if rc != 0:
            raise ValueError("emu error %d" % rc)

    lanes = 1  # > 1: shape pairs run through lane groups of that many threads (tests/emu lanesim)

    def _run(self, fn, dtype, h1, tf1, h2, tf2, req, want_guess):
        h1 = np.ascontiguousarray(h1, dtype=np.uint32)
        h2 = np.ascontiguousarray(h2, dtype=np.uint32)
        tf1 = np.ascontiguousarray(tf1, dtype=P.transform_dtype)
        tf2 = np.ascontiguousarray(tf2, dtype=P.transform_dtype)
        n = h1.shape[0]
        out = np.zeros(n, dtype=dtype)
        g = gg = gh = None
        if want_guess:
            gg = np.zeros((n, 3))
            gh = np.zeros((n, 2), dtype=np.int32)
            g = P.GuessOut(_ptr(gg), _ptr(gh))
        if self.lanes > 1:
            lfn = self.L.emu_batch_distance_lanes if fn is self.L.emu_batch_distance else self.L.emu_batch_collide_lanes
            lfn.restype = C.c_long
            lfn.argtypes = [C.c_void_p, C.c_int, C.c_size_t] + [C.c_void_p] * 7
            rc = lfn(self.h, self.lanes, n, _ptr(h1), _ptr(tf1), _ptr(h2), _ptr(tf2), C.byref(req), _ptr(out),
                     C.byref(g) if g is not None else None)
            if rc == -1:
                raise RuntimeError("a lane of a group never reached a barrier (divergent control flow)")
            if rc > 0:
                raise RuntimeError("the lanes of a group disagreed on %d pairs" % rc)
            if rc == -2:  # meshes in the batch (one lane per query on the device as well) or a special request
                rc = fn(self.h, n, _ptr(h1), _ptr(tf1), _ptr(h2), _ptr(tf2), C.byref(req), _ptr(out),
                        C.byref(g) if g is not None else None)
        else:
            rc = fn(self.h, n, _ptr(h1), _ptr(tf1), _ptr(h2), _ptr(tf2), C.byref(req), _ptr(out),
                    C.byref(g) if g is not None else None)
        if rc != 0:
            raise ValueError("emu error %d" % rc)
        return (out, gg, gh) if want_guess else out

    def batch_distance(self, h1, tf1, h2, tf2, req=None, want_guess=False):
        return self._run(self.L.emu_batch_distance, P.distance_result_dtype, h1, tf1, h2, tf2,
                         req or P.DistanceRequestPOD(), want_guess)

    def batch_collide(self, h1, tf1, h2, tf2, req=None, want_guess=False):
        return self._run(self.L.emu_batch_collide, P.contact_dtype, h1, tf1, h2, tf2,
                         req or P.CollisionRequestPOD(), want_guess)

    def batch_collide_contacts(self, h1, tf1, h2, tf2, req=None, max_extra=3):
        req = req or P.CollisionRequestPOD()
        h1 = np.ascontiguousarray(h1, dtype=np.uint32)
        h2 = np.ascontiguousarray(h2, dtype=np.uint32)
        tf1 = np.ascontiguousarray(tf1, dtype=P.transform_dtype)
        tf2 = np.ascontiguousarray(tf2, dtype=P.transform_dtype)
        n = h1.shape[0]
        out = np.zeros(n, dtype=P.contact_dtype)
        extra = np.zeros((n, max(max_extra, 1)), dtype=P.contact_dtype)
        counts = np.zeros(n, dtype=np.uint32)
        fn = self.L.emu_batch_collide_contacts
        fn.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 6 + [C.c_uint32, C.c_void_p, C.c_void_p]
        rc = fn(self.h, n, _ptr(h1), _ptr(tf1), _ptr(h2), _ptr(tf2), C.byref(req), _ptr(out), max_extra, _ptr(extra),
                _ptr(counts))
        if rc != 0:
            raise ValueError("emu error %d" % rc)
        return out, extra[:, :max_extra], counts

    def batch_convex_support(self, ids, dirs):
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        d = np.ascontiguousarray(dirs, dtype=np.float64).reshape(-1, 3)
        idx = np.zeros(ids.shape[0], dtype=np.int32)
        sup = np.zeros((ids.shape[0], 3))
        rc = self.L.emu_batch_convex_support(self.h, ids.shape[0], _ptr(ids), _ptr(d), _ptr(idx), _ptr(sup))
        assert rc == 0
        return idx, sup


class MultiScene:
    """Registers identical geometry in every backend given."""

    def __init__(self, backends):
        self.b = backends  # dict name -> scene object

    def register_convex(self, points, tris=None):
        ids = set()
        for name, s in self.b.items():
            if name == "oracle":
                ids.add(int(s.register_convex(points, tris)))
            elif name == "ref":  # Convex<Triangle> needs its faces; a TriangleP's vertex set is a bare point set
                ids.add(int(s.register_points(points) if tris is None else s.register_convex(points, tris)))
            else:
                ids.add(int(s.register_convex(points)))
        assert len(ids) == 1
        return ids.pop()

    def register_bvh(self, vertices, triangles):
        """The oracle builds the tree with the reference's builder; the other backends get the exported
        node array through the product ABI (what a binding copies out of BVHModel<OBBRSS>::bvs)."""
        bid, nodes = self.b["oracle"].register_bvh(vertices, triangles)
        for name, s in self.b.items():
            if name == "ref":  # (builds its own tree: the reference's builder, which the oracle's restates)
                assert s.register_bvh(vertices, triangles)[0] == bid
            elif name != "oracle":
                assert s.register_bvh_obbrss(nodes, vertices, triangles) == bid
        return bid, nodes

    def register_bvh_obb(self, vertices, triangles):
        """a plain BVHModel<OBB> of the mesh: in the oracle and the reference build a model serves both kinds (its id
        is shared), the product registers the node array a second time as an OBB model"""
        bid, nodes = self.b["oracle"].register_bvh(vertices, triangles)
        for name, s in self.b.items():
            if name == "ref":
                assert s.register_bvh(vertices, triangles)[0] == bid
            elif name != "oracle":
                assert s.register_bvh_obb(nodes, vertices, triangles) == bid
        return bid, nodes

    def register_shapes(self, shapes):
        hs = [s.register_shapes(shapes) for s in self.b.values()]
        for h in hs[1:]:
            assert np.array_equal(h, hs[0])
        return hs[0]

    def register_halfspaces(self, kind, n_d, ssr=None):
        hs = [s.register_halfspaces(kind, n_d, ssr) for s in self.b.values()]
        for h in hs[1:]:
            assert np.array_equal(h, hs[0])
        return hs[0]

    def commit(self):
        for name, s in self.b.items():
            if hasattr(s, "commit"):
                s.commit()


def make_scenes(gpu=False, emu=True, ref=False):
    """ref=True adds the reference build (oracle/_ref, or its recorded answers where it is not built): the
    known-answer tests then check their literal numbers on records the reference's own code agrees with bit for bit"""
    b = {"oracle": oracle_lib.OracleScene(P)}
    if ref:
        from tests.recorded_reference import reference_scene
        b["ref"] = reference_scene(P)
    if emu:
        b["emu"] = EmuScene()
    if gpu:
        b["gpu"] = hf.Engine(0)
    return MultiScene(b)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def compare_distance(ref, got, rtol=1e-6, exact=True, what=""):
    """north_star bar: status/flags/indices bit-exact; distances, points, normals within
    1e-6 relative.  With exact=True additionally require bitwise-identical doubles
    (oracle and device code execute the same IEEE operation sequence)."""
    assert ref.shape == got.shape
    assert np.array_equal(ref["status"], got["status"]), "%s: status words differ at %s" % (
        what, np.nonzero(ref["status"] != got["status"])[0][:10])
    if exact:
        assert np.array_equal(ref["iterations"], got["iterations"]), "%s: iteration counts differ" % what
    assert np.array_equal(ref["b1"], got["b1"]) and np.array_equal(ref["b2"], got["b2"])
    dname = "min_distance" if "min_distance" in ref.dtype.names else "distance"
    for f in (dname, "p1", "p2", "normal") + (("pos", "distance_lower_bound") if "pos" in ref.dtype.names else ()):
        a, b = ref[f], got[f]
        assert np.array_equal(np.isnan(a), np.isnan(b)), "%s: NaN pattern differs in %s" % (what, f)
        if exact:
            bad = _bits(a) != _bits(b)
            bad &= ~(np.isnan(a) & np.isnan(b))
            bad &= ~((a == 0) & (b == 0))
            assert not bad.any(), "%s: %s not bit-identical at rows %s (max abs diff %g)" % (
                what, f, np.unique(np.nonzero(bad)[0])[:10], np.nanmax(np.abs(a - b)))
        else:
            m = ~np.isnan(a)
            scale = np.maximum(1.0, np.abs(a[m]))
            assert np.all(np.abs(a[m] - b[m]) <= rtol * scale), "%s: %s exceeds rtol" % (what, f)
    if "num_contacts" in ref.dtype.names:
        assert np.array_equal(ref["num_contacts"], got["num_contacts"]), "%s: collide flags differ" % what


def ref_agrees(sc, fn, ro, args, what, fields=None):
    """the reference build returns the same bits (it leaves `distance` of a collide() without a contact unset).
    `fields`: compare only these (mesh queries: the BV / leaf test counters and the path byte of the record are the
    oracle's own, and the reference writes no normal on the mesh-mesh distance path)"""
    if "ref" not in sc.b:
        return
    rr = getattr(sc.b["ref"], fn)(*args)
    if fields is not None:
        for f in fields:
            x, y = rr[f], ro[f]
            ok = (x == y) | (np.isnan(x) & np.isnan(y)) if x.dtype.kind == "f" else x == y
            assert np.all(ok), "%s (reference build): field %s differs at rows %s" % (what, f, np.unique(np.nonzero(~ok)[0])[:8])
        return
    a, b = rr.copy(), ro.copy()
    if "num_contacts" in a.dtype.names:
        nc = a["num_contacts"] == 0
        a["distance"][nc] = 0
        b["distance"][nc] = 0
    compare_distance(a, b, what=what + " (reference build)")


def compare_hill_climb(ref, got):
    """Exhaustive-argmax device code vs the reference's hill-climbing support (hulls > 32
    vertices).  The chosen vertex can differ only on maxima tied to rounding, i.e. at GJK/EPA
    convergence; the solver may then stop one iteration earlier or later.  Bar: status words and
    collide flags bit-exact; distances within 1e-6 (north_star); witness points / normals equal
    to 1e-9 on all but a vanishing fraction of pairs (tolerance-limited early stops), and within
    the solver's own accuracy (1e-3) everywhere."""
    assert np.array_equal(ref["status"], got["status"])
    assert np.array_equal(ref["num_contacts"], got["num_contacts"])
    m = ~np.isnan(ref["p1"][:, 0])
    assert np.array_equal(m, ~np.isnan(got["p1"][:, 0]))
    assert np.all(np.abs(ref["distance"][m] - got["distance"][m]) <= 1e-6 * np.maximum(1, np.abs(ref["distance"][m])))
    for f in ("p1", "p2", "normal"):
        d = np.abs(ref[f][m] - got[f][m]).max(axis=1)
        assert (d > 1e-9).mean() < 1e-3, f
        assert d.max() < 1e-3, f
