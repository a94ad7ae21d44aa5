"""ORACLE -- TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/liboracle.so (the CPU restatement of the hpp-fcl hot
path) and of oracle/_ref/libhppfcl_ref.so (the reference's own sources compiled in
place, `make -C oracle ref`).  Imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs ONLY; the product package never
imports this module.  The restatement is pinned against the reference's known-answer
tests (tests/test_oracle_golden.py) and, bit for bit, against the reference build
(tests/test_reference_build.py).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".cpp", ".hpp"))]
    srcs.append(os.path.join(_HERE, "..", "include", "hppfcl_b200.h"))
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(so):
            build()
        L = C.CDLL(so)
        L.oracle_scene_create.restype = C.c_void_p
        L.oracle_scene_destroy.argtypes = [C.c_void_p]
        L.oracle_register_convex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
        L.oracle_register_convex.restype = C.c_int
        L.oracle_register_shapes.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.oracle_register_shapes.restype = C.c_int64
        L.oracle_register_halfspaces.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t]
        L.oracle_register_halfspaces.restype = C.c_int64
        for name in ("oracle_batch_distance", "oracle_batch_collide"):
            f = getattr(L, name)
            f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
            f.restype = C.c_int
        L.oracle_batch_convex_support.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
        L.oracle_batch_convex_support_log.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                                      C.c_void_p]
        L.oracle_max_threads.restype = C.c_int
        L.oracle_register_bvh.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
        L.oracle_register_bvh.restype = C.c_int
        L.oracle_bvh_export.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32]
        L.oracle_bvh_export.restype = C.c_int
        _LIB = L
    return _LIB


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class OracleScene:
    """Mirror of the product's geometry arena for the oracle."""

    def __init__(self, pod):
        self.pod = pod  # the product's _pod module (layouts only)
        self.L = lib()
        self.h = C.c_void_p(self.L.oracle_scene_create())

    def close(self):
        if self.h:
            self.L.oracle_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def register_convex(self, points, tris=None):
        pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        t = None if tris is None else np.ascontiguousarray(tris, dtype=np.uint32).reshape(-1, 3)
        cid = self.L.oracle_register_convex(self.h, _ptr(pts), pts.shape[0], _ptr(t),
                                            0 if t is None else t.shape[0])
        return cid

    def register_bvh(self, vertices, triangles):
        """Builds a BVHModel<OBBRSS> with the reference's builder; returns (bvh id, exported nodes)."""
        v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, dtype=np.uint32).reshape(-1, 3)
        bid = self.L.oracle_register_bvh(self.h, _ptr(v), v.shape[0], _ptr(t), t.shape[0])
        n = self.L.oracle_bvh_export(self.h, bid, None, 0)
        nodes = np.zeros(n, dtype=self.pod.bvh_node_dtype)
        self.L.oracle_bvh_export(self.h, bid, _ptr(nodes), n)
        return bid, nodes

    def register_shapes(self, shapes):
        shapes = np.ascontiguousarray(shapes, dtype=self.pod.shape_dtype)
        first = self.L.oracle_register_shapes(self.h, _ptr(shapes), shapes.shape[0])
        if first < 0:
            raise ValueError("oracle_register_shapes failed")
        return np.arange(first, first + shapes.shape[0], dtype=np.uint32)

    _halfspaces_fn = "oracle_register_halfspaces"

    def register_halfspaces(self, kind, n_d, ssr=None):
        """kind: GEOM_PLANE or GEOM_HALFSPACE; n_d: (count, 4) rows (n.x, n.y, n.z, d); ssr: count radii or None"""
        nd = np.ascontiguousarray(n_d, dtype=np.float64).reshape(-1, 4)
        r = None if ssr is None else np.ascontiguousarray(ssr, dtype=np.float64).reshape(-1)
        assert r is None or r.shape[0] == nd.shape[0]
        first = getattr(self.L, self._halfspaces_fn)(self.h, int(kind), _ptr(nd), None if r is None else _ptr(r), nd.shape[0])
        if first < 0:
            raise ValueError(self._halfspaces_fn + " failed")
        return np.arange(first, first + nd.shape[0], dtype=np.uint32)

    def _run(self, fn, out_dtype, h1, tf1, h2, tf2, req, want_guess, nthreads):
        h1 = np.ascontiguousarray(h1, dtype=np.uint32)
        h2 = np.ascontiguousarray(h2, dtype=np.uint32)
        tf1 = np.ascontiguousarray(tf1, dtype=self.pod.transform_dtype)
        tf2 = np.ascontiguousarray(tf2, dtype=self.pod.transform_dtype)
        n = h1.shape[0]
        out = np.zeros(n, dtype=out_dtype)
        g = None
        gg = gh = None
        if want_guess:
            gg = np.zeros((n, 3), dtype=np.float64)
            gh = np.zeros((n, 2), dtype=np.int32)
            g = self.pod.GuessOut(_ptr(gg), _ptr(gh))
        rc = fn(self.h, n, _ptr(h1), _ptr(tf1), _ptr(h2), _ptr(tf2), C.byref(req), _ptr(out),
                C.byref(g) if g is not None else None, nthreads)
        if rc != 0:
            raise ValueError("oracle error code %d" % rc)
        if want_guess:
            return out, gg, gh
        return out

    def batch_distance(self, h1, tf1, h2, tf2, req=None, want_guess=False, nthreads=1):
        req = req or self.pod.DistanceRequestPOD()
        return self._run(self.L.oracle_batch_distance, self.pod.distance_result_dtype, h1, tf1, h2, tf2,
                         req, want_guess, nthreads)

    def batch_collide(self, h1, tf1, h2, tf2, req=None, want_guess=False, nthreads=1):
        req = req or self.pod.CollisionRequestPOD()
        return self._run(self.L.oracle_batch_collide, self.pod.contact_dtype, h1, tf1, h2, tf2, req,
                         want_guess, nthreads)

    _contacts_fn = "oracle_batch_collide_contacts"

    def batch_collide_contacts(self, h1, tf1, h2, tf2, req=None, max_extra=3, nthreads=1):
        """-> (out, extra[n, max_extra], counts): see hfb_batch_collide_contacts in include/hppfcl_b200.h"""
        req = req or self.pod.CollisionRequestPOD()
        h1 = np.ascontiguousarray(h1, dtype=np.uint32)
        h2 = np.ascontiguousarray(h2, dtype=np.uint32)
        tf1 = np.ascontiguousarray(tf1, dtype=self.pod.transform_dtype)
        tf2 = np.ascontiguousarray(tf2, dtype=self.pod.transform_dtype)
        n = h1.shape[0]
        out = np.zeros(n, dtype=self.pod.contact_dtype)
        extra = np.zeros((n, max(max_extra, 1)), dtype=self.pod.contact_dtype)
        counts = np.zeros(n, dtype=np.uint32)
        fn = getattr(self.L, self._contacts_fn)
        fn.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 6 + [C.c_uint32, C.c_void_p, C.c_void_p, C.c_int]
        rc = fn(self.h, n, _ptr(h1), _ptr(tf1), _ptr(h2), _ptr(tf2), C.byref(req), _ptr(out), max_extra, _ptr(extra),
                _ptr(counts), nthreads)
        if rc != 0:
            raise ValueError("error code %d" % rc)
        return out, extra[:, :max_extra], counts

    def batch_convex_support(self, convex_ids, dirs, log=False):
        ids = np.ascontiguousarray(convex_ids, dtype=np.uint32)
        d = np.ascontiguousarray(dirs, dtype=np.float64).reshape(-1, 3)
        idx = np.zeros(ids.shape[0], dtype=np.int32)
        if log:
            self.L.oracle_batch_convex_support_log(self.h, ids.shape[0], _ptr(ids), _ptr(d), _ptr(idx))
            return idx
        sup = np.zeros((ids.shape[0], 3), dtype=np.float64)
        rc = self.L.oracle_batch_convex_support(self.h, ids.shape[0], _ptr(ids), _ptr(d), _ptr(idx), _ptr(sup))
        if rc != 0:
            raise ValueError("oracle error code %d" % rc)
        return idx, sup

    def gjk_lowlevel(self, h0, tf0, h1, tf1, gjk_max_it=128, gjk_tol=1e-6, variant=0, criterion=0,
                     criterion_type=0, guess=(1, 0, 0), run_epa=False, epa_max_it=64, epa_tol=1e-6,
                     epa_guess=(1, 0, 0)):
        tf0 = np.ascontiguousarray(tf0, dtype=self.pod.transform_dtype).reshape(1)
        tf1 = np.ascontiguousarray(tf1, dtype=self.pod.transform_dtype).reshape(1)
        out = np.zeros(14, dtype=np.float64)
        istat = np.zeros(5, dtype=np.int32)
        g = np.asarray(guess, dtype=np.float64)
        eg = np.asarray(epa_guess, dtype=np.float64)
        f = self.L.oracle_gjk_lowlevel
        f.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_double,
                      C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_uint32, C.c_double, C.c_void_p,
                      C.c_void_p, C.c_void_p]
        f(self.h, int(h0), _ptr(tf0), int(h1), _ptr(tf1), gjk_max_it, gjk_tol, variant, criterion,
          criterion_type, _ptr(g), int(run_epa), epa_max_it, epa_tol, _ptr(eg), _ptr(out), _ptr(istat))
        return dict(w0=out[0:3].copy(), w1=out[3:6].copy(), normal=out[6:9].copy(), ray=out[9:12].copy(),
                    distance=out[12], epa_depth=out[13], gjk_status=int(istat[0]), epa_status=int(istat[1]),
                    gjk_iterations=int(istat[2]), epa_iterations=int(istat[3]), rank=int(istat[4]))

    def project(self, *pts):
        pts = [np.asarray(p, dtype=np.float64) for p in pts]
        param = np.zeros(4)
        sqr = C.c_double()
        enc = C.c_uint()
        fn = {2: self.L.oracle_project_line_origin, 3: self.L.oracle_project_triangle_origin,
              4: self.L.oracle_project_tetrahedra_origin}[len(pts)]
        fn(*[_ptr(p) for p in pts], _ptr(param), C.byref(sqr), C.byref(enc))
        return param, sqr.value, enc.value


# ---------------------------------------------------------------------------------------------------
# The reference itself (oracle/_ref/libhppfcl_ref.so: hpp-fcl's sources compiled in place, see
# oracle/Makefile target `ref` and oracle/ref_driver.cpp).  Same interface as OracleScene.
_REF = None


def ref_available():
    return os.path.exists(os.path.join(_HERE, "_ref", "libhppfcl_ref.so"))


def build_ref():
    """(re)builds oracle/_ref where the reference's sources are present (oracle/Makefile REF); a no-op elsewhere"""
    subprocess.check_call(["make", "-C", _HERE, "-s", "ref"])
    return ref_available()


def ref_lib():
    global _REF
    if _REF is None:
        L = C.CDLL(os.path.join(_HERE, "_ref", "libhppfcl_ref.so"))
        L.ref_scene_create.restype = C.c_void_p
        L.ref_scene_destroy.argtypes = [C.c_void_p]
        L.ref_register_convex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
        L.ref_register_bvh.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
        L.ref_bvh_export.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32]
        L.ref_register_shapes.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.ref_register_shapes.restype = C.c_int64
        L.ref_register_halfspaces.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t]
        L.ref_register_halfspaces.restype = C.c_int64
        for name in ("ref_batch_distance", "ref_batch_collide"):
            f = getattr(L, name)
            f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
            f.restype = C.c_int
        L.ref_max_threads.restype = C.c_int
        _REF = L
    return _REF


class RefScene(OracleScene):
    """The reference's own collide()/distance() behind the interface of OracleScene."""

    def __init__(self, pod):
        self.pod = pod
        self.L = ref_lib()
        self.h = C.c_void_p(self.L.ref_scene_create())

    def close(self):
        if self.h:
            self.L.ref_scene_destroy(self.h)
            self.h = None

    def register_convex(self, points, tris=None):
        if tris is None:
            raise ValueError("the reference needs the hull's triangles (Convex<Triangle>)")
        pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        t = np.ascontiguousarray(tris, dtype=np.uint32).reshape(-1, 3)
        return self.L.ref_register_convex(self.h, _ptr(pts), pts.shape[0], _ptr(t), t.shape[0])

    def register_points(self, points):
        """a bare point set (TriangleP vertices)"""
        pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        t = np.zeros((0, 3), dtype=np.uint32)
        return self.L.ref_register_convex(self.h, _ptr(pts), pts.shape[0], _ptr(t), 0)

    def register_bvh(self, vertices, triangles):
        v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, dtype=np.uint32).reshape(-1, 3)
        bid = self.L.ref_register_bvh(self.h, _ptr(v), v.shape[0], _ptr(t), t.shape[0])
        n = self.L.ref_bvh_export(self.h, bid, None, 0)
        nodes = np.zeros(n, dtype=self.pod.bvh_node_dtype)
        self.L.ref_bvh_export(self.h, bid, _ptr(nodes), n)
        return bid, nodes

    def register_shapes(self, shapes):
        shapes = np.ascontiguousarray(shapes, dtype=self.pod.shape_dtype)
        first = self.L.ref_register_shapes(self.h, _ptr(shapes), shapes.shape[0])
        if first < 0:
            raise ValueError("ref_register_shapes failed")
        return np.arange(first, first + shapes.shape[0], dtype=np.uint32)

    def batch_distance(self, h1, tf1, h2, tf2, req=None, want_guess=False, nthreads=1):
        req = req or self.pod.DistanceRequestPOD()
        return self._run(self.L.ref_batch_distance, self.pod.distance_result_dtype, h1, tf1, h2, tf2,
                         req, want_guess, nthreads)

    def batch_collide(self, h1, tf1, h2, tf2, req=None, want_guess=False, nthreads=1):
        req = req or self.pod.CollisionRequestPOD()
        return self._run(self.L.ref_batch_collide, self.pod.contact_dtype, h1, tf1, h2, tf2, req,
                         want_guess, nthreads)

    def object_aabbs(self, handles, tfs):
        """CollisionObject(geometry, pose).getAABB() of the reference: (n, 6) rows min xyz, max xyz"""
        h = np.ascontiguousarray(handles, dtype=np.uint32)
        tf = np.ascontiguousarray(tfs, dtype=self.pod.transform_dtype)
        out = np.zeros((len(h), 6))
        self.L.ref_object_aabbs.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
        if self.L.ref_object_aabbs(self.h, len(h), _ptr(h), _ptr(tf), _ptr(out)) != 0:
            raise ValueError("ref_object_aabbs failed")
        return out

    def bvh_obb_is_obbrss_half(self, bvh_id):
        """1 when the plain BVHModel<OBB> of model `bvh_id` is the OBB half of its BVHModel<OBBRSS>"""
        self.L.ref_bvh_obb_is_obbrss_half.argtypes = [C.c_void_p, C.c_int]
        return self.L.ref_bvh_obb_is_obbrss_half(self.h, int(bvh_id))

    _contacts_fn = "ref_batch_collide_contacts"
    _halfspaces_fn = "ref_register_halfspaces"
