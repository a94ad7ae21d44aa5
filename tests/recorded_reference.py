"""The reference build's answers, stored, for machines that cannot build it.

oracle/_ref (hpp-fcl's own sources compiled in place, `make -C oracle ref`) needs the reference's source tree.  Where
it is missing, `reference_scene()` returns a RecordedReference instead: it runs every call on the oracle and accepts
the oracle's answer only if it is the answer the reference build gave to the same inputs, as recorded in
tests/golden/reference_answers.npz.  What a test compares against is then the reference's answer, as before.

A recording keeps, per call, a digest of the inputs (the scene's registrations so far, the method, its arguments and
the data a request points to) and a digest of the reference's output.  Records in which a field of the reference's
output differs from the oracle's (fields it never writes, pairs it does not support, rows it reads from uninitialised
memory) are listed per field in a bit mask, left out of the digest and stored as they are; a replay puts them back.
The `distance` of a contact record without a contact, which the reference leaves unset, is left out by rule and
returned bit-inverted, so that a comparison that reads it fails as it would against the reference.  Floats are
compared as the tests compare them: every NaN is one value and -0 equals +0.  Registrations that return ids are not
stored: their results enter the digest of every later call.

Recording (needs oracle/_ref): HFB_RECORD_REFERENCE=tests/golden/reference_answers.npz python -m pytest tests ...
adds the answers of every reference call the run makes to that file.
"""
import atexit
import ctypes as C
import hashlib
import os

import numpy as np

from oracle import oracle_lib

STORE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_answers.npz")
_REGISTRATIONS = ("register_shapes", "register_halfspaces", "register_convex", "register_points", "register_bvh")


def reference_scene(pod):
    """the reference build where oracle/_ref exists (recording its answers when HFB_RECORD_REFERENCE names a file),
    else its recorded answers"""
    if oracle_lib.ref_available():
        if os.environ.get("HFB_RECORD_REFERENCE"):
            return RecordedReference(pod, oracle_lib.RefScene(pod))
        return oracle_lib.RefScene(pod)
    return RecordedReference(pod)


class _Store:
    """input digest -> (output digest, {field number: (packed mask of records, empty: by rule; the reference's bytes
    of the field in those records)}, int value or None)"""

    def __init__(self):
        self.path = os.environ.get("HFB_RECORD_REFERENCE") or STORE
        self.recording = bool(os.environ.get("HFB_RECORD_REFERENCE"))
        self.entries = {}
        if os.path.exists(self.path):
            z = np.load(self.path)
            keys, digests = z["keys"], z["digests"]
            values = dict(zip(z["value_entry"].tolist(), z["value"].tolist()))
            masks = {}
            mo, vo = z["mask_offsets"], z["mask_value_offsets"]
            for k, (e, c) in enumerate(zip(z["mask_entry"], z["mask_field"])):
                masks.setdefault(int(e), {})[int(c)] = (z["mask_bits"][mo[k]:mo[k + 1]],
                                                        z["mask_values"][vo[k]:vo[k + 1]].tobytes())
            for i in range(len(keys)):
                self.entries[keys[i].tobytes()] = (digests[i].tobytes(), masks.get(i, {}), values.get(i))
        if self.recording:
            atexit.register(self.save)

    def save(self):
        keys = sorted(self.entries)
        me, mc, offs, bits, voffs, vals, ve, vv = [], [], [0], [], [0], [], [], []
        for i, k in enumerate(keys):
            _, masks, value = self.entries[k]
            for c, (m, v) in sorted(masks.items()):
                me.append(i)
                mc.append(c)
                bits.append(m)
                offs.append(offs[-1] + len(m))
                vals.append(np.frombuffer(v, np.uint8))
                voffs.append(voffs[-1] + len(v))
            if value is not None:
                ve.append(i)
                vv.append(value)
        np.savez_compressed(
            self.path, keys=np.array([np.frombuffer(k, np.uint8) for k in keys], dtype=np.uint8).reshape(-1, 8),
            digests=np.array([np.frombuffer(self.entries[k][0], np.uint8) for k in keys], dtype=np.uint8).reshape(-1, 8),
            value_entry=np.array(ve, dtype=np.uint32), value=np.array(vv, dtype=np.int64),
            mask_entry=np.array(me, dtype=np.uint32), mask_field=np.array(mc, dtype=np.uint8),
            mask_offsets=np.array(offs, dtype=np.uint64), mask_value_offsets=np.array(voffs, dtype=np.uint64),
            mask_bits=np.concatenate(bits) if bits else np.zeros(0, dtype=np.uint8),
            mask_values=np.concatenate(vals) if vals else np.zeros(0, dtype=np.uint8))


_STORE = None


def _store():
    global _STORE
    if _STORE is None:
        _STORE = _Store()
    return _STORE


def _feed(h, x, rows):
    """the inputs of a call, as bytes: arrays by dtype, shape and contents; a request by its fields, with the
    cached guesses of its `rows` pairs that it points to in place of the pointers"""
    if isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        h.update(b"A" + str(a.dtype.descr).encode() + str(a.shape).encode())
        h.update(a.tobytes())
    elif isinstance(x, C.Structure):
        r = type(x).from_buffer_copy(x)
        q = getattr(r, "q", None)
        guess = None
        if q is not None and q.cached_gjk_guess:
            guess = (q.cached_gjk_guess, q.cached_support_func_guess)
            q.cached_gjk_guess = q.cached_support_func_guess = None
        h.update(b"S" + type(x).__name__.encode() + bytes(r))
        if guess is not None:
            h.update(b"G")
            h.update(C.string_at(guess[0], 24 * rows))
            h.update(C.string_at(guess[1], 8 * rows))
    elif isinstance(x, (list, tuple)):
        h.update(b"L%d" % len(x))
        for y in x:
            _feed(h, y, rows)
    else:
        h.update(b"V" + repr(x).encode())


def _parts(out):
    """an output (an id, an array or a tuple of them) as a list of arrays, copied"""
    return [np.array([p], dtype=np.int64) if isinstance(p, (int, np.integer)) else np.array(p, copy=True)
            for p in (out if isinstance(out, tuple) else (out,))]


def _fields(parts):
    """every field of every array as (view, record shape, rule): a plain array has one record per row; `rule` marks
    the records in which the reference leaves the field unset (the distance of a contact without a contact)"""
    out = []
    for a in parts:
        if not a.dtype.names:
            out.append((a, a.shape[:1], None))
            continue
        rule = (a["num_contacts"] == 0).reshape(-1) if "num_contacts" in a.dtype.names else None
        out += [(a[f], a.shape, rule if f == "distance" else None) for f in a.dtype.names if not f.startswith("_")]
    return out


def _cells(view, shape):
    """one row per record, floats with NaN made one value and -0 made +0"""
    c = np.ascontiguousarray(view).reshape(int(np.prod(shape)), -1).copy()
    if c.dtype.kind == "f":
        c[np.isnan(c)] = np.nan
        c[c == 0] = 0.0
    return c


def _masked(fields, masks):
    """field number -> boolean mask of its records"""
    out = {}
    for c, (m, _) in masks.items():
        view, shape, rule = fields[c]
        out[c] = rule if len(m) == 0 else np.unpackbits(m, count=int(np.prod(shape))).astype(bool)
    return out


def _digest(fields, masked):
    h = hashlib.blake2b(digest_size=8)
    for c, (view, shape, _) in enumerate(fields):
        a = _cells(view, shape)
        if c in masked:
            a[masked[c]] = 0
        h.update(a.tobytes())
    return h.digest()


class RecordedReference(oracle_lib.OracleScene):
    """oracle_lib.RefScene's interface over the oracle, checked call by call against the reference's recorded
    answers (or, given the reference build as `ref`, recording them)."""

    def __init__(self, pod, ref=None):
        self.pod = pod
        self.orc = oracle_lib.OracleScene(pod)
        self.ref = ref
        self.history = b""
        self.calls = []  # registrations, replayed into a host build of the device code for object_aabbs
        self._emu = None

    def close(self):
        pass

    def _key(self, method, args):
        h = hashlib.blake2b(self.history, digest_size=8)
        h.update(method.encode())
        _feed(h, list(args), len(args[0]) if args and isinstance(args[0], (np.ndarray, list)) else 0)
        return h.digest()

    def _oracle(self, method, args):
        if method == "register_points":
            return self.orc.register_convex(args[0])
        if method == "object_aabbs":
            return self._emu_scene().scene_aabbs(*args)
        if method == "bvh_obb_is_obbrss_half":
            return None
        if method.startswith("batch_"):
            return getattr(self.orc, method)(*args, nthreads=0)
        return getattr(self.orc, method)(*args)

    def _emu_scene(self):
        if self._emu is None:
            from tests.common import EmuScene
            self._emu = EmuScene()
            for method, args, out in self.calls:
                if method in ("register_convex", "register_points"):
                    self._emu.register_convex(args[0])
                elif method == "register_bvh":
                    self._emu.register_bvh_obbrss(out[1], *args)
                else:
                    getattr(self._emu, method)(*args)
        return self._emu

    def _call(self, method, *args):
        key = self._key(method, args)
        mine = self._oracle(method, args)
        if method in _REGISTRATIONS and method != "register_bvh":
            if self.ref is not None:
                theirs = getattr(self.ref, method)(*args)
                if _digest(_fields(_parts(theirs)), {}) != _digest(_fields(_parts(mine)), {}):
                    raise AssertionError("%s: the oracle's ids are not the reference build's" % method)
            self.history = hashlib.blake2b(key + _digest(_fields(_parts(mine)), {}), digest_size=8).digest()
            self.calls.append((method, args, mine))
            self._emu = None
            return mine
        st = _store()
        if self.ref is not None:
            theirs = getattr(self.ref, method)(*args, **({"nthreads": 0} if method.startswith("batch_") else {}))
            tf = _fields(_parts(theirs))
            masks = {}
            if mine is not None:
                for c, ((a, sa, rule), (b, sb, _)) in enumerate(zip(tf, _fields(_parts(mine)))):
                    x, y = _cells(a, sa), _cells(b, sb)
                    if x.shape != y.shape:
                        raise AssertionError("%s: the oracle's answer has another shape than the reference's" % method)
                    ne = ((x != y) & ~(np.isnan(x) & np.isnan(y)) if x.dtype.kind == "f" else x != y).any(axis=1)
                    if rule is not None and ne.any() and not (ne & ~rule).any():
                        masks[c] = (np.zeros(0, np.uint8), b"")
                    elif ne.any():
                        masks[c] = (np.packbits(ne), np.ascontiguousarray(a[ne.reshape(sa)]).tobytes())
            st.entries[key] = (_digest(tf, _masked(tf, masks)), masks,
                               int(theirs) if isinstance(theirs, (int, np.integer)) else None)
            out = theirs
        else:
            if key not in st.entries:
                raise AssertionError(
                    "%s: no recorded answer of the reference build for these inputs (tests/golden/reference_answers.npz "
                    "holds the calls the tests made when it was recorded; see tests/recorded_reference.py)" % method)
            digest, masks, value = st.entries[key]
            if mine is None:
                out = value
            else:
                parts = _parts(mine)
                fields = _fields(parts)
                masked = _masked(fields, masks)
                if _digest(fields, masked) != digest:
                    raise AssertionError("%s: the oracle's answer is not the reference build's recorded answer to the "
                                         "same inputs" % method)
                for c, m in masked.items():
                    view, shape, _ = fields[c]
                    sel = m.reshape(shape)
                    if len(masks[c][0]):  # the reference's own values
                        view[sel] = np.frombuffer(masks[c][1], view.dtype).reshape((-1,) + view.shape[len(shape):])
                    else:
                        bits = view.view(np.uint64 if view.dtype.itemsize == 8 else np.uint32)
                        bits[sel] = ~bits[sel]
                out = tuple(p if isinstance(p, (int, np.integer)) else q for p, q in zip(mine, parts)) \
                    if isinstance(mine, tuple) else parts[0]
        if method == "register_bvh":
            self.history = key
            self.calls.append((method, args, out))
            self._emu = None
        return out

    def register_shapes(self, shapes):
        return self._call("register_shapes", shapes)

    def register_halfspaces(self, kind, n_d, ssr=None):
        return self._call("register_halfspaces", kind, n_d, ssr)

    def register_convex(self, points, tris=None):
        if tris is None:
            raise ValueError("the reference needs the hull's triangles (Convex<Triangle>)")
        return self._call("register_convex", points, tris)

    def register_points(self, points):
        return self._call("register_points", points)

    def register_bvh(self, vertices, triangles):
        return self._call("register_bvh", vertices, triangles)

    def batch_distance(self, h1, tf1, h2, tf2, req=None, want_guess=False, nthreads=0):
        return self._call("batch_distance", h1, tf1, h2, tf2, req or self.pod.DistanceRequestPOD(), want_guess)

    def batch_collide(self, h1, tf1, h2, tf2, req=None, want_guess=False, nthreads=0):
        return self._call("batch_collide", h1, tf1, h2, tf2, req or self.pod.CollisionRequestPOD(), want_guess)

    def batch_collide_contacts(self, h1, tf1, h2, tf2, req=None, max_extra=3, nthreads=0):
        return self._call("batch_collide_contacts", h1, tf1, h2, tf2, req or self.pod.CollisionRequestPOD(), max_extra)

    def object_aabbs(self, handles, tfs):
        return self._call("object_aabbs", handles, tfs)

    def bvh_obb_is_obbrss_half(self, bvh_id):
        return self._call("bvh_obb_is_obbrss_half", bvh_id)
