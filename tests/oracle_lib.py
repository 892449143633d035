"""ctypes wrappers for the two CPU checkers (TEST INFRASTRUCTURE ONLY).

* ``RefMap``    -> oracle/_ref/libufo_ref.so   (the unmodified reference, see
                  oracle/ref_harness.cpp) where it has been built; elsewhere the
                  restatement below, every answer checked against the digest of
                  the reference's answer to the same question after the same
                  history (tests/golden/reference/answers.npz).  Regenerate that
                  ledger with the reference built: delete it, then run the whole
                  suite with UFO_REFERENCE_RECORD=<repo>/tests/golden/reference/answers.npz.
* ``OracleMap`` -> oracle/libufo_oracle.so     (plain-C restatement, oracle/ufo_oracle.c)

Both expose the same methods; state is compared as a *value field*
(``value_field()``: every depth-0 voxel with a non-default payload), never as
tree shape (SURVEY.md Appendix A.7).
"""
import atexit
import ctypes as C
import functools
import hashlib
import os
import subprocess
import threading

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libufo_ref.so")
ORACLE_SO = os.path.join(ORACLE_DIR, "libufo_oracle.so")
LEDGER = os.path.join(ROOT, "tests", "golden", "reference", "answers.npz")

DEFAULT_MODEL = dict(occupied_thres=0.5, free_thres=0.5, prob_hit=0.7, prob_miss=0.4,
                     clamping_thres_min=0.1192, clamping_thres_max=0.971)


def build_oracle(force=False):
    """Compile oracle/libufo_oracle.so (and oracle/_ref when /root/reference exists)."""
    if force or not os.path.exists(ORACLE_SO) or (
            os.path.getmtime(ORACLE_SO) < os.path.getmtime(os.path.join(ORACLE_DIR, "ufo_oracle.c"))):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "libufo_oracle.so"],
                              stdout=subprocess.DEVNULL)
    if os.path.isdir("/root/reference/ufomap/include") and (
            force or not os.path.exists(REF_SO) or
            os.path.getmtime(REF_SO) < os.path.getmtime(os.path.join(ORACLE_DIR, "ref_harness.cpp"))):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "_ref/libufo_ref.so"],
                              stdout=subprocess.DEVNULL)


def have_ref():
    return os.path.exists(REF_SO)


_libs = {}


def _load(path, prefix):
    key = (path, prefix)
    if key in _libs:
        return _libs[key]
    lib = C.CDLL(path)
    vp, sz, dbl, u32, i32, u64 = C.c_void_p, C.c_size_t, C.c_double, C.c_uint, C.c_int, C.c_uint64

    def sig(name, res, args):
        f = getattr(lib, prefix + name)
        f.restype = res
        f.argtypes = args
        return f

    api = dict(
        create=sig("create", vp, [dbl, u32, i32, dbl, dbl, dbl, dbl, dbl, dbl, i32]),
        destroy=sig("destroy", None, [vp]),
        insert=sig("insert", dbl, [vp, vp, vp, vp, sz, dbl, u32, i32, u32, i32, i32]),
        walk=sig("walk", sz, [vp, i32]),
        walk_fetch=sig("walk_fetch", None, [vp, vp, vp, vp, vp, vp]),
        node=sig("node", i32, [vp, u64, u32, vp, vp, vp, vp]),
        compute_ray=sig("compute_ray", sz, [vp, vp, vp, dbl, u32, vp, sz]),
        free_set=sig("free_set", sz, [vp, vp, vp, sz, u32, i32, u32, vp, sz]),
        to_key=sig("to_key", None, [vp, vp, u32, vp]),
        to_code=sig("to_code", u64, [vp, vp, u32]),
        key_to_code=sig("key_to_code", u64, [vp, u32]),
        code_to_key=sig("code_to_key", None, [u64, u32, vp]),
        key_to_coord=sig("key_to_coord", None, [vp, vp, u32, vp]),
        move_line_inside=sig("move_line_inside", i32, [vp, vp, vp]),
        change_bbox=sig("change_bbox", None, [vp, vp, vp]),
        reset_change_bbox=sig("reset_change_bbox", None, [vp]),
        sensor_model=sig("sensor_model", None, [vp, vp]),
        memory_usage=sig("memory_usage", sz, [vp]),
        set_value_volume=sig("set_value_volume", None, [vp, vp, dbl, u32]),
        read_data=sig("read_data", i32, [vp, vp, vp, sz]),
        write=sig("write", sz, [vp, vp, sz]),
        write_data=sig("write_data", sz, [vp, vp, u32, vp, sz]),
        transform=sig("transform", None, [vp, vp, sz, vp]),
        pose_from_rpy=sig("pose_from_rpy", None, [dbl, dbl, dbl, dbl, dbl, dbl, vp]),
    )
    if prefix == "ufo_ref_":
        api["read"] = sig("read", i32, [vp, vp, sz])
        api["write_region"] = sig("write_region", sz, [vp, vp, u32, vp, sz])
        api["clear"] = sig("clear", None, [vp, dbl, u32])
        api["field"] = sig("field", sz, [vp, vp, vp, vp, sz])
        api["node_batch"] = sig("node_batch", None, [vp, vp, vp, sz, vp, vp, vp, vp])
        api["leaves"] = sig("leaves", sz, [vp, i32, i32, i32, vp, u32, vp, vp, vp, sz])
        api["write_compressed"] = sig("write_compressed", sz, [vp, u32, i32, i32, vp, sz])
        api["enable_changes"] = sig("enable_changes", None, [vp, i32])
        api["reset_changes"] = sig("reset_changes", None, [vp])
        api["changes"] = sig("changes", sz, [vp, vp, vp, sz])
    if prefix == "ufo_oracle_":
        api["last_counters"] = sig("last_counters", None, [vp, vp])
        api["cast_ray"] = sig("cast_ray", i32, [vp, vp, vp, i32, dbl, u32, vp])
        api["canonicalize"] = sig("canonicalize", None, [vp])
    _libs[key] = api
    return api


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class _CpuMap:
    _path = None
    _prefix = None

    def __init__(self, resolution, depth_levels=16, automatic_pruning=True, color=False, **model):
        self.api = _load(self._path, self._prefix)
        mdl = dict(DEFAULT_MODEL)
        mdl.update(model)
        self.color = bool(color)
        self.resolution = resolution
        self.depth_levels = depth_levels
        self.h = self.api["create"](resolution, depth_levels, int(automatic_pruning),
                                    mdl["occupied_thres"], mdl["free_thres"], mdl["prob_hit"],
                                    mdl["prob_miss"], mdl["clamping_thres_min"],
                                    mdl["clamping_thres_max"], int(color))
        if not self.h:
            raise ValueError("depth_levels has to be [2, 21]")

    def close(self):
        if self.h:
            self.api["destroy"](self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- integration ------------------------------------------------------
    def insert(self, origin, xyz, rgb=None, max_range=-1.0, depth=0, simple=False,
               early_stopping=0, discrete=False):
        o = _f64(origin)
        p = _f64(xyz).reshape(-1, 3)
        c = None
        if rgb is not None:
            c = np.ascontiguousarray(rgb, dtype=np.uint8).reshape(-1, 3)
            assert len(c) == len(p)
        secs = self.api["insert"](self.h, o.ctypes.data, p.ctypes.data,
                                  c.ctypes.data if c is not None else None, len(p),
                                  float(max_range), int(depth), int(simple), int(early_stopping),
                                  int(discrete), 0)
        if secs < 0:
            raise RuntimeError("entry point not instantiable in the reference")
        return secs

    # -- state ------------------------------------------------------------
    def walk(self, leaves=True):
        n = self.api["walk"](self.h, int(leaves))
        codes = np.empty(n, np.uint64)
        depths = np.empty(n, np.uint32)
        occ = np.empty(n, np.float32)
        rgb = np.empty((n, 3), np.uint8)
        flags = np.empty(n, np.uint8)
        self.api["walk_fetch"](self.h, codes.ctypes.data, depths.ctypes.data, occ.ctypes.data,
                               rgb.ctypes.data, flags.ctypes.data)
        return codes, depths, occ, rgb, flags

    def value_field(self):
        """(codes u64 sorted, occ f32, rgb u8[n,3]) of all depth-0 voxels whose payload is
        not the default (0.0, black); collapsed leaves are expanded."""
        codes, depths, occ, rgb, _ = self.walk(True)
        return expand_value_field(codes, depths, occ, rgb)

    def inner_nodes(self):
        """dict-like arrays of nodes that have children: (codes, depths, occ, rgb, flags)."""
        return self.walk(False)

    def node(self, code, depth):
        occ = C.c_float()
        rgb = (C.c_uint8 * 3)()
        flags = C.c_uint8()
        fd = C.c_uint()
        exact = self.api["node"](self.h, int(code), int(depth), C.byref(occ), rgb, C.byref(flags),
                                 C.byref(fd))
        return bool(exact), np.float32(occ.value), tuple(rgb), int(flags.value), int(fd.value)

    # -- geometry -----------------------------------------------------------
    def compute_ray(self, origin, end, max_range=-1.0, depth=0):
        o, e = _f64(origin), _f64(end)
        n = self.api["compute_ray"](self.h, o.ctypes.data, e.ctypes.data, float(max_range),
                                    int(depth), None, 0)
        out = np.empty(n, np.uint64)
        if n:
            self.api["compute_ray"](self.h, o.ctypes.data, e.ctypes.data, float(max_range),
                                    int(depth), out.ctypes.data, n)
        return out

    def free_set(self, origin, ends, depth=0, simple=False, early_stopping=0):
        o, e = _f64(origin), _f64(ends).reshape(-1, 3)
        cap = 1 << 16
        while True:
            out = np.empty(cap, np.uint64)
            n = self.api["free_set"](self.h, o.ctypes.data, e.ctypes.data, len(e), int(depth),
                                     int(simple), int(early_stopping), out.ctypes.data, cap)
            if n <= cap:
                return out[:n].copy()
            cap = int(n)

    def to_key(self, xyz, depth=0):
        p = _f64(xyz)
        k = np.empty(3, np.uint32)
        self.api["to_key"](self.h, p.ctypes.data, int(depth), k.ctypes.data)
        return k

    def to_code(self, xyz, depth=0):
        p = _f64(xyz)
        return int(self.api["to_code"](self.h, p.ctypes.data, int(depth)))

    def key_to_code(self, key, depth=0):
        k = np.ascontiguousarray(key, dtype=np.uint32)
        return int(self.api["key_to_code"](k.ctypes.data, int(depth)))

    def code_to_key(self, code, depth=0):
        k = np.empty(3, np.uint32)
        self.api["code_to_key"](int(code), int(depth), k.ctypes.data)
        return k

    def key_to_coord(self, key, depth=0):
        k = np.ascontiguousarray(key, dtype=np.uint32)
        p = np.empty(3, np.float64)
        self.api["key_to_coord"](self.h, k.ctypes.data, int(depth), p.ctypes.data)
        return p

    def move_line_inside(self, a, b):
        a, b = _f64(a).copy(), _f64(b).copy()
        ok = self.api["move_line_inside"](self.h, a.ctypes.data, b.ctypes.data)
        return bool(ok), a, b

    def change_bbox(self):
        mn, mx = np.empty(3), np.empty(3)
        self.api["change_bbox"](self.h, mn.ctypes.data, mx.ctypes.data)
        return mn, mx

    def reset_change_bbox(self):
        self.api["reset_change_bbox"](self.h)

    def sensor_model(self):
        out = np.empty(6)
        self.api["sensor_model"](self.h, out.ctypes.data)
        return out

    def memory_usage(self):
        return int(self.api["memory_usage"](self.h))

    def read_data(self, data, box=None):
        """Octree::readData(stream, AABB(min, max) or none): merge a node stream into the map."""
        b = None if box is None else np.ascontiguousarray(np.concatenate([box[0], box[1]]), np.float64)
        buf = np.frombuffer(data, np.uint8)
        return bool(self.api["read_data"](self.h, None if b is None else b.ctypes.data,
                                          buf.ctypes.data if len(buf) else None, len(buf)))

    def set_value_volume(self, box, occupancy, min_depth=0):
        """setValueVolume(AABB(min, max), occupancy probability, min_depth)."""
        b = np.ascontiguousarray(np.concatenate([box[0], box[1]]), np.float64)
        self.api["set_value_volume"](self.h, b.ctypes.data, float(occupancy), int(min_depth))

    def write_data(self, box=None, min_depth=0):
        """Octree::writeData(stream, AABB(min, max) or the whole map, False, min_depth): node stream."""
        b = None if box is None else np.ascontiguousarray(np.concatenate([box[0], box[1]]), np.float64)
        bp = None if b is None else b.ctypes.data
        n = self.api["write_data"](self.h, bp, int(min_depth), None, 0)
        buf = np.empty(max(n, 1), np.uint8)
        assert self.api["write_data"](self.h, bp, int(min_depth), buf.ctypes.data, n) == n
        return buf[:n].tobytes()

    def write(self):
        """Octree::write(ostream, compress=False): the complete file image as bytes."""
        n = self.api["write"](self.h, None, 0)
        buf = np.empty(n, np.uint8)
        assert self.api["write"](self.h, buf.ctypes.data, n) == n
        return buf.tobytes()


def _feed(h, value):
    """Canonical encoding of a (nested) call argument or answer into a hash."""
    if isinstance(value, (tuple, list)):
        h.update(b"(%d" % len(value))
        for v in value:
            _feed(h, v)
        h.update(b")")
    elif isinstance(value, dict):
        _feed(h, sorted(value.items()))
    elif isinstance(value, (bytes, bytearray)):
        h.update(b"B%d:" % len(value))
        h.update(value)
    elif value is None or isinstance(value, str):
        h.update(repr(value).encode())
    else:
        a = np.ascontiguousarray(value)
        h.update(("A%s%s:" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())


def _digest(*values):
    """64-bit SHA-256 prefix of the canonical encoding of `values`."""
    h = hashlib.sha256()
    _feed(h, values)
    return int.from_bytes(h.digest()[:8], "little")


class _Answers:
    """The reference's answers to questions asked of a map after a given history.

    tests/golden/reference/answers.npz holds ``answers``: the sorted 64-bit digests of every
    (construction, history of state changes, question, answer) the reference was seen to give.
    With UFO_REFERENCE_RECORD=<path> every answer the compiled reference gives is added to the
    ledger at <path> when the process exits."""

    def __init__(self):
        self._ledger = None
        self._new = set()
        self._lock = threading.Lock()

    def ledger(self):
        if self._ledger is None:
            self._ledger = _read_ledger(LEDGER)
        return self._ledger

    def record(self, entry):
        with self._lock:
            if not self._new:
                atexit.register(self._flush)
            self._new.add(entry)

    def _flush(self):
        path = os.environ["UFO_REFERENCE_RECORD"]
        answers = np.union1d(_read_ledger(path), np.array(sorted(self._new), np.uint64))
        np.savez_compressed(path, answers=answers)


def _read_ledger(path):
    if not os.path.exists(path):
        return np.empty(0, np.uint64)
    with np.load(path) as z:
        return z["answers"]


_ANSWERS = _Answers()


def _ask(real, state, question, args, compute):
    """The reference's answer to `question(args)` on the map whose history hashes to `state`.

    `compute` runs on the compiled reference when `real` (and its answer is recorded when
    UFO_REFERENCE_RECORD is set), otherwise on the C restatement, whose answer must then be
    the one the reference gave to the same question."""
    answer = compute()
    entry = _digest(_digest(state, question, args), _digest(answer))
    if real:
        if os.environ.get("UFO_REFERENCE_RECORD"):
            _ANSWERS.record(entry)
        return answer
    answers = _ANSWERS.ledger()
    i = np.searchsorted(answers, np.uint64(entry))
    assert i < len(answers) and answers[i] == entry, (
        "the C restatement's answer to %s is not one the reference gave on this history" % question)
    return answer


def ref_pose_from_rpy(*xyzrpy):
    """The reference's Pose6(x, y, z, roll, pitch, yaw) as (x, y, z, qw, qx, qy, qz)."""
    def compute():
        out = np.empty(7)
        _load(REF_SO if have_ref() else ORACLE_SO,
              "ufo_ref_" if have_ref() else "ufo_oracle_")["pose_from_rpy"](*xyzrpy, out.ctypes.data)
        return out
    return _ask(have_ref(), b"", "pose_from_rpy", [float(v) for v in xyzrpy], compute)


def ref_transform(pose, pts):
    """The reference's PointCloud::transform of float64 points by a pose of ref_pose_from_rpy."""
    pose, pts = _f64(pose), _f64(pts)

    def compute():
        out = np.empty_like(pts)
        _load(REF_SO if have_ref() else ORACLE_SO,
              "ufo_ref_" if have_ref() else "ufo_oracle_")["transform"](pose.ctypes.data, pts.ctypes.data,
                                                                         len(pts), out.ctypes.data)
        return out
    return _ask(have_ref(), b"", "transform", [pose, pts], compute)


def _asked(stand_in=None):
    """Route a RefMap query through _ask (see there).  `stand_in` names the method that answers
    it without the reference where the restatement has no entry point of that name."""
    def wrap(fn):
        @functools.wraps(fn)
        def method(self, *args, **kw):
            compute = fn if self._real or stand_in is None else getattr(RefMap, stand_in)
            return _ask(self._real, self._state, fn.__name__, [args, kw], lambda: compute(self, *args, **kw))
        return method
    return wrap


def _changes_state(fn):
    """A RefMap call that changes the map: folded into the history the answers are keyed by."""
    @functools.wraps(fn)
    def method(self, *args, **kw):
        self._state = _digest(self._state, fn.__name__, args, kw)
        return fn(self, *args, **kw)
    return method


class RefMap(_CpuMap):
    """The unmodified reference (oracle/_ref/libufo_ref.so).  Where it has not been built, the C
    restatement stands in for it and every answer is checked against the reference's recorded
    answer to the same question after the same history (tests/golden/reference/answers.npz)."""
    _path = REF_SO
    _prefix = "ufo_ref_"

    def __init__(self, resolution, depth_levels=16, automatic_pruning=True, color=False, **model):
        self._real = have_ref()
        self._tracking, self._changed = False, []   # change detection of the stand-in
        if not self._real:
            self._path, self._prefix = ORACLE_SO, "ufo_oracle_"
        self._kw = dict(automatic_pruning=automatic_pruning, color=color, **model)
        self._state = _digest("RefMap", float(resolution), int(depth_levels), self._kw)
        super().__init__(resolution, depth_levels, **self._kw)

    set_value_volume = _changes_state(_CpuMap.set_value_volume)
    read_data = _changes_state(_asked()(_CpuMap.read_data))
    walk = _asked()(_CpuMap.walk)
    node = _asked()(_CpuMap.node)
    compute_ray = _asked()(_CpuMap.compute_ray)
    to_key = _asked()(_CpuMap.to_key)
    to_code = _asked()(_CpuMap.to_code)
    key_to_code = _asked()(_CpuMap.key_to_code)
    code_to_key = _asked()(_CpuMap.code_to_key)
    key_to_coord = _asked()(_CpuMap.key_to_coord)
    move_line_inside = _asked()(_CpuMap.move_line_inside)
    change_bbox = _asked()(_CpuMap.change_bbox)
    sensor_model = _asked()(_CpuMap.sensor_model)
    write_data = _asked()(_CpuMap.write_data)
    write = _asked()(_CpuMap.write)

    @_asked()
    def free_set(self, origin, ends, depth=0, simple=False, early_stopping=0):
        """The free set, sorted (the reference and the restatement list it in different orders)."""
        return np.sort(_CpuMap.free_set(self, origin, ends, depth, simple, early_stopping))

    @_asked("_oracle_write_region")
    def write_region(self, box=None, min_depth=0):
        """Octree::write(stream, AABB(min, max) or whole map, False, min_depth): file image."""
        b = None if box is None else np.ascontiguousarray(np.concatenate([box[0], box[1]]), np.float64)
        bp = None if b is None else b.ctypes.data
        n = self.api["write_region"](self.h, bp, int(min_depth), None, 0)
        buf = np.empty(n, np.uint8)
        assert self.api["write_region"](self.h, bp, int(min_depth), buf.ctypes.data, n) == n
        return buf.tobytes()

    def _oracle_header(self, compressed, size):
        image = _CpuMap.write(self)
        return image[:image.index(b"compressed ")] + b"compressed %d\nuncompressed_data_size %d\ndata\n" % (
            compressed, size)

    def _oracle_write_region(self, box=None, min_depth=0):
        data = _CpuMap.write_data(self, box, min_depth)
        return self._oracle_header(0, len(data)) + data

    @_asked("_oracle_value_field")
    def value_field(self):
        """Same result as _CpuMap.value_field, produced by the harness in one ordered tree walk
        (no numpy expansion / sort: full-size maps hold ~10^8 voxels)."""
        n = self.api["field"](self.h, None, None, None, 0)
        codes = np.empty(n, np.uint64)
        occ = np.empty(n, np.float32)
        rgb = np.zeros((n, 3), np.uint8)
        if n:
            got = self.api["field"](self.h, codes.ctypes.data, occ.ctypes.data,
                                    rgb.ctypes.data if self.color else None, n)
            assert got == n
        return codes, occ, rgb

    def _oracle_value_field(self):
        return expand_value_field(*_CpuMap.walk(self, True)[:4])

    @_asked("_oracle_leaves")
    def leaves(self, occupied=True, free=True, unknown=False, box=None, min_depth=0):
        """The reference's beginLeaves(...) iteration: (codes, depths, occ), sorted by code."""
        b = None if box is None else np.ascontiguousarray(np.concatenate([box[0], box[1]]), np.float64)
        bp = None if b is None else b.ctypes.data
        n = self.api["leaves"](self.h, int(occupied), int(free), int(unknown), bp, int(min_depth), None, None, None, 0)
        codes = np.empty(n, np.uint64)
        depths = np.empty(n, np.uint32)
        occ = np.empty(n, np.float32)
        if n:
            self.api["leaves"](self.h, int(occupied), int(free), int(unknown), bp, int(min_depth), codes.ctypes.data,
                               depths.ctypes.data, occ.ctypes.data, n)
        order = np.argsort(codes, kind="stable")
        return codes[order], depths[order], occ[order]

    def _oracle_leaves(self, occupied=True, free=True, unknown=False, box=None, min_depth=0):
        """Leaves at or below min_depth and the nodes at min_depth, filtered by state and box."""
        lc, ld, lo, _, _ = _CpuMap.walk(self, True)
        ic, idp, io, _, _ = _CpuMap.walk(self, False)
        top = idp == min_depth
        low = ld >= min_depth
        codes = np.concatenate([lc[low], ic[top]])
        depths = np.concatenate([ld[low], idp[top]]).astype(np.uint32)
        occ = np.concatenate([lo[low], io[top]])
        occ_thr, free_thr = _CpuMap.sensor_model(self)[:2]
        o64 = occ.astype(np.float64)
        is_occ, is_free = o64 > occ_thr, o64 < free_thr
        keep = (occupied & is_occ) | (free & is_free) | (unknown & ~is_occ & ~is_free)
        if box is not None:
            key = np.zeros((len(codes), 3), np.float64)
            for i in range(21):
                for a in range(3):
                    key[:, a] += ((codes >> np.uint64(3 * i + a)) & np.uint64(1)).astype(np.float64) * float(1 << i)
            lo = (key - float(1 << (self.depth_levels - 1))) * self.resolution
            size = (self.resolution * np.ldexp(1.0, depths.astype(np.int32)))[:, None]
            keep &= ((lo <= np.asarray(box[1])) & (lo + size >= np.asarray(box[0]))).all(axis=1)
        codes, depths, occ = codes[keep], depths[keep], occ[keep]
        order = np.argsort(codes, kind="stable")
        return codes[order], depths[order], occ[order]

    @_asked("_oracle_write_compressed")
    def write_compressed(self, min_depth=0, acceleration=1, level=0):
        """Octree::write(ostream, compress=True, ...): LZ4-compressed file image (b"" on failure)."""
        n = self.api["write_compressed"](self.h, int(min_depth), int(acceleration), int(level), None, 0)
        buf = np.empty(max(n, 1), np.uint8)
        if n:
            assert self.api["write_compressed"](self.h, int(min_depth), int(acceleration), int(level), buf.ctypes.data, n) == n
        return buf[:n].tobytes()

    def _oracle_write_compressed(self, min_depth=0, acceleration=1, level=0):
        """The node stream through the liblz4 calls the reference makes (octree.h compressData)."""
        data = _CpuMap.write_data(self, None, min_depth)
        lz4 = C.CDLL("liblz4.so.1")
        bound = lz4.LZ4_compressBound(len(data))
        out = C.create_string_buffer(max(bound, 1))
        if level <= 0:
            n = lz4.LZ4_compress_fast(data, out, len(data), bound, int(acceleration))
        else:
            n = lz4.LZ4_compress_HC(data, out, len(data), bound, int(level))
        return self._oracle_header(1, len(data)) + out.raw[:n] if n >= 0 else b""

    @_changes_state
    def enable_change_detection(self, enable=True):
        if self._real:
            self.api["enable_changes"](self.h, int(enable))
        else:
            self._tracking = enable

    @_changes_state
    def reset_change_detection(self):
        if self._real:
            self.api["reset_changes"](self.h)
        else:
            self._changed = []

    @_changes_state
    def insert(self, origin, xyz, rgb=None, max_range=-1.0, depth=0, **kw):
        kw.update(rgb=rgb, max_range=max_range, depth=depth)
        if self._real or not self._tracking:
            return _CpuMap.insert(self, origin, xyz, **kw)
        before = self._oracle_value_field()
        secs = _CpuMap.insert(self, origin, xyz, **kw)
        after = self._oracle_value_field()
        # voxels whose value is not what it was: new ones, and old ones with another value
        changed = np.ones(len(after[0]), bool)
        if len(before[0]):
            i = np.minimum(np.searchsorted(before[0], after[0]), len(before[0]) - 1)
            changed = (before[0][i] != after[0]) | (before[1][i].view(np.uint32) != after[1].view(np.uint32))
        changed = after[0][changed]
        if depth:
            # the reference records the hit voxels at depth 0 and the free space as the depth-d
            # nodes it updated (a depth-d code has its 3 d low bits set)
            pts = _f64(xyz).reshape(-1, 3)
            if max_range >= 0:
                pts = pts[np.linalg.norm(pts - _f64(origin), axis=1) <= max_range]
            hits = np.unique(np.array([_CpuMap.to_code(self, q, 0) for q in pts], np.uint64))
            low = np.uint64((1 << (3 * depth)) - 1)
            free = np.unique((np.setdiff1d(changed, hits) & ~low) | low)
            self._changed.append((np.intersect1d(changed, hits), 0))
            self._changed.append((free, depth))
        else:
            self._changed.append((changed, 0))
        return secs

    @_asked("_oracle_changed_codes")
    def changed_codes(self):
        """(codes, depths) of the reference's changes_ set, sorted by code, then depth."""
        n = self.api["changes"](self.h, None, None, 0)
        codes = np.empty(n, np.uint64)
        depths = np.empty(n, np.uint32)
        if n:
            self.api["changes"](self.h, codes.ctypes.data, depths.ctypes.data, n)
        order = np.lexsort((depths, codes))
        return codes[order], depths[order]

    def _oracle_changed_codes(self):
        codes = np.concatenate([c for c, _ in self._changed] + [np.empty(0, np.uint64)])
        depths = np.concatenate([np.full(len(c), d, np.uint32) for c, d in self._changed] + [np.empty(0, np.uint32)])
        both = np.unique(np.stack([codes, depths.astype(np.uint64)], axis=1), axis=0)
        return both[:, 0].copy(), both[:, 1].astype(np.uint32)

    @_asked("_oracle_field_count")
    def field_count(self):
        """Number of non-default depth-0 voxels (collapsed nodes counted as 8^depth)."""
        return int(self.api["field"](self.h, None, None, None, 0))

    def _oracle_field_count(self):
        _, depths, occ, rgb, _ = _CpuMap.walk(self, True)
        keep = (occ != 0) | rgb.any(axis=1)
        return int((np.uint64(1) << (np.uint64(3) * depths[keep].astype(np.uint64))).sum())

    @_asked("_oracle_node_batch")
    def node_batch(self, codes, depths=0):
        """Deepest existing node on the path to each code: (occ f32, rgb u8[n,3], flags, depth found)."""
        codes = np.ascontiguousarray(codes, dtype=np.uint64)
        depths = np.ascontiguousarray(np.broadcast_to(depths, codes.shape), dtype=np.uint32)
        n = len(codes)
        occ = np.empty(n, np.float32)
        rgb = np.zeros((n, 3), np.uint8)
        flags = np.empty(n, np.uint8)
        fd = np.empty(n, np.uint32)
        self.api["node_batch"](self.h, codes.ctypes.data, depths.ctypes.data, n, occ.ctypes.data,
                               rgb.ctypes.data, flags.ctypes.data, fd.ctypes.data)
        return occ, rgb, flags, fd

    def _oracle_node_batch(self, codes, depths=0):
        codes = np.ascontiguousarray(codes, dtype=np.uint64)
        depths = np.broadcast_to(depths, codes.shape)
        occ = np.empty(len(codes), np.float32)
        rgb = np.zeros((len(codes), 3), np.uint8)
        flags = np.empty(len(codes), np.uint8)
        fd = np.empty(len(codes), np.uint32)
        for i in range(len(codes)):
            _, occ[i], rgb[i], flags[i], fd[i] = _CpuMap.node(self, codes[i], depths[i])
        return occ, rgb, flags, fd

    @_changes_state
    def clear(self, resolution, depth_levels):
        """Octree::clear(resolution, depth_levels)."""
        if self._real:
            self.api["clear"](self.h, float(resolution), int(depth_levels))
        else:
            self.close()
            _CpuMap.__init__(self, resolution, depth_levels, **self._kw)

    @_changes_state
    @_asked("_oracle_read")
    def read(self, image):
        """Octree::read(istream): replace the map's content by a file image."""
        buf = np.frombuffer(image, np.uint8)
        return bool(self.api["read"](self.h, buf.ctypes.data, len(buf)))

    def _oracle_read(self, image):
        """The node stream behind the header into an emptied map of the same geometry."""
        self.close()
        _CpuMap.__init__(self, self.resolution, self.depth_levels, **self._kw)
        return _CpuMap.read_data(self, image[image.index(b"data\n") + 5:])


class OracleMap(_CpuMap):
    _path = ORACLE_SO
    _prefix = "ufo_oracle_"

    def cast_rays(self, origins, directions, ignore_unknown=False, max_range=-1.0, depth=0):
        """castRay (intended semantics) for every (origin, direction): (hit bool[n], code u64[n])."""
        o, d = _f64(origins).reshape(-1, 3), _f64(directions).reshape(-1, 3)
        hit = np.zeros(len(o), bool)
        codes = np.zeros(len(o), np.uint64)
        c = C.c_uint64()
        for i in range(len(o)):
            if self.api["cast_ray"](self.h, o[i].ctypes.data, d[i].ctypes.data, int(ignore_unknown),
                                    float(max_range), int(depth), C.byref(c)):
                hit[i] = True
                codes[i] = c.value
        return hit, codes

    def canonicalize(self):
        """Collapse every collapsible node: the canonical minimal tree of the value field."""
        self.api["canonicalize"](self.h)

    def last_counters(self):
        out = np.empty(4, np.uint64)
        self.api["last_counters"](self.h, out.ctypes.data)
        return dict(rays=int(out[0]), visits=int(out[1]), unique_free=int(out[2]),
                    unique_hits=int(out[3]))


def expand_value_field(codes, depths, occ, rgb):
    """Expand leaves at depth>0 into their depth-0 voxels, drop default payloads,
    return arrays sorted by code."""
    keep = (occ != 0) | (rgb.any(axis=1))
    codes, depths, occ, rgb = codes[keep], depths[keep], occ[keep], rgb[keep]
    if len(codes) and depths.max() > 0:
        reps = (np.uint64(1) << (np.uint64(3) * depths.astype(np.uint64))).astype(np.int64)
        total = int(reps.sum())
        if total > 400_000_000:
            raise MemoryError("value field too large to expand (%d voxels)" % total)
        base = np.repeat(codes, reps)
        starts = np.cumsum(reps) - reps
        offs = np.arange(total, dtype=np.int64) - np.repeat(starts, reps)
        codes = base + offs.astype(np.uint64)
        occ = np.repeat(occ, reps)
        rgb = np.repeat(rgb, reps, axis=0)
    order = np.argsort(codes, kind="stable")
    return codes[order], occ[order], rgb[order]


def aggregate_level(codes, occ, rgb, level, model, color=False):
    """Pure-function inner aggregates of a value field at `level` (>=1):
    returns (parent_codes (code>>3*level), max_occ, contains_free, contains_unknown).
    Untouched voxels count as 0.0 / unknown (SURVEY.md 8(e), Appendix A.8)."""
    occ_thr, free_thr = model[0], model[1]
    parents = codes >> np.uint64(3 * level)
    uniq, inv, counts = np.unique(parents, return_inverse=True, return_counts=True)
    mx = np.full(len(uniq), -np.inf, np.float32)
    np.maximum.at(mx, inv, occ)
    full = counts == (1 << (3 * level))
    mx = np.where(full, mx, np.maximum(mx, np.float32(0)))
    o64 = occ.astype(np.float64)
    free = np.zeros(len(uniq), bool)
    np.logical_or.at(free, inv, o64 < free_thr)
    unk = np.zeros(len(uniq), bool)
    np.logical_or.at(unk, inv, (o64 >= free_thr) & (o64 <= occ_thr))
    default_unknown = (0.0 >= free_thr) and (0.0 <= occ_thr)
    default_free = 0.0 < free_thr
    unk |= (~full) & default_unknown
    free |= (~full) & default_free
    return uniq, mx, free, unk
