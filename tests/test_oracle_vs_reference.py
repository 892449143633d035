"""Pins the plain-C restatement (oracle/ufo_oracle.c) to the UNMODIFIED reference
(oracle/_ref/libufo_ref.so): every node of the two trees must agree -- value field, inner
aggregates, flags, colours, change bbox.  Where the reference is not built, RefMap checks the
restatement's answers against the reference's recorded ones (tests/golden/reference/answers.npz)."""
import numpy as np
import pytest

from oracle_lib import OracleMap, RefMap
from ufomap_b200 import scans


def _same_trees(map_kw, inserts, color=False):
    r = RefMap(color=color, **map_kw)
    o = OracleMap(color=color, **map_kw)
    for ins in inserts:
        r.insert(**ins)
        o.insert(**ins)
    for leaves in (True, False):
        a, b = r.walk(leaves), o.walk(leaves)
        ka = np.lexsort((a[0], a[1]))
        kb = np.lexsort((b[0], b[1]))
        assert len(a[0]) == len(b[0])
        for x, y in zip(a, b):
            x, y = x[ka], y[kb]
            if x.dtype == np.float32:
                x, y = x.view(np.uint32), y.view(np.uint32)
            assert np.array_equal(x, y)
    assert all(np.array_equal(x, y) for x, y in zip(r.change_bbox(), o.change_bbox()))
    assert np.array_equal(r.sensor_model(), o.sensor_model())


def test_plain_and_discrete_shell():
    o, p = scans.random_shell()
    _same_trees(dict(resolution=0.16), [dict(origin=o, xyz=p, max_range=5.0)])
    _same_trees(dict(resolution=0.16, automatic_pruning=False),
                [dict(origin=o, xyz=p, max_range=5.0, discrete=True)])


def test_velodyne_stream():
    ins = []
    for k in range(3):
        o, p = scans.velodyne64(k=k, rings=16, azimuths=256)
        ins.append(dict(origin=o, xyz=p, max_range=30.0))
    _same_trees(dict(resolution=0.1), ins)


def test_color_discrete_and_depths():
    o, p, c = scans.rgbd(width=80, height=60)
    o2, p2, c2 = scans.rgbd(k=1, width=80, height=60)
    _same_trees(dict(resolution=0.02),
                [dict(origin=o, xyz=p, rgb=c, max_range=5.0, discrete=True),
                 dict(origin=o2, xyz=p2, rgb=c2, max_range=5.0, discrete=True)], color=True)
    _same_trees(dict(resolution=0.02),
                [dict(origin=o, xyz=p, rgb=c, max_range=3.0, discrete=True, depth=2),
                 dict(origin=o2, xyz=p2, rgb=c2, max_range=3.0, discrete=True, depth=1)], color=True)
    _same_trees(dict(resolution=0.05),
                [dict(origin=o, xyz=p, max_range=3.0, depth=3),
                 dict(origin=o2, xyz=p2, max_range=4.0, simple=True)])


def test_early_stopping_and_sensor_model():
    o, p = scans.velodyne64(rings=8, azimuths=256)
    _same_trees(dict(resolution=0.2, occupied_thres=0.6, free_thres=0.3, prob_hit=0.8, prob_miss=0.45,
                     clamping_thres_min=0.2, clamping_thres_max=0.9),
                [dict(origin=o, xyz=p, max_range=25.0, early_stopping=2)] * 4)


def test_out_of_map_rays():
    o = np.array([0.3, -0.2, 0.1])
    rng = np.random.default_rng(7)
    p = rng.uniform(-40, 40, size=(3000, 3))
    for disc in (False, True):
        _same_trees(dict(resolution=0.5, depth_levels=6), [dict(origin=o, xyz=p, discrete=disc)])
        _same_trees(dict(resolution=0.5, depth_levels=6), [dict(origin=o, xyz=p, max_range=25.0, discrete=disc)])
    _same_trees(dict(resolution=0.5, depth_levels=6), [dict(origin=[30.0, 2.0, 1.0], xyz=p[:500])])


def test_indexing_and_rays():
    r, o = RefMap(0.05), OracleMap(0.05)
    rng = np.random.default_rng(3)
    pts = np.concatenate([rng.uniform(-100, 100, (300, 3)), [[0, 0, 0], [0.05, 0.05, 0.05], [-0.05, 0, 0.025]]])
    for p in pts:
        for d in (0, 1, 3, 7):
            k = r.to_key(p, d)
            assert np.array_equal(k, o.to_key(p, d))
            assert r.to_code(p, d) == o.to_code(p, d)
            assert np.array_equal(r.key_to_coord(k, d), o.key_to_coord(k, d))
            assert r.key_to_code(k, d) == o.key_to_code(k, d)
            assert np.array_equal(r.code_to_key(r.key_to_code(k, d), d), o.code_to_key(o.key_to_code(k, d), d))
    for a, b in zip(pts[:60], pts[60:120]):
        for d, mr in ((0, -1.0), (0, 20.0), (2, -1.0)):
            assert np.array_equal(r.compute_ray(a / 10, b / 10, mr, d), o.compute_ray(a / 10, b / 10, mr, d))
    ends = pts[:200] / 5
    for d, simple in ((0, False), (1, False), (0, True)):
        assert np.array_equal(np.sort(r.free_set([0.01, 0.02, 0.03], ends, d, simple)),
                              np.sort(o.free_set([0.01, 0.02, 0.03], ends, d, simple)))


def test_cloud_frame_transform():
    """Pose6(x,y,z,r,p,y) and PointCloud::transform: oracle and the C ABI's host helpers against the
    reference, bit for bit, over random poses (incl. identity, gimbal lock, large angles)."""
    from oracle_lib import ORACLE_SO, _load, ref_pose_from_rpy, ref_transform
    from ufomap_b200 import capi
    orc = _load(ORACLE_SO, "ufo_oracle_")
    rng = np.random.default_rng(5)
    rpys = [np.zeros(3), np.array([0.0, np.pi / 2, 0.0]), np.array([np.pi, 0.0, -np.pi])]
    rpys += list(rng.uniform(-3.3, 3.3, (60, 3)))
    for rpy in rpys:
        t = rng.uniform(-50, 50, 3)
        po = np.empty(7)
        pr = ref_pose_from_rpy(*t, *rpy)
        orc["pose_from_rpy"](*t, *rpy, po.ctypes.data)
        assert pr.tobytes() == po.tobytes() == capi.pose_from_rpy(*t, *rpy).tobytes()
        pts = rng.uniform(-40, 40, (300, 3)).astype(np.float32).astype(np.float64)
        pts[0] = 0.0
        a, b = ref_transform(pr, pts), np.empty_like(pts)
        orc["transform"](pr.ctypes.data, pts.ctypes.data, len(pts), b.ctypes.data)
        assert a.tobytes() == b.tobytes()
        assert a.tobytes() == capi.transform_points(pr, pts).tobytes()
        assert a.tobytes() == capi.transform_points(pr, pts, dtype=np.float32).tobytes()


@pytest.mark.parametrize("color", [False, True])
@pytest.mark.parametrize("pruning", [True, False])
def test_file_image(color, pruning):
    """Octree::write (header + pre-order node stream): the oracle's restatement is byte-identical to
    the reference's file, and the reference reads it back to the same map."""
    kw = dict(resolution=0.1, automatic_pruning=pruning)
    ref, orc = RefMap(color=color, **kw), OracleMap(color=color, **kw)
    assert ref.write() == orc.write()          # empty map
    for k in range(3):
        o, p, c = scans.rgbd(k=k, width=40, height=30)
        for m in (ref, orc):
            m.insert(origin=o, xyz=p, rgb=c if color else None, max_range=3.0,
                     discrete=bool(k & 1) or color, depth=1 if k == 2 else 0)
    image = ref.write()
    assert image == orc.write()
    back = RefMap(color=color, **kw)
    assert back.read(image)
    a, b = back.value_field(), ref.value_field()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    assert np.array_equal(a[2], b[2])


def test_reference_tree_is_canonical_here():
    """The reference's file equals the canonical minimal tree of its value field on the histories
    the GPU export tests use (automatic pruning on or off) -- which is why ufo_b200_write can be
    compared byte for byte there."""
    cases = []
    ins = []
    for k in range(3):
        o, p = scans.velodyne64(k=k, rings=8, azimuths=128)
        ins.append(dict(origin=o, xyz=p, max_range=25.0))
    cases.append((dict(resolution=0.2), ins, False))
    ins = []
    for k in range(2):
        o, p, c = scans.rgbd(k=k, width=48, height=36)
        ins.append(dict(origin=o, xyz=p, rgb=c, max_range=3.0, discrete=True))
    cases.append((dict(resolution=0.04), ins, True))
    o, p = scans.random_shell(n=1500)
    cases.append((dict(resolution=0.16, depth_levels=12), [dict(origin=o, xyz=p, max_range=5.0)], False))
    for kw, inserts, color in cases:
        for pruning in (True, False):
            ref = RefMap(color=color, automatic_pruning=pruning, **kw)
            orc = OracleMap(color=color, automatic_pruning=pruning, **kw)
            for i in inserts:
                ref.insert(**i)
                orc.insert(**i)
            image = ref.write()
            assert image == orc.write()
            orc.canonicalize()
            assert image == orc.write()


@pytest.mark.parametrize("color", [False, True])
def test_partial_and_truncated_stream(color):
    """Octree::writeData(stream, AABB, false, min_depth): oracle restatement == reference bytes."""
    kw = dict(resolution=0.05)
    ref, orc = RefMap(color=color, **kw), OracleMap(color=color, **kw)
    for k in range(2):
        o, p, c = scans.rgbd(k=k, width=48, height=36)
        for m in (ref, orc):
            m.insert(origin=o, xyz=p, rgb=c if color else None, max_range=3.0, discrete=True)
    image = ref.write()
    assert ref.write_data(None, 0) == image[image.index(b"data\n") + 5:]
    rng = np.random.default_rng(1)
    mn, mx = ref.change_bbox()
    boxes = [None, (mn, mx), (np.array([100.0, 100, 100]), np.array([101.0, 101, 101])),
             (np.array([1e4, 1e4, 1e4]), np.array([2e4, 2e4, 2e4]))]
    for _ in range(8):
        lo = rng.uniform(-1, 2, 3)
        boxes.append((lo, lo + rng.uniform(0.05, 2.0, 3)))
    for box in boxes:
        for md in (0, 1, 2, 3, 4, 5, 7, 16):
            assert ref.write_data(box, md) == orc.write_data(box, md), (box, md)


@pytest.mark.parametrize("color", [False, True])
@pytest.mark.parametrize("pruning", [True, False])
def test_set_value_volume(color, pruning):
    """setValueVolume(AABB, p, min_depth) interleaved with scans: the oracle's tree stays
    node-for-node equal to the reference's (compared through the file image)."""
    kw = dict(resolution=0.05, automatic_pruning=pruning)
    ref, orc = RefMap(color=color, **kw), OracleMap(color=color, **kw)
    rng = np.random.default_rng(2)
    for k in range(2):
        o, p, c = scans.rgbd(k=k, width=48, height=36)
        for m in (ref, orc):
            m.insert(origin=o, xyz=p, rgb=c if color else None, max_range=3.0, discrete=True)
        for t in range(3):
            lo = rng.uniform(-0.5, 2, 3)
            hi = lo + rng.uniform(0.05, 0.8, 3)
            md, val = [0, 1, 2, 3, 4, 0][3 * k + t], [0.1192, 0.7, 0.5, 0.1192, 0.99, 0.3][3 * k + t]
            for m in (ref, orc):
                m.set_value_volume((lo, hi), val, md)
            assert ref.write() == orc.write(), (k, t, md)
    o, p, c = scans.rgbd(k=3, width=48, height=36)
    for m in (ref, orc):
        m.insert(origin=o, xyz=p, rgb=c if color else None, max_range=3.0, discrete=True)
    assert ref.write() == orc.write()


@pytest.mark.parametrize("color", [False, True])
def test_read_data_merges_streams(color):
    """Octree::readData (msgToUfo): whole-map and change-box streams written by one map are merged
    into another, differently filled map; oracle restatement == reference, byte for byte."""
    kw = dict(resolution=0.05)
    src = RefMap(color=color, **kw)
    dst_r, dst_o = RefMap(color=color, **kw), OracleMap(color=color, **kw)
    for k in range(2):
        o, p, c = scans.rgbd(k=k, width=48, height=36)
        src.insert(origin=o, xyz=p, rgb=c if color else None, max_range=3.0, discrete=True)
    o, p, c = scans.rgbd(k=5, width=32, height=24)
    for m in (dst_r, dst_o):
        m.insert(origin=o, xyz=p, rgb=c if color else None, max_range=2.0, discrete=True)
    mn, mx = src.change_bbox()
    mid = (mn + mx) / 2
    for box in [(mid - 0.4, mid + 0.3), (mn, mid), None]:
        data = src.write_data(box, 0)
        assert dst_r.read_data(data, box) and dst_o.read_data(data, box)
        assert dst_r.write() == dst_o.write(), box
    assert dst_r.write() == src.write()     # after the whole-map stream the copy is complete


def test_randomised_differential():
    """Seeded random configurations -- resolution, tree depth, sensor model, map type, insert mode,
    depth, ray casting, early stopping, max range, pruning -- each a short sequence of scans (and a
    volume set); after every step the oracle's tree must equal the reference's byte for byte."""
    rng = np.random.default_rng(20260923)
    for case in range(64):
        res = float(rng.choice([0.05, 0.08, 0.1, 0.2, 0.25]))
        levels = int(rng.choice([10, 12, 16]))
        color = bool(rng.integers(0, 2))
        model = dict(prob_hit=float(rng.choice([0.7, 0.85, 0.6])), prob_miss=float(rng.choice([0.4, 0.3, 0.45])),
                     clamping_thres_min=float(rng.choice([0.1192, 0.05])),
                     clamping_thres_max=float(rng.choice([0.971, 0.9])),
                     occupied_thres=float(rng.choice([0.5, 0.6])), free_thres=float(rng.choice([0.5, 0.4])))
        kw = dict(resolution=res, depth_levels=levels, automatic_pruning=bool(rng.integers(0, 2)), **model)
        ref, orc = RefMap(color=color, **kw), OracleMap(color=color, **kw)
        for step in range(3):
            n = int(rng.integers(1, 400))
            o = rng.uniform(-1, 1, 3)
            d = rng.normal(size=(n, 3))
            d /= np.linalg.norm(d, axis=1, keepdims=True)
            p = (o + d * rng.uniform(0.3, 40 * res, (n, 1))).astype(np.float32).astype(np.float64)
            c = rng.integers(0, 256, (n, 3), dtype=np.uint8)
            discrete = bool(rng.integers(0, 2)) or color     # colour + non-discrete is uninstantiable (G5)
            ins = dict(origin=o, xyz=p, rgb=c if color else None, discrete=discrete,
                       max_range=float(rng.choice([-1.0, 12 * res, 25 * res])),
                       depth=int(rng.choice([0, 0, 1, 2, 3])), simple=bool(rng.integers(0, 4) == 0),
                       early_stopping=int(rng.choice([0, 0, 2])))
            ref.insert(**ins)
            orc.insert(**ins)
            assert ref.write() == orc.write(), (case, step, ins["depth"], ins["simple"], discrete)
            if step == 1:
                lo = o + rng.uniform(-1, 1, 3)
                box = (lo, lo + rng.uniform(res, 20 * res, 3))
                md = int(rng.choice([0, 1, 2]))
                ref.set_value_volume(box, 0.2, md)
                orc.set_value_volume(box, 0.2, md)
                assert ref.write() == orc.write(), (case, "volume", md)
        assert np.array_equal(ref.change_bbox()[0], orc.change_bbox()[0])
        assert np.array_equal(ref.change_bbox()[1], orc.change_bbox()[1])
