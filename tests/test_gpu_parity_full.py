"""GPU parity at the BASELINE configs' REAL sizes against the compiled, unmodified reference
(oracle/_ref/libufo_ref.so; where it is not built, the C restatement checked against the
reference's recorded answers: tests/oracle_lib.py RefMap).  The whole value field is compared bit
for bit (log-odds) / +-1 (colour), inner aggregates on random samples of every level, and the change box.

The reference needs minutes per case on one core (BASELINE.md section 4: ~1 k points/s), so
all cases are integrated on the CPU concurrently in background threads (the harness calls
release the GIL) while the GPU side runs; the file costs about as long as its slowest case.

  #2  OccupancyMap 2 cm, one full 131 072-pt Velodyne-64 scan, max_range 30 m
  #4  OccupancyMap 5 cm, two consecutive full 131 072-pt scans, max_range 100 m
  #3r OccupancyMapColor 2 mm, 160x120 RGB-D (SURVEY.md 8(d) "#3-reduced"), discrete, depth 0
  #3  OccupancyMapColor 2 mm, full 640x480 RGB-D at insert depth 4 (the depth at which the CPU
      path can run the full-size config at all), two scans, colour included
  #5  OccupancyMap 1 cm, two sensors of the 8-sensor ring, every 8th point, applied in sensor order
  and the 1-vs-2 shard union on #4.
"""
import concurrent.futures as cf

import numpy as np
import pytest

from helpers import assert_value_fields_equal, check_inner_sampled, sorted_field_large
from oracle_lib import RefMap
from ufomap_b200 import scans
from ufomap_b200.capi import Map

pytestmark = pytest.mark.gpu


def _cases():
    c = {}
    o, p = scans.velodyne64(k=0)
    c["c2"] = dict(map_kw=dict(resolution=0.02), color=False,
                   inserts=[dict(origin=o, xyz=p, max_range=30.0)])
    ins = []
    for k in range(2):
        o, p = scans.velodyne64(k=k)
        ins.append(dict(origin=o, xyz=p, max_range=100.0))
    c["c4"] = dict(map_kw=dict(resolution=0.05), color=False, inserts=ins)
    o, p, g = scans.rgbd(k=0, width=160, height=120)
    c["c3r"] = dict(map_kw=dict(resolution=0.002), color=True,
                    inserts=[dict(origin=o, xyz=p, rgb=g, max_range=5.0, discrete=True)])
    ins = []
    for k in range(2):
        o, p, g = scans.rgbd(k=k)
        ins.append(dict(origin=o, xyz=p, rgb=g, max_range=5.0, discrete=True, depth=4))
    # 2 * 10^9 voxels when expanded: compared by voxel count + 2 M sampled voxels, not as a field
    c["c3d4"] = dict(map_kw=dict(resolution=0.002), color=True, inserts=ins, sampled=True)
    # the reference's only fast regime at 2 mm (SURVEY.md 6.2): insert depth 6 (64^3-voxel free nodes)
    c["c3d6"] = dict(map_kw=dict(resolution=0.002), color=True, sampled=True,
                     inserts=[dict(i, depth=6) for i in ins])
    ins = []
    for s in range(2):
        so = scans.sensor_ring(s, 8)
        o, p = scans.velodyne64(k=0, origin=so, seed=88172645463325252 + 7919 * s)
        ins.append(dict(origin=o, xyz=p[::8], max_range=30.0))
    c["c5"] = dict(map_kw=dict(resolution=0.01), color=False, inserts=ins)
    return c


def _cpu_run(case):
    m = RefMap(color=case["color"], **case["map_kw"])
    secs = 0.0
    for ins in case["inserts"]:
        secs += m.insert(**ins)
    bbox = m.change_bbox()
    model = m.sensor_model()
    if case.get("sampled"):
        return dict(map=m, bbox=bbox, model=model, secs=secs, kind="RefMap")
    field = m.value_field()
    m.close()
    return dict(field=field, bbox=bbox, model=model, secs=secs, kind="RefMap")


@pytest.fixture(scope="module")
def cpu_results():
    cases = _cases()
    pool = cf.ThreadPoolExecutor(max_workers=len(cases))
    futures = {k: pool.submit(_cpu_run, v) for k, v in cases.items()}
    yield cases, futures
    pool.shutdown(wait=True)


def _gpu_field(case, shard=None, bricks=1 << 17):
    gpu = Map(color=case["color"], initial_bricks=bricks, **case["map_kw"])
    if shard:
        gpu.set_shard(*shard)
    for ins in case["inserts"]:
        gpu.insert(dtype=np.float32, **ins)  # float32 payload, as a PointCloud2 delivers it
    field = sorted_field_large(gpu)
    return gpu, field


def _compare(name, cpu_results, color_tol=0, levels=(1, 2, 3, 4, 5, 6, 9, 16)):
    cases, futures = cpu_results
    gpu, field = _gpu_field(cases[name])
    ref = futures[name].result()
    assert_value_fields_equal(field, ref["field"], color_tol=color_tol, what="%s vs %s" % (name, ref["kind"]))
    check_inner_sampled(gpu, ref["field"], ref["model"], levels=levels)
    mn, mx = gpu.change_bbox()
    assert np.array_equal(mn, ref["bbox"][0]) and np.array_equal(mx, ref["bbox"][1])
    st = gpu.stats()
    gpu.close()
    print("%s: %d voxels identical to %s (%.1f s of CPU)" % (name, len(field[0]), ref["kind"], ref["secs"]))
    return st, ref


def test_config2_full_scan(cpu_results):
    st, _ = _compare("c2", cpu_results)
    assert st["rays"] == 131072


def test_config4_two_full_scans_100m(cpu_results):
    st, _ = _compare("c4", cpu_results)
    assert st["rays"] == 131072


def test_config3_reduced_2mm_color(cpu_results):
    _compare("c3r", cpu_results, color_tol=1)


@pytest.mark.parametrize("name", ["c3d4", "c3d6"])
def test_config3_full_size_coarse_insert_color(cpu_results, name):
    """Full-size #3 at insert depth 4 / 6: number of non-default voxels, and occupancy (bit-exact) +
    colour (+-1) of 2 M voxels sampled along the rays (free space) and at the end points (hits)."""
    cases, futures = cpu_results
    case = cases[name]
    gpu = Map(color=True, initial_bricks=1 << 19, **case["map_kw"])
    rng = np.random.default_rng(3)
    pts = []
    for ins in case["inserts"]:
        gpu.insert(dtype=np.float32, **ins)
        o, p = ins["origin"], ins["xyz"]
        idx = rng.integers(0, len(p), 1_000_000)
        frac = np.concatenate([rng.uniform(0.02, 1.0, len(idx) // 2), np.ones(len(idx) - len(idx) // 2)])
        pts.append(o + (p[idx] - o) * frac[:, None])
    pts = np.concatenate(pts)
    res = 1.0 / case["map_kw"]["resolution"]
    keys = (np.floor(pts * res).astype(np.int64) + 32768).astype(np.uint64)
    spread = lambda v: sum(((v >> np.uint64(i)) & np.uint64(1)) << np.uint64(3 * i) for i in range(16))
    codes = spread(keys[:, 0]) | (spread(keys[:, 1]) << np.uint64(1)) | (spread(keys[:, 2]) << np.uint64(2))
    assert int(codes[0]) == gpu.to_code(pts[0], 0)
    occ, flags, rgb = gpu.query(codes, 0)
    ref = futures[name].result()
    rocc, rrgb, _, _ = ref["map"].node_batch(codes, 0)
    assert np.array_equal(occ.view(np.uint32), rocc.view(np.uint32))
    assert np.abs(rgb.astype(np.int32) - rrgb.astype(np.int32)).max() <= 1
    assert (occ > 0).sum() > 100000 and (occ < 0).sum() > 100000
    st = gpu.stats()
    print("%s: gpu %.3f ms/scan vs %.3f s/scan on the CPU" % (name, st["ms_total"], ref["secs"] / len(case["inserts"])))
    n_gpu = gpu.value_field_count()
    assert n_gpu == ref["map"].field_count()
    mn, mx = gpu.change_bbox()
    assert np.array_equal(mn, ref["bbox"][0]) and np.array_equal(mx, ref["bbox"][1])
    ref["map"].close()
    gpu.close()


def test_config5_two_sensors_in_order(cpu_results):
    _compare("c5", cpu_results)


def test_config4_shard_union(cpu_results):
    """1-vs-2 spatial shards on #4: the union of the two ranks' fields is the reference's field."""
    cases, futures = cpu_results
    parts = []
    for r in range(2):
        gpu, field = _gpu_field(cases["c4"], shard=(r, 2))
        parts.append(field)
        gpu.close()
    assert len(np.intersect1d(parts[0][0], parts[1][0])) == 0
    codes = np.concatenate([parts[0][0], parts[1][0]])
    order = np.argsort(codes, kind="stable")
    union = (codes[order], np.concatenate([parts[0][1], parts[1][1]])[order],
             np.concatenate([parts[0][2], parts[1][2]])[order])
    assert_value_fields_equal(union, futures["c4"].result()["field"], what="shard union")
