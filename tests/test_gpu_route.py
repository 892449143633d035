"""Routed multi-GPU mode (ufo_b200_route_*, SURVEY.md 8(e) variant 2) on ONE device: several maps
play the ranks, their inboxes are connected by plain device pointers (the same kernels write
through NVLink-mapped peer pointers when the ranks are processes on different GPUs -- bench.py
--mode route), and a stream synchronisation stands in for the barrier.

  * one scan split over the ranks by rays: union of the ranks' value fields == single-GPU map
  * BASELINE config #5 shape: one sensor per rank, owner applies the sensors in sensor order:
    union == single-GPU map that inserts the sensors' scans one after the other == CPU reference
"""
import numpy as np
import pytest

from helpers import assert_value_fields_equal
from oracle_lib import OracleMap, RefMap
from ufomap_b200 import capi, scans
from ufomap_b200.capi import Map

pytestmark = pytest.mark.gpu


def _ranks(world, resolution, bricks=1 << 15, **kw):
    maps = [Map(resolution, initial_bricks=bricks) for _ in range(world)]
    ptrs = [m.route_setup(r, world, **kw) for r, m in enumerate(maps)]
    for m in maps:
        m.route_connect(ptrs)
    return maps


def _union(maps):
    parts = [m.value_field() for m in maps]
    codes = np.concatenate([p[0] for p in parts])
    assert len(np.unique(codes)) == len(codes), "ranks own disjoint bricks"
    order = np.argsort(codes, kind="stable")
    return codes[order], np.concatenate([p[1] for p in parts])[order], np.concatenate([p[2] for p in parts])[order]


def _barrier(maps):
    for m in maps:
        m.wait()


@pytest.mark.parametrize("world", [2, 4])
def test_one_scan_split_by_rays(world):
    res, rng_max = 0.05, 30.0
    maps = _ranks(world, res)
    single = Map(res, initial_bricks=1 << 15)
    cpu = OracleMap(res)
    for k in range(3):
        o, p = scans.velodyne64(k=k, rings=32, azimuths=1024)
        buf, layout = capi.pack_points(p, None, np.float32)
        single.insert(o, p, max_range=rng_max, dtype=np.float32)
        cpu.insert(o, p, max_range=rng_max)
        keep = []
        for r, m in enumerate(maps):
            part = np.ascontiguousarray(buf[r::world])  # any split of the rays works
            keep.append(part)
            m.route_mark(o, part.ctypes.data, len(part), layout, max_range=rng_max)
        _barrier(maps)
        for m in maps:
            m.route_apply(0, world, True)
        _barrier(maps)
    ref = single.value_field()
    assert_value_fields_equal(_union(maps), ref, what="routed union vs single GPU")
    assert_value_fields_equal(ref, cpu.value_field(), what="single GPU vs oracle")
    st = [m.stats() for m in maps]
    assert sum(s["touched_voxels"] for s in st) == single.stats()["touched_voxels"]


def test_sensors_merged_in_sensor_order():
    """Config #5 shape at 4 cm: two sensors 10 m apart see overlapping space; every time step the
    owner applies sensor 0's marks, then sensor 1's."""
    res, world = 0.04, 2
    maps = _ranks(world, res, bricks=1 << 16)
    single = Map(res, initial_bricks=1 << 16)
    cpus = [OracleMap(res), RefMap(res)]
    for k in range(2):
        keep = []
        for s, m in enumerate(maps):
            base = scans.sensor_ring(s, 8) + np.array([0.25 * k, 0.10 * k, 0.0])
            o, p = scans.velodyne64(k=k, rings=32, azimuths=512, origin=base, seed=88172645463325252 + 7919 * s)
            single.insert(o, p, max_range=30.0, dtype=np.float32)
            for c in cpus:
                c.insert(o, p, max_range=30.0)
            buf, layout = capi.pack_points(p, None, np.float32)
            keep.append(buf)
            m.route_mark(o, buf.ctypes.data, len(buf), layout, max_range=30.0, self_too=True)
        _barrier(maps)
        for s in range(world):
            for m in maps:
                m.route_apply(s, 1, s == world - 1)
        _barrier(maps)
    field = _union(maps)
    assert_value_fields_equal(field, single.value_field(), what="merged sensors vs single GPU")
    for c in cpus:
        assert_value_fields_equal(field, c.value_field(), what="merged sensors vs %s" % type(c).__name__)
