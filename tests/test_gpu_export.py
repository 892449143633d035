"""The map in the reference's file format (SURVEY.md 8(f) N2): ufo_b200_write against
Octree::write of the reference / the oracle's restatement of it: byte for byte (the canonical
tree is the reference's tree on these histories), and by reading the image back through the
reference's own Octree::read."""
import numpy as np
import pytest

from oracle_lib import OracleMap, RefMap
from ufomap_b200 import scans
from ufomap_b200.capi import Map

pytestmark = pytest.mark.gpu


def _cpu_maps(color, **kw):
    return [OracleMap(color=color, **kw), RefMap(color=color, **kw)]


def _scenario(name):
    if name == "velodyne":
        ins = []
        for k in range(3):
            o, p = scans.velodyne64(k=k, rings=8, azimuths=128)
            ins.append(dict(origin=o, xyz=p, max_range=25.0))
        return dict(resolution=0.2), ins, False
    if name == "rgbd_color_discrete":
        ins = []
        for k in range(2):
            o, p, c = scans.rgbd(k=k, width=48, height=36)
            ins.append(dict(origin=o, xyz=p, rgb=c, max_range=3.0, discrete=True))
        return dict(resolution=0.04), ins, True
    o, p = scans.random_shell(n=1500)
    return dict(resolution=0.16, depth_levels=12), [dict(origin=o, xyz=p, max_range=5.0)], False


@pytest.mark.parametrize("name", ["velodyne", "rgbd_color_discrete", "shell_small_tree"])
@pytest.mark.parametrize("pruning", [False, True])
def test_image_is_byte_identical(name, pruning, tmp_path):
    """Canonical export == the reference's own file (and the oracle's restatement of it) on
    histories where the reference's tree is canonical (all of these; checked on the CPU side by
    tests/test_oracle_vs_reference.py::test_reference_tree_is_canonical_here)."""
    kw, inserts, color = _scenario(name)
    gpu = Map(color=color, automatic_pruning=pruning, initial_blocks=1 << 12, **kw)
    cpus = _cpu_maps(color, automatic_pruning=pruning, **kw)
    for c in cpus:
        assert gpu.write() == c.write(), "empty map"
    for ins in inserts:
        gpu.insert(**ins)
        for c in cpus:
            c.insert(**ins)
    image = gpu.write()
    for c in cpus:
        assert image == c.write(), type(c).__name__
    path = tmp_path / "map.ufo"
    gpu.write_file(str(path))
    assert path.read_bytes() == image
    gpu.close()


@pytest.mark.parametrize("name,depth", [("velodyne", 0), ("rgbd_color_discrete", 0), ("velodyne", 2)])
@pytest.mark.parametrize("expanded", [False, True])
def test_image_reads_back_in_the_reference(name, depth, expanded):
    """Octree::read of the reference parses the image and ends up with the same value field; the
    canonical image is never larger than the reference's own."""
    kw, inserts, color = _scenario(name)
    gpu = Map(color=color, initial_blocks=1 << 12, **kw)
    ref = RefMap(color=color, **kw)
    for ins in inserts:
        gpu.insert(depth=depth, **ins)
        ref.insert(depth=depth, **ins)
    image = gpu.write(expanded=expanded)
    back = RefMap(color=color, **kw)
    assert back.read(image)
    a, b = back.value_field(), ref.value_field()
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    if color:
        assert np.abs(a[2].astype(int) - b[2].astype(int)).max() <= 1
    if not expanded:
        assert len(image) <= len(ref.write())
    gpu.close()


@pytest.mark.parametrize("name", ["velodyne", "rgbd_color_discrete"])
def test_partial_and_truncated_stream(name):
    """Octree::writeData with a bounding box and/or min_depth -- what ufoToMsg publishes
    (change box of the last scans at depths 0..publish_depth, server.cpp:184-199)."""
    kw, inserts, color = _scenario(name)
    gpu = Map(color=color, initial_blocks=1 << 12, **kw)
    cpus = _cpu_maps(color, **kw)
    for ins in inserts:
        gpu.insert(**ins)
        for c in cpus:
            c.insert(**ins)
    rng = np.random.default_rng(17)
    mn, mx = cpus[0].change_bbox()
    span = mx - mn
    boxes = [None, (mn, mx), (mn + 0.4 * span, mn + 0.6 * span), (mn - 5.0, mn - 4.0),
             (np.array([1e4, 1e4, 1e4]), np.array([2e4, 2e4, 2e4]))]
    for _ in range(6):
        lo = mn + rng.uniform(-0.1, 0.9, 3) * span
        boxes.append((lo, lo + rng.uniform(0.01, 0.6, 3) * span))
    res = kw["resolution"]
    boxes.append((np.array([3 * res, 0.0, 0.0]), np.array([3 * res, 4 * res, res])))   # faces on voxel borders
    for box in boxes:
        for md in range(5):
            got = gpu.write_data(box, md)
            for c in cpus:
                assert got == c.write_data(box, md), (type(c).__name__, box, md, len(got))
    gpu.close()


def test_region_file_and_reset(tmp_path):
    """save_map (Octree::write(filename, bounding volume, compress, depth), server.cpp:381-392) and
    reset (Octree::clear(resolution, depth_levels), server.cpp:364-378)."""
    kw, inserts, color = _scenario("velodyne")
    gpu = Map(color=color, initial_blocks=1 << 12, **kw)
    ref = RefMap(color=color, **kw)
    for ins in inserts:
        gpu.insert(**ins)
        ref.insert(**ins)
    mn, mx = ref.change_bbox()
    mid = (mn + mx) / 2
    for box, md in [((mn, mid), 0), ((mid - 1.0, mid + 2.0), 3), (None, 2),
                    ((np.array([1e4, 1e4, 1e4]), np.array([2e4, 2e4, 2e4])), 0)]:
        expect = ref.write_region(box, md)
        assert gpu.write(box=box, min_depth=md) == expect, (box, md)
        path = tmp_path / "region.ufo"
        gpu.write_file(str(path), box=box, min_depth=md)
        assert path.read_bytes() == expect
    # reset to another geometry, then map again
    gpu.clear_resize(0.1, 14)
    ref.clear(0.1, 14)
    assert gpu.write() == ref.write()
    for ins in inserts[:2]:
        gpu.insert(**ins)
        ref.insert(**ins)
    assert gpu.write() == ref.write()
    a, b = gpu.value_field(), ref.value_field()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    gpu.close()


@pytest.mark.parametrize("name", ["velodyne", "rgbd_color_discrete"])
def test_compressed_image_matches_the_reference(name):
    """write(compress=True): one LZ4 block behind the header (octree.h:1428-1456).  The same liblz4
    on both sides -> byte-identical to the reference's own compressed file, for the fast and the
    HC compressor; the data-only form decompresses to the uncompressed node stream."""
    import ctypes
    kw, inserts, color = _scenario(name)
    gpu, ref = Map(color=color, initial_blocks=1 << 12, **kw), RefMap(color=color, **kw)
    for ins in inserts:
        gpu.insert(**ins)
        ref.insert(**ins)
    for accel, level in ((1, 0), (4, 0), (1, 6)):
        image, usize = gpu.write_compressed(acceleration=accel, level=level)
        want = ref.write_compressed(acceleration=accel, level=level)
        assert len(want) > 0 and image == want, (accel, level, len(image), len(want))
        assert b"compressed 1\n" in image[:300] and (b"uncompressed_data_size %d\n" % usize) in image[:300]
    raw = gpu.write_data()
    packed, usize = gpu.write_compressed(data_only=True)
    assert usize == len(raw) and len(packed) < len(raw)
    lz4 = ctypes.CDLL("liblz4.so.1")
    out = ctypes.create_string_buffer(usize)
    n = lz4.LZ4_decompress_safe(packed, out, len(packed), usize)
    assert n == usize and out.raw == raw
    gpu.close()


@pytest.mark.parametrize("name", ["velodyne", "rgbd_color_discrete"])
def test_read_data_merges_like_the_reference(name):
    """Octree::readData: a node stream written by one map is merged into another map that already
    holds different content -- whole stream, a stream truncated at min_depth 2 (its leaves overwrite
    whole blocks), and a stream / read restricted to a box -- and the result is the reference's,
    value for value; inner aggregates follow."""
    from helpers import assert_value_fields_equal, check_inner_against_field
    kw, inserts, color = _scenario(name)
    src = Map(color=color, initial_blocks=1 << 12, **kw)
    for ins in inserts:
        src.insert(**ins)
    lo = np.array(inserts[0]["origin"]) - 1.5
    box = (lo, lo + np.array([4.0, 3.0, 2.5]))
    for stream_kw in (dict(), dict(min_depth=2), dict(box=box), dict(box=box, min_depth=1)):
        data = src.write_data(**stream_kw)
        gpu = Map(color=color, initial_blocks=1 << 12, **kw)
        cpus = _cpu_maps(color, **kw)
        # other content first: the second half of the scenario seen from a shifted pose
        other = dict(inserts[-1])
        other["origin"] = np.array(other["origin"]) + np.array([0.37, -0.21, 0.05])
        gpu.insert(**other)
        for c in cpus:
            c.insert(**other)
        gpu.read_data(data, box=stream_kw.get("box"))
        for c in cpus:
            assert c.read_data(data, box=stream_kw.get("box"))
        field = gpu.value_field()
        for c in cpus:
            assert_value_fields_equal(field, c.value_field(), color_tol=0, what="%s %s" % (type(c).__name__, stream_kw.keys()))
        check_inner_against_field(gpu, cpus[0].value_field(), cpus[0].sensor_model(), levels=(1, 2, 3, 4, 5, 7))
        # and the merged map keeps integrating scans like the reference's
        gpu.insert(**inserts[0])
        for c in cpus:
            c.insert(**inserts[0])
        assert_value_fields_equal(gpu.value_field(), cpus[0].value_field(), color_tol=1 if color else 0, what="scan after merge")
        gpu.close()
    src.close()
