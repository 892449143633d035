"""Randomised cross-check of the library's host-side indexing and ray enumeration (the same
UFO_HD code the kernels run) against the oracle, over resolutions, tree depths and awkward
coordinates (voxel borders, map faces, axis-parallel and degenerate rays).  No GPU needed."""
import numpy as np
import pytest

from oracle_lib import OracleMap, RefMap
from ufomap_b200.capi import Map

def _checkers(res, levels):
    """the oracle, and the reference (or its recorded answers where it is not built)"""
    return [OracleMap(res, depth_levels=levels), RefMap(res, depth_levels=levels)]


CASES = [(0.02, 16), (0.05, 16), (0.16, 12), (0.1, 8), (0.01, 18), (0.25, 21), (0.002, 16)]


def _points(rng, res, levels, n):
    ext = res * (1 << (levels - 1))
    span = min(ext * 0.98, 400.0 * res)
    pts = rng.uniform(-span, span, (n, 3))
    k = n // 4
    pts[:k] = np.round(pts[:k] / res) * res                       # exactly on voxel borders
    pts[k:2 * k] = (np.round(pts[k:2 * k] / res) + 0.5) * res      # exactly on voxel centres
    pts[2 * k] = 0.0
    pts[2 * k + 1] = [ext, -ext, ext - res]                       # on / next to the map faces
    pts[2 * k + 2] = [-ext, ext - res / 2, -ext + res / 2]
    return pts


@pytest.mark.parametrize("res,levels", CASES)
def test_indexing_matches_oracle(res, levels):
    rng = np.random.default_rng(int(res * 1e4) + levels)
    lib = Map(res, depth_levels=levels, device=-2)
    for orc in _checkers(res, levels):
        for p in _points(rng, res, levels, 64):
            for d in (0, 1, 3, min(levels - 1, 7)):
                k = lib.to_key(p, d)
                assert np.array_equal(k, orc.to_key(p, d)), (p, d)
                assert lib.to_code(p, d) == orc.to_code(p, d)
                assert np.array_equal(lib.key_to_coord(k, d), orc.key_to_coord(k, d))
                c = lib.key_to_code(k, d)
                assert c == orc.key_to_code(k, d)
                assert np.array_equal(lib.code_to_key(c, d), orc.code_to_key(c, d))
    lib.close()


@pytest.mark.parametrize("res,levels", CASES)
def test_compute_ray_matches_oracle(res, levels):
    rng = np.random.default_rng(7 * levels + int(res * 1e4))
    lib = Map(res, depth_levels=levels, device=-2)
    span = min(res * (1 << (levels - 1)) * 0.9, 60.0 * res)
    a = rng.uniform(-span, span, (40, 3))
    b = rng.uniform(-span, span, (40, 3))
    b[:6] = a[:6]
    b[:3, 0] += np.array([5, -7, 9]) * res         # axis-parallel
    b[3:6, 2] += np.array([3.5, -0.25, 12]) * res
    a[6] = np.round(a[6] / res) * res               # start on a voxel corner
    b[7] = a[7]                                     # degenerate: zero length
    b[8] = a[8] + res * 1e-3                        # same voxel
    a[9] = np.round(a[9] / res) * res
    b[9] = a[9] + np.array([8, 8, 8]) * res         # exact diagonal: three-way ties at every corner
    for orc in _checkers(res, levels):
        for x, y in zip(a, b):
            for d, mr in ((0, -1.0), (0, 11.3 * res), (1, -1.0), (2, 20 * res)):
                assert np.array_equal(lib.compute_ray(x, y, mr, d), orc.compute_ray(x, y, mr, d)), (x, y, d, mr)
    lib.close()
