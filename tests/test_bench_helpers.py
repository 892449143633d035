"""Host-side pieces of bench.py that the driver's run depends on (no GPU needed)."""
import importlib.util
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_algorithmic_bytes_formula():
    """SURVEY.md 8(d): N*P_in + U*S_leaf + D1*8*S_leaf + sum_{l>=1} D_l*S_inner + sum_{l>=2} D_l*8*S_inner."""
    b = _bench()
    st = dict(points=10, touched_voxels=100, touched_octets=40, touched_blocks=20, touched_d3=8,
              touched_bricks=3, upper_nodes=5)
    mono = 10 * 12 + 100 * 4 + 40 * 8 * 4 + (40 + 20 + 8 + 3 + 5) * 8 + (20 + 8 + 3 + 5) * 8 * 8
    assert b.algorithmic_bytes(st, False, 12) == mono
    upd = 100 * 4 + 40 * 8 * 4 + (40 + 20 + 8 + 3) * 8 + (20 + 8 + 3) * 8 * 8
    assert b.algorithmic_bytes(st, False, 12, part="update") == upd
    color = 10 * 16 + 100 * 8 + 40 * 8 * 8 + (40 + 20 + 8 + 3 + 5) * 12 + (20 + 8 + 3 + 5) * 8 * 12
    assert b.algorithmic_bytes(st, True, 16) == color


def test_committed_measurement_files_are_readable():
    """bench.py folds three committed measurement files into its JSON line."""
    b = _bench()
    traffic, src = b.measured_traffic()
    assert traffic > 1e9 and "profiles/" in src
    ceil = b.atomic_ceiling()
    assert ceil and ceil["l2_resident_gops"] > ceil["at_128mb_gops"] > 0
    sc = b.sector_ceiling()
    assert sc and sc["k3_all_ms"] > sc["k3_leaf_ms"] > 0
    assert sc["rmw_gbs_at_density_1.0"] > sc["rmw_gbs_at_density_0.24"] > sc["rmw_gbs_at_density_0.06"]
    peak, peak_src = b.measured_peak()
    assert 1000.0 < peak < 10000.0 and peak_src


def test_clock_sampler_never_raises_without_a_gpu():
    b = _bench()
    s = b.ClockSampler(0)
    s.start()
    out = s.stop()
    assert set(("sm_mhz", "sm_max_mhz", "reasons", "samples")) <= set(out)
    json.dumps(out)


def test_configs_match_baseline_json():
    """--config 2|3|4 are BASELINE.json's single-GPU configurations."""
    b = _bench()
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert set(b.CONFIGS) == {2, 3, 4}
    assert b.CONFIGS[2]["resolution"] == 0.02 and b.CONFIGS[2]["max_range"] == 30.0 and not b.CONFIGS[2]["color"]
    assert b.CONFIGS[3]["resolution"] == 0.002 and b.CONFIGS[3]["color"]
    assert b.CONFIGS[4]["resolution"] == 0.05 and b.CONFIGS[4]["max_range"] == 100.0
    assert "points" in json.dumps(base).lower()


def test_dump_outputs_writes_the_field_and_counters(tmp_path):
    """--dump-outputs: keys decoded from the voxel codes, float dtypes, a sample of a field above the
    cap that does not depend on the order the device emitted the voxels in."""
    import numpy as np
    b = _bench()
    rng = np.random.default_rng(0)
    keys = rng.integers(0, 1 << 16, (3000, 3)).astype(np.uint64)
    codes = np.zeros(len(keys), np.uint64)
    for i in range(16):
        for a in range(3):
            codes |= ((keys[:, a] >> np.uint64(i)) & np.uint64(1)) << np.uint64(3 * i + a)
    codes, idx = np.unique(codes, return_index=True)
    keys = keys[idx]

    class FakeMap:
        def __init__(self, perm):
            self.perm = perm

        def wait(self):
            pass

        def value_field(self, sort=True):
            occ = (codes % np.uint64(97)).astype(np.float32)
            rgb = np.stack([(codes % np.uint64(251)).astype(np.uint8)] * 3, axis=1)
            return codes[self.perm], occ[self.perm], rgb[self.perm]

        def stats(self):
            return {k: i for i, k in enumerate(b.COUNTER_NAMES)}

    b.dump_outputs(str(tmp_path / "all"), FakeMap(np.arange(len(codes))), True)
    k = np.load(tmp_path / "all" / "voxel_keys.npy")
    assert k.dtype == np.float64 and np.array_equal(k, keys.astype(np.float64))
    assert np.load(tmp_path / "all" / "log_odds.npy").dtype == np.float32
    assert np.load(tmp_path / "all" / "rgb.npy").dtype == np.float32
    assert list(np.load(tmp_path / "all" / "scan_counters.npy")) == list(range(len(b.COUNTER_NAMES)))
    b.DUMP_MAX_VOXELS = 500
    for name in ("a", "b"):
        b.dump_outputs(str(tmp_path / name), FakeMap(rng.permutation(len(codes))), False)
    a_, b_ = (np.load(tmp_path / n / "voxel_keys.npy") for n in ("a", "b"))
    assert 300 < len(a_) < 700 and np.array_equal(a_, b_)
    assert not (tmp_path / "a" / "rgb.npy").exists()
