"""Device buffers of a map: what a map reports holding, and its change set, do not depend on the
order in which its buffers were sized, grown, or switched off and on.

The host-side test runs the change-detection history on the reference alone (RefMap); its answers
are recorded in tests/golden/reference/answers.npz, against which the GPU test checks the CUDA map
where the reference is not built."""
import numpy as np
import pytest

from oracle_lib import RefMap
from ufomap_b200 import scans
from ufomap_b200.capi import Map

# (change detection on, scan k, max_range): a scan, a pause during which the map grows, a resume
PAUSED_HISTORY = ((True, 0, 3.0), (False, 1, 30.0), (True, 2, 12.0))


def run_paused_history(m, after_insert=lambda: None):
    for on, k, max_range in PAUSED_HISTORY:
        m.enable_change_detection(on)
        o, p = scans.velodyne64(k=k, rings=16, azimuths=256)
        m.insert(o, p, max_range=max_range)
        after_insert()


def test_reference_keeps_the_change_set_while_paused():
    """enableChangeDetection(false) only stops the recording (occupancy_map_base.h:783): nothing is
    added while it is off, and the set recorded before is still there after it is on again."""
    ref = RefMap(0.1)
    sets = []
    run_paused_history(ref, lambda: sets.append(ref.changed_codes()[0]))
    assert len(sets[0]) > 1000
    assert np.array_equal(sets[1], sets[0])
    assert len(sets[2]) > len(sets[0]) and np.isin(sets[0], sets[2]).all()


@pytest.mark.gpu
def test_change_detection_survives_pause_growth_and_resume():
    """The change mask grows with the brick pool while recording is off, and recording resumes into
    the kept set: after the history the set is the reference's."""
    gpu, ref = Map(0.1, initial_bricks=16), RefMap(0.1)
    regrows = []
    run_paused_history(gpu, lambda: regrows.append(gpu.stats()["regrows"]))
    run_paused_history(ref)
    assert regrows[1] > 0, "the pools did not grow while change detection was off"
    rc, rd = ref.changed_codes()
    assert rd.max() == 0
    assert np.array_equal(gpu.changed_codes(0), rc)
    gpu.close()


@pytest.mark.gpu
def test_device_bytes_do_not_depend_on_history():
    """A scan volume sized for 5 m and re-sized for 30 m: the map then holds what a map that scanned
    at 30 m from the start holds (both staging buffers, the same ray capacity, a 43^3-brick volume),
    and reports the same number of bytes."""
    device_bytes = []
    for ranges in ((5.0, 30.0), (30.0, 30.0)):
        m = Map(0.1, initial_bricks=1 << 16)
        for k, max_range in enumerate(ranges):
            o, p = scans.velodyne64(k=k, rings=16, azimuths=256)
            m.insert(o, p, max_range=max_range)
            st = m.stats()
            assert st["regrows"] == 0
        device_bytes.append(st["device_bytes"])
        m.close()
    assert device_bytes[0] == device_bytes[1]
