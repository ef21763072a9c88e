"""The oracle against its pins: skimage KATs, golden traces of the real reference, and
(in the build container) the live reference."""
import numpy as np
import pytest

from oracle import traces
from oracle.disk import disk
from tests import trace_util as tu


# ---- skimage.draw.disk known answers (upstream docstrings; SURVEY 8(c)) -----------------
def test_disk_kat_docstring():
    img = np.zeros((10, 10), np.uint8)
    rr, cc = disk((4, 4), 5)
    img[rr, cc] = 1
    want = np.zeros((10, 10), np.uint8)
    want[0, 2:7] = want[8, 2:7] = 1
    want[1, 1:8] = want[7, 1:8] = 1
    want[2:7, 0:9] = 1
    assert np.array_equal(img, want)


def test_disk_kat_clipped_corner():
    img = np.zeros((4, 4), np.uint8)
    rr, cc = disk((0, 0), 2, shape=(4, 4))
    img[rr, cc] = 1
    want = np.zeros((4, 4), np.uint8)
    want[0:2, 0:2] = 1
    assert np.array_equal(img, want)


@pytest.mark.parametrize("center,radius,count", [((200, 200), 8, 193), ((100, 37), 2, 9),
                                                 ((0, 0), 8, 56), ((400, 400), 8, 41)])
def test_disk_pixel_counts(center, radius, count):
    rr, cc = disk(center, radius, shape=(400, 400))
    assert len(rr) == count


def test_disk_ship_halfwidths():
    rr, cc = disk((50, 60), 8, shape=(400, 400))
    for dr, hw in enumerate([7, 7, 7, 7, 6, 6, 5, 3]):
        cols = cc[rr == 50 + dr]
        assert cols.min() == 60 - hw and cols.max() == 60 + hw


def test_disk_offmap_is_empty():
    rr, cc = disk((-5.5, 100.0), 2, shape=(400, 400))
    assert len(rr) == 0


# ---- restatements vs golden traces of the real reference ----------------------------------
@pytest.mark.parametrize("path", tu.golden_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_c_restatement_matches_reference_trace(path):
    gold = tu.load_golden(path)
    bad = tu.run_engine(tu.COracleEngine, gold, n_copies=2)
    assert bad == []


@pytest.mark.parametrize("name", ["default_s7_seed0", "stress_s32_seed0", "lattice_s7_seed2"])
def test_py_restatement_matches_reference_trace(name):
    gold = tu.load_golden(tu.GOLDEN_DIR + "/" + name + ".npz")
    tr = traces.run_py(gold["spawn"], gold["actions"], map_frames=tuple(gold["map_frames"]))
    for k in tu.STATE_KEYS + ("n_lasers", "kills", "deaths", "map_crc", "maps", "final_scores"):
        assert np.array_equal(tr[k], gold[k]), k
    n = gold["laser_x"].shape[-1]
    for k in tu.LASER_KEYS:
        assert np.array_equal(tr[k][..., :n], gold[k]), k
    assert np.array_equal(tr["obs_vec"].astype(np.float32), gold["obs_vec"])


def test_golden_files_cover_quirks():
    """The fixtures really exercise the load-bearing quirks (SURVEY section 0)."""
    g = tu.load_golden(tu.GOLDEN_DIR + "/default_s7_seed0.npz")
    # reset(x=0) keeps the old x; spawn 400 is off-map until the first thrust
    assert g["spawn"][1, 0, 0] == 0 and tuple(g["spawn"][1, 2]) == (400, 400)
    assert g["ship_x"][1, 0, 0] != 0 or g["ship_x"][0, -1, 0] == 0
    # hull is never restored: some ship starts episode 1 with hull <= 0
    assert (g["ship_hull"][1, 0] <= 0).any()
    # destroyed lasers stay listed for exactly one observation
    assert g["laser_destroyed"].any()
    s = tu.load_golden(tu.GOLDEN_DIR + "/stress_s32_seed0.npz")
    assert s["n_lasers"].max() > 200 and s["ship_alive"][0, -1].sum() == 0


LIVE_CASES = [("random", 7, 120, 11), ("stress", 16, 40, 12), ("lattice", 9, 80, 13)]


@pytest.mark.parametrize("kind,S,T,seed", LIVE_CASES)
def test_py_and_c_restatements_agree_on_the_live_reference_scenes(kind, S, T, seed):
    """The scenes of the live-reference test below, which include ship counts no stored trace has (16-ship stress,
    9-ship lattice): the two restatements, each pinned to the reference by the stored traces, agree bit for bit on every
    frame's observation heads, ship and laser state, events and maps."""
    spawn, actions = traces.make_tapes(seed, 2, T, S, kind)
    tr = traces.run_py(spawn, actions, map_frames=(0, 7))
    tr.update(spawn=spawn.astype(np.int32), actions=actions.astype(np.int16))
    assert tu.run_engine(tu.COracleEngine, tr) == []


# ---- live reference (needs the original source tree, OFB_REFERENCE_ROOT) --------------------
@pytest.mark.reference
@pytest.mark.parametrize("kind,S,T,seed", LIVE_CASES)
def test_py_restatement_matches_live_reference(kind, S, T, seed):
    spawn, actions = traces.make_tapes(seed, 2, T, S, kind)
    ref = traces.run_reference(spawn, actions, vector_ships=(0,), map_frames=(0, 7))
    py = traces.run_py(spawn, actions, map_frames=(0, 7))
    assert traces.compare(ref, py) == []
