"""The multi-GPU path's host planner against the numpy model of tests/dist_model.py, and the argument checks of the
partition and histogram entry points that return before any CUDA call (no GPU needed).

Every rejected partition call here has n = 0: a check that let the call through would still enqueue nothing, so a
broken check shows up as B200SORT_OK, never as device work."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import dist_model as dm  # noqa: E402
from b200sort import datagen  # noqa: E402
from b200sort._lib import lib  # noqa: E402

OK, INVALID, WORKSPACE = 0, 1, 2
BITS = list(range(4, 15))


def host_plan(all_hist, rank, bits):
    all_hist = np.ascontiguousarray(all_hist, dtype=np.uint64)
    world = all_hist.shape[0]
    owner = np.full(1 << bits, -1, dtype=np.int32)
    recv, send, offs = (np.full(world, 0xDEAD, dtype=np.uint64) for _ in range(3))
    st = lib().b200sort_dist_plan(all_hist.ctypes.data, world, rank, bits, owner.ctypes.data, recv.ctypes.data,
                                  send.ctypes.data, offs.ctypes.data)
    assert st == OK
    return owner, recv, send, offs


def assert_plan(all_hist, bits, what):
    world = all_hist.shape[0]
    for rank, want in enumerate(dm.plans(all_hist)):
        owner, recv, send, offs = host_plan(all_hist, rank, bits)
        w = f"{what} world={world} bits={bits} rank={rank}"
        if not (owner == want["owner"]).all():
            b = int(np.flatnonzero(owner != want["owner"])[0])
            raise AssertionError(f"{w}: owner of bin {b} is {owner[b]}, model {want['owner'][b]} "
                                 f"(model boundaries {want['bound']})")
        assert (recv == want["recv"]).all(), (w, recv, want["recv"])
        assert (send == want["send"]).all(), (w, send, want["send"])
        assert (offs == want["offs"]).all(), (w, offs, want["offs"])


@pytest.mark.parametrize("bits", BITS)
def test_host_planner_matches_numpy_model_on_synthetic_histograms(bits):
    """Every world 1-16 and rank, on histograms with per-rank totals up to 2^30 (global counts up to 2^34), empty
    source ranks, ranks that own nothing, one bin holding every key, a few heavy bins, and no keys at all."""
    for world in range(1, 17):
        for i, kind in enumerate(dm.SYNTHETIC):
            all_hist = dm.synthetic_histograms(kind, world, bits, seed=1000 * bits + 17 * world + i)
            assert_plan(all_hist, bits, kind)


@pytest.mark.parametrize("bits", [4, 5, 7, 8, 9, 12, 14])
@pytest.mark.parametrize("dist_name", ["uniform", "skewed90", "all_equal", "ascending", "edge_mix"])
def test_host_planner_matches_numpy_model_on_keys(dist_name, bits):
    for world in (1, 2, 3, 5, 8, 16):
        srcs = [datagen.make(dist_name, 3000 + 101 * s, seed=30 + s) for s in range(world)]
        assert_plan(np.stack([dm.histogram(k, bits) for k in srcs]), bits, dist_name)


def test_model_reaches_both_sides_of_the_straddle_rule():
    """The synthetic and key-derived histograms above move some boundaries back one bin and keep others: the
    model (and so the planner it is compared with) is exercised on both sides of the half-bin rule."""
    moved = kept = 0
    for world in range(2, 17):
        for i, kind in enumerate(dm.SYNTHETIC):
            h = dm.synthetic_histograms(kind, world, 8, seed=1000 * 8 + 17 * world + i).sum(axis=0)
            cum = [0] + np.cumsum(h.astype(object)).tolist()
            total = cum[-1]
            for k, b in enumerate(dm.boundaries(h, world)[1:-1], start=1):
                first = next(i for i, c in enumerate(cum) if c * world >= total * k)
                moved += b == first - 1
                kept += b == first and first > 0 and cum[first - 1] > 0
    assert moved > 0 and kept > 0, (moved, kept)


def test_model_on_a_hand_made_histogram():
    # 4 bins of 10, 30, 50, 10 keys, two ranks: target 50 falls in bin 2 ([40, 90)), 40 of its 50 keys lie beyond
    # the target, so bin 2 goes to rank 1
    h = np.array([[10, 30, 50, 10]], dtype=np.uint64)
    assert dm.boundaries(h[0], 2) == [0, 2, 4]
    # 10, 60, 20, 10: target 50 falls in bin 1 ([10, 70)); 20 of its 60 keys lie beyond it, so bin 1 stays with rank 0
    assert dm.boundaries(np.array([10, 60, 20, 10]), 2) == [0, 2, 4]
    # everything in bin 0: no boundary moves back to 0 keys
    assert dm.boundaries(np.array([100, 0, 0, 0]), 4) == [0, 1, 1, 1, 4]
    p = dm.plans(np.array([[5, 0, 7, 1], [0, 3, 2, 0]], dtype=np.uint64))
    assert p[0]["owner"].tolist() == [0, 0, 1, 1] and p[1]["offs"].tolist() == [5, 8]
    assert p[1]["send"].tolist() == [3, 2] and p[0]["recv"].tolist() == [8, 10]


# ---- argument checks before any CUDA call ---------------------------------------------------------------------
ALIGNED = [0x7f0000000000 + 0x10000 * r for r in range(17)]


def partition(bits=8, world=2, base=ALIGNED, owner=0x7f1000000000, offs="ok", ws=0x7f2000000000, ws_bytes=256):
    table = None if base is None else (ctypes.c_void_p * 17)(*base)
    offsets = np.zeros(17, dtype=np.uint64)
    return lib().b200sort_dist_partition_i32(0x7f3000000000, 0, bits, world, table, owner,
                                             offsets.ctypes.data if offs == "ok" else None, ws, ws_bytes, None)


def test_partition_accepts_valid_arguments_with_no_keys():
    for bits in (4, 14):
        for world in (1, 16):
            assert partition(bits=bits, world=world) == OK


@pytest.mark.parametrize("case,want", [
    (dict(bits=3), INVALID), (dict(bits=15), INVALID), (dict(world=0), INVALID), (dict(world=17), INVALID),
    (dict(world=-1), INVALID), (dict(base=None), INVALID), (dict(owner=None), INVALID), (dict(offs=None), INVALID),
    (dict(base=ALIGNED[:1] + [ALIGNED[1] + 4] + ALIGNED[2:]), INVALID),
    (dict(base=ALIGNED[:15] + [ALIGNED[15] + 8] + ALIGNED[16:], world=16), INVALID),
    (dict(ws=None), WORKSPACE), (dict(ws_bytes=255), WORKSPACE),
], ids=["bits3", "bits15", "world0", "world17", "world-1", "null_table", "null_owner", "null_offsets",
        "base_plus_4_bytes", "base15_plus_8_bytes", "null_workspace", "workspace_255"])
def test_partition_rejects_bad_arguments(case, want):
    assert partition(**case) == want


@pytest.mark.parametrize("bits", [-1, 0, 3, 15, 16, 32])
def test_histogram_rejects_bits_out_of_range(bits):
    hist = np.full(1 << 17, 7, dtype=np.uint64)        # host memory, and n = 0: a call that got through would not launch
    keys = np.zeros(16, dtype=np.int32)
    assert lib().b200sort_dist_histogram_i32(keys.ctypes.data, 0, bits, hist.ctypes.data, None) == INVALID
    assert lib().b200sort_dist_histogram_i32(keys.ctypes.data, 0, 8, None, None) == INVALID
    assert (hist == 7).all()
