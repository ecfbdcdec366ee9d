"""The multi-GPU path's kernels on ONE GPU, every simulated rank's receive buffer a guarded local region: the
partition in each of its four compiled shapes, the device planner's record, the source histograms, the error flag,
the MSD histogram and the argument checks of the planned entry points.

Everything goes through the C-ABI; torch only owns device memory.  The reference is the numpy model of
tests/dist_model.py (checked against the host planner on the CPU by tests/test_dist_partition_cpu.py):
- the destination of a key is owner[(key ^ 0x80000000) >> (32 - bits)];
- source s's block in destination r is the multiset of s's keys destined to r;
- src_hist[r][p] is the histogram of byte p of key ^ 0x80000000 over those keys, p = 0..2, and row 3 is zero;
- top_hist of rank r is the histogram of the top byte of every key rank r owns, counted from the keys.

The partition's compiled shapes: "bulk" (512 threads, bulk copies: the default), "stores" (512 threads, 128-bit
stores: B200SORT_DIST_TMA=0), "stores256" (256 threads, stores: B200SORT_DIST_SHAPE=1) and "bulk_hist" (512 threads,
bulk copies, source histograms: whenever d_src_hist is given).  The environment picks a shape once per process, so
"stores" and "stores256" run in a subprocess that imports this module.
"""
import ctypes
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

import digit_patterns as dp
import dist_model as dm
import oracle
from b200sort import datagen
from b200sort import dist as b200dist
from b200sort._lib import ALGO_RADIX, check, lib
from helpers import stream_ptr

pytestmark = pytest.mark.gpu

OK, INVALID, WORKSPACE = 0, 1, 2
PLAN_BYTES, PLAN_M_OFFSET, PLAN_TOP_OFFSET = 1424, 384, 400
SHAPE_ENV = {"bulk": {}, "stores": {"B200SORT_DIST_TMA": "0"}, "stores256": {"B200SORT_DIST_SHAPE": "1"}}
# more tiles than either grid (148 SMs x 2 CTAs of 8192-key tiles, 148 x 4 of 4096-key tiles): CTAs loop and share
# the destination cursors
N_BIG = 148 * 2 * 8192 + 3 * 8192 + 5
GUARD, GAP = 16, 8                 # canary words around every receive region and between consecutive source blocks

# (world, bits, keys per source, distribution, word offset of every source's keys): every world, bin width, size
# class, distribution and key offset appears; n = 1000 and 5 lie below one tile, 4095/4097 and 8191/8193 straddle
# the 256- and 512-thread tiles
CASES = [
    (1, 4, 1000, "uniform", 1),
    (2, 5, 8191, "skewed90", 2),
    (3, 7, 8193, "all_equal", 3),
    (5, 8, 4095, "ascending", 0),
    (8, 9, 4097, "edge_mix", 1),
    (16, 12, 1000, "uniform", 2),
    (16, 14, 8193, "skewed90", 3),
    (16, 4, 4095, "edge_mix", 0),
    (5, 12, 8191, "all_equal", 2),
    (8, 8, 8193, "uniform", 3),
    (1, 14, 8191, "ascending", 0),
    (3, 8, 5, "edge_mix", 1),
    (2, 9, 0, "uniform", 0),
    (3, 14, N_BIG, "uniform", 1),
    (2, 8, N_BIG, "skewed90", 2),
]


def case_id(c):
    world, bits, n, dist_name, koff = c
    return f"world{world}-bits{bits}-n{n}-{dist_name}-keys_at_word{koff}"


def _aligned(nbytes: int, fill: int):
    """A uint8 device tensor and a 256-byte aligned pointer to nbytes of it."""
    import torch
    t = torch.full((nbytes + 256,), fill, dtype=torch.uint8, device="cuda")
    return t, t.data_ptr() + (-t.data_ptr()) % 256


class Workspace:
    """One workspace for the module, filled with 0xFF once and never cleared; the GUARD bytes past each call's
    ws_bytes must not change."""
    GUARD = 1024

    def __init__(self):
        self.cap = lib().b200sort_dist_workspace_bytes(0, 15) + self.GUARD        # room for a bits = 15 call
        self.t, self.ptr = _aligned(self.cap, 0xFF)
        self.lo = self.ptr - self.t.data_ptr()

    def guard(self, nbytes: int):
        return self.t[self.lo + nbytes:self.lo + nbytes + self.GUARD].cpu()


@functools.lru_cache(maxsize=None)
def workspace() -> Workspace:
    return Workspace()


def assert_no_check_failures():
    """Checked library (B200SORT_LIB=libb200sort_checked.so): the partition kernel's staging-slot (site 9) and
    bulk-copy alignment (site 10) checks, and every other site, counted nothing."""
    L = lib()
    if L.b200sort_debug_checked_build() == 1:
        per = (ctypes.c_ulonglong * 16)()
        total = L.b200sort_debug_check_failures_by_site(per)
        assert per[9] == 0 and per[10] == 0 and total == 0, list(per)


@pytest.fixture(scope="module", autouse=True)
def _no_check_failures():
    yield
    assert_no_check_failures()


def device_words(a: np.ndarray):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int32).copy()).cuda()


def keys_at(keys: np.ndarray, koff: int):
    """(tensor, pointer) of keys placed koff words past a 16-byte boundary."""
    import torch
    t = torch.zeros(keys.size + 4, dtype=torch.int32, device="cuda")
    if keys.size:
        t[koff:koff + keys.size] = torch.from_numpy(keys).cuda()
    return t, t.data_ptr() + 4 * koff


def record(p: dict, offs, error: int = 0):
    """A plan record laid out as include/b200sort.h states (recv, send, dst_offset, m, error, top_hist)."""
    rec = np.zeros(PLAN_BYTES // 8, dtype=np.uint64)
    w = len(offs)
    rec[:w], rec[16:16 + w], rec[32:32 + w] = p["recv"], p["send"], np.asarray(offs, dtype=np.uint64)
    u32 = rec.view(np.uint32)
    u32[PLAN_M_OFFSET // 4], u32[PLAN_M_OFFSET // 4 + 1] = p["m"] & 0xFFFFFFFF, error
    return device_words(rec)


def parse_record(rec: np.ndarray, world: int) -> dict:
    u64, u32 = rec.view(np.uint64), rec.view(np.uint32)
    return {"recv": u64[:world], "send": u64[16:16 + world], "offs": u64[32:32 + world],
            "m": int(u32[PLAN_M_OFFSET // 4]), "error": int(u32[PLAN_M_OFFSET // 4 + 1]),
            "top": u32[PLAN_TOP_OFFSET // 4:PLAN_TOP_OFFSET // 4 + 256], "tail16": (u64[world:16], u64[16 + world:32],
                                                                             u64[32 + world:48])}


@functools.lru_cache(maxsize=8)
def sources(world: int, n: int, dist_name: str):
    return tuple(datagen.make(dist_name, n, seed=100 + s) for s in range(world))


# ---- guarded receive regions --------------------------------------------------------------------------------------
class Regions:
    """The receive regions of every destination in one canary-filled device buffer.  Region r starts on a 16-byte
    boundary (the API requires it); source s's block in it starts at GUARD + (the model's offset) + GAP * s +
    (s + 2r) % 4 words, so every block has canary words before and after it, and block starts take every
    alignment."""

    def __init__(self, plans: list, salt: int):
        import torch
        world = len(plans)
        recv = plans[0]["recv"]
        self.world = world
        self.start = np.zeros(world, dtype=np.int64)
        self.off = np.zeros((world, world), dtype=np.int64)               # [source][destination], words
        pos = 0
        for r in range(world):
            self.start[r] = pos
            for s in range(world):
                self.off[s, r] = GUARD + int(plans[s]["offs"][r]) + GAP * s + (s + 2 * r) % 4
            pos += (GUARD + int(recv[r]) + GAP * world + GUARD + 3) // 4 * 4
        self.fill = dp.canary(pos, salt)
        self.t = torch.from_numpy(self.fill.view(np.int32).copy()).cuda()
        self.bases = (ctypes.c_void_p * world)(*[self.t.data_ptr() + 4 * int(a) for a in self.start])
        self.words = self.fill.copy()                                      # what the buffer holds after the last check

    def read(self) -> np.ndarray:
        return self.t.cpu().numpy().view(np.uint32)

    def check_source(self, s: int, blocks: list, what: str) -> None:
        """After source s's call: every word outside its blocks unchanged, each block a permutation of the model's."""
        got = self.read()
        mine = np.zeros(got.size, dtype=bool)
        for r, b in enumerate(blocks):
            a = self.start[r] + self.off[s, r]
            mine[a:a + b.size] = True
        bad = np.flatnonzero((got != self.words) & ~mine)
        if bad.size:
            k = int(bad[0])
            r = int(np.searchsorted(self.start, k, side="right")) - 1
            raise AssertionError(f"{what}: source {s} changed {bad.size} words outside its blocks, first at word "
                                 f"{k - self.start[r]} of destination {r}'s region (its block there: "
                                 f"[{self.off[s, r]}, {self.off[s, r] + blocks[r].size}))")
        for r, b in enumerate(blocks):
            a = self.start[r] + self.off[s, r]
            if np.sort(got[a:a + b.size].view(np.int32)).tobytes() != np.sort(b).tobytes():
                raise AssertionError(f"{what}: source {s}'s block in destination {r} ({b.size} keys at word "
                                     f"{self.off[s, r]}) is not the model's multiset")
        self.words = got.copy()

    def assert_unchanged(self, what: str) -> None:
        got = self.read()
        bad = np.flatnonzero(got != self.words)
        assert bad.size == 0, f"{what}: {bad.size} words of the receive regions changed, first at {bad[0]}"


# ---- the guarded block layout in every shape ----------------------------------------------------------------------
def run_case(case, path: str, shape: str = "bulk") -> None:
    """Every source of `case` partitioned one at a time into guarded regions, checked after each call.

    path: "host" (b200sort_dist_partition_i32 with the regions' offsets), "planned"
    (b200sort_dist_partition_planned_i32 with a record that holds the same offsets) or "planned_hist" (the same with
    d_src_hist: the bulk_hist shape, bits >= 8)."""
    import torch
    L = lib()
    world, bits, n, dist_name, koff = case
    what = f"shape {shape if path != 'planned_hist' else 'bulk_hist'} via {path} {case_id(case)}"
    srcs = sources(world, n, dist_name)
    all_hist = np.stack([dm.histogram(k, bits) for k in srcs])
    plans = dm.plans(all_hist)
    owner = plans[0]["owner"]
    reg = Regions(plans, salt=world * 31 + bits)
    d_owner = torch.from_numpy(owner).cuda()
    ws = workspace()
    hist = torch.empty(world * 1024 + 64, dtype=torch.int32, device="cuda")
    for s in range(world):
        dest = owner[dm.bins(srcs[s], bits)]
        blocks = [srcs[s][dest == r] for r in range(world)]
        assert [b.size for b in blocks] == [int(x) for x in plans[s]["send"]]
        kt, kp = keys_at(srcs[s], koff)
        hist.fill_(-1)
        before = ws.guard(256)
        if path == "host":
            offs = reg.off[s].astype(np.uint64)
            st = L.b200sort_dist_partition_i32(kp, n, bits, world, reg.bases, d_owner.data_ptr(), offs.ctypes.data,
                                               ws.ptr, 256, stream_ptr())
        else:
            rec = record(plans[s], reg.off[s])
            st = L.b200sort_dist_partition_planned_i32(kp, n, bits, world, reg.bases, d_owner.data_ptr(),
                                                       rec.data_ptr(), hist.data_ptr() if path == "planned_hist"
                                                       else None, ws.ptr, 256, stream_ptr())
        check(st)
        torch.cuda.synchronize()
        reg.check_source(s, blocks, what)
        assert torch.equal(ws.guard(256), before), f"{what}: workspace written past 256 bytes"
        h = hist.cpu().numpy().view(np.uint32)
        assert (h[world * 1024:] == 0xFFFFFFFF).all(), f"{what}: source histograms written past world x 1024"
        if path == "planned_hist":
            h = h[:world * 1024].reshape(world, 4, 256)
            for r in range(world):
                want = dm.digit_rows(blocks[r])
                assert (h[r] == want).all(), (f"{what}: source {s}'s histograms for destination {r} differ in rows "
                                              f"{sorted(set(np.nonzero(h[r] != want)[0].tolist()))}")
        else:
            assert (h == 0xFFFFFFFF).all(), f"{what}: d_src_hist = NULL, yet histograms were written"


PATH_CASES = [pytest.param(c, p, id=f"{'bulk_hist' if p == 'planned_hist' else 'bulk'}-{p}-{case_id(c)}")
              for p in ("host", "planned", "planned_hist")
              for c in CASES if p != "planned_hist" or c[1] >= 8]


@pytest.mark.parametrize("case,path", PATH_CASES)
def test_partition_guarded_blocks(case, path):
    """The default bulk-copy shape (host-planned and planned entry points) and the bulk_hist shape."""
    run_case(case, path)


def shape_matrix(shape: str) -> None:
    """Every case through both entry points, and the error path, in the shape the environment selected."""
    for case in CASES:
        for path in ("host", "planned"):
            run_case(case, path, shape)
    for case in ERROR_CASES:
        run_error_path(case, with_hist=False, shape=shape)


def _subprocess(code: str, env: dict):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prog = ("import sys; sys.path.insert(0, '.'); sys.path.insert(0, 'tests')\n"
            "import test_dist_partition_gpu as t\n" + code + "\nt.assert_no_check_failures()\nprint('ok')\n")
    r = subprocess.run([sys.executable, "-c", prog], cwd=root, env={**os.environ, **env}, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("shape", ["stores", "stores256"])
def test_partition_shapes_selected_by_the_environment(shape):
    """The 128-bit store write-out at 512 and at 256 threads: tiles of 8192 and 4096 keys, grids of 296 and 592
    CTAs, vector and scalar stores at every head/body/tail split."""
    _subprocess(f"t.shape_matrix({shape!r})\n", SHAPE_ENV[shape])


# ---- the plan record ----------------------------------------------------------------------------------------------
def device_plans(all_hist: np.ndarray, bits: int, cap: int, ranks):
    """(owner int32[len(ranks)][nbins], records) from b200sort_dist_plan_device, one call per rank, one sync."""
    import torch
    L = lib()
    world, nbins = all_hist.shape
    d_hist = torch.from_numpy(all_hist.astype(np.int64).reshape(-1)).cuda()
    owners = torch.full((len(ranks), nbins), -1, dtype=torch.int32, device="cuda")
    recs = torch.full((len(ranks), PLAN_BYTES // 8), -1, dtype=torch.int64, device="cuda")   # the planner clears it
    ws = workspace()
    need = L.b200sort_dist_workspace_bytes(0, bits)
    before = ws.guard(need)
    for i, rank in enumerate(ranks):
        check(L.b200sort_dist_plan_device(d_hist.data_ptr(), world, rank, bits, cap, owners[i].data_ptr(),
                                          recs[i].data_ptr(), ws.ptr, need, stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(ws.guard(need), before), f"planner wrote past ws_bytes = {need}"
    return owners.cpu().numpy(), recs.cpu().numpy()


def assert_device_plans(all_hist: np.ndarray, bits: int, what: str, top_from_keys=None) -> None:
    """Every rank's device plan against the host planner and the model; top_hist against `top_from_keys`
    ([world][256], counted from the keys) or, without keys, against the bins."""
    world = all_hist.shape[0]
    model = dm.plans(all_hist)
    recv = model[0]["recv"]
    cap = int(recv.max())
    owners, recs = device_plans(all_hist, bits, cap, range(world))
    for rank in range(world):
        w = f"{what} world={world} bits={bits} rank={rank}"
        want = model[rank]
        owner_h, recv_h, send_h, offs_h = b200dist.plan(all_hist, rank, bits)
        assert (owner_h == want["owner"]).all() and (recv_h == want["recv"]).all(), w + ": host planner vs model"
        assert (send_h == want["send"]).all() and (offs_h == want["offs"]).all(), w + ": host planner vs model"
        if not (owners[rank] == want["owner"]).all():
            b = int(np.flatnonzero(owners[rank] != want["owner"])[0])
            raise AssertionError(f"{w}: device owner of bin {b} is {owners[rank][b]}, host {want['owner'][b]}")
        got = parse_record(recs[rank], world)
        for field in ("recv", "send", "offs"):
            assert (got[field] == want[field]).all(), (w, field, got[field], want[field])
        assert all((x == 0).all() for x in got["tail16"]), w + ": counts past `world` not cleared"
        assert got["error"] == 0, w + f": error flag with cap = the largest recv ({cap})"
        if want["m"] < 1 << 32:
            assert got["m"] == want["m"], (w, got["m"], want["m"])
            if bits < 8:
                assert (got["top"] == 0).all(), w + ": top_hist below 8 bits must be zero"
            else:
                top = top_from_keys[rank] if top_from_keys is not None else dm.top_hist_from_bins(
                    all_hist, want["owner"], rank, bits)
                if not (got["top"] == top).all():
                    t = int(np.flatnonzero(got["top"] != top)[0])
                    raise AssertionError(f"{w}: top_hist[{t}] = {got['top'][t]}, model {top[t]}")
    if cap > 0:                                         # one key more than the cap somewhere: the flag, nothing else
        _, recs = device_plans(all_hist, bits, cap - 1, [world - 1])
        got = parse_record(recs[0], world)
        assert got["error"] == 1, f"{what} world={world} bits={bits}: cap = largest recv - 1, no error flag"
        assert (got["recv"] == recv).all() and (got["offs"] == model[world - 1]["offs"]).all()


KEY_DISTS = ("uniform", "skewed90", "all_equal", "ascending", "edge_mix")


@pytest.mark.parametrize("bits", range(4, 15))
def test_device_plan_record(bits):
    """World 1-16, every rank: the key-derived cases of the partition tests and synthetic histograms (per-rank totals
    of 2^30, empty ranks, one bin with every key, a few heavy bins, no keys)."""
    for world in range(1, 17):
        for dist_name in KEY_DISTS:
            srcs = [datagen.make(dist_name, 3000 + 101 * s, seed=30 + s) for s in range(world)]
            all_hist = np.stack([dm.histogram(k, bits) for k in srcs])
            everything = np.concatenate(srcs)
            dest = dm.plans(all_hist)[0]["owner"][dm.bins(everything, bits)]
            top = np.bincount(dest * 256 + (dm.images(everything) >> np.uint32(24)).astype(np.int64),
                              minlength=world * 256).reshape(world, 256)
            assert_device_plans(all_hist, bits, dist_name, top_from_keys=top)
        for i, kind in enumerate(dm.SYNTHETIC):
            assert_device_plans(dm.synthetic_histograms(kind, world, bits, seed=5000 + 100 * bits + 17 * world + i),
                                bits, kind)


# ---- the error flag: nothing written ------------------------------------------------------------------------------
ERROR_CASES = [c for c in CASES if c[2] > 0 and c[0] > 1 and c[2] < N_BIG]


def run_error_path(case, with_hist: bool, shape: str = "bulk") -> None:
    """A device plan whose cap is one key short: the planned partition leaves every region word as it was and the
    source histograms all zero."""
    import torch
    L = lib()
    world, bits, n, dist_name, koff = case
    if with_hist and bits < 8:
        return
    what = f"error path shape {shape if not with_hist else 'bulk_hist'} {case_id(case)}"
    srcs = sources(world, n, dist_name)
    all_hist = np.stack([dm.histogram(k, bits) for k in srcs])
    plans = dm.plans(all_hist)
    cap = int(plans[0]["recv"].max()) - 1
    reg = Regions(plans, salt=7 + bits)
    hist = torch.full((world * 1024,), -1, dtype=torch.int32, device="cuda")
    for s in range(world):
        owners, recs = device_plans(all_hist, bits, cap, [s])
        assert parse_record(recs[0], world)["error"] == 1, what
        d_owner, d_rec = torch.from_numpy(owners[0]).cuda(), torch.from_numpy(recs[0]).cuda()
        kt, kp = keys_at(srcs[s], koff)
        ws = workspace()
        check(L.b200sort_dist_partition_planned_i32(kp, n, bits, world, reg.bases, d_owner.data_ptr(), d_rec.data_ptr(),
                                                    hist.data_ptr() if with_hist else None, ws.ptr, 256, stream_ptr()))
        torch.cuda.synchronize()
        reg.assert_unchanged(f"{what} source {s}")
        h = hist.cpu().numpy()
        assert (h == 0).all() if with_hist else (h == -1).all(), f"{what} source {s}: source histograms"
        hist.fill_(-1)


@pytest.mark.parametrize("with_hist", [False, True], ids=["bulk", "bulk_hist"])
@pytest.mark.parametrize("case", ERROR_CASES, ids=case_id)
def test_error_flag_writes_nothing(case, with_hist):
    run_error_path(case, with_hist)


# ---- the source histograms of a call with no keys -----------------------------------------------------------------
@pytest.mark.parametrize("bits", [8, 14])
def test_source_histograms_cleared_when_a_rank_sends_nothing(bits):
    """d_src_hist is overwritten by every call, n == 0 included: a rank that contributes no keys after a call in
    which it did must not hand its old counts to the reduce-scatter."""
    import torch
    L = lib()
    world, n = 4, 30000
    srcs = sources(world, n, "uniform")
    all_hist = np.stack([dm.histogram(k, bits) for k in srcs])
    plans = dm.plans(all_hist)
    reg = Regions(plans, salt=3)
    d_owner = torch.from_numpy(plans[0]["owner"]).cuda()
    hist = torch.full((world * 1024,), -1, dtype=torch.int32, device="cuda")
    s = 1
    rec = record(plans[s], reg.off[s])
    kt, kp = keys_at(srcs[s], 0)
    ws = workspace()
    check(L.b200sort_dist_partition_planned_i32(kp, n, bits, world, reg.bases, d_owner.data_ptr(), rec.data_ptr(),
                                                hist.data_ptr(), ws.ptr, 256, stream_ptr()))
    torch.cuda.synchronize()
    dest = plans[0]["owner"][dm.bins(srcs[s], bits)]
    reg.check_source(s, [srcs[s][dest == r] for r in range(world)], f"bits={bits} n={n}")
    assert int(hist.sum().item()) == 3 * n                 # rows 0..2 count every key once
    check(L.b200sort_dist_partition_planned_i32(kp, 0, bits, world, reg.bases, d_owner.data_ptr(), rec.data_ptr(),
                                                hist.data_ptr(), ws.ptr, 256, stream_ptr()))
    torch.cuda.synchronize()
    h = hist.cpu().numpy()
    assert (h == 0).all(), f"bits={bits}: n = 0 left {int(np.count_nonzero(h))} nonzero counts of the previous call"
    reg.assert_unchanged(f"bits={bits} n=0")


# ---- plan -> partition -> local sort with the source histograms ---------------------------------------------------
def sync_free_round(srcs, bits, bufs, src_hists, radix_ws, what):
    """One distributed sort of `srcs` on one GPU: device plans, planned partitions with source histograms into
    `bufs` (canary-filled regions of cap words), then every destination's histogram summed over the sources (the
    reduce-scatter) with row 3 from its record, checked, and handed to b200sort_radix_copy_devn_i32."""
    import torch
    L = lib()
    world = len(srcs)
    cap = bufs.shape[1] - 2 * GUARD
    all_hist = np.stack([dm.histogram(k, bits) for k in srcs])
    plans = dm.plans(all_hist)
    owner = plans[0]["owner"]
    assert int(plans[0]["recv"].max()) <= cap
    fill = dp.canary(bufs.numel(), world).view(np.int32).reshape(bufs.shape)
    bufs.copy_(torch.from_numpy(fill))
    base = (ctypes.c_void_p * world)(*[bufs[r].data_ptr() + 4 * GUARD for r in range(world)])
    recs, owners = [], []
    for s in range(world):
        o, r_ = device_plans(all_hist, bits, cap, [s])
        owners.append(torch.from_numpy(o[0]).cuda())
        recs.append(torch.from_numpy(r_[0]).cuda())
        kt, kp = keys_at(srcs[s], s % 4)
        check(L.b200sort_dist_partition_planned_i32(kp, srcs[s].size, bits, world, base, owners[s].data_ptr(),
                                                    recs[s].data_ptr(), src_hists[s].data_ptr(), workspace().ptr, 256,
                                                    stream_ptr()))
    torch.cuda.synchronize()
    everything = np.concatenate(srcs)
    dest = owner[dm.bins(everything, bits)]
    got_bufs = bufs.cpu().numpy()
    wsb, ws_ptr = radix_ws
    for r in range(world):
        w = f"{what} destination {r}"
        want = np.sort(everything[dest == r])
        m = want.size
        assert parse_record(recs[r].cpu().numpy(), world)["m"] == m, w
        row = got_bufs[r]
        assert (row[:GUARD] == fill[r, :GUARD]).all() and (row[GUARD + m:] == fill[r, GUARD + m:]).all(), \
            w + ": receive buffer written outside its first m words"
        assert np.sort(row[GUARD:GUARD + m]).tobytes() == want.tobytes(), w + ": received keys"
        mine = torch.stack([h.view(world, 1024)[r] for h in src_hists]).sum(0).to(torch.int32).contiguous()
        assert int(mine[768:].abs().sum().item()) == 0, w + ": row 3 counted at the source"
        mine[768:] = recs[r].view(torch.int32)[PLAN_TOP_OFFSET // 4:PLAN_TOP_OFFSET // 4 + 256]
        # checked before the sort uses it: a wrong histogram would misplace keys, and stale counts could overrun
        assert (mine.cpu().numpy().astype(np.uint64).reshape(4, 256) == oracle.digit_histograms(want)).all(), \
            w + ": summed source histograms + top_hist"
        for d_hist in (None, mine.data_ptr()):
            out = torch.full((cap,), -9, dtype=torch.int32, device="cuda")
            tmp = torch.empty_like(out)
            check(L.b200sort_radix_copy_devn_i32(bufs[r].data_ptr() + 4 * GUARD, out.data_ptr(), tmp.data_ptr(), cap,
                                                 recs[r].data_ptr() + PLAN_M_OFFSET, d_hist, ws_ptr, wsb,
                                                 stream_ptr()))
            torch.cuda.synchronize()
            assert out.cpu().numpy()[:m].tobytes() == want.tobytes(), f"{w} sorted, d_hist={d_hist is not None}"


@pytest.mark.parametrize("radix_shape", [0, 3])
@pytest.mark.parametrize("world", [3, 16])
@pytest.mark.parametrize("bits", [8, 9, 12, 14])
def test_sync_free_path_with_source_histograms(bits, world, radix_shape):
    """Two rounds on the same buffers, as DistSorter reuses them: every source sends keys, then source 1 sends
    none.  In the second round source 1's histograms must hold zeros, not the first round's counts."""
    import torch
    L = lib()
    if radix_shape >= L.b200sort_radix_num_variants():
        pytest.skip("shape not compiled")
    for dist_name in ("uniform", "skewed90"):
        rounds = [[datagen.make(dist_name, 20000 + 311 * s, seed=200 + s) for s in range(world)]]
        rounds.append([k[:0] if s == 1 else k for s, k in enumerate(rounds[0])])
        most = max(int(dm.plans(np.stack([dm.histogram(k, bits) for k in srcs]))[0]["recv"].max()) for srcs in rounds)
        cap = (most + 64 + 3) // 4 * 4                  # keeps every buffer row 16-byte aligned
        bufs = torch.empty((world, cap + 2 * GUARD), dtype=torch.int32, device="cuda")
        src_hists = [torch.full((world * 1024,), -1, dtype=torch.int32, device="cuda") for _ in range(world)]
        nb = L.b200sort_workspace_bytes(cap, ALGO_RADIX)
        sws, sws_ptr = _aligned(nb, 0)
        check(L.b200sort_radix_set_variant(radix_shape))
        try:
            for i, srcs in enumerate(rounds):
                sync_free_round(srcs, bits, bufs, src_hists, (nb, sws_ptr), f"{dist_name} bits={bits} world={world} "
                                f"radix shape {radix_shape} round {i + 1}{', source 1 empty' if i else ''}")
        finally:
            L.b200sort_radix_set_variant(0)


# ---- the MSD histogram --------------------------------------------------------------------------------------------
HIST_SIZES = (0, 1, 2, 3, 4, 5, 7, (1 << 20) + 3)


@pytest.mark.parametrize("bits", range(4, 15))
def test_msd_histogram_every_bin_width(bits):
    """Keys at word offsets 0-3 (every head/body/tail split of the 128-bit loads) in a guarded buffer; the histogram
    in a guarded buffer that starts as canary words (it is overwritten, also for n = 0)."""
    import torch
    L = lib()
    nbins = 1 << bits
    for n in HIST_SIZES:
        keys = datagen.uniform(n, seed=n + bits)
        keys[::7] = datagen.edge_mix(keys[::7].size, seed=n)
        want = dm.histogram(keys, bits)
        for koff in range(4):
            what = f"bits={bits} n={n} keys at word {koff}"
            gk = dp.guarded(n, koff, salt=1)
            full = gk.fill.copy()
            full[gk.start:gk.end] = keys.view(np.uint32)
            tk = device_words(full)
            gh = dp.guarded(nbins, 0, itemsize=8, salt=2)
            th = device_words(gh.fill)
            check(L.b200sort_dist_histogram_i32(tk.data_ptr() + 4 * gk.start, n, bits, th.data_ptr() + 4 * gh.start,
                                                stream_ptr()))
            torch.cuda.synchronize()
            hk = tk.cpu().numpy().view(np.uint32)
            assert hk.tobytes() == full.tobytes(), what + ": keys buffer changed"
            h = th.cpu().numpy().view(np.uint32)
            gh.check(h, what + " histogram")
            got = h[gh.start:gh.end].view(np.uint64)
            if not (got == want).all():
                b = int(np.flatnonzero(got != want)[0])
                raise AssertionError(f"{what}: bin {b} = {got[b]}, numpy {want[b]}")


# ---- the planned entry points reject bad arguments before any device work -----------------------------------------
def test_planned_entry_points_reject_bad_arguments():
    """Every buffer is sized for the largest call the arguments could claim (world 17, bits 15), and the partition's
    record has its error flag set, so a check that let a call through could write nothing out of place; the test
    then sees the status, a launch, or a changed buffer."""
    import torch
    L = lib()
    check(L.b200sort_device_check())
    world, bits, n = 4, 8, 4096
    d_all = torch.ones(17 << 15, dtype=torch.int64, device="cuda")
    owner = torch.zeros(1 << 15, dtype=torch.int32, device="cuda")
    plan_rec = torch.full((PLAN_BYTES // 8,), -1, dtype=torch.int64, device="cuda")
    ws = workspace()
    ws_before = ws.t.cpu()
    need = L.b200sort_dist_workspace_bytes(0, bits)
    keys = torch.from_numpy(datagen.uniform(n, 9)).cuda()
    plans = dm.plans(np.stack([dm.histogram(k, bits) for k in sources(16, 64, "uniform")]))
    reg = Regions(plans, salt=11)
    err_rec = record(plans[0], reg.off[0], error=1)
    src_hist = torch.full((17 * 1024,), -1, dtype=torch.int32, device="cuda")

    def table(r=None, shift=0):                         # 17 receive bases; base r moved by `shift` bytes
        t = (ctypes.c_void_p * 17)(*reg.bases, reg.bases[0])
        if r is not None:
            t[r] = t[r] + shift
        return t
    base, shifted, last = table(), table(2, 4), table(world - 1, 8)

    def plan(bits=bits, world=world, rank=0, rec=plan_rec.data_ptr(), wsp=ws.ptr, wsb=need, hist=d_all.data_ptr(),
             own=owner.data_ptr()):
        return L.b200sort_dist_plan_device(hist, world, rank, bits, 1 << 40, own, rec, wsp, wsb, stream_ptr())

    def part(bits=bits, world=world, rec=err_rec.data_ptr(), table=base, wsp=ws.ptr, wsb=256, sh=None,
             own=owner.data_ptr()):
        return L.b200sort_dist_partition_planned_i32(keys.data_ptr(), n, bits, world, table, own, rec, sh, wsp, wsb,
                                                     stream_ptr())

    cases = [
        ("plan bits=3", lambda: plan(bits=3), INVALID), ("plan bits=15", lambda: plan(bits=15), INVALID),
        ("plan world=0", lambda: plan(world=0), INVALID), ("plan world=17", lambda: plan(world=17), INVALID),
        ("plan rank=world", lambda: plan(rank=world), INVALID), ("plan rank=-1", lambda: plan(rank=-1), INVALID),
        ("plan NULL plan", lambda: plan(rec=None), INVALID), ("plan NULL counts", lambda: plan(hist=None), INVALID),
        ("plan NULL owner", lambda: plan(own=None), INVALID),
        ("plan NULL workspace", lambda: plan(wsp=None), WORKSPACE),
        ("plan workspace one byte short", lambda: plan(wsb=need - 1), WORKSPACE),
        ("plan bits=14 workspace of bits=8", lambda: plan(bits=14), WORKSPACE),
        ("partition bits=3", lambda: part(bits=3), INVALID), ("partition bits=15", lambda: part(bits=15), INVALID),
        ("partition world=0", lambda: part(world=0), INVALID), ("partition world=17", lambda: part(world=17), INVALID),
        ("partition NULL plan", lambda: part(rec=None), INVALID),
        ("partition NULL table", lambda: part(table=None), INVALID),
        ("partition NULL owner", lambda: part(own=None), INVALID),
        ("partition base 2 at +4 bytes", lambda: part(table=shifted), INVALID),
        ("partition last base at +8 bytes", lambda: part(table=last), INVALID),
        ("partition NULL workspace", lambda: part(wsp=None), WORKSPACE),
        ("partition workspace of 255 bytes", lambda: part(wsb=255), WORKSPACE),
    ] + [(f"partition d_src_hist with bits={b}", functools.partial(part, bits=b, sh=src_hist.data_ptr()), INVALID)
         for b in (4, 5, 6, 7)]
    for what, call, want in cases:
        L.b200sort_launch_count_reset()
        st = call()
        assert st == want, f"{what}: status {st}, want {want}"
        assert L.b200sort_launch_count() == 0, f"{what}: launched a kernel"
    torch.cuda.synchronize()
    assert (plan_rec.cpu().numpy() == -1).all(), "a rejected plan call wrote the record"
    assert (owner.cpu().numpy() == 0).all(), "a rejected call wrote the owner table"
    assert torch.equal(ws.t.cpu(), ws_before), "a rejected call wrote the workspace"
    assert (src_hist.cpu().numpy() == -1).all(), "a rejected call wrote the source histograms"
    reg.assert_unchanged("rejected partition calls")
    # the same calls with good arguments go through: one launch each, and the partition, whose record carries the
    # error flag, only clears the histograms
    for what, call in (("plan", plan), ("partition bits=8 with d_src_hist", lambda: part(sh=src_hist.data_ptr()))):
        L.b200sort_launch_count_reset()
        check(call())
        assert L.b200sort_launch_count() == 1, what
    torch.cuda.synchronize()
    assert (src_hist.cpu().numpy()[:world * 1024] == 0).all() and (src_hist.cpu().numpy()[world * 1024:] == -1).all()
    reg.assert_unchanged("partition with the error flag")
