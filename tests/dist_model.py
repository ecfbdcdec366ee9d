"""numpy model of the multi-GPU path's planner and partition (test infrastructure only, numpy only).

Written from the rules include/b200sort.h states, not from the C code, so that the host planner
(b200sort_dist_plan), the device planner (b200sort_dist_plan_device) and the partition kernel all have a
reference that is not the function they share:

- a key's bin is the top `bits` bits of key ^ 0x80000000;
- rank k's range ends at the first bin boundary whose cumulative count reaches k/world of all keys, moved back
  one bin when more than half of the bin that straddles the target lies beyond it (never back to a boundary with
  no keys before it);
- every source rank's block sits in a destination's receive buffer after the blocks of the lower source ranks.
"""
from __future__ import annotations

import bisect
from fractions import Fraction

import numpy as np


def images(keys: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(keys).view(np.uint32) ^ np.uint32(0x80000000)


def bins(keys: np.ndarray, bits: int) -> np.ndarray:
    return (images(keys) >> np.uint32(32 - bits)).astype(np.int64)


def histogram(keys: np.ndarray, bits: int) -> np.ndarray:
    return np.bincount(bins(keys, bits), minlength=1 << bits).astype(np.uint64)


def boundaries(global_hist: np.ndarray, world: int) -> list:
    """bound[0..world]: rank k owns bins [bound[k], bound[k + 1])."""
    counts = [int(c) for c in global_hist]
    cum = [0]
    for c in counts:
        cum.append(cum[-1] + c)
    total, nbins = cum[-1], len(counts)
    bound = [0]
    for k in range(1, world):
        target = Fraction(total * k, world)
        b = bisect.bisect_left(cum, target)                              # first boundary with cum >= target
        # bin b - 1 straddles the target; it goes to rank k when more than half of it lies beyond the target
        if b > 0 and cum[b - 1] > 0 and Fraction(cum[b] + cum[b - 1], 2) > target:
            b -= 1
        bound.append(b)
    bound.append(nbins)
    return bound


def plans(all_hist: np.ndarray, cap: int | None = None) -> list:
    """The plan of every rank over all_hist[world][nbins]: owner, recv, send, offs (uint64[world]), m, error."""
    all_hist = np.asarray(all_hist, dtype=np.uint64)
    world, nbins = all_hist.shape
    bound = boundaries(all_hist.sum(axis=0, dtype=np.uint64), world)
    owner = np.zeros(nbins, dtype=np.int32)
    for k in range(world):
        owner[bound[k]:bound[k + 1]] = k
    per_dest = np.zeros((world, world), dtype=np.uint64)                  # [source][destination]
    for r in range(world):
        per_dest[:, r] = all_hist[:, bound[r]:bound[r + 1]].sum(axis=1, dtype=np.uint64)
    recv = per_dest.sum(axis=0, dtype=np.uint64)
    error = int(cap is not None and int(recv.max()) > cap)
    return [{"owner": owner, "bound": bound, "recv": recv, "send": per_dest[rank].copy(),
             "offs": per_dest[:rank].sum(axis=0, dtype=np.uint64), "m": int(recv[rank]), "error": error}
            for rank in range(world)]


def top_hist_from_bins(all_hist: np.ndarray, owner: np.ndarray, rank: int, bits: int) -> np.ndarray:
    """Top-byte histogram of what `rank` owns, from bin counts (bits >= 8: a bin lies inside one top byte)."""
    assert bits >= 8
    g = np.asarray(all_hist, dtype=np.uint64).sum(axis=0, dtype=np.uint64)
    out = np.zeros(256, dtype=np.uint64)
    mine = np.flatnonzero(owner == rank)
    np.add.at(out, mine >> (bits - 8), g[mine])
    return out


def top_byte_histogram(keys: np.ndarray) -> np.ndarray:
    return np.bincount((images(keys) >> np.uint32(24)).astype(np.int64), minlength=256).astype(np.uint64)


def digit_rows(keys: np.ndarray) -> np.ndarray:
    """[4][256] histograms of bytes 0..2 of key ^ 0x80000000 and a zero row 3: what the partition counts per
    destination at the source."""
    img = images(keys)
    out = np.zeros((4, 256), dtype=np.uint64)
    for p in range(3):
        out[p] = np.bincount(((img >> np.uint32(8 * p)) & np.uint32(255)).astype(np.int64), minlength=256)
    return out


def synthetic_histograms(kind: str, world: int, bits: int, seed: int) -> np.ndarray:
    """all_hist[world][2^bits] without keys behind it:
      max_totals   every rank holds 2^30 keys (the largest n), so the global count reaches world * 2^30;
      empty_ranks  the odd source ranks hold nothing, and every key sits in two bins, so most ranks own nothing;
      one_bin      every key of every rank in one bin;
      spiky        up to 2^30 keys per rank in a few dozen heavy bins, so most targets fall inside a heavy bin;
      zero         no keys at all."""
    rng = np.random.default_rng(seed)
    nbins = 1 << bits
    h = np.zeros((world, nbins), dtype=np.uint64)
    if kind == "max_totals":
        for r in range(world):
            p = rng.dirichlet(np.full(nbins, 0.3))
            h[r] = rng.multinomial(1 << 30, p)
    elif kind == "empty_ranks":
        pick = rng.choice(nbins, 2, replace=False)
        for r in range(0, world, 2):
            h[r, pick] = rng.integers(1, 1 << 20, 2)
    elif kind == "one_bin":
        b = int(rng.integers(0, nbins))
        h[:, b] = (1 << 30) - rng.integers(0, 3, world)
    elif kind == "spiky":
        pick = rng.choice(nbins, min(nbins, 40), replace=False)
        for r in range(world):
            h[r, pick] = rng.multinomial(int(rng.integers(1, 1 << 30)), rng.dirichlet(np.full(pick.size, 0.5)))
    else:
        assert kind == "zero", kind
    return h


SYNTHETIC = ("max_totals", "empty_ranks", "one_bin", "spiky", "zero")
