"""The references of tests/test_largest_sizes_gpu.py checked without a GPU, at small n and in small chunks.

Every closed form (construction D and T, 1-D and segmented) must equal the numpy stable argsort of tests/key_orders*.py,
every checker must accept that reference, and every checker must reject each way a sort can be subtly wrong: two
equal-key values swapped, the last element left where the input had it, indices wrapped modulo a power of two, a key
replaced by its neighbour, a segment left unsorted, a segment's keys moved into the next segment.  This is what makes a
pass of the 2^30 cases mean something."""
import numpy as np
import pytest
import torch

import large_refs as R

SIZES = [4099, 1 << 12, 3 * (1 << 10) + 7]
ORDERS = [(kt, d) for kt in sorted(R.BITS) for d in (0, 1)]
ORDER_IDS = [f"{R.NAMES[kt]}_{'desc' if d else 'asc'}" for kt, d in ORDERS]
CH = 1000                                  # chunks much smaller than n: chunk edges are crossed everywhere
T = 3


def np_keys(t, kt):
    """A CPU tensor of keys as numpy, in the dtype of tests/key_orders*.py (bfloat16 as its uint16 patterns)."""
    return R.ints(t, kt).numpy().view(R.KEY_ORDERS[kt].DTYPES[kt])


def np_order(keys, kt, desc, offsets=None):
    """Stable argsort of the images (per segment when offsets are given)."""
    img = R.KEY_ORDERS[kt].image(keys, kt, desc)
    if offsets is None:
        return np.argsort(img, kind="stable")
    seg = np.repeat(np.arange(offsets.size - 1), np.diff(offsets))
    return np.lexsort((img, seg))


def rejects(fn, *args, **kw):
    with pytest.raises(AssertionError):
        fn(*args, **kw)


def random_keys(n, kt, seed):
    """Random bit patterns with -0.0, +0.0 and NaNs of both signs planted."""
    b = R.BITS[kt]
    g = torch.Generator().manual_seed(seed)
    w = torch.randint(-(1 << 62), 1 << 62, (n,), dtype=torch.int64, generator=g) * 2 + torch.randint(0, 2, (n,), generator=g)
    w = w.to(R.int_dtype(torch, kt)) if b < 64 else w
    top = -(1 << (b - 1))
    w[:4] = torch.tensor([top, 0, -1, (1 << (b - 1)) - 1], dtype=w.dtype)  # -0.0, +0.0, -NaN, +NaN patterns
    return w.view(R.torch_dtype(torch, kt))


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kt,desc", ORDERS, ids=ORDER_IDS)
def test_images_and_inverse_match_key_orders(n, kt, desc):
    b = R.BITS[kt]
    keys = random_keys(n, kt, n + kt)
    img_np = R.KEY_ORDERS[kt].image(np_keys(keys, kt), kt, desc)
    centred = (img_np ^ img_np.dtype.type(1 << (b - 1))).view({16: np.int16, 32: np.int32, 64: np.int64}[b])
    img = R.image(keys, kt, desc)
    assert img.dtype == torch.int64 and np.array_equal(img.numpy(), centred.astype(np.int64))
    assert torch.equal(R.ints(R.inverse(img, kt, desc), kt), R.ints(keys, kt))


@pytest.mark.parametrize("n", SIZES)
def test_g_spreads_every_digit_and_straddles_the_top_bit(n):
    for b in (16, 32, 64):
        for t in (0, T):
            g = R.groups(n, t)
            if g > 1 << b:
                continue
            q = torch.arange(g, dtype=torch.int64)
            f = R.G(q, g, b)
            assert bool((f[1:] > f[:-1]).all()) and int(f[0]) >= -(1 << (b - 1)) and int(f[-1]) < 1 << (b - 1)
            assert int(f[0]) < 0 <= int(f[-1]), "images straddle the top bit"
            u = f ^ -(1 << (b - 1))                                   # the image's bits (two's complement)
            for d in range(b // 8):
                assert ((u >> (8 * d)) & 255).unique().numel() > 1, f"b={b} digit {d} constant"
    # the top of the range: 2^30 keys of 32 and 64 bits, 2^16 values of 16 bits
    assert R.spread(1 << 30, 32) == 3 and R.spread(1 << 16, 16) == 1 and R.spread(1 << 30, 64) == (1 << 34) - 1
    for g, b in (((1 << 30), 32), ((1 << 30) - 3, 32), ((1 << 29) + 1, 64), ((1 << 30), 64), (1 << 16, 16)):
        ends = R.G(torch.tensor([0, g - 1]), g, b)
        assert -(1 << (b - 1)) <= int(ends[0]) < 0 <= int(ends[1]) < 1 << (b - 1)


@pytest.mark.parametrize("n", SIZES + [1 << 30, (1 << 30) - 3, (1 << 29) + 1])
def test_permutation_and_inverse(n):
    a = R.multiplier(n)
    assert a < 1 << 31 and np.gcd(a, n) == 1
    m = min(n, 1 << 16)
    i = torch.cat([torch.arange(m // 2), torch.arange(n - m // 2, n)]).to(torch.int64)
    assert torch.equal(R.perm_inv(R.perm(i, n, a), n, a), i)
    if n < 1 << 20:
        p = R.perm(torch.arange(n, dtype=torch.int64), n, a)
        assert torch.equal(torch.sort(p).values, torch.arange(n))


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kt,desc", ORDERS, ids=ORDER_IDS)
def test_closed_forms_equal_numpy(n, kt, desc):
    for t in (None, T):
        keys, case = R.build(n, kt, desc, t, "cpu", chunk=CH)
        k = np_keys(keys, kt)
        p = np_order(k, kt, desc)
        out = torch.from_numpy(R.ints(keys, kt).numpy()[p].copy()).view(keys.dtype)
        v = torch.from_numpy(p.astype(np.int64))
        want = torch.cat([R.expected_keys(case, s, min(n, s + CH), "cpu") for s in range(0, n, CH)])
        assert torch.equal(R.ints(want, kt), R.ints(out, kt)), f"t={t}: closed-form keys differ from numpy"
        R.check_keys(out, case, "numpy", chunk=CH)
        R.check_pairs(keys, out, v, kt, desc, "numpy", chunk=CH)
        R.check_pairs(keys, out, v.to(torch.int32), kt, desc, "numpy", chunk=CH)
        if t is None:
            want_v = R.perm_inv(torch.arange(n, dtype=torch.int64), n, case.a)
            assert torch.equal(want_v, v), "closed-form values differ from numpy's stable argsort"
            R.check_values_d(v, case, "numpy", chunk=CH)
            assert R.image(keys, kt, desc).unique().numel() == n, "construction D has distinct keys"
        else:
            assert R.image(keys, kt, desc).unique().numel() == case.g and case.g < n


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kt,desc", ORDERS, ids=ORDER_IDS)
def test_random_data_checker_against_numpy(n, kt, desc):
    keys = random_keys(n, kt, 7 * n + kt + desc)
    out = torch.from_numpy(R.ints(keys, kt).numpy()[np_order(np_keys(keys, kt), kt, desc)].copy()).view(keys.dtype)
    R.check_sorted_like_torch(out, keys, kt, desc, "numpy", chunk=CH)
    bad = out.clone()
    j = next(j for j in range(CH - 1, n - 1) if R.ints(bad, kt)[j] != R.ints(bad, kt)[j + 1])
    bad[j] = bad[j + 1]
    rejects(R.check_sorted_like_torch, bad, keys, kt, desc, chunk=CH)
    bad = out.clone()
    bad[-1] = keys[-1]
    if int(R.ints(bad, kt)[-1]) != int(R.ints(out, kt)[-1]):
        rejects(R.check_sorted_like_torch, bad, keys, kt, desc, chunk=CH)


def _sorted_1d(n, kt, desc, t):
    keys, case = R.build(n, kt, desc, t, "cpu", chunk=CH)
    p = np_order(np_keys(keys, kt), kt, desc)
    out = torch.from_numpy(R.ints(keys, kt).numpy()[p].copy()).view(keys.dtype)
    return keys, case, out, torch.from_numpy(p.astype(np.int64))


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kt,desc", ORDERS, ids=ORDER_IDS)
def test_1d_checkers_reject_corrupted_outputs(n, kt, desc):
    # two equal-key values swapped (construction T)
    keys, case, out, v = _sorted_1d(n, kt, desc, T)
    bad = v.clone(); bad[[CH, CH + 1]] = bad[[CH + 1, CH]]
    assert int(R.ints(out, kt)[CH]) == int(R.ints(out, kt)[CH + 1])
    rejects(R.check_pairs, keys, out, bad, kt, desc, chunk=CH)
    # construction D: the last element left as the input had it, wrapped indices, a key replaced by its neighbour
    keys, case, out, v = _sorted_1d(n, kt, desc, None)
    assert int(R.ints(keys, kt)[-1]) != int(R.ints(out, kt)[-1])
    bad_k, bad_v = out.clone(), v.clone()
    bad_k[-1], bad_v[-1] = keys[-1], n - 1
    rejects(R.check_keys, bad_k, case, chunk=CH)
    rejects(R.check_values_d, bad_v, case, chunk=CH)
    rejects(R.check_pairs, keys, bad_k, bad_v, kt, desc, chunk=CH)
    k = (n - 1).bit_length() - 1                                      # 2^k < n
    wrapped = v % (1 << k)
    rejects(R.check_values_d, wrapped, case, chunk=CH)
    rejects(R.check_permutation, wrapped, n, chunk=CH)
    rejects(R.check_pairs, keys, out, wrapped, kt, desc, chunk=CH)
    for j in (0, CH - 1, n - 2):                                      # at the front, across a chunk edge, at the end
        bad_k = out.clone(); bad_k[j] = bad_k[j + 1]
        rejects(R.check_keys, bad_k, case, chunk=CH)
        rejects(R.check_pairs, keys, bad_k, v, kt, desc, chunk=CH)
    # the all-skipped shape: equal keys must keep 0..n-1
    rejects(R.check_pairs, torch.zeros(n, dtype=keys.dtype), torch.zeros(n, dtype=keys.dtype),
            torch.arange(n).flip(0), kt, desc, chunk=CH)


def ragged(n, seed):
    """Offsets summing to n: empty segments, length 1, short and long ones, and two adjacent of different length."""
    rng = np.random.default_rng(seed)
    lens = [0, 1, 0, 0, 2, 1, 129, 300, 0, 1025, 57]
    while sum(lens) < n:
        lens.append(int(rng.choice([0, 1, 3, 31, 128, 129, 700, 1500])))
    lens[-1] -= sum(lens) - n
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kt,desc", ORDERS, ids=ORDER_IDS)
def test_segmented_closed_forms_equal_numpy(n, kt, desc):
    offs_np = ragged(n, n + kt)
    for dtype in (torch.int32, torch.int64):
        offs = torch.from_numpy(offs_np).to(dtype)
        for t in (None, T):
            keys, case = R.build_segmented(offs, kt, desc, t, chunk=CH)
            assert case.t == (t or 0) and case.g == R.groups(int(np.diff(offs_np).max()), case.t)
            p = np_order(np_keys(keys, kt), kt, desc, offs_np)
            out = torch.from_numpy(R.ints(keys, kt).numpy()[p].copy()).view(keys.dtype)
            loc = R.local_positions(offs, chunk=CH)
            assert torch.equal(loc.to(torch.int64), torch.arange(n) - torch.from_numpy(
                np.repeat(offs_np[:-1], np.diff(offs_np))))
            v = loc[torch.from_numpy(p)]
            R.check_seg_keys(out, offs, case, "numpy", chunk=CH)
            R.check_seg_pairs(keys, out, v, offs, kt, desc, "numpy", chunk=CH)
            R.check_seg_pairs(keys, out, v.to(torch.int64), offs, kt, desc, "numpy", chunk=CH)


def test_segment_lengths_pick_the_shift():
    assert R.shift_for(1 << 30, 16) == 14 and R.shift_for((1 << 30) - 3, 16) == 14 and R.shift_for(1 << 16, 16) == 0
    assert R.shift_for((1 << 16) + 1, 16) == 1 and R.shift_for(1 << 30, 32) == 0 and R.shift_for(1 << 17, 16) == 1


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kt,desc", ORDERS, ids=ORDER_IDS)
def test_segmented_checkers_reject_corrupted_outputs(n, kt, desc):
    offs_np = ragged(n, 3 * n + kt)
    offs = torch.from_numpy(offs_np).to(torch.int32)
    lens = np.diff(offs_np)
    keys, case = R.build_segmented(offs, kt, desc, T, chunk=CH)
    p = np_order(np_keys(keys, kt), kt, desc, offs_np)
    out = torch.from_numpy(R.ints(keys, kt).numpy()[p].copy()).view(keys.dtype)
    v = R.local_positions(offs, chunk=CH)[torch.from_numpy(p)]
    R.check_seg_pairs(keys, out, v, offs, kt, desc, chunk=CH)
    # two equal-key values swapped
    o = int(offs_np[np.flatnonzero(lens >= 2 << T)[0]])
    bad = v.clone(); bad[[o, o + 1]] = bad[[o + 1, o]]
    assert int(R.ints(out, kt)[o]) == int(R.ints(out, kt)[o + 1])
    rejects(R.check_seg_pairs, keys, out, bad, offs, kt, desc, chunk=CH)
    # the last element left as it was in the input
    bad_k, bad_v = out.clone(), v.clone()
    bad_k[-1], bad_v[-1] = keys[-1], lens[-1] - 1
    if int(R.ints(bad_k, kt)[-1]) != int(R.ints(out, kt)[-1]):
        rejects(R.check_seg_keys, bad_k, offs, case, chunk=CH)
        rejects(R.check_seg_pairs, keys, bad_k, bad_v, offs, kt, desc, chunk=CH)
    # indices wrapped modulo 2^k, 2^k below the longest segment
    k = (int(lens.max()) - 1).bit_length() - 1
    rejects(R.check_seg_pairs, keys, out, v % (1 << k), offs, kt, desc, chunk=CH)
    # one key replaced by its neighbour (a different one)
    j = next(j for j in range(CH - 1, n - 1) if R.ints(out, kt)[j] != R.ints(out, kt)[j + 1])
    bad_k = out.clone(); bad_k[j] = bad_k[j + 1]
    rejects(R.check_seg_keys, bad_k, offs, case, chunk=CH)
    rejects(R.check_seg_pairs, keys, bad_k, v, offs, kt, desc, chunk=CH)
    # one segment left unsorted: the longest one keeps its input keys and positions
    s = int(np.argmax(lens))
    a, b = int(offs_np[s]), int(offs_np[s + 1])
    bad_k, bad_v = out.clone(), v.clone()
    bad_k[a:b], bad_v[a:b] = keys[a:b], torch.arange(b - a, dtype=v.dtype)
    rejects(R.check_seg_keys, bad_k, offs, case, chunk=CH)
    rejects(R.check_seg_pairs, keys, bad_k, bad_v, offs, kt, desc, chunk=CH)
    # one segment's keys moved into the next segment: two adjacent segments of different lengths, each holding more
    # than one group of equal keys
    s = next(s for s in range(lens.size - 1) if 2 << T < lens[s] != lens[s + 1] > 2 << T)
    a, b = int(offs_np[s]), int(offs_np[s + 2])
    bad_k, bad_v = out.clone(), v.clone()
    bad_k[a:b], bad_v[a:b] = out[a:b].roll(int(lens[s])), v[a:b].roll(int(lens[s]))
    rejects(R.check_seg_keys, bad_k, offs, case, chunk=CH)
    rejects(R.check_seg_pairs, keys, bad_k, bad_v, offs, kt, desc, chunk=CH)
    # a whole-array sort that ignores the boundaries
    p_all = np_order(np_keys(keys, kt), kt, desc)
    glob = torch.from_numpy(R.ints(keys, kt).numpy()[p_all].copy()).view(keys.dtype)
    rejects(R.check_seg_keys, glob, offs, case, chunk=CH)
