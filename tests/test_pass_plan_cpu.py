"""The generators of tests/digit_patterns.py do what they promise (no GPU needed): the pass-plan tests on the GPU
(tests/test_pass_plan_gpu.py) reach the skipped-pass sets, near-constant and hot digits they name only if so."""
import itertools

import numpy as np
import pytest

import digit_patterns as dp
import key_orders as ko32
import key_orders64 as ko64

ORDERS32 = ko32.ORDERS
ORDERS64 = ko64.ORDERS
ALL_ORDERS = ORDERS32 + ORDERS64
ORDER_IDS = [f"{(ko64 if kt in ko64.DTYPES else ko32).NAMES[kt]}_{'desc' if d else 'asc'}" for kt, d in ALL_ORDERS]


def _image(keys, order):
    kt, desc = order
    return dp.orders_module(kt).image(keys, kt, desc)


def _subsets(passes):
    return [frozenset(s) for r in range(passes + 1) for s in itertools.combinations(range(passes), r)]


@pytest.mark.parametrize("order", ALL_ORDERS, ids=ORDER_IDS)
def test_image_of_inverse_is_the_identity(order):
    kt, desc = order
    m = dp.orders_module(kt)
    w = dp.random_images(4099, kt, np.random.default_rng(kt * 2 + desc))
    top = np.iinfo(w.dtype).max
    edges = np.array([0, 1, top, top - 1, top >> 1, (top >> 1) + 1], dtype=w.dtype)
    for img in (w, edges):
        keys = m.inverse(img, kt, desc)
        assert keys.dtype == m.DTYPES[kt]
        assert m.image(keys, kt, desc).tobytes() == img.tobytes()


@pytest.mark.parametrize("order", ALL_ORDERS, ids=ORDER_IDS)
def test_constant_digits_give_exactly_the_set(order):
    kt, _ = order
    passes = dp.passes_of(kt)
    n = 3 * 4096 + 17
    for i, S in enumerate(_subsets(passes)):
        for consts in (None, 0, 255):
            keys = dp.with_constant_digits(n, S, order, seed=i, consts=consts)
            img = _image(keys, order)
            assert dp.constant_passes(img, passes) == S, (sorted(S), consts)
            for p in S:
                if consts is not None:
                    assert int(dp.digit(img[:1], p)[0]) == consts
    # two keys are enough for every set, and the same seed gives the same keys
    for S in _subsets(passes):
        assert dp.constant_passes(_image(dp.with_constant_digits(2, S, order, 5), order), passes) == S
    a, b = (dp.with_constant_digits(1000, {1}, order, 3) for _ in range(2))
    assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("order", [(ko32.KEY_I32, 0), (ko32.KEY_F32, 1), (ko64.KEY_I64, 0), (ko64.KEY_F64, 1)],
                         ids=["i32_asc", "f32_desc", "i64_asc", "f64_desc"])
def test_near_constant_digit_must_be_sorted_by_that_pass(order):
    kt, desc = order
    passes = dp.passes_of(kt)
    n, tile = 3 * 4096 + 17, 4096
    for p in range(passes):
        for where in dp.WHERE:
            keys, i, c = dp.near_constant(n, p, where, order, tile=tile, seed=p)
            img = _image(keys, order)
            d = dp.digit(img, p)
            assert int((d == c).sum()) == n - 1 and int(d[i]) != c
            assert i == {"first": 0, "last": n - 1, "last_tile": 3 * 4096}[where]
            assert p not in dp.constant_passes(img, passes)
            # a sort that skipped pass p (stable by the other digits only) gives a different order
            full = np.argsort(img, kind="stable")
            skipped = np.argsort(dp.set_digit(img, p, 0), kind="stable")
            assert not np.array_equal(full, skipped), (p, where)


@pytest.mark.parametrize("order", [(ko32.KEY_I32, 0), (ko32.KEY_U32, 1), (ko64.KEY_U64, 0)],
                         ids=["i32_asc", "u32_desc", "u64_asc"])
def test_hot_digit_counts(order):
    kt, _ = order
    for n in (8191, 8193, 33 * 16384 + 4099):
        for p in range(dp.passes_of(kt)):
            for value in (0, 0x80, 255):
                for fraction in dp.HOT_FRACTIONS:
                    img = _image(dp.hot_digit(n, p, value, fraction, order, seed=p + value), order)
                    want = dp.hot_count(n, fraction)
                    counts = np.bincount(dp.digit(img, p), minlength=256)
                    assert counts[value] == want and counts[value] * 8 > n
                    assert counts.sum() - counts[value] == n - want
    assert dp.hot_count(8192, "eighth_plus") * 8 > 8192 and (dp.hot_count(8192, "eighth_plus") - 1) * 8 == 8192


def test_locally_hot_runs_without_a_globally_hot_digit():
    for kt in (ko32.KEY_I32, ko64.KEY_I64):
        for n in (8191, 33 * 16384 + 4099):
            for p in range(dp.passes_of(kt)):
                img = _image(dp.locally_hot(n, p, (kt, 0), seed=p), (kt, 0))
                d = dp.digit(img, p)
                assert np.bincount(d, minlength=256).max() * 8 <= n
                runs = d[: n // 64 * 64].reshape(-1, 2, 32)
                assert bool((runs[:, 0, :] == runs[:, 0, :1]).all())          # every even run agrees
                assert not bool((runs[:, 1, :] == runs[:, 1, :1]).all())      # the odd runs do not


# 2-byte items: 16-bit words, 2, 6 and 14 bytes past a 16-byte boundary
@pytest.mark.parametrize("word_offset,itemsize", [(0, 4), (1, 4), (2, 4), (3, 4), (0, 8), (2, 8),
                                                  (0, 2), (1, 2), (3, 2), (7, 2)])
def test_guard_catches_a_changed_word_on_either_side(word_offset, itemsize):
    n = 1001
    g = dp.guarded(n, word_offset, itemsize=itemsize)
    word = min(itemsize, 4)
    assert g.fill.dtype.itemsize == word
    assert (g.start * word) % 16 == word_offset * word and (g.end - g.start) * word == n * itemsize
    assert (g.total * word) % 16 == 0
    assert g.total - g.end >= 16 and g.start >= 16
    buf = g.fill.copy()
    buf[g.start:g.end] = 0                                                     # the array itself may change
    g.check(buf)
    for k, side in ((g.start - 1, "before"), (0, "before"), (g.end, "after"), (g.total - 1, "after")):
        bad = buf.copy()
        bad[k] ^= 1
        with pytest.raises(AssertionError, match=f"guard word {side}"):
            g.check(bad, "test")
        if word == 2:                                                          # a byte of the word next to the array
            raw = buf.copy().view(np.uint8)
            raw[2 * k + 1] ^= 0x80
            with pytest.raises(AssertionError, match=f"guard word {side}"):
                g.check(raw, "test")
    assert len(np.unique(g.fill)) == g.total                                   # no two canary words alike
    assert dp.guarded(n, word_offset, itemsize=itemsize, salt=1).fill.tobytes() != g.fill.tobytes()


def test_guard_rejects_offsets_past_a_16_byte_boundary():
    for word_offset, itemsize in ((4, 4), (4, 8), (8, 2), (-1, 2)):
        with pytest.raises(AssertionError):
            dp.guarded(100, word_offset, itemsize=itemsize)
