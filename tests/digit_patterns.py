"""Key generators that steer the radix sorts' device-side pass plan, canary-guarded buffer layouts, and the guarded
device buffers and never-cleared workspace the GPU tests build from them (test infrastructure only; numpy, and torch
only inside DevBuf and Workspace).

The histogram kernel of every 1-D radix sort skips a pass when one digit value holds all n keys, picks the buffer
each executed pass reads and writes from the number of executed passes, and flags a pass as hot when one digit value
holds more than n/8 keys.  The host never sees that plan, so these generators build keys whose image digits
(tests/key_orders.py, tests/key_orders64.py) are constant, near-constant or hot in exactly the passes a test names.
Digit p of an image is bits [8p, 8p + 8): 4 passes for 32-bit keys, 8 for 64-bit keys.
"""
from __future__ import annotations

import numpy as np

import key_orders as ko32
import key_orders64 as ko64

HOT_FRACTIONS = ("eighth_plus", "half", "all_but_one")
WHERE = ("first", "last", "last_tile")


def orders_module(key_type: int):
    """key_orders for 32-bit key types, key_orders64 for 64-bit ones."""
    return ko64 if key_type in ko64.DTYPES else ko32


def passes_of(key_type: int) -> int:
    return 8 if key_type in ko64.DTYPES else 4


def _word(key_type: int):
    return np.uint64 if key_type in ko64.DTYPES else np.uint32


def digit(img: np.ndarray, p: int) -> np.ndarray:
    return ((img >> img.dtype.type(8 * p)) & img.dtype.type(255)).astype(np.uint32)


def set_digit(img: np.ndarray, p: int, d) -> np.ndarray:
    """img with digit p replaced by d (a scalar or an array broadcast against img), in a new array."""
    t = img.dtype.type
    d = np.asarray(d).astype(img.dtype)
    return (img & ~t(255 << (8 * p))) | (d << t(8 * p))


def constant_passes(img: np.ndarray, passes: int) -> set:
    """The passes whose digit takes one value over all of img (every pass for fewer than two keys)."""
    out = set()
    for p in range(passes):
        d = digit(img, p)
        if d.size == 0 or bool((d == d[0]).all()):
            out.add(p)
    return out


def random_images(n: int, key_type: int, rng: np.random.Generator) -> np.ndarray:
    w = _word(key_type)
    return rng.integers(0, np.iinfo(w).max, n, dtype=w, endpoint=True)


def keys_of(img: np.ndarray, order) -> np.ndarray:
    """The keys of `order` = (key_type, descending) whose images are img."""
    kt, desc = order
    return orders_module(kt).inverse(img, kt, desc)


def with_constant_digits(n: int, S, order, seed: int, consts=None) -> np.ndarray:
    """Keys of `order` whose image digits are constant in exactly the passes of S and take at least two values in
    every other pass (n >= 2 unless S holds every pass).

    consts: None = a random constant per pass; an int = that digit in every pass of S; a dict {pass: digit}."""
    kt, _ = order
    passes = passes_of(kt)
    S = set(S)
    assert S <= set(range(passes)), S
    rng = np.random.default_rng(seed)
    img = random_images(n, kt, rng)
    for p in range(passes):
        if p in S:
            c = (int(rng.integers(0, 256)) if consts is None else
                 consts if isinstance(consts, int) else consts[p])
            img = set_digit(img, p, c)
        elif n >= 2 and bool((digit(img, p) == digit(img, p)[0]).all()):
            img[1:2] = set_digit(img[1:2], p, digit(img[:1], p) ^ 1)
    got = constant_passes(img, passes)
    assert got == S or n < 2, (sorted(got), sorted(S))
    return keys_of(img, order)


def near_constant(n: int, p: int, where: str, order=(ko32.KEY_I32, 0), tile: int = 4096, seed: int = 0):
    """Keys of `order` whose digit p is one value c in every key but one.  Returns (keys, odd index, c).

    The odd key sits first, last, or at the start of the last tile of `tile` keys.  Its other digits are copied from a
    twin elsewhere in the array, and its digit p is chosen so that the sorted order of the two is the reverse of their
    input order: a sort that skipped pass p would keep them in input order and be wrong."""
    kt, _ = order
    assert 0 <= p < passes_of(kt) and n >= 3 and where in WHERE
    rng = np.random.default_rng(seed)
    img = random_images(n, kt, rng)
    c = int(rng.integers(1, 255))
    img = set_digit(img, p, c)
    i = {"first": 0, "last": n - 1, "last_tile": (n - 1) // tile * tile}[where]
    if i == 0:
        j, odd = int(rng.integers(1, n)), int(rng.integers(c + 1, 256))        # twin after it: the odd key goes after
    else:
        j, odd = int(rng.integers(0, i)), int(rng.integers(0, c))              # twin before it: the odd key goes before
    img[i] = set_digit(img[j:j + 1], p, odd)[0]
    return keys_of(img, order), i, c


def hot_count(n: int, fraction: str) -> int:
    """Keys that get the hot digit: just above n/8 (the plan's threshold is count * 8 > n), half, or all but one."""
    return {"eighth_plus": n // 8 + 1, "half": n // 2, "all_but_one": n - 1}[fraction]


def hot_digit(n: int, p: int, value: int, fraction: str, order=(ko32.KEY_I32, 0), seed: int = 0) -> np.ndarray:
    """Keys of `order` in which exactly hot_count(n, fraction) keys, at random positions, have digit `value` in pass p;
    the others have a random digit other than `value` there, and every other digit is random."""
    kt, _ = order
    rng = np.random.default_rng(seed)
    img = random_images(n, kt, rng)
    other = rng.integers(0, 255, n).astype(np.uint32)
    other = other + (other >= value)                                           # uniform over the 255 other values
    hot = np.zeros(n, bool)
    hot[rng.choice(n, hot_count(n, fraction), replace=False)] = True
    img = set_digit(img, p, np.where(hot, np.uint32(value), other))
    return keys_of(img, order)


def locally_hot(n: int, p: int, order=(ko32.KEY_I32, 0), seed: int = 0, run: int = 32) -> np.ndarray:
    """Keys of `order` in runs of `run` consecutive keys: even runs share one random digit in pass p (a whole warp's
    load agrees on it), odd runs are random.  No digit value holds more than n/8 keys overall."""
    kt, _ = order
    rng = np.random.default_rng(seed)
    img = random_images(n, kt, rng)
    d = digit(img, p)
    runs = (np.arange(n) // run)
    shared = rng.integers(0, 256, runs[-1] + 1 if n else 0).astype(np.uint32)
    d = np.where(runs % 2 == 0, shared[runs], d)
    return keys_of(set_digit(img, p, d), order)


def canary(words: int, salt: int = 0) -> np.ndarray:
    """A word pattern that differs from word to word (so a shifted or duplicated copy of it shows)."""
    i = np.arange(words, dtype=np.uint64) + np.uint64(salt * 7919)
    return ((i * np.uint64(0x9E3779B1)) ^ np.uint64(0xA5A5A5A5)).astype(np.uint32)


class Guarded:
    """Layout of a buffer of words that holds n items of `itemsize` bytes starting `word_offset` words past a
    16-byte boundary, with at least `guard_words` words on each side.  A word is 32 bits for items of 4 and 8 bytes
    and 16 bits for items of 2 bytes (2-byte keys may begin 2, 6 or 14 bytes past a boundary: word offsets 1, 3, 7).
    Whatever allocates the buffer (a 16-byte aligned numpy array or device tensor of `total` words of `self.dtype`)
    fills it with `self.fill` and puts the array at word `self.start`; `check` asserts that every word outside the
    array still holds its canary."""

    def __init__(self, n: int, word_offset: int, guard_words: int = 16, itemsize: int = 4, salt: int = 0):
        assert itemsize in (2, 4, 8)
        self.word = min(itemsize, 4)                                   # bytes per word
        self.dtype = np.uint16 if self.word == 2 else np.uint32
        line = 16 // self.word                                         # words per 16 bytes
        assert guard_words % line == 0 and 0 <= word_offset < line
        self.n, self.word_offset, self.itemsize = n, word_offset, itemsize
        self.start = guard_words + word_offset
        self.end = self.start + n * itemsize // self.word
        self.total = (self.end + guard_words + line - 1) // line * line
        self.fill = canary(self.total, salt).astype(self.dtype)      # 16-bit: i * odd stays distinct below 2^16 words

    def check(self, words: np.ndarray, what: str = "") -> None:
        words = np.ascontiguousarray(words).view(self.dtype)
        assert words.size == self.total, (words.size, self.total)
        for side, lo, hi in (("before", 0, self.start), ("after", self.end, self.total)):
            bad = np.flatnonzero(words[lo:hi] != self.fill[lo:hi])
            if bad.size:
                k = lo + int(bad[0])
                where = k - self.start if side == "before" else k - self.end
                w = 2 + 2 * self.word
                raise AssertionError(f"{what}: guard word {side} the array changed ({bad.size} words), first at "
                                     f"word {where:+d} from the array's {'start' if side == 'before' else 'end'}: "
                                     f"{int(words[k]):#0{w}x}, canary {int(self.fill[k]):#0{w}x}")


def guarded(n: int, word_offset: int, guard_words: int = 16, itemsize: int = 4, salt: int = 0) -> Guarded:
    return Guarded(n, word_offset, guard_words, itemsize, salt)


# ---- device buffers of the GPU tests (torch is imported only when one is made) ---------------------------------------
class DevBuf:
    """n items of `itemsize` bytes at `word_offset` words past a 16-byte boundary inside a canary-filled device buffer
    (Guarded)."""

    def __init__(self, n: int, word_offset: int, itemsize: int, salt: int):
        import torch
        self.g = guarded(n, word_offset, itemsize=itemsize, salt=salt)
        self.t = torch.empty(self.g.total, dtype=torch.int16 if self.g.word == 2 else torch.int32, device="cuda")
        assert self.t.data_ptr() % 16 == 0
        self.ptr = self.t.data_ptr() + self.g.word * self.g.start

    def load(self, words=None):
        """Canaries everywhere, `words` (any dtype of the item size) in the array if given."""
        import torch
        full = self.g.fill.copy()
        if words is not None:
            full[self.g.start:self.g.end] = np.ascontiguousarray(words).view(self.g.dtype)
        self.t.copy_(torch.from_numpy(full.view(np.int16 if self.g.word == 2 else np.int32)))
        return self

    def read(self, what: str) -> np.ndarray:
        """The array's words (uint32, or uint16 for 2-byte items), after checking every guard word."""
        full = self.t.cpu().numpy().view(self.g.dtype)
        self.g.check(full, what)
        return full[self.g.start:self.g.end].copy()


class Workspace:
    """One workspace of `cap` bytes (256-byte aligned) for a whole test module, filled with 0xFF bytes once and never
    cleared: every call finds what the calls before it (other sizes, other paths, other plans) left there.
    guard(nbytes) is the stretch of GUARD bytes just past one call's ws_bytes, which that call must not change;
    check_tail asserts that the bytes past the last such stretch still hold 0xFF."""
    GUARD = 1024

    def __init__(self, cap: int):
        import torch
        self.cap = cap + self.GUARD
        self.t = torch.full((self.cap + 256 + self.GUARD,), 0xFF, dtype=torch.uint8, device="cuda")
        self.lo = (-self.t.data_ptr()) % 256
        self.ptr = self.t.data_ptr() + self.lo

    def guard(self, nbytes: int):
        return self.t[self.lo + nbytes:self.lo + nbytes + self.GUARD]

    def check_tail(self):
        tail = self.t[self.lo + self.cap:].cpu().numpy()
        assert bool((tail == 0xFF).all()), "workspace written past every call's ws_bytes"
