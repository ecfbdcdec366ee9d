"""Exact references for sorts of up to 2^30 keys that cost O(n) on the device (test infrastructure only).

Nothing here sorts: inputs are built so that their sorted output is known in closed form, and outputs are checked
against that form or against an exact characterization of the stable sort.  Everything is torch tensor arithmetic
(int64 where products need it), on whatever device the tensors live, in chunks so that temporaries stay small.

Orders.  Every key order is image(k) = k ^ (top bit of k set ? neg : pos) sorted as an unsigned b-bit integer
(tests/key_orders.py, key_orders16.py, key_orders64.py).  Here an image is held as ``image - 2^(b-1)`` in int64 (the
"centred image"), so that torch's signed compare is the unsigned order of the images for every width, 64 included.

Permutation.  pi(i) = (a*i + c) mod n with gcd(a, n) = 1 and a < 2^31, so a*i fits in int64; its inverse is
pi^-1(j) = a^-1 * (j - c) mod n.  In a segment of length L the same a and c act modulo L.

Construction D (distinct keys): image(i) = G(pi(i)); construction T (ties): image(i) = G(pi(i) >> t), groups of 2^t
equal keys.  G(q) = m * (q - g // 2) centred, for q < g values, with the largest spread m that keeps every image in b
bits: every 8-bit digit takes more than one value, the images straddle the top bit (so both masks of an order apply),
and for 64-bit keys all eight digits vary.  The sorted keys are then inverse(G(j >> t)) at position j (per segment:
at local position j), and for D the values are pi^-1(j).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import key_orders as ko32
import key_orders16 as ko16
import key_orders64 as ko64

CHUNK = 1 << 26                   # elements per chunk of every construction and check
A0 = 1_000_000_007                # a prime below 2^31: coprime with every n < 2^31 except its own multiples
C0 = 0x2545F491                   # the permutation's shift (taken mod n)

KEY_ORDERS = {**{k: ko32 for k in ko32.DTYPES}, **{k: ko16 for k in ko16.DTYPES}, **{k: ko64 for k in ko64.DTYPES}}
BITS = {**{k: 32 for k in ko32.DTYPES}, **{k: 16 for k in ko16.DTYPES}, **{k: 64 for k in ko64.DTYPES}}
NAMES = {**ko32.NAMES, **ko16.NAMES, **ko64.NAMES}


def torch_dtype(torch, kt: int):
    return {ko32.KEY_I32: torch.int32, ko32.KEY_U32: torch.uint32, ko32.KEY_F32: torch.float32,
            ko64.KEY_I64: torch.int64, ko64.KEY_U64: torch.uint64, ko64.KEY_F64: torch.float64,
            ko16.KEY_I16: torch.int16, ko16.KEY_U16: torch.uint16, ko16.KEY_F16: torch.float16,
            ko16.KEY_BF16: torch.bfloat16}[kt]


def int_dtype(torch, kt: int):
    return {16: torch.int16, 32: torch.int32, 64: torch.int64}[BITS[kt]]


def ints(t, kt: int):
    """The keys' bit patterns as signed integers of their width (a view, no copy)."""
    import torch
    return t.view(int_dtype(torch, kt))


def _sext(x: int, b: int) -> int:
    """The b-bit pattern x as a signed integer."""
    return x - (1 << b) if x >> (b - 1) & 1 else x


def _masks(kt: int, desc: int):
    b = BITS[kt]
    neg, pos = KEY_ORDERS[kt].MASKS[(kt, desc)]
    top = 1 << (b - 1)
    set_mask, clear_mask = (neg, pos) if not neg & top else (pos, neg)
    return b, neg, pos, top, set_mask, clear_mask


# ---- images ---------------------------------------------------------------------------------------------------------
def image(keys, kt: int, desc: int):
    """Centred images (int64) of a tensor of keys of type kt: their order is the order (kt, desc)."""
    import torch
    b, neg, pos, top, _, _ = _masks(kt, desc)
    w = ints(keys, kt).to(torch.int64)
    return w ^ torch.where(w < 0, _sext(neg ^ top, b), _sext(pos ^ top, b))


def inverse(img, kt: int, desc: int):
    """The keys (as their torch dtype) whose centred images are ``img`` (int64): tests/key_orders*.inverse."""
    import torch
    b, _, _, top, set_mask, clear_mask = _masks(kt, desc)
    w = img ^ torch.where(img >= 0, _sext(set_mask ^ top, b), _sext(clear_mask ^ top, b))
    return w.to(int_dtype(torch, kt)).view(torch_dtype(torch, kt))


def spread(g: int, b: int) -> int:
    """G's step for g values in b bits: m * (g // 2) <= 2^(b-1) and m * (ceil(g / 2) - 1) < 2^(b-1), so G stays in the
    centred b-bit range; for b = 64 and g >= 2, m < 2^63 fits int64.  m is odd, so the lowest digit changes from one
    value to the next."""
    m = ((1 << b) - 1) // g if g > 1 else 1
    return max(1, m - 1 + m % 2)


def G(q, g: int, b: int):
    """Centred images of q in [0, g): strictly increasing in q, spread over the b-bit range, straddling its middle."""
    return (q - g // 2) * spread(g, b)


def groups(length: int, t: int) -> int:
    """Distinct values among ``length`` keys of construction T with shift t."""
    return ((length - 1) >> t) + 1 if length > 0 else 0


def shift_for(length: int, b: int) -> int:
    """The smallest t for which ``length`` keys of b bits can be built (g <= 2^b)."""
    t = 0
    while groups(length, t) > 1 << b:
        t += 1
    return t


# ---- the permutation ------------------------------------------------------------------------------------------------
def multiplier(n: int) -> int:
    a = A0
    while math.gcd(a, n) != 1:
        a += 2
    assert a < 1 << 31
    return a


def perm(i, n, a: int, c: int = C0):
    """pi(i) = (a*i + c) mod n; n an int or a tensor of per-element moduli (segment lengths)."""
    return (i * a + c) % n


def perm_inv(j, n: int, a: int, c: int = C0):
    return ((j - c) % n) * pow(a, -1, n) % n


def _chunks(n: int, chunk: int):
    for s in range(0, n, chunk):
        yield s, min(n, s + chunk)


# ---- 1-D constructions ----------------------------------------------------------------------------------------------
@dataclass
class Case:
    """What a construction promises: n keys of type kt, order desc, shift t (None: construction D), permutation a."""
    n: int
    kt: int
    desc: int
    t: int | None
    a: int

    @property
    def g(self) -> int:
        return groups(self.n, self.t or 0)


def build(n: int, kt: int, desc: int, t: int | None, device, chunk: int = CHUNK):
    """(keys, Case): construction D (t None) or T (t >= 0) of n keys of type kt for the order (kt, desc)."""
    import torch
    case = Case(n, kt, desc, t, multiplier(n))
    b = BITS[kt]
    assert case.g <= 1 << b, f"{n} keys of {b} bits cannot hold {case.g} distinct values"
    keys = torch.empty(n, dtype=torch_dtype(torch, kt), device=device)
    for s, e in _chunks(n, chunk):
        q = perm(torch.arange(s, e, dtype=torch.int64, device=device), n, case.a) >> (t or 0)
        keys[s:e] = inverse(G(q, case.g, b), kt, desc)
    return keys, case


def expected_keys(case: Case, s: int, e: int, device):
    """Keys s..e of the sorted output of a construction."""
    import torch
    j = torch.arange(s, e, dtype=torch.int64, device=device) >> (case.t or 0)
    return inverse(G(j, case.g, BITS[case.kt]), case.kt, case.desc)


def check_keys(out, case: Case, what: str = "", chunk: int = CHUNK) -> None:
    """The sorted keys of a construction, bit for bit."""
    import torch
    for s, e in _chunks(case.n, chunk):
        got = ints(out[s:e], case.kt)
        want = ints(expected_keys(case, s, e, out.device), case.kt)
        if not torch.equal(got, want):
            j = s + int(torch.nonzero(got != want)[0])
            raise AssertionError(f"{what}: keys differ from the closed form first at {j} of {case.n}: "
                                 f"got {int(ints(out[j:j + 1], case.kt))}, want {int(want[j - s])}")


def check_values_d(v, case: Case, what: str = "", chunk: int = CHUNK) -> None:
    """Values (input positions) of construction D: pi^-1(j) at position j."""
    import torch
    assert case.t is None
    for s, e in _chunks(case.n, chunk):
        want = perm_inv(torch.arange(s, e, dtype=torch.int64, device=v.device), case.n, case.a)
        got = v[s:e].to(torch.int64)
        if not torch.equal(got, want):
            j = s + int(torch.nonzero(got != want)[0])
            raise AssertionError(f"{what}: value at {j} of {case.n} is {int(got[j - s])}, want {int(want[j - s])}")


def _first(mask) -> int:
    return int(mask.nonzero()[0])


def check_permutation(v, n: int, what: str = "", chunk: int = CHUNK) -> None:
    """v holds every integer of [0, n) once: in range (checked before any indexing), then a bool seen[v]."""
    import torch
    seen = torch.zeros(n, dtype=torch.bool, device=v.device)
    for s, e in _chunks(n, chunk):
        x = v[s:e].to(torch.int64)
        bad = (x < 0) | (x >= n)
        if bool(bad.any()):
            j = s + _first(bad)
            raise AssertionError(f"{what}: value {int(v[j])} at {j} is outside [0, {n})")
        seen[x] = True
    if not bool(seen.all()):
        raise AssertionError(f"{what}: values are not a permutation of [0, {n}): {int((~seen).sum())} missing, "
                             f"first {_first(~seen)}")


def check_pairs(keys_in, keys_out, v, kt: int, desc: int, what: str = "", chunk: int = CHUNK) -> None:
    """The stable sort of (key, position) pairs, exactly: v is a permutation of [0, n), keys_out == keys_in[v] bit for
    bit, the images of keys_out never decrease, and v increases strictly wherever two adjacent images are equal."""
    import torch
    n = keys_out.numel()
    check_permutation(v, n, what, chunk)
    kin = ints(keys_in, kt)
    for s, e in _chunks(n, chunk):
        x = v[s:e].to(torch.int64)
        if not torch.equal(kin[x], ints(keys_out[s:e], kt)):
            raise AssertionError(f"{what}: keys do not follow their values, first at "
                                 f"{s + _first(kin[x] != ints(keys_out[s:e], kt))}")
        e1 = min(n, e + 1)
        img = image(keys_out[s:e1], kt, desc)
        down = img[1:] < img[:-1]
        if bool(down.any()):
            raise AssertionError(f"{what}: keys decrease at {s + _first(down)}")
        tie = img[1:] == img[:-1]
        vv = v[s:e1].to(torch.int64)
        unstable = tie & (vv[1:] <= vv[:-1])
        if bool(unstable.any()):
            raise AssertionError(f"{what}: equal keys out of input order at {s + _first(unstable)}")


def check_sorted_like_torch(keys_out, keys_in, kt: int, desc: int, what: str = "", chunk: int = CHUNK) -> None:
    """Keys-only result of random data: its images equal torch.sort of the input's images, element for element.
    Frees what it builds before returning."""
    import torch
    want = torch.sort(image(keys_in, kt, desc)).values
    n = keys_out.numel()
    for s, e in _chunks(n, chunk):
        got = image(keys_out[s:e], kt, desc)
        if not torch.equal(got, want[s:e]):
            raise AssertionError(f"{what}: differs from torch.sort of the images first at {s + _first(got != want[s:e])}")
    del want
    if keys_out.is_cuda:
        torch.cuda.empty_cache()


# ---- segmented constructions ----------------------------------------------------------------------------------------
SEG_MIX = 0x9E3779B1               # segment s shifts its values by (s * SEG_MIX) mod (span - g + 1)


@dataclass
class SegCase:
    """Every segment holds construction D or T of its own length, with the same a and c: the keys of segment s are
    G(c_s + (pi_L(j) >> t)) for its local positions j, where g = the groups of the longest segment, G spans
    span = min(2^b, g + 2^20) values and c_s = (s * SEG_MIX) mod (span - g + 1).  Segments of one key thus differ from
    their neighbours, and segments overlap in value, so a sort across segment boundaries gives another result."""
    n: int
    kt: int
    desc: int
    t: int
    g: int
    span: int
    a: int = A0

    def shift(self, seg):
        return seg * SEG_MIX % (self.span - self.g + 1)


def _segment_of(offsets, s: int, e: int):
    """(segment id, segment begin, segment length) of positions s..e, int64; offsets int32 or int64."""
    import torch
    p = torch.arange(s, e, dtype=offsets.dtype, device=offsets.device)
    seg = torch.searchsorted(offsets, p, right=True).to(torch.int64) - 1
    o0 = offsets[seg].to(torch.int64)
    return seg, o0, offsets[seg + 1].to(torch.int64) - o0


def longest(offsets) -> int:
    return int((offsets[1:] - offsets[:-1]).max()) if offsets.numel() > 1 else 0


def build_segmented(offsets, kt: int, desc: int, t: int | None = None, chunk: int = CHUNK):
    """(keys, SegCase) for segments given by ``offsets`` (a sorted tensor of S + 1 integers from 0 to n).  t None: the
    smallest shift the key width allows (D where it can be)."""
    import torch
    n, b = int(offsets[-1]), BITS[kt]
    lmax = longest(offsets)
    t = shift_for(lmax, b) if t is None else t
    g = groups(lmax, t)
    assert g <= 1 << b
    case = SegCase(n, kt, desc, t, g, min(1 << b, g + (1 << 20)), A0)
    keys = torch.empty(n, dtype=torch_dtype(torch, kt), device=offsets.device)
    for s, e in _chunks(n, chunk):
        seg, o0, ln = _segment_of(offsets, s, e)
        loc = torch.arange(s, e, dtype=torch.int64, device=offsets.device) - o0
        keys[s:e] = inverse(G(case.shift(seg) + (perm(loc, ln, case.a) >> t), case.span, b), kt, desc)
    return keys, case


def local_positions(offsets, chunk: int = CHUNK):
    """int32 position of every element inside its segment (the values of the pairs sorts)."""
    import torch
    n = int(offsets[-1])
    v = torch.empty(n, dtype=torch.int32, device=offsets.device)
    for s, e in _chunks(n, chunk):
        _, o0, _ = _segment_of(offsets, s, e)
        v[s:e] = (torch.arange(s, e, dtype=torch.int64, device=offsets.device) - o0).to(torch.int32)
    return v


def check_seg_keys(out, offsets, case: SegCase, what: str = "", chunk: int = CHUNK) -> None:
    """Every segment's sorted keys, bit for bit: G(c_s + (j >> t)) at local position j of segment s."""
    import torch
    for s, e in _chunks(case.n, chunk):
        seg, o0, _ = _segment_of(offsets, s, e)
        loc = torch.arange(s, e, dtype=torch.int64, device=out.device) - o0
        want = ints(inverse(G(case.shift(seg) + (loc >> case.t), case.span, BITS[case.kt]), case.kt, case.desc), case.kt)
        got = ints(out[s:e], case.kt)
        if not torch.equal(got, want):
            j = s + _first(got != want)
            raise AssertionError(f"{what}: keys differ from the closed form first at {j} of {case.n}: "
                                 f"got {int(got[j - s])}, want {int(want[j - s])}")


def check_seg_pairs(keys_in, keys_out, v, offsets, kt: int, desc: int, what: str = "", chunk: int = CHUNK) -> None:
    """check_pairs per segment: v holds local positions (v < the segment's length) and off[seg] + v is a permutation
    of [0, n); keys_out == keys_in[off[seg] + v]; within a segment images never decrease and v increases strictly
    between equal images.  Nothing is compared across a segment boundary."""
    import torch
    n = keys_out.numel()
    seen = torch.zeros(n, dtype=torch.bool, device=keys_out.device)
    kin = ints(keys_in, kt)
    for s, e in _chunks(n, chunk):
        e1 = min(n, e + 1)
        seg, o0, ln = _segment_of(offsets, s, e1)
        x = v[s:e1].to(torch.int64)
        bad = (x < 0) | (x >= ln)
        if bool(bad.any()):
            j = s + _first(bad)
            raise AssertionError(f"{what}: value {int(v[j])} at {j} is outside its segment of length {int(ln[j - s])}")
        src = o0 + x
        seen[src[:e - s]] = True
        if not torch.equal(kin[src[:e - s]], ints(keys_out[s:e], kt)):
            raise AssertionError(f"{what}: keys do not follow their values, first at "
                                 f"{s + _first(kin[src[:e - s]] != ints(keys_out[s:e], kt))}")
        img = image(keys_out[s:e1], kt, desc)
        same = seg[1:] == seg[:-1]
        down = same & (img[1:] < img[:-1])
        if bool(down.any()):
            raise AssertionError(f"{what}: keys decrease inside a segment at {s + _first(down)}")
        unstable = same & (img[1:] == img[:-1]) & (x[1:] <= x[:-1])
        if bool(unstable.any()):
            raise AssertionError(f"{what}: equal keys out of input order at {s + _first(unstable)}")
    if not bool(seen.all()):
        raise AssertionError(f"{what}: values are not a permutation of every segment's positions: "
                             f"{int((~seen).sum())} positions missing, first {_first(~seen)}")
