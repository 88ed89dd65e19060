"""The two primitives every stage of the filter runs on, tested directly against plain NumPy: the stable one-sweep LSD radix sort
(csrc/radix_sort.cuh: rs_sort_pairs, and rs_sort_packed with its pack pass and gap-layout squeeze) and the one-pass scans
(csrc/scan.cuh: scan_apply, scan_flags, scan_segmax, compact_unordered).

tests/primitives_harness.cu drives the header code the way the pipeline does and is compiled here, with the product's nvcc
flags, into a temporary directory.  The sizes sit on the boundaries where the kernels change code path: one warp's 14 x 32
sort items, the 5376-pair sort tile (full tiles rank with shared-memory match masks and a MATCH.ALL shortcut, the last partial
tile with ballots), the 8-tile look-back window of the sort, the 2048-element scan tile and the scans' 32-tile look-back.
The key patterns steer the ranking and histogram shortcuts (warp-uniform digits, 32 distinct digits per warp, half-uniform
warps).  At the top of each contract (2^30 - 1 sorted pairs, whose digit counts fill the 30-bit tile status words, and
2^31 - 1 scanned elements, the context's record limit) the harness generates the input on the device and checks it there
against closed forms and a one-thread-per-segment walk.

A failed comparison here points at one primitive and one shape, where a whole-filter mismatch points at the pipeline.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__

HERE = os.path.dirname(os.path.abspath(__file__))
HARNESS = os.path.join(HERE, "primitives_harness.cu")

RS_TILE = 5376      # sort tile: 384 threads x 14 items
RS_WARP_ITEMS = 448  # one warp's 14 x 32 items
SC_TILE = 2048      # scan tile: 256 threads x 8 items
PH_NOMEM = 2

SORT_SIZES = [0, 1, 2, 31, 32, 33, RS_WARP_ITEMS - 1, RS_WARP_ITEMS, RS_WARP_ITEMS + 1, RS_TILE - 1, RS_TILE, RS_TILE + 1,
              2 * RS_TILE - 1, 2 * RS_TILE + 1, 8 * RS_TILE - 1, 8 * RS_TILE + 1, 9 * RS_TILE, 100_007]
SORT_SIZES_LARGE = [1 << 20, (1 << 24) + 3]
KEY_BITS = [1, 7, 8, 9, 16, 17, 31, 32, 33, 53, 56, 63, 64]
PATTERNS = ["random", "equal", "all_ones", "ascending", "descending", "runs32", "distinct32", "half_uniform", "digits_0_255",
            "skewed", "top_digit"]
PACKED_IB = [1, 8, 13, 21, 24, 31, 32]
SCAN_SIZES = [0, 1, 255, 256, 257, 1023, 1024, 1025, SC_TILE - 1, SC_TILE, SC_TILE + 1, 32 * SC_TILE - 1, 32 * SC_TILE + 1,
              33 * SC_TILE, 1_000_003, 1 << 27]
FLAG_PATTERNS = ["none", "all", "alternating", "last_only", "one_per_tile", "random", "sparse"]
HEAD_PATTERNS = ["every", "none", "first_only", "tile_edges", "off_tile_edges", "random", "multi_tile"]
HOST_BIG = 1 << 24  # from here on the host reference dominates the run time: fewer patterns per size


def _some(n, patterns, few):
    return [p for p in patterns if p in few] if n >= HOST_BIG else patterns


def _compile(out_dir):
    out = os.path.join(str(out_dir), "libprimitives_harness.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    r = subprocess.run([nvcc] + __graft_entry__.NVCC_FLAGS + ["-shared", "-o", out, HARNESS], capture_output=True, text=True)
    assert r.returncode == 0, f"the primitives harness does not compile:\n{r.stderr}"
    return out


@pytest.fixture(scope="module")
def harness_so(tmp_path_factory):
    return _compile(tmp_path_factory.mktemp("primitives_harness"))


def test_harness_compiles(harness_so):
    """The harness builds against the current headers for sm_100a (no GPU needed): a header change that breaks the
    primitives' driver interface shows on machines without one."""
    assert os.path.getsize(harness_so) > 0


@pytest.fixture(scope="module")
def ph(harness_so):
    lib = C.CDLL(harness_so)
    P, U32, INT = C.c_void_p, C.c_uint32, C.c_int
    for name, args in {"ph_sort_pairs": [U32, INT, P, P, P, P], "ph_sort_packed": [U32, INT, INT, INT, P, P, P, P],
                       "ph_scan_apply": [U32, P, P, P, P, P], "ph_scan_flags": [U32, P, P, P, P, P],
                       "ph_scan_segmax": [U32, P, P, P, P], "ph_compact_unordered": [U32, P, P, P, P],
                       "ph_big_sort": [U32, INT, P, P], "ph_big_scan": [INT, P, P, P]}.items():
        f = getattr(lib, name)
        f.argtypes = args + [P, INT]
        f.restype = C.c_int
    return lib


def _p(a):
    return a.ctypes.data


def _run(fn, *args):
    msg = C.create_string_buffer(512)
    rc = fn(*args, C.addressof(msg), 512)
    text = msg.value.decode(errors="replace")
    if rc == PH_NOMEM:
        pytest.skip(f"{fn.__name__}: {text}")
    assert rc == 0, f"{fn.__name__} returned {rc}: {text}"


# ---- calls -----------------------------------------------------------------------------------------------------------------------
def dev_sort_pairs(ph, keys, bits):
    n = len(keys)
    vals = np.arange(n, dtype=np.uint32)
    ko, vo = np.empty(n, np.uint64), np.empty(n, np.uint32)
    _run(ph.ph_sort_pairs, n, bits, _p(keys), _p(vals), _p(ko), _p(vo))
    return ko, vo


def dev_sort_packed(ph, keys, vals, key_bits, ib, gap_cb=0):
    n = len(keys)
    words, info = np.empty(n, np.uint64), np.zeros(4, np.int32)
    _run(ph.ph_sort_packed, n, key_bits, ib, gap_cb, _p(keys), _p(vals), _p(words), _p(info))
    return words, dict(zip(("c0", "passes", "pack_pass", "timed_passes"), (int(x) for x in info)))


def dev_scan(fn, inp):
    n = len(inp)
    excl, seen, calls, total = (np.empty(n, np.uint32), np.empty(n, np.uint32), np.empty(n, np.uint32), np.zeros(1, np.uint32))
    _run(fn, n, _p(inp), _p(excl), _p(seen), _p(calls), _p(total))
    return excl, seen, calls, int(total[0])


def dev_segmax(ph, head, val):
    n = len(head)
    out, calls = np.empty(n, np.uint32), np.empty(n, np.uint32)
    _run(ph.ph_scan_segmax, n, _p(head), _p(val), _p(out), _p(calls))
    return out, calls


def dev_compact(ph, pred):
    n = len(pred)
    slot, calls, count = np.empty(n, np.uint32), np.empty(n, np.uint32), np.zeros(1, np.uint32)
    _run(ph.ph_compact_unordered, n, _p(pred), _p(slot), _p(calls), _p(count))
    return slot, calls, int(count[0])


# ---- references and checks (plain NumPy; each raises AssertionError naming the property that fails) -----------------------------
def check_sorted_pairs(keys, ko, vo):
    """(ko, vo): the device's sort of (keys, payload = index)."""
    n = len(keys)
    assert len(ko) == n and len(vo) == n
    assert np.array_equal(np.sort(vo), np.arange(n, dtype=np.uint32)), "the payloads are not a permutation of the input positions"
    assert np.array_equal(ko, keys[vo]), "a key left its payload"
    assert np.all(ko[1:] >= ko[:-1]), "keys out of order"
    tie = ko[1:] == ko[:-1]
    assert np.all(vo[1:][tie] > vo[:-1][tie]), "equal keys out of input order (not stable)"
    assert np.array_equal(vo, np.argsort(keys, kind="stable")), "differs from numpy's stable argsort"


def rs_packed_c0(key_bits, ib):
    """radix_sort.cuh rs_packed_c0: the smallest multiple of the 8-bit digit with key_bits - c0 + ib <= 64."""
    c0 = 0
    while key_bits - c0 + ib > 64:
        c0 += 8
    return c0


def packed_expect(key_bits, ib):
    c0 = rs_packed_c0(key_bits, ib)
    passes = (key_bits + 7) // 8
    pk = 0 if c0 == 0 else c0 // 8 - 1
    timed = passes - pk - 1
    return {"c0": c0, "passes": passes, "pack_pass": pk, "timed_passes": timed if timed > 0 else passes}


def squeeze(keys, gap_cb):
    """The gap layout (high << 32) | low with low < 2^gap_cb, as the contiguous key (high << gap_cb) | low."""
    return keys if gap_cb == 0 else ((keys >> np.uint64(32)) << np.uint64(gap_cb)) | (keys & np.uint64(0xFFFFFFFF))


def check_packed(keys, vals, words, c0, ib, gap_cb=0):
    k = squeeze(keys, gap_cb)
    order = np.argsort(k, kind="stable")
    want = ((k[order] >> np.uint64(c0)) << np.uint64(ib)) | vals[order].astype(np.uint64)
    assert len(words) == len(keys)
    assert np.array_equal(np.sort(words & np.uint64((1 << ib) - 1)), np.sort(vals.astype(np.uint64))), "payloads lost or duplicated"
    assert np.all((words[1:] >> np.uint64(ib)) >= (words[:-1] >> np.uint64(ib))), "keys out of order"
    assert np.array_equal(words, want), "differs from ((key >> c0) << ib) | payload in numpy's stable order"


def check_scan(inp, excl, seen, calls, total):
    v = inp.astype(np.uint64)
    csum = np.cumsum(v)
    assert np.all(calls == 1), "out() not called exactly once per element"
    assert np.array_equal(seen, inp.astype(np.uint32)), "out() received a value other than the element's"
    assert np.array_equal(excl.astype(np.uint64), csum - v), "exclusive prefix differs from cumsum"
    assert total == (int(csum[-1]) if len(v) else 0), "total differs"


def segmax_ref(head, val):
    """Per-segment maximum.accumulate (a segment starts at every head; elements before the first head form one segment)."""
    seg = np.cumsum(head != 0, dtype=np.uint64)
    comb = (seg << np.uint64(32)) | val.astype(np.uint64)
    return (np.maximum.accumulate(comb) & np.uint64(0xFFFFFFFF)).astype(np.uint32) if len(val) else np.empty(0, np.uint32)


def check_segmax(head, val, out, calls):
    assert np.all(calls == 1), "out() not called exactly once per element"
    assert np.array_equal(out, segmax_ref(head, val)), "segmented max differs from the per-segment maximum.accumulate"


def check_compact(pred, slot, calls, count):
    sel = pred != 0
    assert count == int(sel.sum()), "count differs from the number of selected elements"
    assert np.all(calls[sel] == 1) and np.all(calls[~sel] == 0), "out() not called exactly once per selected element"
    assert np.all(slot[~sel] == 0xFFFFFFFF), "an element that was not selected got a slot"
    assert np.array_equal(np.sort(slot[sel]), np.arange(count, dtype=np.uint32)), "the slots are not exactly [0, count)"


# ---- inputs ----------------------------------------------------------------------------------------------------------------------
def _rand64(rng, n):
    return (rng.integers(0, 1 << 32, n, dtype=np.uint64) << np.uint64(32)) | rng.integers(0, 1 << 32, n, dtype=np.uint64)


def sort_keys(pattern, n, bits, rng):
    """Keys below 2^bits (the drivers' contract) that steer the ranking and histogram paths."""
    mask = np.uint64((1 << bits) - 1)
    lane = np.arange(n, dtype=np.uint64) % np.uint64(32)
    rows = np.repeat(_rand64(rng, n // 32 + 1), 32)[:n]   # one value per 32-key row: every warp item holds one key
    if pattern == "random":
        k = _rand64(rng, n)
    elif pattern == "equal":
        k = np.full(n, _rand64(rng, 1)[0], np.uint64)
    elif pattern == "all_ones":  # 2^bits - 1; at 64 bits 0xFFFF...F, the value invalid lanes of a partial tile carry
        k = np.full(n, mask, np.uint64)
    elif pattern == "ascending":
        k = np.sort(_rand64(rng, n) & mask)
    elif pattern == "descending":
        k = np.sort(_rand64(rng, n) & mask)[::-1].copy()
    elif pattern == "runs32":  # the MATCH.ALL shortcut of the full-tile ranking, the 64-at-once histogram shortcut
        k = rows
    elif pattern == "distinct32":  # every digit of a row differs across its 32 lanes
        k = np.zeros(n, np.uint64)
        for j in range(8):
            s = np.uint64(8 * j)
            k |= (((rows >> s) + lane) & np.uint64(0xFF)) << s
    elif pattern == "half_uniform":  # lanes 0-15 share a key, 16-31 random
        k = np.where(lane < np.uint64(16), rows, _rand64(rng, n))
    elif pattern == "digits_0_255":
        r = _rand64(rng, n)
        k = np.zeros(n, np.uint64)
        for j in range(8):
            k |= ((r >> np.uint64(j)) & np.uint64(1)) * np.uint64(0xFF << (8 * j))
    elif pattern == "skewed":  # 99.9 % one key
        k = np.full(n, _rand64(rng, 1)[0], np.uint64)
        odd = rng.random(n) < 0.001
        k[odd] = _rand64(rng, int(odd.sum()))
    elif pattern == "top_digit":  # equal below the digit of the last pass
        low = np.uint64((1 << (8 * ((bits + 7) // 8 - 1))) - 1)
        k = (_rand64(rng, 1)[0] & low) | (_rand64(rng, n) & ~low)
    else:
        raise ValueError(pattern)
    return k & mask


def flag_input(pattern, n, rng):
    i = np.arange(n)
    if pattern == "none":
        f = np.zeros(n, bool)
    elif pattern == "all":
        f = np.ones(n, bool)
    elif pattern == "alternating":
        f = i % 2 == 1
    elif pattern == "last_only":
        f = i == n - 1
    elif pattern == "one_per_tile":  # one flag at a random place in every 2048-element tile
        f = i % SC_TILE == rng.integers(0, SC_TILE, (n + SC_TILE - 1) // SC_TILE).repeat(SC_TILE)[:n]
    elif pattern == "random":
        f = rng.random(n) < 0.5
    elif pattern == "sparse":
        f = rng.random(n) < 0.001
    else:
        raise ValueError(pattern)
    return f.astype(np.uint8)


def head_input(pattern, n, rng):
    i = np.arange(n)
    if pattern == "every":
        h = np.ones(n, bool)
    elif pattern == "none":
        h = np.zeros(n, bool)
    elif pattern == "first_only":
        h = i == 0
    elif pattern == "tile_edges":
        h = i % SC_TILE == 0
    elif pattern == "off_tile_edges":
        h = (i % SC_TILE == 1) | (i % SC_TILE == SC_TILE - 1)
    elif pattern == "random":
        h = rng.random(n) < 0.01
    elif pattern == "multi_tile":  # segments of several tiles: the look-back stops at a predecessor tile holding a head
        h = rng.random(n) < 1.0 / (5 * SC_TILE)
    else:
        raise ValueError(pattern)
    return h.astype(np.uint8)


def segmax_values(kind, n, rng):
    if kind == "hashed":  # the whole u32 range, 0 and 0xFFFFFFFF frequent
        v = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
        r = rng.random(n)
        v[r < 0.01] = 0xFFFFFFFF
        v[(r >= 0.01) & (r < 0.02)] = 0
        return v
    return (0xFFFFFFFF - np.arange(n, dtype=np.uint64)).astype(np.uint32)  # descending: the carry into a tile decides its max


def apply_values(pattern, n, rng):
    if pattern == "zeros":
        return np.zeros(n, np.uint32)
    if pattern == "ones":
        return np.ones(n, np.uint32)
    if pattern == "to_u32_max":  # random values, one of them raised so that the total is exactly 2^32 - 1
        v = rng.integers(0, max(1, (1 << 32) // (2 * max(n, 1))), n, dtype=np.uint64)
        if n:
            j = int(rng.integers(0, n))
            v[j] = 0
            v[j] = (1 << 32) - 1 - int(v.sum())
        return v.astype(np.uint32)
    if pattern == "sparse_big":  # mostly 0, a few values near 2^31 (at most 2 of them)
        v = np.zeros(n, np.uint64)
        idx = rng.choice(n, size=min(n, 2), replace=False) if n else np.empty(0, int)
        v[idx] = rng.integers(1 << 30, 1 << 31, len(idx), dtype=np.uint64)
        return v.astype(np.uint32)
    raise ValueError(pattern)


# ---- the sort --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", SORT_SIZES)
def test_sort_pairs(ph, n):
    """rs_sort_pairs at every key width and digit pattern against numpy's stable argsort: order, stability, permutation."""
    for pi, pattern in enumerate(PATTERNS):
        for bits in KEY_BITS:
            keys = sort_keys(pattern, n, bits, np.random.default_rng([n, pi, bits]))
            ko, vo = dev_sort_pairs(ph, keys, bits)
            try:
                check_sorted_pairs(keys, ko, vo)
            except AssertionError as e:
                raise AssertionError(f"n={n} bits={bits} pattern={pattern}: {e}") from None


@pytest.mark.gpu
@pytest.mark.parametrize("n,pattern", [(n, p) for n in SORT_SIZES_LARGE
                                       for p in _some(n, PATTERNS, ("random", "runs32", "half_uniform", "skewed", "top_digit"))])
def test_sort_pairs_large(ph, n, pattern):
    for bits in ((64,) if n >= HOST_BIG else (17, 64)):
        keys = sort_keys(pattern, n, bits, np.random.default_rng([n, bits, PATTERNS.index(pattern)]))
        ko, vo = dev_sort_pairs(ph, keys, bits)
        try:
            check_sorted_pairs(keys, ko, vo)
        except AssertionError as e:
            raise AssertionError(f"n={n} bits={bits}: {e}") from None


def _packed_case(ph, n, key_bits, ib, gap_cb, rng, pattern="pool"):
    """One packed sort: keys with repeats (so stability shows), payloads the index where it fits ib bits, else random."""
    if pattern == "pool":
        pool = sort_keys("random", max(1, n // 4), key_bits, rng)
        keys = pool[rng.integers(0, len(pool), n)]
    else:
        keys = sort_keys(pattern, n, key_bits, rng)
    if gap_cb:  # store the contiguous key in the gap layout
        keys = ((keys >> np.uint64(gap_cb)) << np.uint64(32)) | (keys & np.uint64((1 << gap_cb) - 1))
    vals = np.arange(n, dtype=np.uint32) if n <= (1 << ib) else rng.integers(0, 1 << ib, n, dtype=np.uint64).astype(np.uint32)
    words, info = dev_sort_packed(ph, keys, vals, key_bits, ib, gap_cb)
    want = packed_expect(key_bits, ib)
    if n == 0:  # an empty sort returns before it plans its passes
        want.update(pack_pass=-1, timed_passes=0)
    assert info == want, f"key_bits={key_bits} ib={ib}: the sort reports {info}, the contract says {want}"
    try:
        check_packed(keys, vals, words, info["c0"], ib, gap_cb)
    except AssertionError as e:
        raise AssertionError(f"n={n} key_bits={key_bits} ib={ib} gap_cb={gap_cb} {want} pattern={pattern}: {e}") from None


@pytest.mark.gpu
@pytest.mark.parametrize("key_bits", range(1, 65))
def test_sort_packed_widths(ph, key_bits):
    """rs_sort_packed at every key width against every payload width of PACKED_IB, so every c0 and every pack pass occurs
    (c0 == 0: pass 0 packs and keeps its own digit; the single-pass sort whose pack pass is its last).  Where 0 < c0 <= gap_cb
    the same keys also go in the gap layout, squeezed by the histogram and the pack pass."""
    n = 2 * RS_TILE + RS_WARP_ITEMS + 1  # two full tiles and a partial one
    for ib in PACKED_IB:
        rng = np.random.default_rng([key_bits, ib])
        _packed_case(ph, n, key_bits, ib, 0, rng)
        c0 = rs_packed_c0(key_bits, ib)
        if c0 > 0:
            for gap_cb in sorted({max(c0, key_bits - 32), min(32, key_bits)}):
                if c0 <= gap_cb <= 32 and key_bits - gap_cb <= 32:
                    _packed_case(ph, n, key_bits, ib, gap_cb, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("n", SORT_SIZES + SORT_SIZES_LARGE)
def test_sort_packed_sizes(ph, n):
    """The packed sort as the record sort calls it (payload = record index, ib = bits_for(n - 1)) at the tile boundaries."""
    ib = max(1, int(n - 1).bit_length()) if n > 1 else 1
    for key_bits in ((47,) if n >= HOST_BIG else (17, 47, 64)):
        for pattern in _some(n, ("random", "runs32", "half_uniform", "skewed", "top_digit"), ("random", "runs32")):
            rng = np.random.default_rng([n, key_bits, PATTERNS.index(pattern)])
            _packed_case(ph, n, key_bits, ib, 0, rng, pattern)


@pytest.mark.gpu
@pytest.mark.parametrize("packed", [0, 1], ids=["pairs", "packed"])
@pytest.mark.parametrize("m", [1, 3, 256, 65537])
def test_sort_top_of_contract(ph, m, packed):
    """n = 2^30 - 1 pairs (key i mod m, payload i) sorted by 32 key bits: the high digits are constant, so one digit's running
    count in the tile status words reaches RS_VAL_MASK exactly.  The device checks every output position against the closed
    form r*q + min(r, n mod m) + i div m."""
    bad, first = C.c_ulonglong(), C.c_ulonglong()
    _run(ph.ph_big_sort, m, packed, C.addressof(bad), C.addressof(first))
    assert bad.value == 0, f"{bad.value} positions wrong, the first at {first.value}"


# ---- the scans -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", SCAN_SIZES)
def test_scan_apply(ph, n):
    for pattern in _some(n, ("zeros", "ones", "to_u32_max", "sparse_big"), ("to_u32_max",)):
        v = apply_values(pattern, n, np.random.default_rng([n, len(pattern)]))
        try:
            check_scan(v, *dev_scan(ph.ph_scan_apply, v))
        except AssertionError as e:
            raise AssertionError(f"n={n} values={pattern}: {e}") from None


@pytest.mark.gpu
@pytest.mark.parametrize("n", SCAN_SIZES)
def test_scan_flags(ph, n):
    for pattern in _some(n, FLAG_PATTERNS, ("all", "one_per_tile", "random")):
        f = flag_input(pattern, n, np.random.default_rng([n, FLAG_PATTERNS.index(pattern)]))
        try:
            check_scan(f, *dev_scan(ph.ph_scan_flags, f))
        except AssertionError as e:
            raise AssertionError(f"n={n} flags={pattern}: {e}") from None


@pytest.mark.gpu
@pytest.mark.parametrize("n", SCAN_SIZES)
def test_scan_segmax(ph, n):
    for hp in _some(n, HEAD_PATTERNS, ("tile_edges", "multi_tile")):
        for kind in _some(n, ("hashed", "descending"), ("hashed",)):
            rng = np.random.default_rng([n, HEAD_PATTERNS.index(hp), len(kind)])
            head, val = head_input(hp, n, rng), segmax_values(kind, n, rng)
            try:
                check_segmax(head, val, *dev_segmax(ph, head, val))
            except AssertionError as e:
                raise AssertionError(f"n={n} heads={hp} values={kind}: {e}") from None


@pytest.mark.gpu
@pytest.mark.parametrize("n", SCAN_SIZES)
def test_compact_unordered(ph, n):
    for pattern in _some(n, FLAG_PATTERNS, ("random",)):
        f = flag_input(pattern, n, np.random.default_rng([n, FLAG_PATTERNS.index(pattern), 1]))
        try:
            check_compact(f, *dev_compact(ph, f))
        except AssertionError as e:
            raise AssertionError(f"n={n} pred={pattern}: {e}") from None


BIG_SCANS = {0: "apply_near_u32_total", 1: "apply_mod3", 2: "flags_all", 3: "flags_mod3", 4: "segmax_hashed", 5: "compact_mod3"}


@pytest.mark.gpu
@pytest.mark.parametrize("which", list(BIG_SCANS), ids=list(BIG_SCANS.values()))
def test_scans_top_of_contract(ph, which):
    """n = 2^31 - 1, generated and checked on the device: periodic values and flags against their closed-form prefixes (one
    total within 2^22 of 2^32), the segmented max on hashed heads and values against one thread per segment walking it in
    order (segments of 1 element to several 32-tile look-back rounds, heads on and off the tile edges), the unordered
    compaction against a count of hits per slot."""
    bad, first, total = C.c_ulonglong(), C.c_ulonglong(), C.c_uint32()
    _run(ph.ph_big_scan, which, C.addressof(bad), C.addressof(first), C.addressof(total))
    n = (1 << 31) - 1
    want_total = {0: 2046 * (n // 1024), 1: 3 * (n // 3) + (1 if n % 3 == 2 else 0), 2: n, 3: (n + 2) // 3, 5: n // 3 + 1}
    if which in want_total:
        assert total.value == want_total[which]
    assert bad.value == 0, f"{bad.value} mismatches, the first at index {first.value}"


# ---- the checks reject what they must --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_checks_reject_corrupted_results(ph):
    """Each check, given a copy of a correct device result with one defect a faulty kernel could produce, fails."""
    rng = np.random.default_rng(5)
    n = 2 * RS_TILE + 1
    keys = sort_keys("runs32", n, 8, rng)
    ko, vo = dev_sort_pairs(ph, keys, 8)
    check_sorted_pairs(keys, ko, vo)
    j = int(np.flatnonzero(ko[1:] == ko[:-1])[0])
    swapped = vo.copy()
    swapped[[j, j + 1]] = swapped[[j + 1, j]]               # two payloads of one key exchanged: unstable
    with pytest.raises(AssertionError, match="stable"):
        check_sorted_pairs(keys, ko, swapped)
    dk, dv = ko.copy(), vo.copy()
    dk[j + 1], dv[j + 1] = dk[j], dv[j]                     # one element written over its neighbour: one lost, one twice
    with pytest.raises(AssertionError, match="permutation"):
        check_sorted_pairs(keys, dk, dv)

    vals = np.arange(n, dtype=np.uint32)
    words, info = dev_sort_packed(ph, keys, vals, 8, 32)
    check_packed(keys, vals, words, info["c0"], 32)
    w = words.copy()
    w[[j, j + 1]] = w[[j + 1, j]]
    with pytest.raises(AssertionError, match="stable order"):
        check_packed(keys, vals, w, info["c0"], 32)

    v = apply_values("to_u32_max", 3 * SC_TILE, rng)
    excl, seen, calls, total = dev_scan(ph.ph_scan_apply, v)
    check_scan(v, excl, seen, calls, total)
    broken = excl.copy()
    broken[SC_TILE + 5] += 1                                # one prefix off by one
    with pytest.raises(AssertionError, match="cumsum"):
        check_scan(v, broken, seen, calls, total)

    head, val = head_input("random", 3 * SC_TILE, rng), segmax_values("hashed", 3 * SC_TILE, rng)
    out, calls = dev_segmax(ph, head, val)
    check_segmax(head, val, out, calls)
    k = int(np.flatnonzero(out != 0xFFFFFFFF)[-1])
    broken = out.copy()
    broken[k] += 1                                          # one running max off by one
    with pytest.raises(AssertionError, match="maximum.accumulate"):
        check_segmax(head, val, broken, calls)

    pred = flag_input("random", 3 * SC_TILE, rng)
    slot, calls, count = dev_compact(ph, pred)
    check_compact(pred, slot, calls, count)
    sel = np.flatnonzero(pred)
    broken = slot.copy()
    broken[sel[1]] = broken[sel[0]]                         # two elements in one slot
    with pytest.raises(AssertionError, match=r"\[0, count\)"):
        check_compact(pred, broken, calls, count)
