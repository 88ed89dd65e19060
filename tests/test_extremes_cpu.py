"""The oracle's arithmetic at the edges of the u32 coordinate contract, against a few lines of exact Python integers.

The GPU tests of tests/test_extremes_gpu.py compare the kernels with the oracle bit for bit on tables whose coordinates reach
2^32 - 1 and whose gap / deviation limits reach 2^31 - 1.  This file pins what they are compared with: the chaining gap rule
(`paf_filter.rs:799-833`) at G / G + 1 and G/5 / G/5 + 1, the inversion bound floor(|dev| / sqrt 2) <= G (`:535-597`) and the
rescue distance floor(sqrt(qd^2 + td^2)) <= D (`:690-716`), whose u64 sum wraps past 2^64 as in a release build of the
reference.  The table builders are shared with the GPU file.
"""
import math

import numpy as np
import pytest

import oracle_lib
from workloads.table import Table, prefix_ids

U32_MAX = (1 << 32) - 1
U64 = 1 << 64
SQRT2 = math.sqrt(2.0)  # == M_SQRT2


def build(rows, names, cls=Table):
    """rows: (query id, target id, qs, qe, ts, te, '+' | '-', identity) -> a table (cls: Table or sweepga_b200.MappingTable)."""
    col = lambda k: np.array([r[k] for r in rows], np.int64)
    qs, qe, ts, te = col(2), col(3), col(4), col(5)
    assert all(0 <= int(x) <= U32_MAX for c in (qs, qe, ts, te) for x in c)
    blk = np.maximum(np.maximum(qe - qs, te - ts), 1)
    ident = np.array([r[7] for r in rows], np.float64)
    matches = np.rint(ident * blk).astype(np.int64)
    strand = np.array([ord(r[6]) for r in rows], np.uint8)
    P, P2 = prefix_ids(names)
    return cls(col(0), col(1), qs, qe, ts, te, blk, matches, matches / blk, strand, P, P2, None, list(names))


def pair_names(n_pairs):
    """Two genomes, sequence 2k of the first against sequence 2k + 1 of the second."""
    return [f"{'AB'[i % 2]}#1#c{i // 2}" for i in range(2 * n_pairs)]


# ---- chaining: the gap rule ----------------------------------------------------------------------------------------------
def gap_cases(G):
    """(query step, target step) from record a to record b: >= 0 a gap, < 0 an overlap."""
    g5 = G // 5
    steps = [(G, 0), (G + 1, 0), (0, G), (0, G + 1), (G, G), (G + 1, G), (-g5, 0), (-(g5 + 1), 0), (0, -g5), (0, -(g5 + 1)),
             (-g5, -g5), (-g5, G), (G, -(g5 + 1))]
    return [(dq, dt, s) for s in "+-" for dq, dt in steps]


def gap_rule(G, dq, dt):
    """Exact: do a and b chain?  An overlap counts as its length if it is at most G/5, else as G + 1."""
    g = lambda d: d if d >= 0 else (-d if -d <= G // 5 else G + 1)
    return g(dq) <= G and g(dt) <= G


def gap_table(G, cls=Table, top=True):
    """One (query, target) pair per case, two records a -> b each; every pair moved so that its largest end is 2^32 - 1 (top)
    or its smallest start is 0.  Near the top, a.query_end + G passes 2^32 in every overlap case."""
    L = G // 5 + 1000  # longer than any overlap: b starts after a on the query
    rows, cases = [], gap_cases(G)
    for k, (dq, dt, s) in enumerate(cases):
        aq = (0, L)
        bq = (L + dq, 2 * L + dq)
        if s == "+":
            at = (0, L)
            bt = (L + dt, 2 * L + dt)
        else:  # b precedes a on the target: the gap is a.ts - b.te
            bt = (0, L)
            at = (L + dt, 2 * L + dt)
        lo_q, lo_t = min(aq[0], bq[0]), min(at[0], bt[0])
        hi_q, hi_t = max(aq[1], bq[1]) - lo_q, max(at[1], bt[1]) - lo_t
        sq, st = (U32_MAX - hi_q - lo_q, U32_MAX - hi_t - lo_t) if top else (-lo_q, -lo_t)
        rows.append((2 * k, 2 * k + 1, aq[0] + sq, aq[1] + sq, at[0] + st, at[1] + st, s, 0.95))
        rows.append((2 * k, 2 * k + 1, bq[0] + sq, bq[1] + sq, bt[0] + st, bt[1] + st, s, 0.9))
    return build(rows, pair_names(len(cases)), cls), [gap_rule(G, dq, dt) for dq, dt, _ in cases]


@pytest.mark.parametrize("top", [True, False])
@pytest.mark.parametrize("G", [50_000, 1000, (1 << 31) - 1])
def test_gap_rule_at_G_and_G5(G, top):
    t, joined = gap_table(G, top=top)
    cfg = oracle_lib.Config(scaffold_gap=G, min_scaffold_length=0)
    status, chain, st = oracle_lib.apply_filters(cfg, t)
    assert (status == 1).all()
    for k, j in enumerate(joined):
        assert (chain[2 * k] == chain[2 * k + 1]) == j, (G, gap_cases(G)[k])
    assert st.n_chains == sum(1 if j else 2 for j in joined)
    assert any(joined) and not all(joined)


# ---- inversion capture: floor(|dev| / sqrt 2) <= G -----------------------------------------------------------------------
def inversion_devs(G):
    """|dev| around G sqrt 2 and (G + 1) sqrt 2: perp = G - 1 | G and G | G + 1."""
    out = []
    for m in (G, G + 1):
        c = math.isqrt(2 * m * m)  # floor(m sqrt 2)
        out += [c - 1, c, c + 1, c + 2]
    return out


def inversion_table(G, cls=Table):
    """Per case one pair: a kept '+' chain (20 kb, diagonal 0 or far up) and one 100 bp '-' mapping inside it, its centre
    diagonal `dev` away from the chain's (both signs)."""
    rows, devs = [], []
    k = 0
    for d in inversion_devs(G):
        for sign in (1, -1):
            diag = 0 if sign > 0 else d + 30_000  # the chain's ts - qs
            Q0 = 1_000
            rows.append((2 * k, 2 * k + 1, Q0, Q0 + 20_000, Q0 + diag, Q0 + diag + 20_000, "+", 0.99))
            qs = Q0 + 5_000
            qc = qs + 50
            ts = qc + diag + sign * d - 50
            rows.append((2 * k, 2 * k + 1, qs, qs + 100, ts, ts + 100, "-", 0.9))
            devs.append(sign * d)
            k += 1
    return build(rows, pair_names(k), cls), devs


def perp_kept(G, dev):
    """The reference: (|dev| as f64 / SQRT_2) as u64 <= G."""
    return int(abs(dev) / SQRT2) <= G


@pytest.mark.parametrize("G", [50_000, 7, (1 << 31) - 1])
def test_inversion_perp_bound(G):
    t, devs = inversion_table(G)
    status, chain, st = oracle_lib.apply_filters(oracle_lib.Config(scaffold_gap=G), t)
    for k, dev in enumerate(devs):
        # exact integers agree with the f64 quotient at these deviations: |dev| < (G + 1) sqrt 2  <=>  dev^2 < 2 (G + 1)^2
        assert perp_kept(G, dev) == (dev * dev < 2 * (G + 1) ** 2)
        assert status[2 * k] == 1
        if perp_kept(G, dev):
            assert status[2 * k + 1] == 1 and chain[2 * k + 1] == chain[2 * k], (G, dev)
        else:
            assert status[2 * k + 1] == 0, (G, dev)
    assert 0 < sum(perp_kept(G, d) for d in devs) < len(devs)


# ---- rescue: floor(sqrt(qd^2 + td^2)) <= D, the u64 sum wrapping --------------------------------------------------------
def rescue_dist(qd, td):
    """The reference: ((qd * qd + td * td) as f64).sqrt() as u64, the sum in u64 (wraps)."""
    return int(math.sqrt(float((qd * qd + td * td) % U64)))


def center(s, e):
    return (s + e) // 2


def expected_rescue(t, anchors, D):
    """Per non-anchor record: the chain-giving anchor (smallest distance, then smallest index) or None, by brute force."""
    out = {}
    for i in range(t.n):
        if i in anchors:
            continue
        qc, tc = center(int(t.query_start[i]), int(t.query_end[i])), center(int(t.target_start[i]), int(t.target_end[i]))
        best = None
        for a in anchors:
            if (t.query_id[a], t.target_id[a]) != (t.query_id[i], t.target_id[i]):
                continue
            qd = abs(qc - center(int(t.query_start[a]), int(t.query_end[a])))
            if qd > D:
                continue
            d = rescue_dist(qd, abs(tc - center(int(t.target_start[a]), int(t.target_end[a]))))
            if d <= D and (best is None or (d, a) < best):
                best = (d, a)
        out[i] = None if best is None else best[1]
    return out


ANCHOR = 20_000  # anchor length: one record is a kept chain under the default scaffold mass (10 kb)


def rescue_wrap_table(cls=Table):
    """Rescue where qd^2 + td^2 passes 2^64 (D = 2 * 10^7).  A wrapped sum is below qd^2 (td < 2^32), so an anchor with
    qd <= D whose sum wraps always rescues; the kernel's two shortcuts assume a sum that does not wrap.
    Pair 0: an anchor at q, t [0, 20000), a 100 bp mapping at q ~ 10^7, t ~ 2^32 - 250 (the `td > D` early return drops it).
    Pair 1: the same with the anchor right of the mapping's query centre.
    Pair 2: an unwrapped anchor U 10^5 left of the mapping (distance ~10^6) and a wrapped anchor W 10^7 right of it whose
    wrapped distance is smaller: W wins (scanned first, so only the early return matters).
    Pair 3: a wrapping anchor one base beyond D on the query (not rescued).
    Pair 4: the mirror image of pair 2, U 10^5 right and W 10^7 left: U is scanned first, and the outward scan's stop at
    qd > best + 1 would cut W before it is measured.
    Pair 5: pair 0 upside down on the target axis, the anchor at the top and the mapping at 0."""
    rows = []
    # pair 0
    rows.append((0, 1, 0, ANCHOR, 0, ANCHOR, "+", 0.99))
    rows.append((0, 1, 10_000_000, 10_000_100, U32_MAX - 250, U32_MAX - 150, "+", 0.9))
    # pair 1: anchor right of the mapping on the query
    rows.append((2, 3, 30_000_000, 30_000_000 + ANCHOR, 0, ANCHOR, "+", 0.99))
    rows.append((2, 3, 20_000_000, 20_000_100, U32_MAX - 250, U32_MAX - 150, "+", 0.9))
    # pair 2: mapping centre (qm, tm); unwrapped anchor U at qd = 10^5, td = 10^6; wrapped anchor W at qd = 10^7 with the
    # smallest td that wraps: td = isqrt(2^64 - qd^2) + 1
    qm, tm = 60_000_000, U32_MAX - 200
    qdw = 10_000_000
    tdw = math.isqrt(U64 - qdw * qdw) + 1
    u_qc, u_tc = qm - 100_000, tm - 1_000_000
    w_qc, w_tc = qm + qdw, tm - tdw
    rows.append((4, 5, u_qc - ANCHOR // 2, u_qc + ANCHOR // 2, u_tc - ANCHOR // 2, u_tc + ANCHOR // 2, "+", 0.99))
    rows.append((4, 5, qm - 50, qm + 50, tm - 50, tm + 50, "+", 0.9))
    rows.append((4, 5, w_qc - ANCHOR // 2, w_qc + ANCHOR // 2, w_tc - ANCHOR // 2, w_tc + ANCHOR // 2, "+", 0.99))
    # pair 3: would wrap, but qd = D + 1
    qd3 = 20_000_001
    td3 = U32_MAX - 200 - ANCHOR // 2
    rows.append((6, 7, 0, ANCHOR, 0, ANCHOR, "+", 0.99))
    q3 = ANCHOR // 2 + qd3
    t3 = ANCHOR // 2 + td3
    rows.append((6, 7, q3 - 50, q3 + 50, t3 - 50, t3 + 50, "+", 0.9))
    # pair 4: pair 2 mirrored on the query axis
    u_qc, w_qc = qm + 100_000, qm - qdw
    rows.append((8, 9, u_qc - ANCHOR // 2, u_qc + ANCHOR // 2, u_tc - ANCHOR // 2, u_tc + ANCHOR // 2, "+", 0.99))
    rows.append((8, 9, qm - 50, qm + 50, tm - 50, tm + 50, "+", 0.9))
    rows.append((8, 9, w_qc - ANCHOR // 2, w_qc + ANCHOR // 2, w_tc - ANCHOR // 2, w_tc + ANCHOR // 2, "+", 0.99))
    # pair 5
    rows.append((10, 11, 0, ANCHOR, U32_MAX - ANCHOR - 100, U32_MAX - 100, "+", 0.99))
    rows.append((10, 11, 10_000_000, 10_000_100, 0, 100, "+", 0.9))
    return build(rows, pair_names(6), cls), 20_000_000, {0, 2, 4, 6, 7, 9, 11, 12}


def rescue_limit_table(D, cls=Table):
    """Floored distances D - 1, D, D + 1 (through the f64 root of the rounded sum), anchors tied at equal distance."""
    rows = []
    anchors = set()
    # pair 0: anchor centre (c, c); candidates at (qd, td) around the circle of radius D, a few qd values
    c = ANCHOR // 2
    rows.append((0, 1, 0, ANCHOR, 0, ANCHOR, "+", 0.99))
    anchors.add(0)
    for qd in (0, 1, 3, D // 3, D // 2, D - 7, D, D + 1):
        if qd > U32_MAX - c - 50:
            continue
        r2 = (D + 1) ** 2 - 1 - qd * qd  # td^2 <= r2  <=>  qd^2 + td^2 < (D + 1)^2
        if r2 < 0:
            rows.append((0, 1, c + qd - 50, c + qd + 50, c - 50, c + 50, "+", 0.9))
            continue
        t0 = math.isqrt(r2)
        for td in sorted({max(t0 - 1, 0), t0, t0 + 1, t0 + 2}):
            if c + td + 50 <= U32_MAX:
                rows.append((0, 1, c + qd - 50, c + qd + 50, c + td - 50, c + td + 50, "+", 0.9))
    # pair 1: two anchor chains whose centres are 2x apart on the query, a candidate exactly between them (equal distance).
    # The smaller index lies left of the candidate: an outward scan meets it second, so only the index tie-break picks it.
    x = min(D // 2, 1_000_000)
    rows.append((2, 3, 100_000, 100_000 + ANCHOR, 0, ANCHOR, "+", 0.99))
    anchors.add(len(rows) - 1)
    rows.append((2, 3, 100_000 + 2 * x, 100_000 + 2 * x + ANCHOR, 0, ANCHOR, "+", 0.99))
    anchors.add(len(rows) - 1)
    qm = 100_000 + c + x
    for y in (0, 7, x // 2):
        rows.append((2, 3, qm - 50, qm + 50, c + y - 50, c + y + 50, "+", 0.9))
    return build(rows, pair_names(2), cls), anchors


def check_rescue(t, anchors, D):
    status, chain, st = oracle_lib.apply_filters(oracle_lib.Config(scaffold_max_deviation=D), t)
    exp = expected_rescue(t, anchors, D)
    for a in anchors:
        assert status[a] == 1
    for i, a in exp.items():
        if a is None:
            assert status[i] == 0, i
        else:
            assert status[i] == 2 and chain[i] == chain[a], (i, a, int(status[i]), int(chain[i]), int(chain[a]))
    return status, chain, exp


def test_rescue_wraps_like_the_reference():
    t, D, anchors = rescue_wrap_table()
    status, chain, exp = check_rescue(t, anchors, D)
    # pair 0: rescued onto chain 1 through the wrapped sum, though the true distance is ~4.29e9
    qd, td = 10_000_050 - ANCHOR // 2, (U32_MAX - 200) - ANCHOR // 2
    assert qd * qd + td * td >= U64 and math.isqrt(qd * qd + td * td) > 4 * 10**9
    assert rescue_dist(qd, td) <= D
    assert status[1] == 2 and chain[1] == 1
    assert status[3] == 2 and chain[3] == chain[2]
    assert exp[5] == 6 and chain[5] == chain[6] != chain[4]  # the wrapped anchor beats the near one
    assert exp[8] is None and status[8] == 0
    assert exp[10] == 11 and chain[10] == chain[11] != chain[9]  # ... also when the near anchor is scanned first
    qd, td = 10_000_000, (U32_MAX - 200) - (t.target_start[11] + ANCHOR // 2)
    assert rescue_dist(qd, int(td)) < 10**5 < math.isqrt(qd * qd + int(td) ** 2)
    assert exp[13] == 12 and status[13] == 2 and chain[13] == chain[12]


@pytest.mark.parametrize("D", [(1 << 31) - 1, (1 << 31) - 2, 3_037_000, 1000])
def test_rescue_distance_at_D(D):
    t, anchors = rescue_limit_table(D)
    status, _, exp = check_rescue(t, anchors, D)
    assert 0 < sum(a is not None for a in exp.values()) < len(exp)


def test_rescue_tie_takes_the_smaller_anchor_index():
    t, anchors = rescue_limit_table(1_000_000)
    status, chain, exp = check_rescue(t, anchors, 1_000_000)
    n0 = t.n - 3
    left, right = sorted(anchors - {0})
    assert t.query_start[left] < t.query_start[n0] < t.query_start[right]
    assert exp[n0] == left and status[n0] == 2 and chain[n0] == chain[left] != chain[right]
