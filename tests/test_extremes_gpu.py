"""The CUDA path at the edges of its contract, "u32 coordinates, any n_seq", against the CPU oracle bit for bit.

Every width of the hot path comes from the data: sb = bits_for(n_seq), cb = bits_for(maxcoord), the record key
kb = 2 sb + 1 + cb and the index ib = bits_for(N - 1).  They decide whether the prefilter writes fused keys (2 sb + 1 <= 32),
whether the counting sort by group runs (2 n_seq^2 <= 2^26), whether keys are wide (kb > 64), where the packed LSD sort
starts (kb + ib vs 64) and whether the dead key is all ones or NONE64 (kb == 64).  The tables below sit on both sides of each
of these, with coordinates up to 2^32 - 1 and gap / deviation limits up to 2^31 - 1; each case also asserts the path it is
meant to reach, so that a moved threshold fails here instead of passing untested.  Tables are small enough for the oracle,
except the translated ones of test_translation_invariance, which compare the kernels with themselves.
"""
import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth
from test_extremes_cpu import (U32_MAX, build, expected_rescue, gap_table, inversion_table, rescue_limit_table,
                               rescue_wrap_table)
from test_parity_gpu import check

pytestmark = pytest.mark.gpu

MT = swg.MappingTable
DEFAULT_CASES = {
    "defaults": {},
    "1:1_1:1": dict(num_mappings="1:1", scaffold_filter="1:1"),
    "rescue100k": dict(scaffold_dist="100k"),
    "scaffolds_only": dict(scaffolds_only=True),
}


def bits_for(v):
    return max(int(v).bit_length(), 1)


def cli(**kw):
    return swg.FilterConfig.from_cli(**kw)


# ---- (a) sequence-count boundaries ------------------------------------------------------------------------------------------
def special_ids(n_seq):
    """0, n_seq - 1, n_seq - 2 and the ids next to every power of two below n_seq."""
    ids = {0, 1, n_seq - 1, n_seq - 2}
    for k in range(1, 18):
        ids |= {(1 << k) - 1, 1 << k, (1 << k) + 1}
    return sorted(i for i in ids if 0 <= i < n_seq)


def many_seq_table(n_seq, seed=0, group=4):
    """A few hundred records over `n_seq` sequences named over three genomes (dense prefix ids), rows in aligner order
    (groups of `group` consecutive records), both strands, with the live key of (n_seq - 2, n_seq - 2, '-') - the largest a
    live record can have - among them."""
    rng = np.random.default_rng(seed)
    ids = special_ids(n_seq)
    pairs = {(n_seq - 2, n_seq - 2), (n_seq - 1, n_seq - 1), (0, n_seq - 1), (n_seq - 1, 0), (0, 0), (n_seq - 2, n_seq - 1)}
    while len(pairs) < 60:
        pairs.add((int(rng.choice(ids)), int(rng.choice(ids))))
    rows = []
    for q, t in sorted(pairs):
        for s in "+-":
            base_q, base_t = int(rng.integers(0, 1 << 20)), int(rng.integers(0, 1 << 20))
            for j in range(group):
                qs = base_q + j * 6_000 + int(rng.integers(0, 500))
                ln = int(rng.integers(3_000, 9_000))
                ts = base_t + (j if s == "+" else group - j) * 6_000 + int(rng.integers(0, 500))
                rows.append((q, t, qs, qs + ln, ts, ts + ln + int(rng.integers(-20, 21)), s, float(rng.choice([0.9, 0.95, 0.99]))))
    names = [f"G{i * 3 // n_seq}#1#s{i}" for i in range(n_seq)]
    return build(rows, names, MT)


SEQ_CASES = {
    "defaults": {},
    "self_mass0": dict(keep_self=True, scaffold_mass="0"),
    "1:1_rescue_self": dict(num_mappings="1:1", scaffold_filter="1:1", scaffold_dist="20k", keep_self=True, scaffold_mass="5k"),
    "scaffolds_only_self": dict(scaffolds_only=True, keep_self=True),
}


@pytest.mark.parametrize("n_seq", [5792, 5793, 32767, 32768, 65536, 65537])
def test_sequence_count_boundaries(ctx, n_seq):
    """5792 | 5793: the group table (2 n_seq^2 entries <= 2^26) fits or not; 32767 | 32768: fused prefilter keys (sb 15 -> 16);
    65536 | 65537: 16-bit id columns possible or not."""
    t = many_seq_table(n_seq, seed=n_seq)
    assert t.n_seq == n_seq and set(t.seq_genome_id.tolist()) == {0, 1, 2}
    for name, flags in SEQ_CASES.items():
        cfg = cli(**flags)
        s, c, st = check(ctx, cfg, t, f"n_seq {n_seq} {name}")
        if name == "defaults":
            if 2 * n_seq * n_seq <= 1 << 26:
                assert st.n_sort_passes == 0, "rows in aligner order and the group table fits: the counting sort by group"
            else:
                assert st.n_sort_passes > 0, "the group table does not fit: the LSD passes"
            # fused keys: the prefilter also writes a key (8 B) and an index (4 B) per record
            fused = 2 * bits_for(n_seq) + 1 <= 32
            assert st.prefilter_bytes_per_record == 29 + 8 + 1 + 16 + (12 if fused else 0)
        if n_seq <= 65536:
            s16, c16, st16 = ctx.filter(cfg, swg.with_ids16(t))
            assert np.array_equal(s16, s) and np.array_equal(c16, c), f"16-bit ids differ from 32-bit ids: n_seq {n_seq} {name}"
            assert st16.n_kept == st.n_kept and st16.n_chains == st.n_chains
    if n_seq > 65536:
        with pytest.raises(ValueError):
            swg.with_ids16(t)


# ---- (b) coordinate-width boundaries ----------------------------------------------------------------------------------------
def wide_coord_table(n_seq, maxcoord, n, seed=0, shuffled=False):
    """n records whose largest coordinate is exactly `maxcoord`: most of them in the last few Mbp below it (chains, overlaps,
    equal query starts), plus a record spanning [0, maxcoord], zero-length records at maxcoord, ids 0 and n_seq - 1, both
    strands.  Rows in aligner order, or shuffled (the LSD passes)."""
    rng = np.random.default_rng(seed)
    nq = min(n_seq, 6)
    qids = [0, n_seq - 1] + [int(x) for x in rng.integers(1, n_seq - 1, nq - 2)]
    rows = [(0, n_seq - 1, 0, maxcoord, 0, maxcoord, "+", 0.97),
            (n_seq - 1, 0, maxcoord, maxcoord, maxcoord, maxcoord, "+", 0.9),
            (n_seq - 1, 0, maxcoord, maxcoord, maxcoord - 5, maxcoord - 5, "-", 0.9),
            (0, n_seq - 1, maxcoord - 10_000, maxcoord, maxcoord - 10_000, maxcoord, "-", 0.95)]
    top = maxcoord - 3_000_000
    starts = rng.integers(0, 2_990_000, 40) // 1000 * 1000  # few distinct starts: equal query starts
    while len(rows) < n:
        q = qids[int(rng.integers(0, nq))]
        t = qids[int(rng.integers(0, nq))]
        if q == t:
            t = (t + 1) % n_seq
        qs = top + int(rng.choice(starts))
        ln = int(rng.integers(0, 12_000)) if rng.random() < 0.9 else 0
        ts = min(max(qs + int(rng.integers(-3_000, 3_000)), 0), maxcoord - ln)
        rows.append((q, t, qs, min(qs + ln, maxcoord), ts, ts + ln, "+" if rng.random() < 0.6 else "-",
                     float(rng.choice([0.85, 0.9, 0.95, 1.0]))))
    rows = rows[:n]
    if shuffled:
        rows = [rows[i] for i in rng.permutation(n)]
    else:
        rows.sort(key=lambda r: (r[0], r[1], r[6]))
    names = [f"G{i * 2 // n_seq}#1#s{i}" for i in range(n_seq)]
    t = build(rows, names, MT)
    assert int(max(t.query_end.max(), t.target_end.max())) == maxcoord
    return t


@pytest.mark.parametrize("maxcoord", [(1 << 31) - 1, 1 << 31, U32_MAX])
@pytest.mark.parametrize("n_seq", [32767, 32768])
def test_key_width_63_64_65(ctx, n_seq, maxcoord):
    """kb = 2 sb + 1 + cb: 62 | 63 (sb 15), 64 (sb 16, cb 31: the key fills the word, the dead key is NONE64) and 65 (sb 16,
    cb 32: the wide path, taken without SWG_FORCE_WIDE_KEYS)."""
    kb = 2 * bits_for(n_seq) + 1 + bits_for(maxcoord)
    assert kb in (62, 63, 64, 65)
    for shuffled in (False, True):
        t = wide_coord_table(n_seq, maxcoord, 300, seed=n_seq + maxcoord, shuffled=shuffled)
        for name, flags in DEFAULT_CASES.items():
            check(ctx, cli(**flags), t, f"kb {kb} shuffled={shuffled} {name}")


@pytest.mark.parametrize("n", [64, 65, 128, 129])
def test_packed_sort_start_moves(ctx, n):
    """n_seq 3000 (sb 12) with cb 32: kb = 57, and kb + ib = 63 | 64 | 64 | 65 at N = 64 | 65 | 128 | 129, so the packed
    LSD sort starts packing at a different digit on either side.  Shuffled rows: the LSD passes, not the group sort."""
    t = wide_coord_table(3000, U32_MAX, n, seed=n, shuffled=True)
    for name, flags in DEFAULT_CASES.items():
        _, _, st = check(ctx, cli(**flags), t, f"N {n} {name}")
        if name == "defaults":
            assert st.n_sort_passes > 0


# ---- (c) arithmetic at the limits -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fixpoint", [False, True])
@pytest.mark.parametrize("G", [50_000, 1000, (1 << 31) - 1])
def test_chaining_gap_limits(ctx, G, fixpoint, monkeypatch):
    """Gaps of exactly G and G + 1, overlaps of G/5 and G/5 + 1 on both axes and strands, at the top of the u32 range (where
    a.query_end + G passes 2^32) and at 0; G up to 2^31 - 1, the largest --scaffold-jump accepted.  Once as shipped and once
    through the fixed point, whose target-bucket widths follow from G."""
    if fixpoint:
        monkeypatch.setenv("SWG_FIXPOINT_MIN", "2")
        monkeypatch.setenv("SWG_FIXPOINT_VERIFY", "1")
    for top in (True, False):
        t, joined = gap_table(G, MT, top=top)
        cfg = cli(scaffold_jump=str(G), scaffold_mass="0")
        assert cfg.scaffold_gap == G
        _, chain, st = check(ctx, cfg, t, f"G {G} top={top} fixpoint={fixpoint}")
        assert [chain[2 * k] == chain[2 * k + 1] for k in range(len(joined))] == joined
        check(ctx, cli(scaffold_jump=str(G), scaffold_mass="0", scaffold_dist=str(min(G, (1 << 31) - 1))), t, f"G {G} rescue")


@pytest.mark.parametrize("knobs", ["walk", "grid", "grid_nodiag"])
@pytest.mark.parametrize("G", [50_000, 7, (1 << 31) - 1])
def test_inversion_capture_at_G(ctx, G, knobs, monkeypatch):
    """'-' mappings at floor(|dev| / sqrt 2) = G - 1, G, G + 1 against a kept '+' chain, |dev| up to ~3.04e9: through the
    plain walk and the bucketed capture, with and without the diagonal buckets."""
    if knobs != "walk":
        monkeypatch.setenv("SWG_INV_GRID", "1")
    if knobs == "grid_nodiag":
        monkeypatch.setenv("SWG_INV_NO_DIAG", "1")
    t, devs = inversion_table(G, MT)
    s, c, _ = check(ctx, cli(scaffold_jump=str(G)), t, f"inversion G {G} {knobs}")
    assert 0 < int((s[1::2] == 1).sum()) < len(devs)


def overlap_table():
    """Two long intervals per pair whose overlap / shorter length is a threshold exactly (a tie: not "greater than") or one
    base either side, on the query axis and, in other pairs, on the target axis: 19k / 20k against 0.95 with k = 2^27 (the
    f64 quotient rounds to f64(0.95)) and m / 2m against 0.5 with m = 2^30.  Returns the table and, per pair, (axis, threshold,
    e): e = -1 overlaps by one base more than the tie, e = +1 by one less."""
    k, m = 1 << 27, 1 << 30
    specs = []  # (a, b) intervals on the swept axis, threshold, e
    for e in (-1, 0, 1):
        specs.append(((0, 20 * k), (k + e, 21 * k + e), 0.95, e))
        specs.append(((0, 2 * m), (m + e, 3 * m + e), 0.5, e))
        specs.append(((U32_MAX - 21 * k, U32_MAX - k), (U32_MAX - 20 * k + e, U32_MAX + min(e, 0)), 0.95, e))
    rows, cases = [], []
    p = 0
    for axis in ("q", "t"):
        for a, b, thr, e in specs:
            short_a, short_b = (5_000, 6_000), (3_000_000, 3_001_000)  # the other axis: apart
            for (iv, other, idy) in ((a, short_a, 0.95), (b, short_b, 0.9)):
                q, t = (iv, other) if axis == "q" else (other, iv)
                rows.append((2 * p, 2 * p + 1, q[0], q[1], t[0], t[1], "+", idy))
            cases.append((axis, thr, e))
            p += 1
    return build(rows, [f"{'AB'[i % 2]}#1#c{i // 2}" for i in range(2 * p)], MT), cases


@pytest.mark.parametrize("tree", [False, True])
@pytest.mark.parametrize("mode", ["1:1", "1", "2:2"])
def test_sweep_overlap_ties_with_long_intervals(ctx, mode, tree, monkeypatch):
    """The sweep's overlap test ol / ml > threshold at lengths near 2^32, n = 1 (flat kernel, or every group through the
    segment tree) and n = 2.  Where the swept axis keeps one mapping, the weaker interval b of a pair is dropped one base
    beyond the tie and kept at the tie and one base short of it; with n = 2 (or no limit on that axis, the target axis of
    "1") both stay among the best and the overlap test never runs."""
    if tree:
        monkeypatch.setenv("SWG_SWEEP_TREE_ALL", "1")
    t, cases = overlap_table()
    for thr in (0.95, 0.5):
        for jump in ("0", "50k"):
            s, _, _ = check(ctx, cli(num_mappings=mode, overlap=thr, scaffold_jump=jump, scaffold_mass="0"), t, f"{mode} thr {thr} jump {jump}")
            assert (s[0::2] != 0).all()
            for p, (axis, thr_p, e) in enumerate(cases):
                one = mode == "1:1" or (mode == "1" and axis == "q")
                if thr_p == thr:
                    assert (s[2 * p + 1] != 0) == (not one or e >= 0), f"{mode} thr {thr} jump {jump}: pair {p} ({axis}), e = {e}"


def check_rescue_gpu(ctx, t, anchors, D, what):
    s, c, st = check(ctx, cli(scaffold_dist=str(D)), t, what)
    for i, a in expected_rescue(t, anchors, D).items():
        assert (s[i], c[i]) == ((2, c[a]) if a is not None else (0, 0)), f"{what}: record {i}"
    return s, c, st


def test_rescue_wrapped_distance(ctx):
    """qd^2 + td^2 past 2^64: the reference's u64 sum wraps, and the wrapped distance can rescue a mapping ~4.29e9 away in
    truth.  The anchor on either side of the query centre, and a wrapped anchor further out than a near unwrapped one, on
    either side (each of the kernel's two shortcuts would lose one of these cases)."""
    t, D, anchors = rescue_wrap_table(MT)
    s, c, st = check_rescue_gpu(ctx, t, anchors, D, "wrap")
    assert s[1] == 2 and c[1] == 1 and st.n_rescued == 5
    # the fixed point and the bucketed inversion capture in front of it change nothing
    for k, v in (("SWG_FIXPOINT_MIN", "2"), ("SWG_INV_GRID", "1")):
        with pytest.MonkeyPatch.context() as mp:
            mp.setenv(k, v)
            check_rescue_gpu(ctx, t, anchors, D, f"wrap {k}")


@pytest.mark.parametrize("D", [(1 << 31) - 1, (1 << 31) - 2, 3_037_000, 1_000_000, 1000])
def test_rescue_distance_at_D(ctx, D):
    """Floored distances D - 1, D, D + 1 from the f64 root of the rounded sum; a candidate between two anchors at equal
    distance takes the anchor of the smaller index."""
    t, anchors = rescue_limit_table(D, MT)
    s, c, _ = check_rescue_gpu(ctx, t, anchors, D, f"D {D}")
    assert 0 < int((s == 2).sum()) < t.n - len(anchors)


@pytest.mark.parametrize("field", ["scaffold_gap", "scaffold_max_deviation"])
def test_gap_and_deviation_limits(ctx, field):
    """Both limits are 2^31 - 1: one more is refused with SWG_ERR_RANGE (-2), not computed with a wrapped 32-bit gap."""
    t, _, _ = rescue_wrap_table(MT)
    cfg = swg.FilterConfig(**{field: (1 << 31) - 1})
    check(ctx, cfg, t, f"{field} = 2^31 - 1")
    with pytest.raises(swg.SwgError) as e:
        ctx.filter(swg.FilterConfig(**{field: 1 << 31}), t)
    assert e.value.code == -2


# ---- (d) translation invariance at scale ------------------------------------------------------------------------------------
def shifted_to_top(t):
    """Every coordinate of a sequence moved by one per-sequence constant so that its largest end is 2^32 - 1: no gap,
    overlap, span, centre difference or diagonal difference changes."""
    end = np.zeros(t.n_seq, np.int64)
    np.maximum.at(end, t.query_id, t.query_end.astype(np.int64))
    np.maximum.at(end, t.target_id, t.target_end.astype(np.int64))
    sh = U32_MAX - end
    q, g = sh[t.query_id], sh[t.target_id]
    return MT(t.query_id, t.target_id, t.query_start + q, t.query_end + q, t.target_start + g, t.target_end + g, t.block_length,
              t.matches, t.identity, t.strand, t.seq_genome_id, t.seq_genome2_id, t.score, t.names)


@pytest.mark.parametrize("which", ["pansn3m", "skew200k"])
def test_translation_invariance(ctx, which):
    """Status and chain ids do not move when every sequence is shifted to end at 2^32 - 1 (cb 28 -> 32: every key layout, the
    anchor keys, the diagonal-bucket width and the fixed point's bucket directory change).  The skew table's pile takes the
    fixed point as shipped and the bucketed inversion capture."""
    t = synth.pansn(3_000_000, seed=13, n_hap=12) if which == "pansn3m" else synth.skew(n_pile=200_000, n_tiny_groups=20_000, seed=5)
    t2 = shifted_to_top(t)
    assert int(max(t2.query_end.max(), t2.target_end.max())) == U32_MAX
    for name in ("defaults", "rescue100k", "1:1_1:1"):
        cfg = cli(**DEFAULT_CASES[name])
        s1, c1, st1 = ctx.filter(cfg, t)
        s2, c2, st2 = ctx.filter(cfg, t2)
        bad = np.nonzero((s1 != s2) | (c1 != c2))[0]
        assert bad.size == 0, f"{which} {name}: {bad.size} records differ after the shift, first {bad[:10]}"
        for f in ("n_stage1", "n_after_sweep", "n_chains", "n_chains_after_mass", "n_chains_kept", "n_rescued", "n_kept"):
            assert getattr(st1, f) == getattr(st2, f), f"{which} {name}: {f}"
        assert st1.n_kept > 0


# ---- (e) PAF front ends at the u32 edge -------------------------------------------------------------------------------------
def test_paf_coordinates_at_the_u32_edge(ctx, tmp_path):
    """4294967295 is a coordinate; 4294967296 is beyond the table, an error only if its line passes the retain.  Device
    tokeniser and host front end against the oracle, byte for byte."""
    M = U32_MAX
    good = (f"q#1#c\t{M + 1}\t{M - 5000}\t{M}\t+\tt#1#c\t{M + 1}\t{M - 5000}\t{M}\t4900\t5000\t60\n"
            f"q#1#c\t{M + 1}\t{M - 12000}\t{M - 6000}\t+\tt#1#c\t{M + 1}\t{M - 12010}\t{M - 6010}\t5900\t6000\t60\n"
            f"q#1#c\t{M + 1}\t0\t{M}\t-\tt#1#c\t{M + 1}\t0\t{M}\t{M - 7}\t{M}\t60\n"
            f"q#1#c\t{M + 1}\t{M}\t{M}\t+\tt#1#c\t{M + 1}\t{M}\t{M}\t0\t1\t60\n")
    bad = f"q#1#c\t{M + 1}\t{M - 10}\t{M + 1}\t+\tt#1#c\t{M + 1}\t0\t11\t5\t11\t60\n"  # beyond u32, block length 11
    src, out, ref = tmp_path / "in.paf", tmp_path / "out.paf", tmp_path / "ref.paf"
    src.write_text(good)
    for flags in ({}, dict(scaffold_mass="0"), dict(num_mappings="1:1", scaffold_filter="1:1"), dict(scaffold_dist="100k")):
        f = swg.PafFilter(cli(**flags))
        f._ctx = ctx
        for host in (False, True):
            f.filter_paf(str(src), str(out), host_frontend=host)
            oracle_lib.filter_paf(f.config, str(src), str(ref))
            assert out.read_bytes() == ref.read_bytes(), (flags, host)
    src.write_text(good + bad + good)
    f = swg.PafFilter(cli(min_aln_length="1k", scaffold_mass="0"))
    f._ctx = ctx
    for host in (False, True):
        f.filter_paf(str(src), str(out), host_frontend=host)
        oracle_lib.filter_paf(f.config, str(src), str(ref))
        assert out.read_bytes() == ref.read_bytes() and out.read_bytes().count(b"\n") > 0, host
    f2 = swg.PafFilter(cli(scaffold_mass="0"))
    f2._ctx = ctx
    for host in (False, True):
        with pytest.raises(swg.SwgError) as e:
            f2.filter_paf(str(src), str(out), host_frontend=host)
        assert e.value.code == -2
