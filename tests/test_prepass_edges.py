"""The ANI pre-pass (calculate_ani_stats / calculate_ani_n_percentile, src/main.rs:334-688) and the tree filter
(apply_tree_filter_to_paf, src/tree_filter.rs:205-283) restated in plain Python, at the inputs where their f64 and u64
arithmetic changes behaviour: sums past 2^53 and 2^64, cuts landing exactly on the threshold, NaN and signed-zero keys,
ties decided by stable order or by name, 20-digit columns, fractions at the edges of the hash threshold.

The reference has no tests for either pre-pass, so the restatement here pins the oracle (CPU tests) and the device must
equal both (GPU tests): the same (ani50, n_pairs) bit for bit or all three raise; the same output bytes and
(kept, selected)."""
import functools
import math
import operator
import random
import re
from fractions import Fraction

import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from sweepga_b200._lib import ERR_RANGE

from test_ani_gpu import pansn_paf

U64 = 1 << 64


# ---- the plain restatement --------------------------------------------------------------------------------------
def parse_u64(s):  # str::parse::<u64>: an optional '+', then digits, at most 2^64 - 1
    return int(s) if re.fullmatch(rb"\+?[0-9]+", s) and int(s) < U64 else None


_F64 = re.compile(rb"[+-]?(?:inf|infinity|nan|(?:[0-9]+\.?[0-9]*|\.[0-9]+)(?:e[+-]?[0-9]+)?)", re.I)


def parse_f64(s):  # str::parse::<f64>; float() alone would also take '_' and surrounding whitespace
    return float(s) if _F64.fullmatch(s) else None


def prefix_p(n):  # up to and including the last '#' (main.rs:424-433)
    p = n.rfind(b"#")
    return n if p < 0 else n[: p + 1]


def prefix_p2(n):  # extract_genome_prefix, tree_filter.rs:15-25: the first two '#' fields
    p = n.find(b"#")
    if p < 0:
        return n
    p2 = n.find(b"#", p + 1)
    return n[:p] + b"#" + (n[p + 1:] if p2 < 0 else n[p + 1:p2]) + b"#"


def rust_max(x, y):  # f64::max: a NaN argument yields the other one
    return y if math.isnan(x) else max(x, y)


def rust_ln(x):
    return -math.inf if x == 0 else math.nan if x < 0 or math.isnan(x) else math.log(x)


class Panic(Exception):
    """partial_cmp(..).unwrap() on a NaN: the reference panics."""


def paf_lines(text):  # BufRead::lines() without empty and '#' lines, split on tabs
    for line in text.split(b"\n"):
        line = line[:-1] if line.endswith(b"\r") else line
        if line and line[:1] != b"#":
            yield line, line.split(b"\t")


def ani_ref(text, method, pct=0.0, sort=1, details=None, sort_key=None):
    """method 0 = all, 2 = nX with sort 0 length / 1 identity / 2 score -> (ani50, n_pairs); raises Panic."""
    alns, sizes = [], {}
    for _, f in paf_lines(text):
        if len(f) < 11:
            continue
        qg, tg = prefix_p(f[0]), prefix_p(f[5])
        if qg == tg:
            continue
        if method == 2:  # main.rs:560-575: keyed by genome + the last '#' field, first appearance wins
            for n, g, col in ((f[0], qg, f[1]), (f[5], tg, f[6])):
                sizes.setdefault(g + n.rsplit(b"#", 1)[-1], parse_u64(col) or 0)
        m, b = parse_f64(f[9]), parse_f64(f[10])
        m, b = 0.0 if m is None else m, 1.0 if b is None else b
        fm = m
        for tag in f[11:]:  # the first dv:f: tag that parses
            dv = parse_f64(tag[5:]) if tag[:5] == b"dv:f:" else None
            if dv is not None:
                fm = (1.0 - dv) * b
                break
        alns.append((min(qg, tg), max(qg, tg), fm, b, fm / rust_max(b, 1.0)))
    if not alns:
        return 0.0, 0
    take = len(alns)
    if method == 2:
        key = [lambda a: a[3], lambda a: a[4], lambda a: a[4] * rust_max(rust_ln(a[3]), 1.0)][sort]
        if any(math.isnan(key(a)) for a in alns):
            raise Panic
        alns = sorted(alns, key=sort_key or key, reverse=True)  # stable, like Vec::sort_by
        thr = float(sum(sizes.values())) * (pct / 100.0)  # sizes are kept order-independent by the corpora
        cum, take = 0.0, 0
        for a in alns:  # the alignment that crosses the threshold is counted
            cum += a[3]
            take += 1
            if cum >= thr:
                break
    pairs = {}
    for a in alns[:take]:
        pairs.setdefault((a[0], a[1]), []).append(a)
    ani = []
    for v in pairs.values():
        sm = sb = 0.0
        for a in v:  # sequential f64 sums in accumulation order
            sm += a[2]
            sb += a[3]
        ani.append(sm / sb if sb > 0 else 0.0)
    if any(math.isnan(x) for x in ani):
        raise Panic
    ani.sort()
    mid = len(ani) // 2
    if details is not None:
        details.update(take=take, pairs=pairs, order=alns)
    return ((ani[mid - 1] + ani[mid]) / 2.0 if len(ani) % 2 == 0 and len(ani) > 1 else ani[mid]), len(ani)  # main.rs:490-495


def fsum_seq(xs):  # a sequential f64 sum (the built-in sum() of floats is compensated)
    return functools.reduce(operator.add, xs, 0.0)


def f64_identity(ms, bs):  # tree_filter.rs:58-59: `as f64` addends summed in file order
    sm, sb = fsum_seq(map(float, ms)), fsum_seq(map(float, bs))
    return sm / sb if sb > 0 else 0.0


def tree_ref(text, k_nearest, k_farthest=0, fraction=0.0, identity=f64_identity):
    """-> (output bytes, (kept, selected)).  identity(matches, blocks) of a pair's records in file order: the reference's
    f64 sums unless a model of another implementation is passed."""
    recs = []
    for line, f in paf_lines(text):
        if len(f) < 11:
            continue
        m, b = parse_u64(f[9]), parse_u64(f[10])
        recs.append((line, prefix_p2(f[0]), prefix_p2(f[5]), 0 if m is None else m, 1 if b is None else b))
    sums = {}
    for _, q, t, m, b in recs:
        if q != t:
            s = sums.setdefault((min(q, t), max(q, t)), ([], []))
            s[0].append(m)
            s[1].append(b)
    nb = {}
    for (a, b), (ms, bs) in sums.items():
        ident = identity(ms, bs)
        nb.setdefault(a, []).append((b, ident))
        nb.setdefault(b, []).append((a, ident))
    sel = set()
    for g, v in nb.items():
        v.sort(key=lambda x: (-x[1], x[0]))  # identity descending, then neighbour name as bytes
        near, far = v[:k_nearest], v[::-1][:k_farthest]
        sel.update((min(g, o), max(g, o)) for o, _ in near + far)
    if fraction > 0:
        t = fraction * 2.0 ** 64
        thr = U64 - 1 if t >= 2.0 ** 64 else int(t)  # `as u64` saturates
        sel.update(p for p in sums if oracle_lib.siphash13(p[0] + b"\xff" + p[1] + b"\xff") <= thr)
    out = [line for line, q, t, _, _ in recs if q != t and (min(q, t), max(q, t)) in sel]
    return b"".join(x + b"\n" for x in out), (len(out), len(sel))


def u64_identity(ms, bs):  # u64 sums converted once: wraps past 2^64, rounds differently past 2^53
    sm, sb = sum(ms) % U64, sum(bs) % U64
    return float(sm) / float(sb) if sb > 0 else 0.0


def split_identity(shift=32, limit=1 << 53):
    """The device's fast path: sums of the high and of the low 32-bit halves, rebuilt as hi << shift + lo; a pair total at
    or past `limit` sends the call to the sequential f64 sums.  shift 32 and limit 2^53 are the device's; other values
    model a wrong one."""
    def identity(ms, bs):
        tm = (sum(v >> 32 for v in ms) << shift) + sum(v & 0xFFFFFFFF for v in ms)
        tb = (sum(v >> 32 for v in bs) << shift) + sum(v & 0xFFFFFFFF for v in bs)
        if tm >= limit or tb >= limit:
            return f64_identity(ms, bs)
        return float(tm) / float(tb) if tb > 0 else 0.0
    return identity


def exact_pair_sums(pairs):  # the same sums without rounding: the corpora assert that they differ from the f64 ones
    return {p: (sum(Fraction(a[2]) for a in v), sum(Fraction(a[3]) for a in v)) for p, v in pairs.items()}


# ---- corpora ----------------------------------------------------------------------------------------------------
def L(q, t, m, b, ql=100, tl=100, tags=()):
    return "\t".join([q, str(ql), "0", "10", "+", t, str(tl), "0", "10", str(m), str(b), "60", *tags])


def paf(lines):
    return ("\n".join(lines) + "\n").encode()


def tree_wrap():  # three 9e18 block lengths wrap a u64 sum: A's nearest neighbour would become B instead of C
    big = [L("A#1#c", "B#1#c", 4500000000000000000, 9000000000000000000)] * 3
    return paf(big + [L("A#1#c", "C#1#c", 9, 10), L("B#1#c", "D#1#c", 99, 100), L("C#1#c", "D#1#c", 99, 100)])


def tree_ulp():
    """(2^60 + 100) + 100 in f64 stays 2^60; the exact 2^60 + 200 rounds to 2^60 + 256, one ulp more.  A-B is then a tie
    with A-C at 0.5 (broken by name: B) or just below it (C); B and C both prefer D."""
    ab = [L("A#1#c", "B#1#c", 2 ** 59, 2 ** 60), L("A#1#c", "B#1#c", 0, 100), L("A#1#c", "B#1#c", 0, 100)]
    return paf(ab + [L("A#1#c", "C#1#c", 1, 2), L("B#1#c", "D#1#c", 9, 10), L("C#1#c", "D#1#c", 9, 10)])


def tree_high_halves():
    """Every matches and block length in [2^32, 2^34), pair totals below 2^53: the fast path with non-zero high halves.
    Runs of 40 to 100 records per pair (several warps add into each), identities within 2 % of each other so that the
    neighbour order rests on the low halves as much as on the high ones."""
    rng = random.Random(29)
    lines = []
    gs = "ABCDEFG"
    for i, a in enumerate(gs):
        for b in gs[i + 1:]:
            ident = rng.uniform(0.9, 0.92)
            for _ in range(rng.randrange(40, 101)):
                bl = rng.randrange(1 << 32, 1 << 34)
                m = max(int(bl * rng.uniform(ident - 0.05, min(ident + 0.05, 1.0))), 1 << 32)
                lines.append(L(f"{a}#1#c{rng.randrange(2)}", f"{b}#1#c{rng.randrange(2)}", m, bl))
    rng.shuffle(lines)
    return paf(lines)


def tree_tie_2p53():
    """2^53 + 1 + 1 stays 2^53 in f64; the exact 2^53 + 2 is representable.  A-B is a tie with A-C at 0.5 (broken by name:
    B) in f64 and just below it in exact arithmetic (C): the sequential path must start at 2^53, not above."""
    ab = [L("A#1#c", "B#1#c", 2 ** 52, 2 ** 53), L("A#1#c", "B#1#c", 0, 1), L("A#1#c", "B#1#c", 0, 1)]
    return paf(ab + [L("A#1#c", "C#1#c", 1, 2), L("B#1#c", "D#1#c", 9, 10), L("C#1#c", "D#1#c", 9, 10)])


def tree_u64_columns():  # 20 digits: the host patch (u64::MAX parses, 2^64 is Err -> 0 / 1); 19 digits parse on the device
    mx, over = "18446744073709551615", "18446744073709551616"
    lines = [L("A#1#c", "B#1#c", mx, mx), L("A#1#c", "B#2#c", mx, mx), L("A#1#c", "C#1#c", over, 10), L("A#1#c", "D#1#c", 5, over),
             L("B#1#c", "C#1#c", 9, 10), L("B#1#c", "D#1#c", 3, 4), L("C#1#c", "D#1#c", "00000000000000000007", 10),
             L("C#1#c", "B#2#c", "9999999999999999999", "9999999999999999999"), L("D#1#c", "B#2#c", over, over), L("A#1#d", "B#2#c", mx, 1)]
    return paf(lines)


def tree_names():  # equal identities: neighbours ordered by name as bytes, non-ASCII included
    gs = ["Z", "a", "z", "ä", "é", "Ω", "中", "aé"]
    rng = random.Random(21)
    lines = []
    for i, a in enumerate(gs):
        for b in gs[i + 1:]:
            m, bl = (1, 2) if rng.random() < 0.7 else (rng.randrange(1, 9), 10)
            lines += [L(f"{a}#1#chr{rng.randrange(2)}", f"{b}#1#chr{rng.randrange(2)}", m, bl) for _ in range(rng.randrange(1, 3))]
    rng.shuffle(lines)
    return paf(lines)


def tree_small(seed=22, n_gen=6, n=60):
    rng = random.Random(seed)
    lines = []
    for _ in range(n):
        a, b = rng.randrange(n_gen), rng.randrange(n_gen)
        bl = rng.randrange(1, 1000)
        lines.append(L(f"g{a}#1#c{rng.randrange(3)}", f"g{b}#1#c{rng.randrange(3)}", rng.randrange(bl + 1), bl))
    return paf(lines)


# SipHash-1-3 of b"edge604#1#\xffzz#1#\xff" is 0x319b88bf332468: 53 significant bits, so EDGE * 2^64 is that hash exactly
EDGE_HASH = 0x319B88BF332468
EDGE = EDGE_HASH / 2.0 ** 64


def tree_hash_edge():  # `<=` is inclusive: EDGE selects the pair, the next fraction below does not
    lines = [L("edge604#1#c", "zz#1#c", 5, 10), L("other#1#c", "zz#1#c", 5, 10), L("edge604#1#c", "other#1#c", 5, 10)]
    return paf(lines)


def wide_genomes(n_gen=70000, seed=24):  # more than 65 536 genomes: the pair key is wider than 32 bits
    rng = random.Random(seed)
    lines = []
    for i in range(n_gen):
        for j in (i + 1, rng.randrange(n_gen)):
            bl = rng.randrange(1, 5000)
            lines.append(L(f"g{i}#1#c", f"g{j % n_gen}#1#c", bl - rng.randrange(bl // 3 + 1), bl, ql=64, tl=64))
    return paf(lines)


TREE = {  # corpus: (builder, parameter sets (k_nearest, k_farthest, random_fraction))
    "wrap": (tree_wrap, [(1, 0, 0.0)]),
    "ulp": (tree_ulp, [(1, 0, 0.0), (0, 1, 0.0)]),
    "tie_2p53": (tree_tie_2p53, [(1, 0, 0.0)]),
    "high_halves": (tree_high_halves, [(1, 0, 0.0), (2, 1, 0.0), (3, 0, 0.0)]),
    "u64_columns": (tree_u64_columns, [(1, 0, 0.0), (1, 1, 0.0), (0, 2, 0.0), (2, 0, 0.5)]),
    "names": (tree_names, [(1, 0, 0.0), (1, 1, 0.0), (2, 2, 0.0), (3, 0, 0.0)]),
    "k_beyond": (tree_small, [(100, 0, 0.0), (0, 100, 0.0), (U64 - 1, U64 - 1, 0.0), (5, 5, 0.0)]),
    "fractions": (lambda: tree_small(23, 12, 200), [(0, 0, 0.0), (0, 0, 5e-324), (0, 0, 1.0), (0, 0, 2.0), (1, 0, 5e-324), (0, 0, 0.3)]),
    "hash_edge": (tree_hash_edge, [(0, 0, EDGE), (0, 0, float(np.nextafter(EDGE, 0.0)))]),
    "wide_genomes": (wide_genomes, [(1, 1, 0.0), (0, 0, 0.001)]),
}


def ani_cut(P, side):
    """nX: the cumulative block length reaches thr exactly at sorted position P + side (P around the 1024-record tiles).
    One genome pair, so that every record taken changes the answer."""
    rng = random.Random(P)
    recs = []
    for _ in range(3000):
        bl = rng.randrange(1, 5000)
        recs.append(("%.4f" % (bl * rng.uniform(0.5, 1.0)), bl))
    text = lambda qa, qb: paf([L("A#1#c", "B#1#c", m, bl, ql=qa, tl=qb) for m, bl in recs])
    d = {}
    ani_ref(text(1, 1), 2, 100.0, 1, details=d)
    thr = sum(int(a[3]) for a in d["order"][: P + side + 1])
    return text(2 * thr - 1, 1)  # thr = total * 0.5


def ani_cut_2p53():  # 2^53 + 1 + 1 + ... stays 2^53 in f64: the walk must be the f64 one, never reaching 2^53 + 6
    lines = [L("A#1#c", "B#1#c", "1e15", 2 ** 53, ql=2 ** 53, tl=2)]
    lines += [L("A#1#c", "BC"[i % 2] + "#1#c", "0.%d" % (i % 10), 1, ql=2 ** 53, tl=2 if i % 2 == 0 else 4) for i in range(40)]
    return paf(lines)


SPECIALS = ["12.5", "1e3", "-0.0", "-5", "inf", "-inf", "1e300", "nan", "NaN", "+infinity", "0", "1E-300"]


def ani_special(v, column):
    """One block length (column 11) or one matches value (column 10) outside the integers.  A negative or NaN block
    length keeps its key under f64::max: the identity divides by max(NaN, 1) = 1, ln(-5) is NaN and max(NaN, 1) = 1."""
    rng = random.Random(25)
    lines = [L(f"{a}#1#c", f"{b}#1#c", rng.randrange(50, 100), 100) for a, b in (rng.sample("ABCD", 2) for _ in range(20))]
    lines[7] = L("A#1#c", "B#1#c", 60, v) if column == 11 else L("C#1#c", "D#1#c", v, 80)
    return paf(lines)


def ani_zero_keys():  # identities +0.0 and -0.0 are one key: the cut falls inside their run in file order
    rng = random.Random(26)
    recs = []
    for i in range(400):
        a, b = rng.sample("ABCD", 2)
        bl = rng.randrange(1, 1000)
        recs.append((a, b, rng.choice(["0", "-0.0", "-0"]) if i % 2 else "%.3f" % (bl * rng.uniform(0.5, 1)), bl))
    text = lambda sizes: paf([L(f"{a}#1#c", f"{b}#1#c", m, bl, ql=sizes[a], tl=sizes[b]) for a, b, m, bl in recs])
    d = {}
    ani_ref(text(dict.fromkeys("ABCD", 1)), 2, 100.0, 1, details=d)
    thr = sum(int(a[3]) for a in d["order"][:300])
    return text({"A": 2 * thr - 3, "B": 1, "C": 1, "D": 1})


def ani_stable_ties():  # equal keys (one block length per pair): the file order of the matches decides the last bit
    rng = random.Random(27)
    lines = [L(f"{a}#1#c", f"{b}#1#c", "%.6f" % rng.uniform(1, 700), 700, ql=50000, tl=50000) for a, b in (rng.sample("ABCDE", 2) for _ in range(500))]
    return paf(lines)


def ani_addends():
    """Pairs of 1..7 addends (the tail of k_ani_pair_sums) and one of 2^20 + 7.  A's sequence is 10^8 long, so n100 and
    n50-length cut inside the large pair (its block lengths add up to about 1.5 * 10^8)."""
    rng = random.Random(28)
    lines = [L("P#1#c", f"Q{k}#1#c", "%.5f" % rng.uniform(10, 90), 100, tags=["dv:f:%.7f" % rng.random()]) for k in range(1, 8) for _ in range(k)]
    lines += ["A#1#c\t100000000\t0\t1\t+\tB#1#c\t9\t0\t1\t%d\t%d\t0\tdv:f:0.%04d" % (i % 97, 100 + i % 89, i % 9973) for i in range((1 << 20) + 7)]
    return paf(lines)


ANI = {  # corpus: (builder, --ani-method strings)
    **{f"cut_{P}_{s:+d}": (lambda P=P, s=s: ani_cut(P, s), ["n50"]) for P in (1023, 1024, 1025, 2047) for s in (-1, 0, 1)},
    "cut_2p53": (ani_cut_2p53, ["n100-length", "n100"]),
    **{f"special{c}_{v}": (lambda v=v, c=c: ani_special(v, c), ["all", "n50", "n50-length", "n50-score", "n100-score", "n100-length"])
       for c, vs in ((11, SPECIALS), (10, ["nan", "inf", "-0.0", "-5", "1e300"])) for v in vs},
    "zero_keys": (ani_zero_keys, ["n50"]),
    "stable_ties": (ani_stable_ties, ["n100-length", "n60-length", "all"]),
    "addends": (ani_addends, ["all", "n100", "n50-length"]),
    "wide_genomes": (wide_genomes, ["all", "n50", "n50-length"]),
}
TREE_CASES = [(n, p) for n, (_, ps) in TREE.items() for p in ps]
ANI_CASES = [(n, m) for n, (_, ms) in ANI.items() for m in ms]
_TEXT = {}


def corpus(table, name):  # the text of a corpus, built once per process
    if (id(table), name) not in _TEXT:
        _TEXT[(id(table), name)] = table[name][0]()
    return _TEXT[(id(table), name)]


def write(tmp_path, text):
    p = tmp_path / "in.paf"
    p.write_bytes(text)
    return str(p)


def run(f, *a, panic):  # -> result, or "raises" where f reports the reference's panic in its own way
    try:
        return f(*a)
    except panic as e:
        if isinstance(e, swg.SwgError) and e.code != ERR_RANGE:  # the device: SWG_ERR_RANGE, nothing else
            raise
        return "raises"


def ani_all_ways(tmp_path, text, method, ctx=None):
    m = swg.parse_ani_method(method)
    path = write(tmp_path, text)
    ref = run(ani_ref, text, *m, panic=Panic)
    orc = run(oracle_lib.ani_stats, path, *m, panic=ValueError)  # rc -2
    dev = run(swg.ani_stats, ctx, path, method, panic=swg.SwgError) if ctx is not None else None
    return ref, orc, dev


def tree_all_ways(tmp_path, text, params, ctx=None):
    src = write(tmp_path, text)
    ref = tree_ref(text, *params)
    o = tmp_path / "orc.paf"
    counts = oracle_lib.tree_filter_paf(src, str(o), *params)
    orc = (o.read_bytes(), counts)
    dev = None
    if ctx is not None:
        d = tmp_path / "dev.paf"
        got = swg.apply_tree_filter_to_paf(ctx, src, str(d), *params)
        dev = (d.read_bytes(), got)
    return ref, orc, dev


# ---- CPU: the restatement pins the oracle -----------------------------------------------------------------------
@pytest.mark.parametrize("name,params", TREE_CASES)
def test_tree_reference_equals_oracle(tmp_path, name, params):
    text = corpus(TREE, name)
    ref, orc, _ = tree_all_ways(tmp_path, text, params)
    assert ref == orc, (name, params)


@pytest.mark.parametrize("name,method", ANI_CASES)
def test_ani_reference_equals_oracle(tmp_path, name, method):
    text = corpus(ANI, name)
    ref, orc, _ = ani_all_ways(tmp_path, text, method)
    assert ref == orc and repr(ref) == repr(orc), (name, method)


@pytest.mark.parametrize("method", ["all", "n100", "n50", "n90-length", "n10-identity", "n0.5-length", "n100-length", "n50-score",
                                    "n100-score", "n30-score"])
def test_ani_reference_on_quirk_corpus(tmp_path, method):
    p = tmp_path / "a.paf"
    pansn_paf(str(p), 60000, seed=3)
    ref, orc, _ = ani_all_ways(tmp_path, p.read_bytes(), method)
    assert ref == orc and ref[1] > 10, method


@pytest.mark.parametrize("params", [(1, 0, 0.0), (2, 1, 0.0), (3, 0, 0.1), (0, 2, 0.5), (100, 0, 0.0)])
def test_tree_reference_on_quirk_corpus(tmp_path, params):
    p = tmp_path / "a.paf"
    pansn_paf(str(p), 50000, seed=11)
    ref, orc, _ = tree_all_ways(tmp_path, p.read_bytes(), params)
    assert ref == orc and ref[1][0] > 0, params


def test_corpora_reach_their_edges():
    """Each corpus exercises what it is named for: a wrong but plausible implementation gives another answer."""
    for name in ("wrap", "ulp", "tie_2p53"):  # exact u64 sums converted once select other pairs
        text = corpus(TREE, name)
        assert tree_ref(text, 1) != tree_ref(text, 1, identity=u64_identity), name
    # the split sums of the device's fast path equal the reference on every corpus; a wrong switch point or rebuild shift
    # gives another output on at least one
    out = lambda model: [tree_ref(corpus(TREE, n), *p, identity=model) for n, p in TREE_CASES]
    want = out(f64_identity)
    assert out(split_identity()) == want
    for shift, limit in ((32, 1 << 54), (32, 1 << 60), (31, 1 << 53), (33, 1 << 53)):
        assert out(split_identity(shift, limit)) != want, (shift, limit)
    vals = [int(f[c]) for _, f in paf_lines(corpus(TREE, "high_halves")) for c in (9, 10)]
    assert min(vals) >= 1 << 32 and len(vals) // 2 // 21 > 32
    assert 3 * 9000000000000000000 >= U64 and tree_ref(corpus(TREE, "wrap"), 1)[1] == (3, 3)
    assert Fraction(2 ** 60) + 200 != float(2 ** 60) + 100.0 + 100.0
    assert oracle_lib.siphash13(b"edge604#1#\xffzz#1#\xff") == EDGE_HASH and int(EDGE * 2.0 ** 64) == EDGE_HASH
    text = corpus(TREE, "hash_edge")
    assert tree_ref(text, 0, 0, EDGE)[1] == (1, 1) and tree_ref(text, 0, 0, float(np.nextafter(EDGE, 0.0)))[1] == (0, 0)
    # the nX cut: three thresholds around each position give three answers, taking P, P + 1, P + 2 records
    for P in (1023, 1024, 1025, 2047):
        got = []
        for s in (-1, 0, 1):
            d = {}
            got.append(ani_ref(corpus(ANI, f"cut_{P}_{s:+d}"), 2, 50.0, 1, details=d))
            assert d["take"] == P + s + 1
        assert len(set(got)) == 3, P
    d = {}
    text = corpus(ANI, "cut_2p53")
    ani_ref(text, 2, 100.0, 0, details=d)
    assert d["take"] == 41  # the f64 running sum never reaches 2^53 + 6 ...
    exact = list(np.cumsum([int(a[3]) for a in d["order"]], dtype=object))
    assert exact.index(2 ** 53 + 6) + 1 == 7  # ... the exact one does after 7 records
    # signed zeros: ordering -0.0 behind +0.0 would move the cut onto other records
    text = corpus(ANI, "zero_keys")
    signed = lambda a: (a[4], math.copysign(1.0, a[4]))
    assert ani_ref(text, 2, 50.0, 1) != ani_ref(text, 2, 50.0, 1, sort_key=signed)
    # equal keys: the reversed order would round differently; past 2^53 / with dv: tags the sums are not exact
    d = {}
    ani_ref(corpus(ANI, "stable_ties"), 2, 60.0, 0, details=d)
    assert 100 < d["take"] < 500
    rev = lambda v: fsum_seq(a[2] for a in reversed(v))
    fwd = {p: fsum_seq(a[2] for a in v) for p, v in d["pairs"].items()}
    assert any(rev(v) != fwd[p] for p, v in d["pairs"].items())
    d = {}
    ani_ref(corpus(ANI, "addends"), 0, details=d)
    ex = exact_pair_sums(d["pairs"])
    assert max(len(v) for v in d["pairs"].values()) > 1 << 20
    for m in ((2, 100.0, 1), (2, 50.0, 0)):  # the cuts take a large part of the large pair, not all of it
        dm = {}
        ani_ref(corpus(ANI, "addends"), *m, details=dm)
        assert 1 << 18 < len(dm["pairs"][(b"A#1#", b"B#1#")]) < 1 << 20, m
    assert any(float(ex[p][0]) != fsum_seq(a[2] for a in v) for p, v in d["pairs"].items())


def test_reference_parsers():
    assert [parse_u64(s) for s in (b"+5", b"18446744073709551615", b"18446744073709551616", b"-1", b"", b"+", b"1_0", b" 1")] == \
        [5, U64 - 1, None, None, None, None, None, None]
    ok = [b"1", b"+1.5", b"-.5", b"1.", b"1e3", b"1E-3", b"inf", b"-Infinity", b"NaN", b"+nan"]
    assert all(parse_f64(s) is not None for s in ok)
    assert all(parse_f64(s) is None for s in (b"", b".", b"1_0", b" 1", b"1e", b"e3", b"0x10", b"infinit", b"1.5 "))
    assert rust_max(math.nan, 1.0) == 1.0 and rust_ln(0.0) == -math.inf and math.isnan(rust_ln(-5.0))
    assert prefix_p(b"a#1#b#c") == b"a#1#b#" and prefix_p2(b"a#1#b#c") == b"a#1#" and prefix_p2(b"a#1") == b"a#1#"


# ---- GPU: the device equals both --------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dctx():
    with swg.Context(0) as c:
        yield c


@pytest.mark.gpu
@pytest.mark.parametrize("name,params", TREE_CASES)
def test_tree_device(dctx, tmp_path, name, params):
    text = corpus(TREE, name)
    ref, orc, dev = tree_all_ways(tmp_path, text, params, dctx)
    assert dev == ref == orc, (name, params)


@pytest.mark.gpu
@pytest.mark.parametrize("name,method", ANI_CASES)
def test_ani_device(dctx, tmp_path, name, method):
    text = corpus(ANI, name)
    ref, orc, dev = ani_all_ways(tmp_path, text, method, dctx)
    assert dev == ref == orc and repr(dev) == repr(ref), (name, method)


@pytest.mark.gpu
def test_score_key_near_tie(dctx, tmp_path, monkeypatch):
    """Two records whose nX-score keys tie under one logarithm and not under the other; the cut takes only the first, so
    the answer is the identity of whichever sorts first.  With the glibc port the device's key is the host's; with
    CUDA's log() (SWG_LOG_IMPL=cuda) it is not, and the answer changes: the test sees a wrong logarithm."""
    assert dctx.log_matches_host()
    monkeypatch.setenv("SWG_LOG_IMPL", "cuda")
    Ls = np.arange(2000, 400_000, dtype=np.uint32)
    zero = np.zeros(len(Ls), np.uint32)
    cuda = dctx.score_column(np.ones(len(Ls)), zero, Ls, 3)  # 1.0 * ln(L) with CUDA's log
    host = oracle_lib.score_column(zero, Ls, np.ones(len(Ls)), 3)
    found = None
    for k in np.nonzero(cuda != host)[0].tolist():
        T = min(float(cuda[k]), float(host[k]))
        for lb in range(int(Ls[k]) + 200, int(Ls[k]) + 4000):
            for m in (T / math.log(lb) * lb, float(np.nextafter(T / math.log(lb) * lb, 0.0)), float(np.nextafter(T / math.log(lb) * lb, 1e9))):
                if (m / lb) * math.log(lb) == T and lb - 2000 < len(Ls) and cuda[lb - 2000] == host[lb - 2000]:
                    found = (int(Ls[k]), m, lb)
                    break
            if found:
                break
        if found:
            break
    assert found, "no record hits the other key exactly"
    la, mb, lb = found
    # B first in the file: a tie keeps it first, a strictly larger key for A puts A first; thr = 100 * 1 % = 1
    text = paf([L("G1#1#c", "G2#1#c", repr(mb), lb, ql=50, tl=50), L("G1#1#c", "G2#1#c", la, la, ql=50, tl=50)])
    path = write(tmp_path, text)
    monkeypatch.setenv("SWG_LOG_IMPL", "cuda")
    cuda_ans = swg.ani_stats(dctx, path, "n1-score")
    monkeypatch.delenv("SWG_LOG_IMPL")
    ref, orc, dev = ani_all_ways(tmp_path, text, "n1-score", dctx)
    assert dev == ref == orc and ref[1] == 1
    assert cuda_ans != ref, "CUDA's log() did not flip the order of the two keys"
