"""The claim behind csrc/chain_fixpoint.cuh, checked on the CPU in plain Python: the reference's sequential best-buddy loop
(src/paf_filter.rs:784-851) is the unique solution of

    pick(i) = first arg-min_j { d(i,j) : d(i,j) < B(i,j) },   B(i,j) = min { d(i',j) : i' < i, pick(i') = j }

and re-evaluating all positions against a snapshot of the picks (Jacobi rounds), starting from the unconstrained arg-min,
ends exactly there.  Also the re-evaluation test of k_fx_check_warp: a position has to be re-evaluated iff its pick is now
blocked or a candidate ranking before its pick has become eligible.  No GPU, no product code: a model of the algorithm."""
import numpy as np
import pytest

NONE = -1


def gaps(a, b, fwd, G):
    """d(i,j) under the gap rule of paf_filter.rs:799-843, or None."""
    g5 = G // 5
    q = b[0] - a[1] if b[0] >= a[1] else (a[1] - b[0] if a[1] - b[0] <= g5 else G + 1)
    if fwd:
        r = b[2] - a[3] if b[2] >= a[3] else (a[3] - b[2] if a[3] - b[2] <= g5 else G + 1)
    else:
        r = a[2] - b[3] if a[2] >= b[3] else (b[3] - a[2] if b[3] - a[2] <= g5 else G + 1)
    return q * q + r * r if q <= G and r <= G else None


def candidates(rec, fwd, G):
    n = len(rec)
    out = []
    for i in range(n):
        c = []
        for j in range(i + 1, n):
            if rec[j][0] > rec[i][1] + G:
                break
            d = gaps(rec[i], rec[j], fwd, G)
            if d is not None:
                c.append((d, j))
        out.append(c)
    return out


def sequential(cands):
    """The reference's loop: strict '<' on both tests, first minimal j wins, the displaced predecessor gets no second pick."""
    n = len(cands)
    bps = [None] * n
    pick = [NONE] * n
    for i in range(n):
        best = None
        for d, j in cands[i]:
            if (best is None or d < best[0]) and (bps[j] is None or d < bps[j]):
                best = (d, j)
        if best:
            bps[best[1]] = best[0]
            pick[i] = best[1]
    return pick


def evaluate(i, cands, pickers):
    """arg-min over the candidates of i that are eligible against the snapshot `pickers[j]` = [(i', d')]."""
    best = None
    for d, j in cands[i]:
        blocked = any(ip < i and dp <= d for ip, dp in pickers[j])
        if not blocked and (best is None or (d, j) < best):
            best = (d, j)
    return best


def fixed_point(cands, exact_test):
    n = len(cands)
    cur = [min(c) if c else None for c in cands]  # unconstrained arg-min: smallest d, then smallest j
    rounds = evals = 0
    while True:
        pickers = [[] for _ in range(n)]
        for i, b in enumerate(cur):
            if b:
                pickers[b[1]].append((i, b[0]))
        todo = []
        for i in range(n):
            if exact_test:
                b = cur[i]
                need = b is not None and any(ip < i and dp <= b[0] for ip, dp in pickers[b[1]])
                if not need:  # X(i): the candidates ranking before the pick
                    for d, j in cands[i]:
                        if (b is None or (d, j) < b) and not any(ip < i and dp <= d for ip, dp in pickers[j]):
                            need = True
                            break
                if need:
                    todo.append(i)
            else:
                todo.append(i)
        changed = 0
        new = list(cur)
        for i in todo:
            new[i] = evaluate(i, cands, pickers)
            changed += new[i] != cur[i]
        evals += len(todo)
        if exact_test:
            assert changed == len(todo), "the re-evaluation test listed a position whose pick did not change"
        cur = new
        rounds += 1
        if changed == 0:
            return [b[1] if b else NONE for b in cur], rounds, evals
        assert rounds <= n + 1


def random_group(rng, n, span, max_len, jitter):
    qs = np.sort(rng.integers(0, span, n))
    ln = rng.integers(1, max_len + 1, n)
    diag = rng.random(n) < 0.6
    ts = np.where(diag, qs + rng.integers(-jitter, jitter + 1, n), rng.integers(0, span, n))
    ts = np.maximum(ts, 0)
    return [(int(a), int(a + l), int(t), int(t + l)) for a, l, t in zip(qs, ln, ts)]


@pytest.mark.parametrize("seed", range(24))
def test_jacobi_rounds_end_in_the_sequential_picks(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(2, 220))
    rec = random_group(rng, n, span=[300, 2000, 20000][seed % 3], max_len=[20, 200][seed % 2], jitter=[3, 40][(seed // 2) % 2])
    G = [50, 400, 5000][seed % 3]
    for fwd in (True, False):
        c = candidates(rec, fwd, G)
        ref = sequential(c)
        full, rounds, _ = fixed_point(c, exact_test=False)
        assert full == ref
        lean, rounds2, evals = fixed_point(c, exact_test=True)
        assert lean == ref and rounds2 == rounds  # the exact test re-evaluates fewer positions, never different ones


def test_ties_and_duplicates():
    # identical records: every d ties, "first minimal j" decides; the chain 0 -> 1 -> 2 -> ... comes out of round 0
    rec = [(100, 110, 100, 110)] * 40
    c = candidates(rec, True, 50)
    assert fixed_point(c, True)[0] == sequential(c) == list(range(1, 40)) + [NONE]
    # a contested successor: the closer, later predecessor displaces the earlier one, which gets no second pick
    rec = [(0, 10, 0, 10), (2, 12, 2, 12), (30, 40, 30, 40), (31, 41, 200, 210)]
    c = candidates(rec, True, 50)
    assert fixed_point(c, True)[0] == sequential(c)


# ---- the search in target-bucket order (fx_bucket_pass) and the verdict from the packed snapshot (fx_eligible_packed) -------------

def packed_verdict(i, d, lst):
    """`lst` = pickers of j in position order [(i', d')].  The shortcuts of fx_eligible_packed, then the binary search over the
    prefix minima; must equal the plain rule 'no earlier picker with d' <= d'."""
    if not lst:
        return True
    minpd = min(dp for _, dp in lst)
    if d < minpd:
        return True
    minpi = min(ip for ip, dp in lst if dp == minpd)
    fp, fd = lst[0]
    if minpi < i:
        return False
    if minpi == i or fp >= i:
        return True
    if fd <= d:
        return False
    if len(lst) <= 2:
        return True
    pm, m = [], None
    for _, dp in lst:
        m = dp if m is None else min(m, dp)
        pm.append(m)
    lo, hi = 0, len(lst)
    while lo < hi:  # first entry at or after i
        mid = (lo + hi) // 2
        if lst[mid][0] < i:
            lo = mid + 1
        else:
            hi = mid
    return not (lo > 0 and pm[lo - 1] <= d)


def bucket_search(i, rec, fwd, G, pickers, shift, rounds_of=4):
    """pick of position i: buckets of the candidate's target coordinate t' (start on '+', end on '-') visited outwards from the one
    that holds i's own te / ts, a direction ends at the first bucket whose nearest edge is further than sqrt(best d); inside a
    bucket the entries are in position order, scanned outwards from the first with query_start >= query_end(i) in rounds, pruned
    by q_gap^2 + r_min^2 > best d at the START of a round (the kernel prunes per round too).  Returns ((d, j) or None, visited)."""
    n = len(rec)
    g5 = G // 5
    a = rec[i]
    tp = [r[2] if fwd else r[3] for r in rec]
    buckets = {}
    for k in range(n):
        buckets.setdefault(tp[k] >> shift, []).append(k)  # position order inside a bucket
    c = a[3] if fwd else a[2]
    below, above = (g5, G) if fwd else (G, g5)
    blo, bhi = max(c - below, 0) >> shift, (c + above) >> shift
    bc = c >> shift
    W = 1 << shift
    best = None
    visited = 0

    def consider(j):
        nonlocal best
        d = gaps(a, rec[j], fwd, G)
        if d is not None and j > i and (best is None or (d, j) < best) and packed_verdict(i, d, pickers[j]):
            best = (d, j)

    live = [True, True]
    step = 0
    while live[0] or live[1]:
        for side in (0, 1):
            if (side and step == 0) or not live[side]:
                continue
            b = bc - step if side else bc + step
            if b < blo or b > bhi:
                live[side] = False
                continue
            rmin = 0 if step == 0 else (c - ((b + 1) * W - 1) if side else b * W - c)
            if best is not None and rmin * rmin > best[0]:
                live[side] = False
                continue
            ent = buckets.get(b, [])
            org = 0
            while org < len(ent) and rec[ent[org]][0] < a[1]:
                org += 1
            x = org
            while x < len(ent):  # right of the origin
                bd = best[0] if best else None
                chunk = ent[x:x + rounds_of]
                for j in chunk:
                    qg = rec[j][0] - a[1]
                    if qg <= G and (bd is None or qg * qg + rmin * rmin <= bd):
                        visited += 1
                        consider(j)
                qg = rec[chunk[-1]][0] - a[1]
                if len(chunk) < rounds_of or not (qg <= G and (bd is None or qg * qg + rmin * rmin <= bd)):
                    break
                x += rounds_of
            x = org
            while x > 0:  # left of the origin: overlaps, positions descend
                bd = best[0] if best else None
                chunk = ent[max(0, x - rounds_of):x][::-1]
                ok = True
                for j in chunk:
                    ov = a[1] - rec[j][0]
                    ok = ov <= g5 and (bd is None or ov * ov + rmin * rmin <= bd) and j > i
                    if ok:
                        visited += 1
                        consider(j)
                if len(chunk) < rounds_of or not ok:
                    break
                x -= rounds_of
        step += 1
    return best, visited


@pytest.mark.parametrize("seed", range(16))
def test_bucket_order_search_equals_the_window_scan(seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(2, 160))
    rec = random_group(rng, n, span=[300, 2000, 20000][seed % 3], max_len=[20, 200][seed % 2], jitter=[3, 40][(seed // 2) % 2])
    if seed % 4 == 0:  # zero-length records share a start with earlier positions
        rec = sorted(rec + [(r[0], r[0], r[2], r[2]) for r in rec[::5]])
        n = len(rec)
    G = [50, 400, 5000][seed % 3]
    for fwd in (True, False):
        c = candidates(rec, fwd, G)
        # a snapshot in the middle of the iteration: the sequential picks of a random half, unconstrained picks elsewhere
        seq = sequential(c)
        pickers = [[] for _ in range(n)]
        for i in range(n):
            b = None
            if rng.random() < 0.5:
                b = next(((d, j) for d, j in c[i] if j == seq[i]), None)
            elif c[i]:
                b = min(c[i])
            if b:
                pickers[b[1]].append((i, b[0]))
        total = 0
        for shift in (0, 3, 6, 20):
            for i in range(n):
                want = evaluate(i, c, pickers)
                got, visited = bucket_search(i, rec, fwd, G, pickers, shift)
                assert got == want, (seed, fwd, shift, i)
                total += visited
        for j in range(n):  # the packed verdict against the plain rule, every (i, d) that can be asked
            for i in range(n):
                for d, jj in c[i]:
                    if jj == j:
                        assert packed_verdict(i, d, pickers[j]) == (not any(ip < i and dp <= d for ip, dp in pickers[j]))
