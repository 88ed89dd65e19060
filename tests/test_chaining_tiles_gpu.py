"""Chaining at the edges of its tiles and windows, against the CPU oracle (-m gpu).

The chain numbering resolves ancestors in 32-position chunks (registers), 256-position warp ranges (shared memory) and
2048-position tiles, and leaves a position whose ancestor lies in an earlier tile to the aggregate pass; the candidate pass
scans a linear window of up to 48 successors before it searches outwards.  The tables here put chains and windows on those
boundaries: collinear groups whose chains cross the 32-, 256- and 2048-position boundaries or span
many tiles (warp walk and fixed point), chains of exactly one chunk, predecessors far back (an interleaved sparse chain), windows
of 3 to 49 successors, ties in the squared gap, windows that end at the group end, groups of 1 and 2 positions, position counts
around multiples of 2048, and swg_filter_batch over several of these tables.  Every check compares status, chain id and counts.
"""
import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from batch_util import check_batch

pytestmark = pytest.mark.gpu

G = swg.FilterConfig().scaffold_gap  # 50 kbp
LEN = 1000


def step_for(window):
    """Query/target step of a collinear run whose every position sees exactly `window` successors (qs_j - qe_i <= G)."""
    s = (G + LEN) // window
    while (G + LEN) // s != window:
        s -= 1
    return s


def run(n, window, q0=1000, t0=1000):
    s = step_for(window)
    qs = q0 + s * np.arange(n, dtype=np.int64)
    return qs, t0 + s * np.arange(n, dtype=np.int64)


def make_table(groups, seed=0):
    """groups: list of (qs, ts) arrays; group g is alone on chromosome pair (G0#1#chr<g>, G1#1#chr<g>), forward strand.
    Records go in shuffled input order."""
    k = len(groups)
    names = [f"G{h}#1#chr{c}" for h in range(2) for c in range(k)]
    qid = np.concatenate([np.full(len(q), g, np.int64) for g, (q, _) in enumerate(groups)])
    tid = qid + k
    qs = np.concatenate([q for q, _ in groups]).astype(np.int64)
    ts = np.concatenate([t for _, t in groups]).astype(np.int64)
    n = qs.size
    perm = np.random.default_rng(seed).permutation(n)
    qid, tid, qs, ts = qid[perm], tid[perm], qs[perm], ts[perm]
    ln = np.full(n, LEN, np.int64)
    matches = (ln * 19) // 20
    strand = np.full(n, ord("+"), np.uint8)
    P, P2 = swg.prefix_ids(names)
    return swg.MappingTable(qid, tid, qs, qs + ln, ts, ts + ln, ln.copy(), matches, matches / ln, strand, P, P2, None, names)


def check(ctx, table, what, chains=None):
    cfg = swg.FilterConfig()
    status, chain, stats = ctx.filter(cfg, table)
    o_status, o_chain, o_stats = oracle_lib.apply_filters(cfg, table)
    bad = np.nonzero(status != o_status)[0]
    assert bad.size == 0, f"{what}: status differs at {bad[:10]} (gpu {status[bad[:10]]}, oracle {o_status[bad[:10]]}) of {table.n}"
    bad = np.nonzero(chain != o_chain)[0]
    assert bad.size == 0, f"{what}: chain id differs at {bad[:10]} (gpu {chain[bad[:10]]}, oracle {o_chain[bad[:10]]})"
    for f in ("n_stage1", "n_after_sweep", "n_kept", "n_chains", "n_chains_after_mass", "n_chains_kept", "n_rescued"):
        assert getattr(stats, f) == getattr(o_stats, f), f"{what}: stats.{f} gpu {getattr(stats, f)} oracle {getattr(o_stats, f)}"
    assert stats.n_after_sweep == table.n, f"{what}: the sweep dropped records, the table does not have the intended shape"
    if chains is not None:
        assert stats.n_chains == chains, f"{what}: {stats.n_chains} chains, the table was built for {chains}"
    return stats


@pytest.mark.parametrize("n", [31, 32, 33, 255, 256, 257, 2047, 2048, 2049, 4095, 4096, 4097, 6200])
def test_one_collinear_chain(ctx, n):
    """One group, one chain from position 0: its end sits just before, on and after the chunk, warp and tile boundaries."""
    check(ctx, make_table([run(n, 8)]), f"collinear n={n}", chains=1)


@pytest.mark.parametrize("size", [32, 33])
def test_chunk_deep_chains(ctx, size):
    """64 groups of 32 (every chunk holds one chain of depth 32) or of 33 (chains straddle every chunk boundary)."""
    groups = [run(size, 5, q0=1000 + 7 * g, t0=2000 + 11 * g) for g in range(64)]
    check(ctx, make_table(groups, seed=size), f"groups of {size}", chains=64)


@pytest.mark.parametrize("n", [16000, 20000], ids=["warp-walk", "fixed-point"])
def test_chain_over_many_tiles(ctx, n):
    """A single collinear chain over 8 or 10 tiles; 20000 positions are a huge group (fixed point, preset roots)."""
    check(ctx, make_table([run(n, 8)]), f"collinear over tiles n={n}", chains=1)


@pytest.mark.parametrize("sparse_every", [3, 40])
def test_pred_far_back(ctx, sparse_every):
    """An off-diagonal repeat inside the group: a sparse chain 200 kbp up the target axis, one record per `sparse_every` of the
    dense chain, interleaved with it in query order: its predecessors lie 3 or ~40 positions back, across chunks and tiles."""
    n = 5000
    qd, td = run(n, 48)
    s = step_for(48)
    m = n // sparse_every
    qr = 1000 + s * sparse_every * np.arange(m, dtype=np.int64) + s // 2
    tr = qr + 200_000
    check(ctx, make_table([(np.concatenate([qd, qr]), np.concatenate([td, tr]))]), f"repeat every {sparse_every}", chains=2)


@pytest.mark.parametrize("window", [3, 4, 5, 8, 47, 48, 49])
def test_window_sizes(ctx, window):
    """Every position sees exactly `window` successors; the group sizes also put the last windows on the group end."""
    groups = [run(n, window, q0=1000 + 13 * i) for i, n in enumerate([window, window + 1, window + 2, 2 * window + 3, 600])]
    check(ctx, make_table(groups, seed=window), f"window {window}", chains=len(groups))


def test_ties_in_gap(ctx):
    """Twins: beside every fifth record of a chain, a record with the same query interval whose target start overlaps the
    predecessor by the gap the original leaves, so both are at the same squared distance: the first minimal position wins."""
    n = 3000
    s = step_for(8)
    q, t = run(n, 8)
    gap = s - LEN
    idx = np.arange(5, n, 5)
    qt = q[idx]
    tt = t[idx - 1] + LEN - gap
    check(ctx, make_table([(np.concatenate([q, qt]), np.concatenate([t, tt]))]), "ties")


def test_tiny_groups(ctx):
    """Groups of 1 and 2 positions among larger ones (every tile sees many heads)."""
    sizes = [1, 2, 1, 1, 2, 2, 3, 1, 40, 2, 1] * 30
    groups = [run(n, 4, q0=1000 + 17 * i) for i, n in enumerate(sizes)]
    check(ctx, make_table(groups, seed=5), "tiny groups", chains=len(sizes))


@pytest.mark.parametrize("total", [2047, 2049, 4095, 4097, 8191, 8193])
def test_positions_around_tiles(ctx, total):
    """Several groups whose positions add up to just below or just above a multiple of 2048."""
    sizes = [700, 300, 45, 1]
    sizes.append(total - sum(sizes))
    groups = [run(n, 6, q0=1000 + 3 * i) for i, n in enumerate(sizes)]
    check(ctx, make_table(groups, seed=total), f"n_m = {total}", chains=len(sizes))


def test_filter_batch(ctx):
    tables = [make_table([run(2049, 8)]), make_table([run(33, 5, q0=1000 + g) for g in range(70)], seed=1),
              make_table([run(n, 48, q0=1000 + 9 * i) for i, n in enumerate([1, 2, 49, 300, 4097])], seed=2),
              make_table([run(16000, 4)], seed=3)]
    check_batch(ctx, swg.FilterConfig(), tables, what="chaining tiles")
