"""The chain-level stage and the anchor tail of the filter against the CPU oracle (-m gpu).

The anchor pass (k_assign) counts the anchors it writes and, when every alive record is a sorted position and the inversion
capture walks chains rather than the buckets of its grid, also emits the inversion candidates; the inversion capture and rescue
count what they write.  There is no separate recount of the status bytes, so every test here also recounts them on the host and
compares with swg_stats.  Covered: reverse-strand heavy tables, scaffolds_only, rescue, the paths that keep the candidate scan
(1:1 modes, k_chain_keys, the LSD record sort, huge groups and the inversion grid), chain counts of 0, 1 and around powers of
two, many genome pairs with many chains each, and swg_filter_batch.
"""
import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth

pytestmark = pytest.mark.gpu


def recount(stats, status):
    assert stats.n_anchors == int((status == 1).sum()), (stats.n_anchors, int((status == 1).sum()))
    assert stats.n_rescued == int((status == 2).sum()), (stats.n_rescued, int((status == 2).sum()))
    assert stats.n_kept == int((status != 0).sum()), (stats.n_kept, int((status != 0).sum()))


def check(ctx, cfg, table, what=""):
    status, chain, stats = ctx.filter(cfg, table)
    o_status, o_chain, o_stats = oracle_lib.apply_filters(cfg, table)
    bad = np.nonzero(status != o_status)[0]
    assert bad.size == 0, f"{what}: status differs at {bad[:10]} (gpu {status[bad[:10]]}, oracle {o_status[bad[:10]]}) of {table.n}"
    bad = np.nonzero(chain != o_chain)[0]
    assert bad.size == 0, f"{what}: chain id differs at {bad[:10]} (gpu {chain[bad[:10]]}, oracle {o_chain[bad[:10]]})"
    for f in ("n_stage1", "n_after_sweep", "n_kept", "n_chains", "n_chains_after_mass", "n_chains_kept", "n_rescued"):
        assert getattr(stats, f) == getattr(o_stats, f), f"{what}: stats.{f} gpu {getattr(stats, f)} oracle {getattr(o_stats, f)}"
    recount(stats, status)
    return status, chain, stats


def reverse_heavy(seed, n=20000, frac_rev=0.6):
    """A yeast-shaped table with most records flipped to the reverse strand: many inversion candidates, many captured."""
    t = synth.yeast_like(n, seed=seed)
    rng = np.random.default_rng(seed + 1000)
    flip = rng.random(t.n) < frac_rev
    t.strand = np.where(flip, np.uint8(ord("-")), t.strand).astype(np.uint8)
    return t


def one_chain_per_pair(k, long_enough=True, n_chr=80):
    """k records, each alone on its own chromosome pair (genome 0 against genome 1): k chains; with long_enough every one passes
    the 10 kbp mass filter and is kept by the scaffold sweep, so C1 = C2 = k; otherwise C1 = C2 = 0."""
    assert k <= n_chr * n_chr
    names = [f"G{g}#1#chr{c}" for g in range(2) for c in range(n_chr)]
    j = np.arange(k, dtype=np.int64)
    qid, tid = j // n_chr, n_chr + j % n_chr
    ln = np.full(k, 20000 if long_enough else 2000, np.int64)
    qs = np.full(k, 1000, np.int64) + (j % 7) * 100
    ts = qs + (j % 3)
    blk = ln.copy()
    matches = (blk * 9) // 10
    identity = matches / blk
    strand = np.where(j % 4 == 3, ord("-"), ord("+")).astype(np.uint8)
    P, P2 = swg.prefix_ids(names)
    return swg.MappingTable(qid, tid, qs, qs + ln, ts, ts + ln, blk, matches, identity, strand, P, P2, None, names)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_reverse_strand_heavy(ctx, seed):
    t = reverse_heavy(seed)
    status, _, _ = check(ctx, swg.FilterConfig(), t, f"reverse-heavy seed {seed}")
    rev = t.strand != ord("+")
    assert (status[rev] == 1).any()


@pytest.mark.parametrize("knobs", [{}, {"SWG_INV_GRID": "1"}], ids=["walk", "grid"])
def test_scaffolds_only(ctx, monkeypatch, knobs):
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    cfg = swg.FilterConfig.from_cli(scaffolds_only=True)
    check(ctx, cfg, reverse_heavy(4), "scaffolds_only")


@pytest.mark.parametrize("table", ["yeast", "reverse"])
def test_rescue(ctx, table):
    t = synth.yeast_like(20000, seed=5) if table == "yeast" else reverse_heavy(5)
    _, _, st = check(ctx, swg.FilterConfig.from_cli(scaffold_dist="100k"), t, f"rescue {table}")
    assert st.n_rescued > 0


# Paths on which the anchor pass does not emit the candidates (not every alive record is a sorted position, or the
# inversion capture takes the buckets of its grid): the capture compacts them with the flag scan over all records.
SCAN_PATHS = {
    "1:1/1:1": ({"num_mappings": "1:1", "scaffold_filter": "1:1"}, {}),
    "1:1 rescue": ({"num_mappings": "1:1", "scaffold_filter": "1:1", "scaffold_dist": "100k"}, {}),
    "k_chain_keys": ({}, {"SWG_NO_FUSED_KEYS": "1"}),
    "lsd record sort": ({}, {"SWG_NO_GROUP_SORT": "1"}),
    "wide keys": ({}, {"SWG_FORCE_WIDE_KEYS": "1"}),
    "huge groups": ({}, {"SWG_FIXPOINT_MIN": "2", "SWG_FIXPOINT_VERIFY": "1"}),
    "inversion grid": ({"scaffold_dist": "100k"}, {"SWG_INV_GRID": "1"}),
}


@pytest.mark.parametrize("name", list(SCAN_PATHS))
def test_candidate_scan_paths(ctx, monkeypatch, name):
    cli, knobs = SCAN_PATHS[name]
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    check(ctx, swg.FilterConfig.from_cli(**cli), reverse_heavy(6, n=12000), name)


def test_skew_pile_grid(ctx):
    """configs[4]-shaped: one pile on a chromosome pair plus many tiny groups; the pile's group is huge, so the inversion
    capture takes the grid."""
    t = synth.skew(n_pile=60_000, n_tiny_groups=3000, seed=7, window=300_000)
    check(ctx, swg.FilterConfig(), t, "skew pile")
    check(ctx, swg.FilterConfig.from_cli(scaffold_dist="100k"), t, "skew pile, rescue")


@pytest.mark.parametrize("k", [1, 2, 255, 256, 257, 1023, 1024, 1025, 4095, 4096, 4097])
def test_chain_counts(ctx, k):
    _, _, st = check(ctx, swg.FilterConfig(), one_chain_per_pair(k), f"{k} chains")
    assert st.n_chains == st.n_chains_after_mass == st.n_chains_kept == k


@pytest.mark.parametrize("k", [1, 256, 4096])
def test_no_chain_passes(ctx, k):
    _, _, st = check(ctx, swg.FilterConfig(), one_chain_per_pair(k, long_enough=False), f"{k} short chains")
    assert st.n_chains == k and st.n_chains_after_mass == 0 and st.n_chains_kept == 0 and st.n_kept == 0


@pytest.mark.parametrize("cli", [{}, {"scaffold_dist": "100k"}, {"scaffold_filter": "1:1"}], ids=["defaults", "rescue", "scaffold 1:1"])
def test_many_pairs_many_chains(ctx, cli):
    t = synth.pansn(150_000, seed=11, n_hap=12)
    _, _, st = check(ctx, swg.FilterConfig.from_cli(**cli), t, f"pansn {cli}")
    assert st.n_chains_kept > 1000


@pytest.mark.parametrize("cli", [{}, {"scaffold_dist": "100k"}, {"num_mappings": "1:1", "scaffold_filter": "1:1"}],
                         ids=["defaults", "rescue", "1:1"])
def test_filter_batch(ctx, cli):
    cfg = swg.FilterConfig.from_cli(**cli)
    tables = [reverse_heavy(21, n=6000), synth.yeast_like(9000, seed=22), one_chain_per_pair(257), synth.pansn(20000, seed=23, n_hap=5),
              one_chain_per_pair(64, long_enough=False)]
    res, counts, stats = ctx.filter_batch(cfg, tables)
    n1 = n2 = 0
    for k, t in enumerate(tables):
        status, chain = res[k][0], res[k][1]
        o_status, o_chain, _ = oracle_lib.apply_filters(cfg, t)
        assert np.array_equal(status, o_status), f"table {k}: status differs from the oracle"
        assert np.array_equal(chain, o_chain), f"table {k}: chain ids differ from the oracle"
        assert counts[k][2] == int((status == 1).sum()) and counts[k][3] == int((status == 2).sum())
        n1 += int((status == 1).sum())
        n2 += int((status == 2).sum())
    assert stats.n_anchors == n1 and stats.n_rescued == n2
