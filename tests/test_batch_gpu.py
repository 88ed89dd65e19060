"""swg_filter_batch on the device (-m gpu): every table of a batch gets, byte for byte, what Context.filter gives it alone
(and what the oracle gives it), wherever it sits in the batch and whatever shares it; the per-table counts match the single
calls; the re-rank, wide-key and fixed-point paths run inside a batch; errors leave the context usable and its prefetches
outstanding."""
import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth, with_ids16

from batch_util import CONFIGS, check_batch, reference_paf_table, self_only, split, union

pytestmark = pytest.mark.gpu


def _no_identity(t):
    import copy
    o = copy.copy(t)
    o.identity = None
    return o


def _mixed_tables():
    """Sizes from 0 to ~20 k records, 16- and 32-bit ids, with and without an identity column."""
    empty = synth.yeast_like(500, seed=3).take(np.zeros(0, np.int64))
    return [
        synth.yeast_like(20000, seed=21),
        with_ids16(synth.yeast_like(4000, seed=22)),
        empty,
        _no_identity(synth.pansn(6000, seed=23, n_hap=6)),
        reference_paf_table(),
        with_ids16(_no_identity(synth.yeast_like(300, seed=24))),
        self_only(synth.yeast_like(700, seed=25)),
        synth.yeast_like(1, seed=26),
        empty,
        synth.pansn(9000, seed=27, n_hap=4),
    ]


@pytest.mark.parametrize("name", list(CONFIGS))
def test_batch_equals_single_calls_and_oracle(ctx, name):
    cfg = swg.FilterConfig.from_cli(**CONFIGS[name])
    check_batch(ctx, cfg, _mixed_tables(), what=name)


def test_position_independence(ctx):
    cfg = swg.FilterConfig.from_cli(scaffold_dist="20k")
    t = synth.yeast_like(8000, seed=31)
    a, b, c = synth.pansn(3000, seed=32, n_hap=5), with_ids16(synth.yeast_like(5000, seed=33)), _no_identity(synth.yeast_like(900, seed=34))
    layouts = [([t, a, b], 0), ([c, b, t, a], 2), ([a, c, t], 2), ([b, a, c, t], 3), ([t], 0)]
    outs = []
    for tables, pos in layouts:
        res, counts, _ = ctx.filter_batch(cfg, tables)
        outs.append((res[pos][0].tobytes(), res[pos][1].tobytes(), counts[pos].tolist()))
    assert all(o == outs[0] for o in outs[1:])
    s, ch, _ = ctx.filter(cfg, t)
    assert outs[0][0] == s.tobytes() and outs[0][1] == ch.tobytes()


@pytest.mark.parametrize("knob", [("SWG_EXACT_SCORES", "always"), ("SWG_FORCE_WIDE_KEYS", "1")])
@pytest.mark.parametrize("name", ["defaults", "1:1_dist50k"])
def test_batch_paths(ctx, monkeypatch, knob, name):
    """The host-log re-rank and the wide-key path, each set for the batch and for the single calls alike."""
    monkeypatch.setenv(*knob)
    cfg = swg.FilterConfig.from_cli(**CONFIGS[name])
    _, _, st = check_batch(ctx, cfg, _mixed_tables(), oracle=False, what=f"{knob[0]} {name}")
    if knob[0] == "SWG_EXACT_SCORES":
        assert st.exact_rerank == 1


def test_fixpoint_inside_a_batch(ctx, monkeypatch):
    """A small skew pile between tiny tables; the pile's group goes through the fixed-point chaining."""
    monkeypatch.setenv("SWG_FIXPOINT_MIN", "1000")
    monkeypatch.setenv("SWG_FIXPOINT_VERIFY", "1")
    pile = synth.skew(n_pile=20_000, n_tiny_groups=2_000, seed=5, window=3_000_000)
    tiny = [synth.yeast_like(150, seed=40 + k) for k in range(4)]
    tables = tiny[:2] + [pile] + tiny[2:]
    for cfg in (swg.FilterConfig(), swg.FilterConfig.from_cli(scaffold_dist="20k")):
        check_batch(ctx, cfg, tables, what="fixpoint")


def test_many_small_tables(ctx):
    """K = 2000 tables of ~200 records: equal to the single calls and to the renumbered union; no launch per table."""
    cfg = swg.FilterConfig()
    tables = [synth.yeast_like(200 + (k % 7) * 10, seed=1000 + k) for k in range(2000)]
    res, counts, bstats = ctx.filter_batch(cfg, tables)
    for k, t in enumerate(tables):
        s, c, st = ctx.filter(cfg, t)
        assert np.array_equal(res[k][0], s) and np.array_equal(res[k][1], c), f"table {k}"
        assert counts[k, swg.TC_STAGE1] == st.n_stage1 and counts[k, swg.TC_CHAINS_KEPT] == st.n_chains_kept
    u, offs = union(tables)
    us, uc, ust = ctx.filter(cfg, u)
    assert bstats.gpu_launches <= ust.gpu_launches + 6, (bstats.gpu_launches, ust.gpu_launches)
    for k, (s, c) in enumerate(split(us, uc, offs)):
        assert np.array_equal(s, res[k][0]) and np.array_equal(c, res[k][1]), f"union, table {k}"


def test_errors_and_context_state(ctx):
    cfg = swg.FilterConfig()
    good = [synth.yeast_like(2000, seed=50 + k) for k in range(5)]
    # an end < start record in table 3 that passes the retain
    import copy
    bad = copy.copy(good[3])
    bad.query_end = bad.query_end.copy()
    i = int(np.nonzero((bad.query_id != bad.target_id) & (bad.query_start > 0))[0][0])
    bad.query_end[i] = bad.query_start[i] - 1
    with pytest.raises(swg.SwgError) as e:
        ctx.filter_batch(cfg, good[:3] + [bad] + good[4:])
    assert e.value.code == swg._lib.ERR_RANGE
    check_batch(ctx, cfg, good, oracle=False, what="after a range error")
    # score in some tables only
    scored = copy.copy(good[1])
    scored.score = oracle_lib.score_column(scored.query_start, scored.query_end, scored.identity)
    with pytest.raises(swg.SwgError) as e:
        ctx.filter_batch(cfg, [good[0], scored])
    assert e.value.code == swg._lib.ERR_ARG and "table 1" in str(e.value)
    # no tables
    res, counts, st = ctx.filter_batch(cfg, [])
    assert res == [] and counts.shape == (0, swg.TC_COUNT) and st.n_input == 0
    # the union's chain numbering is not reported as the last call's
    ctx.filter(cfg, good[0])
    assert len(ctx.last_chain_units()[0]) > 0
    ctx.filter_batch(cfg, good)
    assert len(ctx.last_chain_units()[0]) == 0 and len(ctx.last_chain_keys()[0]) == 0
    # outstanding prefetches survive a batch and are consumed by the following filter
    t = good[2]
    want = ctx.filter(cfg, t)
    try:
        ctx.prefetch(t)
        ctx.prefetch(t)
        ctx.filter_batch(cfg, good)
        with pytest.raises(swg.SwgError):  # still two outstanding
            ctx.prefetch(t)
        got = ctx.filter(cfg, t)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        ctx.prefetch(t)  # one slot free again: the filter consumed one
    finally:
        ctx.prefetch_drop()


def test_thousand_yeast_tables(ctx):
    """1000 tables of ~23 k records: a union of 136 k sequences and 23 M records, whose record sort cannot use the packed LSD
    passes (they would keep the key only from a bit above the coordinate field) and takes the two-stage path."""
    cfg = swg.FilterConfig()
    tables = [synth.yeast_like(26000, seed=k) for k in range(1000)]
    res, counts, st = ctx.filter_batch(cfg, tables)
    n_chains = 0
    for k, t in enumerate(tables):
        s, c, sst = ctx.filter(cfg, t)
        assert np.array_equal(res[k][0], s) and np.array_equal(res[k][1], c), f"table {k}"
        assert counts[k, swg.TC_CHAINS_KEPT] == sst.n_chains_kept
        n_chains += sst.n_chains_kept
    assert st.n_chains_kept == n_chains
