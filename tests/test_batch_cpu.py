"""The premise of swg_filter_batch, pinned on the CPU oracle alone (no GPU): independent tables laid end to end with disjoint
ids (sequence ids offset by the running n_seq, genome-prefix ids by the running genome count) filter to exactly the per-table
results, once every table's chains are renumbered from chain_1 — a table's chains are one consecutive run of the union's
numbering."""
import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth

from batch_util import CONFIGS, oracle_table, reference_paf_table, self_only, split, union


def _random_batch(seed):
    rng = np.random.default_rng(seed)
    tables = []
    for j in range(int(rng.integers(3, 7))):
        kind = rng.integers(0, 3)
        n = int(rng.integers(200, 6000))
        if kind == 0:
            t = synth.yeast_like(n, seed=int(rng.integers(1, 1000)))
        elif kind == 1:
            t = synth.pansn(n, seed=int(rng.integers(1, 1000)), n_hap=int(rng.integers(3, 8)))
        else:
            t = synth.yeast_like(n, seed=int(rng.integers(1, 1000)))
            t.identity = None  # the parser's default identity, derived from matches / block_length
        tables.append(t)
    return tables


def _check(cfg, tables):
    u, offs = union([oracle_table(t) for t in tables])
    us, uc, ust = oracle_lib.apply_filters(cfg, u)
    got = split(us, uc, offs)
    n_chains = 0
    for k, t in enumerate(tables):
        s, c, st = oracle_lib.apply_filters(cfg, oracle_table(t))
        assert np.array_equal(got[k][0], s), f"table {k}: status differs"
        assert np.array_equal(got[k][1], c), f"table {k}: chain id differs"
        n_chains += st.n_chains_kept
    assert ust.n_chains_kept == n_chains


@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("seed", [1, 2])
def test_union_equals_per_table_oracle(name, seed):
    cfg = swg.FilterConfig.from_cli(**CONFIGS[name])
    _check(cfg, _random_batch(100 * seed + len(name)))


@pytest.mark.parametrize("name", list(CONFIGS))
def test_union_with_reference_vector_and_edge_tables(name):
    """The committed PAF vector twice among synthetic tables, an empty table, and a table of self mappings only (nothing of it
    passes the stage-1 retain unless keep_self is set)."""
    cfg = swg.FilterConfig.from_cli(**CONFIGS[name])
    ref = reference_paf_table()
    empty = synth.yeast_like(500, seed=3).take(np.zeros(0, np.int64))
    selfs = self_only(synth.yeast_like(800, seed=4))
    tables = [synth.yeast_like(3000, seed=11), ref, empty, selfs, synth.pansn(2500, seed=12, n_hap=4), ref]
    _check(cfg, tables)


def test_self_only_table_fails_the_retain():
    cfg = swg.FilterConfig()
    t = self_only(synth.yeast_like(800, seed=4))
    s, _, st = oracle_lib.apply_filters(cfg, oracle_table(t))
    assert st.n_stage1 == 0 and not s.any()
