"""Helpers of the batch tests (tests/test_batch_cpu.py, tests/test_batch_gpu.py, tests/test_scale_gpu.py): the union of
independent tables with disjoint ids, built in numpy, the per-table renumbering of a result on that union, and the check of a
batch against the single calls."""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

# the configurations the batch is checked under (FilterConfig.from_cli keyword arguments)
CONFIGS = {
    "defaults": {},
    "1:1": {"num_mappings": "1:1", "scaffold_filter": "1:1"},
    "dist20k": {"scaffold_dist": "20k"},
    "no_scaffold": {"scaffold_jump": "0"},
    "scaffolds_only": {"scaffolds_only": True},
    "1:1_dist50k": {"num_mappings": "1:1", "scaffold_filter": "1:1", "scaffold_dist": "50k"},
    "keep_self": {"keep_self": True},
    "min_identity": {"min_aln_identity": "0.9"},
}


def derived_identity(t):
    """The parser's identity of a record without dv:f: / cg:Z: tags: matches / max(block_length, 1)."""
    return t.matches.astype(np.float64) / np.maximum(t.block_length, 1).astype(np.float64)


def union(tables):
    """The tables end to end: sequence ids offset by the running n_seq, P and P2 by the running genome count
    (max prefix id + 1 per table).  Tables with n == 0 contribute nothing.  Returns (union table, record offsets [K + 1])."""
    from sweepga_b200 import MappingTable
    cols = {f: [] for f in ("query_id", "target_id", "query_start", "query_end", "target_start", "target_end", "block_length",
                            "matches", "identity", "strand", "seq_genome_id", "seq_genome2_id", "score")}
    offs, n, s_off, g_off = [0], 0, 0, 0
    for t in tables:
        if t.n:
            for f in ("query_start", "query_end", "target_start", "target_end", "block_length", "matches", "strand"):
                cols[f].append(getattr(t, f))
            cols["query_id"].append(t.query_id.astype(np.uint64) + s_off)
            cols["target_id"].append(t.target_id.astype(np.uint64) + s_off)
            cols["identity"].append(t.identity if t.identity is not None else derived_identity(t))
            cols["seq_genome_id"].append(t.seq_genome_id.astype(np.uint64) + g_off)
            cols["seq_genome2_id"].append(t.seq_genome2_id.astype(np.uint64) + g_off)
            if t.score is not None:
                cols["score"].append(t.score)
            s_off += t.n_seq
            g_off += int(max(t.seq_genome_id.max(), t.seq_genome2_id.max())) + 1
            n += t.n
        offs.append(n)
    cat = {f: (np.concatenate(v) if v else np.zeros(0)) for f, v in cols.items()}
    u = MappingTable(cat["query_id"], cat["target_id"], cat["query_start"], cat["query_end"], cat["target_start"], cat["target_end"],
                     cat["block_length"], cat["matches"], cat["identity"], cat["strand"], cat["seq_genome_id"], cat["seq_genome2_id"],
                     cat["score"] if cols["score"] else None)
    return u, np.asarray(offs, np.int64)


def split(status, chain, offs):
    """Per-table slices of a union result, each table's chains renumbered from chain_1.  Asserts that a table's chains are one
    consecutive run of the union's numbering (the premise the batch rests on)."""
    out = []
    for k in range(len(offs) - 1):
        s, c = status[offs[k]:offs[k + 1]].copy(), chain[offs[k]:offs[k + 1]].astype(np.int64)
        nz = c[c > 0]
        if nz.size:
            lo, hi = int(nz.min()), int(nz.max())
            assert len(np.unique(nz)) == hi - lo + 1, f"table {k}: its chains are not one consecutive run of the union's numbering"
            c = np.where(c > 0, c - (lo - 1), 0)
        out.append((s, c.astype(np.uint32)))
    return out


def oracle_table(t):
    """The table as the oracle binding takes it (an identity column is required there)."""
    import copy
    if t.identity is not None:
        return t
    o = copy.copy(t)
    o.identity = derived_identity(t)
    return o


def self_only(t):
    """A table whose every record maps a sequence onto itself: nothing passes the stage-1 retain without keep_self."""
    import copy
    o = copy.copy(t)
    o.target_id = t.query_id.copy()
    return o


def reference_paf_table():
    """The table of the committed front-end vector (tests/golden/frontend.paf), parsed by the oracle."""
    import oracle_lib
    return oracle_lib.parse_paf(os.path.join(HERE, "golden", "frontend.paf"))


def check_batch(ctx, cfg, tables, oracle=True, what=""):
    """ctx.filter_batch(cfg, tables) against ctx.filter of every table alone (and the oracle): status, chain numbers and the
    per-table counts; the call's stats against the sums of the counts."""
    import oracle_lib
    import sweepga_b200 as swg
    res, counts, bstats = ctx.filter_batch(cfg, tables)
    assert len(res) == len(tables) and counts.shape == (len(tables), swg.TC_COUNT)
    for k, t in enumerate(tables):
        s, c, st = ctx.filter(cfg, t)
        assert np.array_equal(res[k][0], s), f"{what} table {k}: status differs from the single call"
        assert np.array_equal(res[k][1], c), f"{what} table {k}: chain id differs from the single call"
        want = [st.n_stage1, int((s != 0).sum()), int((s == swg.SCAFFOLD).sum()), int((s == swg.RESCUED).sum()), st.n_chains_kept]
        assert counts[k].tolist() == want, f"{what} table {k}: counts {counts[k].tolist()} != {want}"
        assert st.n_chains_kept == (int(c.max()) if t.n else 0)
        if oracle and t.n:
            os_, oc, _ = oracle_lib.apply_filters(cfg, oracle_table(t))
            assert np.array_equal(s, os_) and np.array_equal(c, oc), f"{what} table {k}: the single call differs from the oracle"
    assert bstats.n_input == sum(t.n for t in tables)
    assert bstats.n_stage1 == int(counts[:, swg.TC_STAGE1].sum())
    assert bstats.n_chains_kept == int(counts[:, swg.TC_CHAINS_KEPT].sum())
    return res, counts, bstats
