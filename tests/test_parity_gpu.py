"""Parity proper: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bit-exact bar: identical status byte and chain number for every record.  Sizes are chosen so that the
single-threaded oracle finishes in seconds.  Full-size parity (20 M and 40 M records, every mode that changes which kernels
run, against the oracle spread over genome-pair units on all host threads) lives in test_scale_gpu.py; size-independent
properties (idempotence, determinism, shard-invariance) are in test_properties_gpu.py.
"""
import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth

pytestmark = pytest.mark.gpu


def fuzz_table(seed, n, n_genomes=3, n_chr=2, span=3000, max_len=400, zero_len_frac=0.02, hashless=False):
    """Dense, tie-rich tables: few sequences, small coordinates, identities from a small set."""
    rng = np.random.default_rng(seed)
    if hashless:
        names = [f"ctg{i}" for i in range(n_genomes * n_chr)]
    else:
        names = [f"G{g}#1#chr{c}" for g in range(n_genomes) for c in range(n_chr)]
    ns = len(names)
    qid = rng.integers(0, ns, n)
    tid = rng.integers(0, ns, n)
    qs = rng.integers(0, span, n)
    ln = rng.integers(1, max_len, n)
    ln[rng.random(n) < zero_len_frac] = 0
    ts = np.where(rng.random(n) < 0.6, qs + rng.integers(-50, 51, n), rng.integers(0, span, n))
    ts = np.maximum(ts, 0)
    tl = np.maximum(ln + rng.integers(-5, 6, n), 0)
    tl[rng.random(n) < zero_len_frac] = 0
    ident = rng.choice([0.8, 0.9, 0.95, 1.0, 0.0], n, p=[0.3, 0.3, 0.2, 0.18, 0.02])
    blk = np.maximum(np.maximum(ln, tl), 1)
    matches = np.rint(ident * blk).astype(np.int64)
    identity = matches / blk
    strand = np.where(rng.random(n) < 0.7, ord("+"), ord("-")).astype(np.uint8)
    P, P2 = swg.prefix_ids(names)
    return swg.MappingTable(qid, tid, qs, qs + ln, ts, ts + tl, blk, matches, identity, strand, P, P2, None, names)


def check(ctx, cfg, table, what=""):
    status, chain, stats = ctx.filter(cfg, table)
    o_status, o_chain, o_stats = oracle_lib.apply_filters(cfg, table)
    bad = np.nonzero(status != o_status)[0]
    assert bad.size == 0, f"{what}: status differs at {bad[:10]} (gpu {status[bad[:10]]}, oracle {o_status[bad[:10]]}) of {table.n}"
    bad = np.nonzero(chain != o_chain)[0]
    assert bad.size == 0, f"{what}: chain id differs at {bad[:10]} (gpu {chain[bad[:10]]}, oracle {o_chain[bad[:10]]})"
    for f in ("n_stage1", "n_after_sweep", "n_kept"):
        assert getattr(stats, f) == getattr(o_stats, f), f"{what}: stats.{f} gpu {getattr(stats, f)} oracle {getattr(o_stats, f)}"
    if cfg.scaffold_gap > 0:
        for f in ("n_chains", "n_chains_after_mass", "n_chains_kept", "n_rescued"):
            assert getattr(stats, f) == getattr(o_stats, f), f"{what}: stats.{f} gpu {getattr(stats, f)} oracle {getattr(o_stats, f)}"
    assert stats.gpu_launches > 0
    return status, chain, stats


CLI_CASES = {
    "defaults": {},
    "1:1_1:1": dict(num_mappings="1:1", scaffold_filter="1:1"),
    "rescue100k": dict(scaffold_dist="100k"),
    "1:1_rescue": dict(num_mappings="1:1", scaffold_filter="1:1", scaffold_dist="20k"),
    "no_scaffold_1:1": dict(num_mappings="1:1", scaffold_jump="0"),
    "no_scaffold_many": dict(scaffold_jump="0"),
    "n3": dict(num_mappings="3", scaffold_jump="0", overlap=0.5),
    "2:3": dict(num_mappings="2:3", scaffold_filter="2:2", scaffold_overlap=0.3),
    "many:1": dict(num_mappings="many:1", scaffold_filter="1:many"),
    "scaffolds_only": dict(scaffolds_only=True),
    "self": dict(keep_self=True, scaffold_mass="0"),
    "identity_scoring": dict(num_mappings="1:1", scaffold_filter="1:1", scoring="ani"),
    "length_scoring": dict(num_mappings="1:1", scaffold_filter="1:1", scoring="length"),
    "length_ani_scoring": dict(num_mappings="1:1", scaffold_filter="1:1", scoring="length-ani"),
    "min_filters": dict(min_aln_length="5k", min_aln_identity="0.95", min_scaffold_identity="0.97"),
    "tight_jump": dict(scaffold_jump="2k", scaffold_mass="1k", scaffold_dist="5k"),
    "mass0": dict(scaffold_mass="0", scaffold_filter="1:1"),
}


@pytest.fixture(scope="module")
def yeast():
    return synth.yeast_like(30000, seed=1)


@pytest.mark.parametrize("case", list(CLI_CASES))
def test_yeast_configs(ctx, yeast, case):
    """BASELINE configs[0] (defaults) and configs[1] (1:1 / 1:1) on the yeast-shaped table, plus flag variants."""
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), yeast, case)


@pytest.mark.parametrize("case", ["defaults", "rescue100k", "1:1_1:1"])
def test_pansn_400k(ctx, case):
    """configs[2]/[3] generator at a size the oracle finishes in seconds."""
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), synth.pansn(400_000, seed=3, n_hap=12), case)


def test_pansn_2m_defaults(ctx):
    check(ctx, swg.FilterConfig(), synth.pansn(2_000_000, seed=4, n_hap=24), "pansn2m")


@pytest.mark.parametrize("case", ["defaults", "rescue100k"])
def test_skew_small(ctx, case):
    """configs[4] shape, scaled so the oracle's O(n*window) chaining finishes: one pile + many tiny groups."""
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), synth.skew(n_pile=20_000, n_tiny_groups=3_000, seed=5, window=3_000_000), case)


@pytest.mark.parametrize("seed", range(160))
def test_fuzz_dense(ctx, seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(2, 600)) if seed < 120 else int(rng.integers(2000, 8000))
    t = fuzz_table(seed, n, hashless=bool(seed % 5 == 0))
    modes = ["1:1", "1", "2:2", "many:many", "3:1", "many:1", "1:many"]
    cfg = swg.FilterConfig.from_cli(
        num_mappings=modes[seed % len(modes)], scaffold_filter=modes[(seed // 3) % len(modes)],
        overlap=[0.0, 0.5, 0.95, 1.0][seed % 4], scaffold_overlap=[0.5, 0.0, 1.0][seed % 3],
        scaffold_jump=str([0, 50, 200, 1000][(seed // 2) % 4]), scaffold_mass=str([0, 100, 500][seed % 3]),
        scaffold_dist=str([0, 100, 1000][(seed // 5) % 3]), keep_self=bool(seed % 2),
        scoring=["log-length-ani", "ani", "length", "length-ani", "matches"][seed % 5])
    check(ctx, cfg, t, f"fuzz{seed}")


@pytest.mark.parametrize("seed", range(8))
def test_dense_windows(ctx, seed):
    """Groups of ~10^3 mappings with hundreds of candidates per window: the chaining leaves the linear scan and
    searches outwards from query_end with the q_gap^2 bound (bb_best_successor), blocked steps included."""
    t = fuzz_table(500 + seed, 6000, n_genomes=1, n_chr=2, span=[4000, 20000][seed % 2], max_len=[400, 60][seed // 4 % 2],
                   zero_len_frac=0.0)
    cfg = swg.FilterConfig.from_cli(scaffold_jump=str([200, 1000, 3000, 50][seed % 4]), scaffold_mass=str([0, 300][seed % 2]),
                                    scaffold_dist=str([0, 500][seed % 2]), keep_self=True)
    check(ctx, cfg, t, f"dense{seed}")


@pytest.mark.parametrize("seed", range(8))
def test_fixpoint_dense_windows(ctx, seed, monkeypatch):
    """The fixed-point chaining (chain_fixpoint.cuh) forced onto EVERY group: same inputs as test_dense_windows."""
    monkeypatch.setenv("SWG_FIXPOINT_MIN", "2")
    monkeypatch.setenv("SWG_FIXPOINT_VERIFY", "1")
    t = fuzz_table(500 + seed, 6000, n_genomes=1, n_chr=2, span=[4000, 20000][seed % 2], max_len=[400, 60][seed // 4 % 2],
                   zero_len_frac=0.0)
    cfg = swg.FilterConfig.from_cli(scaffold_jump=str([200, 1000, 3000, 50][seed % 4]), scaffold_mass=str([0, 300][seed % 2]),
                                    scaffold_dist=str([0, 500][seed % 2]), keep_self=True)
    check(ctx, cfg, t, f"fixpoint-dense{seed}")


@pytest.mark.parametrize("what", ["yeast", "pansn400k", "skew20k", "fuzz"])
def test_fixpoint_everywhere(ctx, yeast, what, monkeypatch):
    """Ordinary inputs with every group of two or more mappings sent through the fixed-point chaining."""
    monkeypatch.setenv("SWG_FIXPOINT_MIN", "2")
    monkeypatch.setenv("SWG_FIXPOINT_VERIFY", "1")
    if what == "yeast":
        check(ctx, swg.FilterConfig(), yeast, what)
        check(ctx, swg.FilterConfig.from_cli(**CLI_CASES["1:1_rescue"]), yeast, what)
    elif what == "pansn400k":
        check(ctx, swg.FilterConfig(), synth.pansn(400_000, seed=3, n_hap=12), what)
    elif what == "skew20k":
        check(ctx, swg.FilterConfig(), synth.skew(n_pile=20_000, n_tiny_groups=3_000, seed=5, window=3_000_000), what)
    else:
        for seed in range(120, 132):
            t = fuzz_table(seed, 5000)
            cfg = swg.FilterConfig.from_cli(scaffold_jump=str([50, 200, 1000][seed % 3]), scaffold_mass=str([0, 100][seed % 2]), keep_self=True)
            check(ctx, cfg, t, f"fixpoint-fuzz{seed}")


@pytest.mark.parametrize("variant", ["narrow0", "narrow6", "narrow12", "narrow5_collect"])
def test_fixpoint_search_orders(ctx, yeast, variant, monkeypatch):
    """The fixed point's searches in target-bucket order with buckets from G + G/5 wide (at most two per search) down to a few
    bases (dozens per search).  Short windows reach the warp search too: the windows that go on past round 0's linear scan,
    every later re-evaluation and the verify pass."""
    monkeypatch.setenv("SWG_FIXPOINT_MIN", "2")
    monkeypatch.setenv("SWG_FIXPOINT_VERIFY", "1")
    if variant.endswith("_collect"):  # X(i) from the separate collecting pass (otherwise only after 1024 blocked candidates)
        monkeypatch.setenv("SWG_FX_FORCE_COLLECT", "1")
        variant = variant[:-8]
    monkeypatch.setenv("SWG_FX_BUCKET_NARROW", variant[6:])
    check(ctx, swg.FilterConfig(), synth.skew(n_pile=20_000, n_tiny_groups=3_000, seed=5, window=3_000_000), variant)
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES["1:1_rescue"]), yeast, variant)
    for seed in (500, 503, 505, 506):
        t = fuzz_table(seed, 6000, n_genomes=1, n_chr=2, span=[4000, 20000][seed % 2], max_len=[400, 60][seed // 4 % 2], zero_len_frac=0.0)
        cfg = swg.FilterConfig.from_cli(scaffold_jump=str([200, 1000, 3000, 50][seed % 4]), scaffold_mass="0", keep_self=True)
        check(ctx, cfg, t, f"{variant}-dense{seed}")
    for seed in range(120, 126):
        cfg = swg.FilterConfig.from_cli(scaffold_jump=str([50, 200, 1000][seed % 3]), scaffold_mass=str([0, 100][seed % 2]), keep_self=True)
        check(ctx, cfg, fuzz_table(seed, 5000), f"{variant}-fuzz{seed}")


def test_fixpoint_round_limit_falls_back_to_the_walk(ctx, monkeypatch):
    """Picks that have not settled after SWG_FIXPOINT_MAX_ROUNDS rounds: the groups go through the sequential warp walk."""
    monkeypatch.setenv("SWG_FIXPOINT_MIN", "2")
    monkeypatch.setenv("SWG_FIXPOINT_MAX_ROUNDS", "2")
    check(ctx, swg.FilterConfig(), synth.skew(n_pile=20_000, n_tiny_groups=3_000, seed=5, window=3_000_000), "round-limit")
    t = fuzz_table(503, 6000, n_genomes=1, n_chr=2, span=4000, max_len=400, zero_len_frac=0.0)
    check(ctx, swg.FilterConfig.from_cli(scaffold_jump="1000", scaffold_mass="0", keep_self=True), t, "round-limit-dense")


@pytest.mark.parametrize("case", ["defaults", "1:1_rescue", "tight_jump"])
def test_fixpoint_and_inversion_grid_with_wide_keys(ctx, yeast, case, monkeypatch):
    """The huge-group paths behind the two-stage (> 64-bit key) sorts: group ids without the strand bit position."""
    monkeypatch.setenv("SWG_FORCE_WIDE_KEYS", "1")
    monkeypatch.setenv("SWG_FIXPOINT_MIN", "2")
    monkeypatch.setenv("SWG_FIXPOINT_VERIFY", "1")
    monkeypatch.setenv("SWG_INV_GRID", "1")
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), yeast, "wide-" + case)


def test_fixpoint_pile_200k(ctx):
    """configs[4] at the largest size the oracle's O(n * window) chaining finishes in seconds: the two 100 k strand groups
    of the pile are above the default threshold, so this is the fixed-point path as shipped."""
    check(ctx, swg.FilterConfig(), synth.skew(n_pile=200_000, n_tiny_groups=20_000, seed=5), "pile200k")


def test_fixpoint_equals_sequential_walk_2m(ctx, monkeypatch):
    """Beyond the oracle's reach: a 2 M pile through the fixed point and through the sequential warp walk (same result).
    SWG_FIXPOINT_VERIFY=1 additionally re-evaluates every position from scratch against the final picks (the call fails if
    one of them would choose differently): the size-independent property that pins the full 50 M configs[4] run."""
    t = synth.skew(n_pile=2_000_000, n_tiny_groups=50_000, seed=6)
    cfg = swg.FilterConfig()
    monkeypatch.setenv("SWG_FIXPOINT_VERIFY", "1")
    s1, c1, st1 = ctx.filter(cfg, t)
    monkeypatch.delenv("SWG_FIXPOINT_VERIFY")
    monkeypatch.setenv("SWG_NO_FIXPOINT", "1")
    s2, c2, st2 = ctx.filter(cfg, t)
    assert np.array_equal(s1, s2) and np.array_equal(c1, c2)
    assert st1.n_chains == st2.n_chains and st1.n_kept == st2.n_kept


@pytest.mark.parametrize("case", ["defaults", "1:1_1:1", "rescue100k", "tight_jump", "self", "mass0"])
def test_inversion_grid_yeast(ctx, yeast, case, monkeypatch):
    """Inversion capture through the bucketed path (taken on its own when a huge group exists), forced onto ordinary input."""
    monkeypatch.setenv("SWG_INV_GRID", "1")
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), yeast, "invgrid-" + case)
    monkeypatch.setenv("SWG_INV_NARROW", "1")  # the narrowest query buckets within budget (default only beyond 65 536 kept chains)
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), yeast, "invgrid-narrow-" + case)


@pytest.mark.parametrize("case", ["defaults", "rescue100k", "tight_jump"])
def test_inversion_grid_without_diagonal_buckets(ctx, yeast, case, monkeypatch):
    """The bucketed inversion capture with query-axis buckets only (what a key beyond 64 bits falls back to)."""
    monkeypatch.setenv("SWG_INV_GRID", "1")
    monkeypatch.setenv("SWG_INV_NO_DIAG", "1")
    if case == "rescue100k":  # ... and the widest query buckets only (the default picks the narrowest width within budget)
        monkeypatch.setenv("SWG_INV_WIDE", "1")
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), yeast, "invgrid-nodiag-" + case)
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), synth.skew(n_pile=20_000, n_tiny_groups=3_000, seed=5, window=3_000_000), "invgrid-nodiag-skew")


@pytest.mark.parametrize("seed", range(0, 160, 4))
def test_inversion_grid_fuzz(ctx, seed, monkeypatch):
    monkeypatch.setenv("SWG_INV_GRID", "1")
    if seed % 8 == 0:
        monkeypatch.setenv("SWG_INV_NARROW", "1")
    test_fuzz_dense(ctx, seed)


def test_edge_cases(ctx):
    cfg = swg.FilterConfig.from_cli(scaffold_mass="0")
    names = ["A#1#c1", "B#1#c1"]
    P, P2 = swg.prefix_ids(names)
    z = lambda *a: np.array(a, dtype=np.int64)
    # empty
    t = swg.MappingTable(z(), z(), z(), z(), z(), z(), z(), z(), np.zeros(0), np.zeros(0, np.uint8), P, P2)
    s, c, st = ctx.filter(cfg, t)
    assert s.size == 0 and st.n_kept == 0
    # one record
    t = swg.MappingTable(z(0), z(1), z(10), z(500), z(10), z(500), z(490), z(480), np.array([480 / 490]), np.array([43], np.uint8), P, P2)
    check(ctx, cfg, t, "single")
    check(ctx, swg.FilterConfig.from_cli(num_mappings="1:1", scaffold_filter="1:1", scaffold_mass="0"), t, "single 1:1")
    # a single self mapping: dropped unless --self
    t = swg.MappingTable(z(0), z(0), z(10), z(500), z(10), z(500), z(490), z(480), np.array([0.98]), np.array([43], np.uint8), P, P2)
    check(ctx, cfg, t, "self dropped")
    # two zero-length records in one group, one alone in its group (size<=1 rule, plane_sweep_exact.rs:274-276)
    t = swg.MappingTable(z(0, 0, 1), z(1, 1, 0), z(5, 5, 7), z(5, 5, 7), z(5, 9, 7), z(5, 9, 7), z(1, 1, 1), z(1, 1, 1), np.array([1.0, 1.0, 1.0]),
                         np.array([43, 43, 43], np.uint8), P, P2)
    check(ctx, cfg, t, "zero-length")
    check(ctx, swg.FilterConfig.from_cli(scaffold_jump="0"), t, "zero-length no scaffold")


def test_range_errors(ctx):
    names = ["A#1#c1", "B#1#c1"]
    P, P2 = swg.prefix_ids(names)
    z = lambda *a: np.array(a, dtype=np.int64)
    t = swg.MappingTable(z(0), z(1), z(500), z(10), z(10), z(500), z(490), z(480), np.array([0.9]), np.array([43], np.uint8), P, P2)
    with pytest.raises(swg.SwgError) as e:
        ctx.filter(swg.FilterConfig(), t)
    assert e.value.code == -2
    # ... but only if the record survives the stage-1 retain (the reference, u64 and unchecked, drops it there too)
    for flags in (dict(min_aln_length="1k"), dict(min_aln_identity="0.95")):
        status, chain, _ = ctx.filter(swg.FilterConfig.from_cli(**flags), t)
        assert status.tolist() == [0] and chain.tolist() == [0]
    t = swg.MappingTable(z(0), z(7), z(10), z(500), z(10), z(500), z(490), z(480), np.array([0.9]), np.array([43], np.uint8), P, P2)
    with pytest.raises(swg.SwgError):
        ctx.filter(swg.FilterConfig(), t)


def test_range_marked_records_through_the_file_front_ends(ctx, tmp_path):
    """A PAF line beyond the u32 table or with end < start is an error only if it passes the retain (ADVICE r1)."""
    good = "q#1#c\t9000\t0\t5000\t+\tt#1#c\t9000\t0\t5000\t4900\t5000\t60\n" * 2
    bad = ("q#1#c\t1\t0\t5000000000\t+\tt#1#c\t1\t0\t10\t5\t10\t60\n"      # beyond u32, block length 10
           "q#1#c\t1\t500\t200\t+\tt#1#c\t1\t0\t10\t5\t10\t60\n")           # end < start, block length 10
    src, out, ref = tmp_path / "in.paf", tmp_path / "out.paf", tmp_path / "ref.paf"
    src.write_text(good + bad + good)
    f = swg.PafFilter(swg.FilterConfig.from_cli(min_aln_length="1k", scaffold_jump="0"))
    f._ctx = ctx
    for host in (False, True):
        f.filter_paf(str(src), str(out), host_frontend=host)
        oracle_lib.filter_paf(f.config, str(src), str(ref))
        assert out.read_bytes() == ref.read_bytes() and out.read_bytes().count(b"\n") == 4
    f2 = swg.PafFilter(swg.FilterConfig.from_cli(scaffold_jump="0"))
    f2._ctx = ctx
    for host in (False, True):
        with pytest.raises(swg.SwgError) as e:
            f2.filter_paf(str(src), str(out), host_frontend=host)
        assert e.value.code == -2


def test_paf_front_end_matches_oracle(ctx, tmp_path):
    """parse + filter + tagged write through swg_filter_paf == the oracle's filter_paf, byte for byte."""
    t = synth.yeast_like(5000, seed=11)
    src = tmp_path / "y.paf"
    synth.write_paf(t, str(src))
    # sprinkle the parser quirks: short line (consumes a rank), CRLF, unparsable number, odd strand, dv after cg
    lines = src.read_text().split("\n")
    lines.insert(3, "short\tline")
    lines.insert(10, "")
    lines[20] = lines[20] + "\r"
    f = lines[30].split("\t"); f[9] = "x12"; lines[30] = "\t".join(f)
    f = lines[31].split("\t"); f[4] = "*"; lines[31] = "\t".join(f)
    f = lines[32].split("\t"); f.append("dv:f:0.25"); lines[32] = "\t".join(f)
    src.write_text("\n".join(lines))
    for flags in ({}, dict(num_mappings="1:1", scaffold_filter="1:1"), dict(scaffold_dist="50k"), dict(scaffold_jump="0")):
        cfg = swg.FilterConfig.from_cli(**flags)
        a, b = tmp_path / "gpu.paf", tmp_path / "orc.paf"
        f = swg.PafFilter(cfg)
        f._ctx = ctx
        f.filter_paf(str(src), str(a))
        oracle_lib.filter_paf(cfg, str(src), str(b))
        assert a.read_bytes() == b.read_bytes(), flags


@pytest.mark.parametrize("case", ["defaults", "1:1_1:1", "rescue100k", "1:1_rescue", "2:3"])
def test_wide_key_paths(ctx, yeast, case, monkeypatch):
    """Keys wider than 64 bits (hundreds of thousands of sequences) take two chained stable sorts instead of one;
    SWG_FORCE_WIDE_KEYS routes an ordinary table through that path."""
    monkeypatch.setenv("SWG_FORCE_WIDE_KEYS", "1")
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), yeast, "wide:" + case)
    for seed in (3, 11, 17):
        t = fuzz_table(seed, 400)
        check(ctx, swg.FilterConfig.from_cli(num_mappings="1:1", scaffold_filter="2:2", scaffold_jump="200", scaffold_mass="0",
                                            scaffold_dist="300"), t, f"wide fuzz{seed}")


@pytest.mark.parametrize("knob", ["SWG_NO_FUSED_KEYS", None])
def test_record_sort_variants(ctx, yeast, knob, monkeypatch):
    """The two forms of the record sort give the same result: (default) keys written by the prefilter pass in the gap layout
    and packed into one word by the third pass; keys from k_chain_keys, packed.
    The default only takes the fused-key path when the key plus the index exceed 64 bits, i.e. on a large table: the PanSN
    table below (12 + 12 + 1 + 28 key bits, 21 index bits) qualifies, the yeast table exercises the other branch."""
    if knob:
        monkeypatch.setenv(knob, "1")
    big = synth.pansn(1_200_000, seed=29, with_names=False)
    for cfg in (swg.FilterConfig(), swg.FilterConfig.from_cli(scaffold_dist="100k"), swg.FilterConfig.from_cli(scaffold_filter="1:1")):
        check(ctx, cfg, big, f"pansn 1.2M {knob}")
    check(ctx, swg.FilterConfig(), yeast, f"yeast {knob}")
    # zero-length intervals among the alive records: the fused keys are discarded and rebuilt after the sweep
    t = fuzz_table(5, 3000)
    check(ctx, swg.FilterConfig.from_cli(scaffold_jump="200", scaffold_mass="0"), t, f"fuzz {knob}")


# ---- the record sort as a counting sort by group (csrc/group_sort.cuh) -------------------------------------------------------
def _shuffled(t, seed):
    t2 = t.take(np.random.default_rng(seed).permutation(t.n))
    return swg.MappingTable(t2.query_id, t2.target_id, t2.query_start, t2.query_end, t2.target_start, t2.target_end, t2.block_length,
                            t2.matches, t2.identity, t2.strand, t2.seq_genome_id, t2.seq_genome2_id)


@pytest.mark.parametrize("knob", [None, "SWG_NO_GROUP_SORT", "SWG_GROUP_SORT_MAX"])
@pytest.mark.parametrize("case", ["defaults", "1:1_1:1", "rescue100k"])
def test_group_sort_paths(ctx, yeast, case, knob, monkeypatch):
    """Default: count + scan + scatter + per-group ordering.  SWG_NO_GROUP_SORT=1: the LSD passes.  SWG_GROUP_SORT_MAX=8: every
    input with a group of more than eight records takes the fallback (table cleaned, keys re-used or rebuilt, LSD passes) —
    the path of a real input with one huge group.  Same result on grouped and on shuffled rows."""
    if knob:
        monkeypatch.setenv(knob, "8" if knob == "SWG_GROUP_SORT_MAX" else "1")
    monkeypatch.setenv("SWG_GROUP_SORT_ALWAYS", "1")  # also for the shuffled rows (by default they would take the LSD passes)
    cfg = swg.FilterConfig.from_cli(**CLI_CASES[case])
    check(ctx, cfg, yeast, f"yeast {knob}")
    check(ctx, cfg, _shuffled(yeast, 1), f"yeast shuffled {knob}")
    big = synth.pansn(300_000, seed=31, n_hap=6)
    check(ctx, cfg, big, f"pansn {knob}")
    check(ctx, cfg, _shuffled(big, 2), f"pansn shuffled {knob}")


@pytest.mark.parametrize("seed", range(6))
def test_group_sort_size_classes(ctx, seed, monkeypatch):
    """Shuffled rows with groups of every size class: one or two records (thread), 3..32 / 33..64 / 65..128 (warp network,
    1 / 2 / 4 words per lane), 129..8192 (CTA in shared memory) and, seed 5, one group beyond that (LSD fallback); many
    equal query starts, so the index tie-break of the stable order is exercised."""
    monkeypatch.setenv("SWG_GROUP_SORT_ALWAYS", "1")
    rng = np.random.default_rng(700 + seed)
    sizes = {0: [1, 2, 3, 5, 31, 32, 33, 63, 64, 65, 100, 127, 128], 1: [129, 200, 256, 257, 1000, 2048, 2049], 2: [8191, 8192, 4097, 3, 1],
             3: list(rng.integers(1, 300, 60)), 4: list(rng.integers(1, 40, 400)), 5: [8193, 50, 2, 1]}[seed]
    names = [f"G{g}#1#c{c}" for g in range(2) for c in range(len(sizes) + 1)]
    nq = len(sizes) + 1
    qid, tid, strand = [], [], []
    for k, sz in enumerate(sizes):
        qid += [k] * sz
        tid += [nq + (k * 7) % nq] * sz
        strand += [ord("+") if k % 3 else ord("-")] * sz
    n = len(qid)
    qs = rng.integers(0, 5000, n) * 100          # many exact ties
    ln = rng.integers(50, 3000, n)
    ts = np.maximum(qs + rng.integers(-2000, 2000, n), 0)
    blk = ln + rng.integers(0, 20, n)
    matches = np.rint(blk * rng.uniform(0.8, 1.0, n)).astype(np.int64)
    P, P2 = swg.prefix_ids(names)
    t = swg.MappingTable(np.array(qid), np.array(tid), qs, qs + ln, ts, ts + ln, blk, matches, matches / blk, np.array(strand, np.uint8), P, P2, None, names)
    t = _shuffled(t, seed)
    for flags in ({}, dict(scaffold_jump="20k", scaffold_mass="0", scaffold_dist="10k"), dict(num_mappings="1:1", scaffold_mass="1k")):
        check(ctx, swg.FilterConfig.from_cli(**flags), t, f"classes seed {seed} {flags}")


def test_group_sort_table_survives_a_failed_call(ctx, yeast):
    """A call that dies after the counting pass (a bad record makes the filter raise) leaves the group table dirty; the next call
    must clear it instead of adding to stale counts."""
    bad = yeast.take(np.arange(yeast.n))
    bad = swg.MappingTable(bad.query_id, bad.target_id, bad.query_start, bad.query_end, bad.target_start, bad.target_end, bad.block_length,
                           bad.matches, bad.identity, bad.strand, bad.seq_genome_id, bad.seq_genome2_id)
    bad.query_end = bad.query_end.copy()
    bad.query_end[yeast.n // 2] = bad.query_start[yeast.n // 2] - 1 if bad.query_start[yeast.n // 2] > 0 else 0
    if bad.query_end[yeast.n // 2] < bad.query_start[yeast.n // 2]:
        with pytest.raises(swg.SwgError):
            ctx.filter(swg.FilterConfig(), bad)
    check(ctx, swg.FilterConfig(), yeast, "after a failed call")


def test_record_sort_method_follows_the_row_order(ctx):
    """Grouped rows (aligner order): counting sort by group, no LSD pass.  The same rows shuffled: the LSD passes (every step of
    the group sort would be a random access).  Same result either way."""
    t = synth.pansn(600_000, seed=41, n_hap=8)
    cfg = swg.FilterConfig()
    s1, c1, st1 = check(ctx, cfg, t, "grouped rows")
    assert st1.n_sort_passes == 0
    perm = np.random.default_rng(5).permutation(t.n)
    t2 = _shuffled(t, 5)
    s2, c2, st2 = check(ctx, cfg, t2, "shuffled rows")
    assert st2.n_sort_passes > 0
    assert np.array_equal(s1[perm], s2)


@pytest.mark.parametrize("n_blocks,group", [(5, 700), (31, 3000), (40, 3000), (7, 6000)])
def test_group_sort_pieces_out_of_place(ctx, n_blocks, group, monkeypatch):
    """A big group whose rows come as a few ascending blocks in the wrong order, separated by rows of other groups (what racing
    slot ranges of a group's runs produce): repaired by putting the pieces into order (up to 32 pieces), by the sorting network
    beyond that and when the blocks interleave."""
    monkeypatch.setenv("SWG_GROUP_SORT_ALWAYS", "1")
    rng = np.random.default_rng(n_blocks * 1000 + group)
    names = [f"G{g}#1#c{c}" for g in range(2) for c in range(4)]
    for interleave in (False, True):
        qs_big = np.sort(rng.integers(0, 3_000_000, group)) * 10
        if interleave:  # blocks = residue classes: every block spans the whole range
            blocks = [qs_big[k::n_blocks] for k in range(n_blocks)]
        else:
            blocks = np.array_split(qs_big, n_blocks)
        order = rng.permutation(n_blocks)
        qid, tid, qs = [], [], []
        for k in order:
            qid += [0] * len(blocks[k]); tid += [4] * len(blocks[k]); qs += list(blocks[k])
            qid += [1, 2]; tid += [5, 6]; qs += list(rng.integers(0, 1000, 2))  # separators: two other groups
        n = len(qid)
        qs = np.array(qs)
        ln = rng.integers(200, 4000, n)
        ts = qs + rng.integers(-500, 500, n) + 1000
        blk = ln + 5
        matches = np.rint(blk * 0.95).astype(np.int64)
        P, P2 = swg.prefix_ids(names)
        t = swg.MappingTable(np.array(qid), np.array(tid), qs, qs + ln, ts, ts + ln, blk, matches, matches / blk, np.full(n, ord("+"), np.uint8), P, P2,
                             None, names)
        _, _, st = check(ctx, swg.FilterConfig.from_cli(scaffold_mass="0"), t, f"pieces {n_blocks} x {group} interleave={interleave}")
        assert st.n_sort_passes == 0 and st.n_unsorted_groups >= 1


# ---- the n = 1 plane sweep of deep piles through the segment tree (csrc/sweep_tree.cuh) ---------------------------------------
@pytest.mark.parametrize("case", ["1:1_1:1", "1:1_rescue", "no_scaffold_1:1", "identity_scoring", "length_scoring", "mass0"])
def test_tree_sweep_everywhere_yeast(ctx, yeast, case, monkeypatch):
    """SWG_SWEEP_TREE_ALL=1: every group of two or more items of an n = 1 sweep is treated as a pile (positions, ranks, segment
    tree, runs of one best item, verdict per item) instead of the neighbour scans of k_sweep_flat1."""
    monkeypatch.setenv("SWG_SWEEP_TREE_ALL", "1")
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), yeast, f"tree sweep {case}")


@pytest.mark.parametrize("seed", range(0, 160, 3))
def test_tree_sweep_everywhere_fuzz(ctx, seed, monkeypatch):
    """Dense, tie-rich fuzz tables (zero-length intervals, equal scores, equal starts) with every n = 1 sweep through the tree."""
    monkeypatch.setenv("SWG_SWEEP_TREE_ALL", "1")
    rng = np.random.default_rng(3000 + seed)
    n = int(rng.integers(2, 600)) if seed < 120 else int(rng.integers(2000, 8000))
    t = fuzz_table(seed, n, hashless=bool(seed % 5 == 0))
    cfg = swg.FilterConfig.from_cli(
        num_mappings=["1:1", "1", "many:1", "1:many"][seed % 4], scaffold_filter=["1:1", "many:many", "1:many"][(seed // 3) % 3],
        overlap=[0.0, 0.5, 0.95, 1.0][seed % 4], scaffold_overlap=[0.5, 0.0, 1.0][seed % 3],
        scaffold_jump=str([0, 50, 200, 1000][(seed // 2) % 4]), scaffold_mass=str([0, 100, 500][seed % 3]),
        scaffold_dist=str([0, 100, 1000][(seed // 5) % 3]), keep_self=bool(seed % 2),
        scoring=["log-length-ani", "ani", "length", "length-ani", "matches"][seed % 5])
    check(ctx, cfg, t, f"tree fuzz{seed}")


@pytest.mark.parametrize("case", ["1:1_1:1", "no_scaffold_1:1"])
def test_tree_sweep_pile(ctx, case):
    """configs[4] shape at a size the oracle finishes: the pile's groups leave the neighbour scans by themselves."""
    t = synth.skew(n_pile=20_000, n_tiny_groups=3_000, seed=5, window=3_000_000)
    check(ctx, swg.FilterConfig.from_cli(**CLI_CASES[case]), t, f"pile {case}")


def test_record_sort_with_more_sequences_than_the_group_table_serves(ctx):
    """6000 sequences: 2 * n_seq^2 entries would exceed the group table's limit, so the record sort runs the LSD passes (the plane
    sweeps' item sort still fits its own, smaller table).  Same result as the oracle either way."""
    t = fuzz_table(77, 5000, n_genomes=6000, n_chr=1, span=200000, max_len=3000, hashless=True)
    for flags in ({}, dict(num_mappings="1:1", scaffold_filter="1:1", scaffold_jump="5000", scaffold_mass="0", scaffold_dist="2000")):
        _, _, st = check(ctx, swg.FilterConfig.from_cli(**flags), t, f"6000 sequences {flags}")
        assert st.n_sort_passes > 0
