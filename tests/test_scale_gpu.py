"""The filter at the sizes users run, where the size-dependent decisions of the pipeline take the branches that small tables
never reach: the width of the record index and the sort path that follows from it, the tile counts of the one-pass scans,
the device PAF writer's 1 GiB windows and the u64 line offsets beyond 4 GiB of text, the batch offsets beyond shared
memory, and the multi-GPU merge helpers.  Every comparison is exact: status byte and chain number of every record, output
bytes, table columns, packed words.

Full-size parity with the oracle lives here: tests/test_parity_gpu.py stops at sizes the single-threaded oracle finishes in
seconds; this file compares 20 M and 40 M record tables against the oracle run over genome-pair units on all host threads
(bench.oracle_mt), after checking that the split reproduces the single-threaded oracle.
"""
import ctypes as C
import hashlib
import os
import shutil

import numpy as np
import pytest

import bench
import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth, with_ids16

from batch_util import check_batch, split, union
from test_paf_device_gpu import COLS
from test_parity_gpu import CLI_CASES, _shuffled

pytestmark = pytest.mark.gpu

THREADS = max(4, os.cpu_count() or 1)  # > 1 always: the genome-pair split is what is under test, not the thread count

# the modes of CLI_CASES that change which kernels run
MODES = ["defaults", "1:1_1:1", "rescue100k", "1:1_rescue", "no_scaffold_1:1", "2:3", "scaffolds_only", "self", "identity_scoring",
         "min_filters"]


def _cfg(mode):
    return swg.FilterConfig.from_cli(**CLI_CASES[mode])


def _first_diff(a, b):
    bad = np.nonzero(a != b)[0]
    return bad[:10], a[bad[:10]], b[bad[:10]]


# ---- A. full-size parity with the oracle, per mode ----------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
def test_oracle_split_equals_single_thread(mode):
    """The reference of the full-size comparisons runs the oracle per genome-pair unit on several threads and merges the chain
    numbers; that is exact only if every grouping of the mode is closed under the genome pair (DESIGN §6)."""
    t = synth.pansn(2_000_000, seed=4, n_hap=24)
    cfg = _cfg(mode)
    s1, c1, _ = oracle_lib.apply_filters(cfg, t)
    _, (s2, c2) = bench.oracle_mt(cfg, t, THREADS, want_result=True)
    bad, x, y = _first_diff(s2, s1)
    assert bad.size == 0, f"{mode}: split status differs at {bad} (split {x}, single {y})"
    bad, x, y = _first_diff(c2, c1)
    assert bad.size == 0, f"{mode}: split chain differs at {bad} (split {x}, single {y})"
    assert int((s1 != 0).sum()) > 0


@pytest.fixture(scope="module")
def pansn20m():
    """The bench workload (configs[2]), rows in aligner order: the counting sort by group."""
    return synth.pansn(20_000_000, seed=3, n_hap=90)


@pytest.fixture(scope="module")
def pansn20m_shuffled(pansn20m):
    """The same rows under a fixed permutation: the LSD passes, every gather random."""
    return _shuffled(pansn20m, 11)


@pytest.fixture(scope="module")
def pansn40m():
    """More than 2^25 records: the record index takes 26 bits."""
    t = synth.pansn(40_000_000, seed=4, n_hap=90)
    assert t.n > 1 << 25
    return t


@pytest.fixture(scope="module")
def pansn40m_shuffled(pansn40m):
    return _shuffled(pansn40m, 12)


def _check_full(ctx, cfg, table, what):
    status, chain, stats = ctx.filter(cfg, table)
    _, (o_status, o_chain) = bench.oracle_mt(cfg, table, THREADS, want_result=True)
    bad, x, y = _first_diff(status, o_status)
    assert bad.size == 0, f"{what}: status differs at {bad} (gpu {x}, oracle {y}) of {table.n}"
    bad, x, y = _first_diff(chain, o_chain)
    assert bad.size == 0, f"{what}: chain id differs at {bad} (gpu {x}, oracle {y})"
    assert stats.n_kept == int((o_status != 0).sum()), f"{what}: n_kept {stats.n_kept}"
    assert stats.n_chains_kept == int(o_chain.max(initial=0)), f"{what}: n_chains_kept {stats.n_chains_kept}"
    assert stats.n_input == table.n and stats.gpu_launches > 0
    return stats


@pytest.mark.parametrize("mode", MODES)
def test_full_size_20m(ctx, pansn20m, mode):
    st = _check_full(ctx, _cfg(mode), pansn20m, f"20M {mode}")
    if mode == "defaults":
        assert st.n_sort_passes == 0, "rows in aligner order: the counting sort by group, no LSD pass"
        assert st.n_chains_kept > 500_000


@pytest.mark.parametrize("mode", ["defaults", "1:1_1:1", "rescue100k"])
def test_full_size_20m_shuffled(ctx, pansn20m_shuffled, mode):
    st = _check_full(ctx, _cfg(mode), pansn20m_shuffled, f"20M shuffled {mode}")
    assert st.n_sort_passes > 0, "shuffled rows: the LSD passes"
    assert st.sort_bytes_per_pair == 16, "the packed LSD sort (one word per record)"


@pytest.mark.parametrize("mode", ["defaults", "1:1_1:1", "rescue100k"])
def test_full_size_40m(ctx, pansn40m, mode):
    st = _check_full(ctx, _cfg(mode), pansn40m, f"40M {mode}")
    assert st.n_sort_passes == 0, "rows in aligner order: the counting sort by group, no LSD pass"


def test_full_size_40m_shuffled(ctx, pansn40m_shuffled):
    """26 index bits in the packed words of the LSD sort."""
    st = _check_full(ctx, _cfg("defaults"), pansn40m_shuffled, "40M shuffled defaults")
    assert st.n_sort_passes > 0 and st.sort_bytes_per_pair == 16


# ---- B. the device PAF front end past its 1 GiB windows and 4 GiB of text -------------------------------------------------------
GiB = 1 << 30
PAF_BYTES = int(4.3 * GiB)  # > 2^32: five output windows
SLACK = 4096                # padding placed this far ahead of a boundary (more than a few block lines)


class _PafBuilder:
    """Copies of one block of PAF lines, the genome names of copy k tagged with k (fixed width, so every copy has the same line
    lengths and the copies are distinct genomes), with lines placed on purpose around given file offsets."""

    def __init__(self, f, block, tag):
        self.f, self.block, self.tag = f, block, tag
        b = np.frombuffer(block, np.uint8)
        self.lo = np.concatenate(([0], np.flatnonzero(b == 10) + 1)).astype(np.int64)
        self.nl = len(self.lo) - 1
        self.pos, self.k, self.i = 0, -1, 0
        self._next_copy()

    def _next_copy(self):
        self.k += 1
        assert self.k < 100
        self.cur = self.block.replace(self.tag, b"%02d#" % self.k)
        self.i = 0

    def put(self, b):
        self.f.write(b)
        self.pos += len(b)

    def lines_until(self, limit):
        """Whole block lines while they end at or before `limit`."""
        while True:
            j = max(self.i, int(np.searchsorted(self.lo, self.lo[self.i] + (limit - self.pos), "right")) - 1)
            if j >= self.nl:
                self.put(self.cur[self.lo[self.i]:])
                self._next_copy()
                continue
            self.put(self.cur[self.lo[self.i]:self.lo[j]])
            self.i = j
            return

    def line(self):
        """The next block line (a record)."""
        if self.i == self.nl:
            self._next_copy()
        b = self.cur[self.lo[self.i]:self.lo[self.i + 1]]
        self.i += 1
        return b

    def pad_to(self, target):
        n = target - self.pos
        assert n >= 2
        self.put(b"#" + b"." * (n - 2) + b"\n")

    def finish(self):
        self.put(self.cur[self.lo[self.i]:])


def _write_big_paf(path, tmp):
    """Returns the boundaries and what sits at each: 'exact' (a record's '\\n' is the last byte before it and the next record
    starts on it) or 'span' (a record starts one byte before it)."""
    t = synth.pansn(2_000_000, seed=5, n_hap=90, with_names=True)
    t.names = [n.replace("#", "@@#", 1) for n in t.names]
    blk = os.path.join(tmp, "block.paf")
    synth.write_paf_fast(t, blk)
    with open(blk, "rb") as f:
        block = f.read()
    os.unlink(blk)
    plan = [(GiB, "span"), (2 * GiB, "exact"), (3 * GiB, "span"), (4 * GiB, "exact")]
    with open(path, "wb") as f:
        w = _PafBuilder(f, block, b"@@#")
        for B, kind in plan:
            w.lines_until(B - SLACK)
            rec = w.line()
            if kind == "exact":
                w.pad_to(B - len(rec))
                w.put(rec)
                assert w.pos == B and rec.endswith(b"\n")
                w.put(w.line())
            else:
                w.pad_to(B - 1)
                w.put(rec)
                assert w.pos > B
            if B == 4 * GiB:  # beyond 2^32: a line for k_tok_long, one for the host patch step, a CRLF line, a short line
                w.put(w.line()[:-1] + b"\tcg:Z:" + b"1=" * 3000 + b"\n")
                w.put(w.line()[:-1] + b"\tdv:f:0.01234567890123456789012345\n")
                w.put(w.line()[:-1] + b"\r\n")
                w.put(b"short\tline\n")
                w.put(w.line())
        w.lines_until(PAF_BYTES)
        w.finish()
        w.put(w.line()[:-1] + b"\tdv:f:0.98765432109876543210987654\r\n")  # the last line: host patch and CRLF at the end
        w.put(b"short\n")
        size = w.pos
    assert size == os.path.getsize(path) > PAF_BYTES
    return plan


def _digest(path):
    """sha256 of the file, streamed, and how many lines carry each status tag."""
    h = hashlib.sha256()
    counts = dict.fromkeys((b"\tst:Z:scaffold\n", b"\tst:Z:rescued\n", b"\tst:Z:unassigned\n"), 0)
    carry = b""
    with open(path, "rb") as f:
        while True:
            b = f.read(64 << 20)
            if not b:
                break
            h.update(b)
            b = carry + b
            cut = b.rfind(b"\n") + 1
            for k in counts:
                counts[k] += b.count(k, 0, cut)
            carry = b[cut:]
    return h.hexdigest(), {k.decode().strip().split(":")[-1]: v for k, v in counts.items()}


def _same_table_columns(a, b):
    assert a.n == b.n
    assert a.names == b.names
    for f in COLS + ("rank",):
        x, y = getattr(a, f), getattr(b, f)
        bad, xv, yv = _first_diff(x, y)
        assert bad.size == 0, f"{f} differs at {bad} (device {xv}, host {yv})"
    bad, xv, yv = _first_diff(a.identity.view(np.uint64), b.identity.view(np.uint64))
    assert bad.size == 0, f"identity bits differ at {bad}"


def test_device_paf_front_end_past_4gib(ctx, tmp_path):
    free0 = shutil.disk_usage(tmp_path).free
    need = int(2.3 * PAF_BYTES)  # the input and one output at a time
    if free0 < need:
        pytest.skip(f"{free0 / 1e9:.1f} GB free under {tmp_path}, {need / 1e9:.1f} GB needed")
    src, out = tmp_path / "big.paf", tmp_path / "out.paf"
    _write_big_paf(str(src), str(tmp_path))
    free_min = shutil.disk_usage(tmp_path).free
    seen = dict(scaffold=0, rescued=0, unassigned=0)
    # scaffold_dist: scaffold and rescued lines, chain numbers of 7 digits; scaffold_jump 0: unassigned lines (no chaining)
    for flags in (dict(scaffold_dist="50k"), dict(scaffold_jump="0")):
        f = swg.PafFilter(swg.FilterConfig.from_cli(**flags))
        f._ctx = ctx
        digests = []
        for host in (False, True):
            st = f.filter_paf(str(src), str(out), host_frontend=host)
            if not host:
                assert st.ms_tokenize > 0, "the device front end fell back to the host front end"
                dev_st = st
            free_min = min(free_min, shutil.disk_usage(tmp_path).free)
            digests.append(_digest(str(out)))
            out.unlink()
        assert digests[0] == digests[1], f"{flags}: device and host front ends wrote different bytes"
        counts = digests[0][1]
        assert sum(counts.values()) == dev_st.n_kept, (flags, counts, dev_st.n_kept)
        if flags.get("scaffold_dist"):
            assert dev_st.n_chains_kept >= 10 ** 6, dev_st.n_chains_kept
        for k, v in counts.items():
            seen[k] += v
    assert all(v > 0 for v in seen.values()), seen
    dev = swg.parse_paf(str(src), ctx)
    host = swg.parse_paf(str(src))
    assert dev.n > 38_000_000 and int(dev.rank[-1]) > 1 << 25
    _same_table_columns(dev, host)
    print(f"\n[scale] PAF input {os.path.getsize(src) / 2**30:.2f} GiB, {dev.n} records; peak disk used under tmp_path "
          f"{(free0 - free_min) / 1e9:.2f} GB")


# ---- C. batches past 8192 tables ------------------------------------------------------------------------------------------------
_NAMES = [f"G{g}#1#c{c}" for g in range(3) for c in range(2)]


def _tiny_tables(seed, K, empty_runs=()):
    """K tables of 1 to 40 records over six sequences (collinear, so chains form); tables in empty_runs are empty; every third
    table has 16-bit id columns, every fifth no identity column."""
    rng = np.random.default_rng(seed)
    P, P2 = swg.prefix_ids(_NAMES)
    empty = set()
    for a, b in empty_runs:
        empty.update(range(a, b))
    tables = []
    for k in range(K):
        n = 0 if k in empty else int(rng.integers(1, 41))
        qid = rng.integers(0, 6, n)
        tid = (qid + rng.integers(1, 6, n)) % 6
        qs = np.sort(rng.integers(0, 200_000, n))
        ln = rng.integers(100, 8000, n)
        ts = qs + rng.integers(0, 3, n) * 1000 + rng.integers(-200, 200, n) + 5000
        blk = ln + rng.integers(0, 30, n)
        matches = np.rint(blk * rng.uniform(0.8, 1.0, n)).astype(np.int64)
        strand = np.where(rng.random(n) < 0.8, ord("+"), ord("-")).astype(np.uint8)
        t = swg.MappingTable(qid, tid, qs, qs + ln, ts, ts + ln, blk, matches, matches / blk, strand, P, P2)
        if k % 5 == 4:
            t.identity = None
        if k % 3 == 1:
            t = with_ids16(t)
        tables.append(t)
    return tables


@pytest.mark.parametrize("flags", [{}, dict(num_mappings="1:1", scaffold_filter="1:1")], ids=["chaining", "1:1"])
@pytest.mark.parametrize("K", [8191, 8192])
def test_batch_at_the_shared_memory_limit(ctx, K, flags):
    """K + 1 record offsets on either side of BATCH_SMEM_TABLES: shared memory, then global memory."""
    check_batch(ctx, swg.FilterConfig.from_cli(**flags), _tiny_tables(K, K), oracle=False, what=f"K={K}")


@pytest.mark.parametrize("flags", [{}, dict(num_mappings="1:1", scaffold_filter="1:1")], ids=["chaining", "1:1"])
def test_batch_of_20000_tiny_tables(ctx, flags):
    K = 20_000
    tables = _tiny_tables(7, K, empty_runs=[(0, 5), (9000, 9040), (K - 7, K)])
    cfg = swg.FilterConfig.from_cli(**flags)
    res, counts, _ = check_batch(ctx, cfg, tables, oracle=False, what="K=20000")
    if not flags:
        assert counts[:, swg.TC_CHAINS_KEPT].sum() > K
    u, offs = union(tables)
    us, uc, _ = ctx.filter(cfg, u)
    for k, (s, c) in enumerate(split(us, uc, offs)):
        assert np.array_equal(s, res[k][0]) and np.array_equal(c, res[k][1]), f"union, table {k}"


# ---- D. the multi-GPU merge helpers on one GPU ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_dev():
    import torch
    return torch, torch.device("cuda", 0)


def _statuses(n, seed):
    """Every status value in every lane position of a 16-record word, then random values."""
    i = np.arange(n)
    s = ((i % 16 + i // 16) % 4).astype(np.uint8)
    if n > 4096:
        s[4096:] = np.random.default_rng(seed).integers(0, 4, n - 4096).astype(np.uint8)
    return s


def _pack_reference(s):
    nw = (len(s) + 15) // 16
    p = np.zeros(nw * 16, np.uint32)
    p[:len(s)] = s & 3
    return (p.reshape(nw, 16) << (2 * np.arange(16, dtype=np.uint32))).sum(axis=1, dtype=np.uint64).astype(np.uint32)


@pytest.mark.parametrize("n", [0, 1, 15, 16, 17, 31, 33, 1_000_007])
def test_pack_status_device(ctx, torch_dev, n):
    torch, dev = torch_dev
    s = _statuses(n, n)
    want = _pack_reference(s)
    nw = len(want)
    sentinel = np.uint32(0xA5A5A5A5)
    for shift in range(16):  # 0: the aligned uint4 path for full words, else the scalar path
        base = torch.zeros(n + 32, dtype=torch.uint8, device=dev)
        assert base.data_ptr() % 16 == 0
        base[shift:shift + n] = torch.from_numpy(s).to(dev)
        packed = torch.from_numpy(np.full(nw + 1, sentinel, np.uint32).view(np.int32)).to(dev)
        torch.cuda.synchronize()
        ctx.pack_status_device(n, base.data_ptr() + shift, packed.data_ptr())
        got = packed.cpu().numpy().view(np.uint32)
        bad = np.nonzero(got[:nw] != want)[0]
        assert bad.size == 0, f"n={n} shift={shift}: words {bad[:8]} = {got[bad[:8]]}, want {want[bad[:8]]}"
        assert got[nw] == sentinel, f"n={n} shift={shift}: the word after the last one was written"


def _renumber_reference(ch, fk, dl):
    if len(fk) == 0:
        return ch.copy()
    ch = ch.astype(np.int64)
    run = np.searchsorted(fk.astype(np.int64), ch, "right") - 1
    out = np.where(ch == 0, 0, ch + dl[np.maximum(run, 0)])
    return (out & 0xFFFFFFFF).astype(np.uint32)


def _renumber_case(ctx, torch, dev, ch, fk, dl, what):
    fk, dl = np.asarray(fk, np.uint32), np.asarray(dl, np.int64)
    want = _renumber_reference(ch, fk, dl)
    d = torch.from_numpy(np.concatenate((ch, [0x5A5A5A5A])).astype(np.uint32).view(np.int32)).to(dev)
    torch.cuda.synchronize()
    ctx.renumber_chains_device(len(ch), d.data_ptr(), fk, dl)
    got = d.cpu().numpy().view(np.uint32)
    bad = np.nonzero(got[:len(ch)] != want)[0]
    assert bad.size == 0, f"{what}: records {bad[:8]} = {got[bad[:8]]}, want {want[bad[:8]]} (from {ch[bad[:8]]})"
    assert got[len(ch)] == 0x5A5A5A5A, f"{what}: the entry after the last one was written"


def test_renumber_chains_device(ctx, torch_dev):
    torch, dev = torch_dev
    rng = np.random.default_rng(9)
    U32MAX = 0xFFFFFFFF
    # one run, positive delta
    ch = rng.integers(0, 5000, 100_003).astype(np.uint32)
    _renumber_case(ctx, torch, dev, ch, [1], [123_456_789], "one run")
    # one run, negative delta down to chain 1
    ch = rng.integers(0, 5000, 1000).astype(np.uint32)
    ch[:3] = [1000, 1001, 4999]
    _renumber_case(ctx, torch, dev, np.where(ch >= 1000, ch, 0).astype(np.uint32), [1000], [-999], "one run, negative")
    # many runs: mixed deltas, chains on the first number of every run and one below the next run's first number
    nu = 3000
    fk = np.concatenate(([1], 1 + np.cumsum(rng.integers(1, 400, nu - 1)))).astype(np.uint32)
    dl = rng.integers(-int(fk[0]), 10 ** 9, nu).astype(np.int64)
    dl[1::2] = -(fk[1::2].astype(np.int64) - 1)  # odd runs move down to start at 1
    last = int(fk[-1]) + 500
    edges = np.concatenate((fk, fk[1:] - 1, [last]))
    ch = np.concatenate((rng.integers(0, last + 1, 1_000_007), edges, np.zeros(17))).astype(np.uint32)
    rng.shuffle(ch)
    _renumber_case(ctx, torch, dev, ch, fk, dl, "many runs")
    # results near 2^32 - 1: large local numbers and deltas that land on the top of the u32 range
    fk = np.array([1, 1000, 0xFFFF0000, 0xFFFFFF00], np.uint32)
    dl = np.array([U32MAX - 999, U32MAX - 1 - 0xFFFEFFFF, 0xFF, -0xFFFFFF00 + 7], np.int64)
    ch = np.array([0, 1, 999, 1000, 0xFFFEFFFF, 0xFFFF0000, 0xFFFFFEFF, 0xFFFFFF00, U32MAX, 0, 5], np.uint32)
    want = _renumber_reference(ch, fk, dl)
    assert want[2] == U32MAX and want[4] == U32MAX - 1 and want[7] == 7 and int(want.max()) == U32MAX
    _renumber_case(ctx, torch, dev, ch, fk, dl, "near 2^32 - 1")
    # nothing to do: no runs, no records
    ch = rng.integers(0, 100, 1000).astype(np.uint32)
    _renumber_case(ctx, torch, dev, ch, np.zeros(0, np.uint32), np.zeros(0, np.int64), "n_units = 0")
    _renumber_case(ctx, torch, dev, np.zeros(0, np.uint32), [1], [5], "n = 0")


def test_merge_helpers_reject_bad_arguments(ctx, torch_dev):
    torch, dev = torch_dev
    lib, h = swg._lib.lib, ctx._h
    buf = torch.zeros(64, dtype=torch.int32, device=dev)
    p = buf.data_ptr()
    fk, dl = np.ones(1, np.uint32), np.ones(1, np.int64)
    fkp, dlp = fk.ctypes.data_as(C.POINTER(C.c_uint32)), dl.ctypes.data_as(C.POINTER(C.c_int64))
    ERR = swg._lib.ERR_ARG
    assert lib.swg_renumber_chains_device(None, 1, p, 1, fkp, dlp) == ERR
    assert lib.swg_renumber_chains_device(h, 1, None, 1, fkp, dlp) == ERR
    assert lib.swg_renumber_chains_device(h, 1, p, 1, None, dlp) == ERR
    assert lib.swg_renumber_chains_device(h, 1, p, 1, fkp, None) == ERR
    assert lib.swg_renumber_chains_device(h, 0x7FFFFFF0, p, 1, fkp, dlp) == ERR
    assert lib.swg_pack_status_device(None, 1, p, p) == ERR
    assert lib.swg_pack_status_device(h, 1, None, p) == ERR
    assert lib.swg_pack_status_device(h, 1, p, None) == ERR
    assert lib.swg_pack_status_device(h, 0x7FFFFFF0, p, p) == ERR
    assert int(buf.abs().sum()) == 0
    # the context is still usable
    assert lib.swg_renumber_chains_device(h, 0, None, 0, None, None) == 0
    assert lib.swg_pack_status_device(h, 0, None, None) == 0
    s = np.array([3, 1, 2], np.uint8)
    st = torch.from_numpy(s).to(dev)
    torch.cuda.synchronize()
    ctx.pack_status_device(3, st.data_ptr(), p)
    assert buf[0].item() == 3 | 1 << 2 | 2 << 4
