"""swg_filter_paf_batch: many PAF files filtered as one union on the device.  Every output must be byte for byte what
swg_filter_paf writes for that file alone (and, for the small files, what the oracle's filter_paf writes), wherever the file
sits and whatever shares the call; the per-file counts match the single calls' stats."""
import gzip
import hashlib
import os
import re
import resource
import shutil

import numpy as np
import pytest

import batch_util
import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
YEAST_NAMES = [f"{g}#{c}" for g in synth.YEAST_GENOMES for c in synth.YEAST_CHROMS]


@pytest.fixture(scope="module")
def ctx():
    with swg.Context(0) as c:
        yield c


def yeast_text(n, seed):
    t = synth.yeast_like(n, seed=seed)
    t.names = YEAST_NAMES
    return t


def write_yeast(path, n, seed, tags=True):
    synth.write_paf(yeast_text(n, seed), str(path), tags=tags)
    return path


def pansn_file(path, n, seed):
    synth.write_paf(synth.pansn(n, seed=seed, n_hap=6, with_names=True), str(path), tags=False)
    return path


def mixed_files(d):
    """The mixed set of test 1, as (name, path)."""
    d.mkdir(exist_ok=True)
    f = {}
    f["yeast_tags"] = write_yeast(d / "yeast_tags.paf", 3000, 1)
    f["pansn"] = pansn_file(d / "pansn.paf", 3000, 3)
    f["golden"] = d / "frontend.paf"
    shutil.copy(os.path.join(HERE, "golden", "frontend.paf"), f["golden"])
    f["share_a"] = write_yeast(d / "share_a.paf", 2000, 5)   # same sequence names as share_b, different records
    f["share_b"] = write_yeast(d / "share_b.paf", 2000, 6)
    f["empty"] = d / "empty.paf"
    f["empty"].write_bytes(b"")
    f["comments"] = d / "comments.paf"
    f["comments"].write_bytes(b"# a comment\nshort\tline\n\n#q\tonly\n")
    data = write_yeast(d / "tmp.paf", 600, 7).read_bytes()
    f["no_final_nl"] = d / "no_final_nl.paf"
    f["no_final_nl"].write_bytes(data.rstrip(b"\n"))
    f["crlf"] = d / "crlf.paf"
    f["crlf"].write_bytes(write_yeast(d / "tmp.paf", 600, 8).read_bytes().replace(b"\n", b"\r\n"))
    f["gz"] = d / "yeast.paf.gz"
    f["gz"].write_bytes(gzip.compress(write_yeast(d / "tmp.paf", 600, 9).read_bytes()))
    # lines above SWG_TOK_LONG (base-level cg:Z:) and dv:f: values the device leaves to the host patch step
    lines = write_yeast(d / "tmp.paf", 400, 10, tags=False).read_bytes().splitlines()
    odd = []
    for i, ln in enumerate(lines):
        if i % 7 == 0:
            ln += b"\tcg:Z:" + b"1=" * (2500 + i)
        elif i % 7 == 3:
            ln += b"\tdv:f:0.0%d23456789012345678901234" % (i % 10)
        odd.append(ln)
    f["long_and_patch"] = d / "long_and_patch.paf"
    f["long_and_patch"].write_bytes(b"\n".join(odd) + b"\n")
    # a self-only file: every record maps a sequence onto itself
    self_lines = []
    for ln in write_yeast(d / "tmp.paf", 300, 11).read_bytes().splitlines():
        c = ln.split(b"\t")
        c[5] = c[0]
        self_lines.append(b"\t".join(c))
    f["self_only"] = d / "self_only.paf"
    f["self_only"].write_bytes(b"\n".join(self_lines) + b"\n")
    (d / "tmp.paf").unlink()
    return list(f.items())


def single(ctx, cfg, src, out):
    f = swg.PafFilter(cfg)
    f._ctx = ctx
    return f.filter_paf(str(src), str(out))


def counts_of(st, out_bytes):
    tags = [ln.rsplit(b"\tst:Z:", 1)[-1] for ln in out_bytes.splitlines()]
    return [st.n_stage1, len(tags), tags.count(b"scaffold"), tags.count(b"rescued"), st.n_chains_kept]


def check_batch(ctx, cfg, files, tmp, what="", oracle=False):
    """Batch over files against the single calls: bytes and counts.  Returns the batch's stats."""
    outs = [tmp / f"batch_{i}.out" for i in range(len(files))]
    counts, bst = ctx.filter_paf_batch(cfg, [str(p) for p in files], [str(o) for o in outs])
    assert counts.shape == (len(files), swg.TC_COUNT)
    for i, (src, o) in enumerate(zip(files, outs)):
        ref = tmp / "single.out"
        st = single(ctx, cfg, src, ref)
        want = ref.read_bytes()
        assert o.read_bytes() == want, f"{what}: file {i} ({src.name}) differs from swg_filter_paf"
        assert counts[i].tolist() == counts_of(st, want), f"{what}: file {i} ({src.name}) counts"
        if oracle and not src.name.endswith(".gz"):  # the oracle reads plain text
            oracle_lib.filter_paf(cfg, str(src), str(ref))
            assert ref.read_bytes() == want, f"{what}: file {i} ({src.name}): swg_filter_paf differs from the oracle"
    assert bst.n_stage1 == int(counts[:, swg.TC_STAGE1].sum())
    assert bst.n_chains_kept == int(counts[:, swg.TC_CHAINS_KEPT].sum())
    return bst


@pytest.fixture(scope="module")
def mixed(tmp_path_factory):
    return mixed_files(tmp_path_factory.mktemp("mixed"))


@pytest.mark.parametrize("name", list(batch_util.CONFIGS))
def test_mixed_files_every_config(ctx, mixed, tmp_path, name):
    cfg = swg.FilterConfig.from_cli(**batch_util.CONFIGS[name])
    paths = [p for _, p in mixed]
    bst = check_batch(ctx, cfg, paths, tmp_path, name, oracle=True)
    assert bst.ms_tokenize > 0, "the batch did not take the device front end"
    if name != "defaults":
        return
    # the namespaces have teeth: the two files that share names, concatenated and filtered as one, give other bytes
    names = dict(mixed)
    cat = tmp_path / "cat.paf"
    cat.write_bytes(names["share_a"].read_bytes() + names["share_b"].read_bytes())
    single(ctx, cfg, cat, tmp_path / "cat.out")
    batch_cat = (tmp_path / f"batch_{paths.index(names['share_a'])}.out").read_bytes() + \
        (tmp_path / f"batch_{paths.index(names['share_b'])}.out").read_bytes()
    assert (tmp_path / "cat.out").read_bytes() != batch_cat


def test_position_independence(ctx, mixed, tmp_path):
    cfg = swg.FilterConfig()
    paths = [p for _, p in mixed]
    target = dict(mixed)["share_b"]
    seen = set()
    rng = np.random.default_rng(3)
    for trial in range(4):
        order = list(rng.permutation(len(paths)))[: 3 + 3 * trial]
        if paths.index(target) not in order:
            order.insert(int(rng.integers(len(order) + 1)), paths.index(target))
        files = [paths[i] for i in order]
        outs = [tmp_path / f"p{trial}_{i}.out" for i in range(len(files))]
        counts, _ = ctx.filter_paf_batch(cfg, [str(p) for p in files], [str(o) for o in outs])
        k = files.index(target)
        seen.add((outs[k].read_bytes(), tuple(counts[k].tolist())))
    assert len(seen) == 1


def _renumber(lines):
    """Chain numbers of a run of output lines from chain_1 (they are one consecutive run of the union's numbering)."""
    nums = [int(m.group(1)) for ln in lines for m in [re.search(rb"\tch:Z:chain_(\d+)", ln)] if m]
    if not nums:
        return lines
    lo = min(nums)
    assert sorted(set(nums)) == list(range(lo, max(nums) + 1))
    return [re.sub(rb"\tch:Z:chain_(\d+)", lambda m: b"\tch:Z:chain_%d" % (int(m.group(1)) - lo + 1), ln) for ln in lines]


def test_union_premise_and_launches(ctx, tmp_path):
    """K = 2000 small files (fewer when the open-file limit cannot hold them in one group): their batch equals one call on
    their concatenation (sequences renamed per file, so that the files stay independent there too), and the batch launches
    no more kernels than that one call plus a constant."""
    limit = resource.getrlimit(resource.RLIMIT_NOFILE)
    soft, hard = limit
    want = 2 * 2000 + 256
    if soft != resource.RLIM_INFINITY and soft < want:
        resource.setrlimit(resource.RLIMIT_NOFILE, (want if hard == resource.RLIM_INFINITY else min(want, hard), hard))
    try:
        soft = resource.getrlimit(resource.RLIMIT_NOFILE)[0]
        # a group holds its inputs and outputs open: (soft - 64) / 2 files, with room for what the test process holds
        K = 2000 if soft == resource.RLIM_INFINITY else min(2000, (soft - 64) // 2 - 64)
        if K < 200:
            pytest.skip(f"an open-file limit of {soft} leaves too few files for one group")
        lines = write_yeast(tmp_path / "all.paf", 30000, 21).read_bytes().splitlines()
        per = len(lines) // K
        files, renamed = [], []
        for k in range(K):
            chunk = lines[k * per:(k + 1) * per]
            p = tmp_path / f"f{k}.paf"
            p.write_bytes(b"\n".join(chunk) + b"\n")
            files.append(p)
            for ln in chunk:
                c = ln.split(b"\t")
                c[0] = b"f%d_" % k + c[0]
                c[5] = b"f%d_" % k + c[5]
                renamed.append(b"\t".join(c))
        cat = tmp_path / "cat.paf"
        cat.write_bytes(b"\n".join(renamed) + b"\n")
        for name in ("defaults", "1:1", "keep_self"):
            cfg = swg.FilterConfig.from_cli(**batch_util.CONFIGS[name])
            outs = [tmp_path / f"o{k}.out" for k in range(K)]
            counts, bst = ctx.filter_paf_batch(cfg, [str(p) for p in files], [str(o) for o in outs])
            sst = single(ctx, cfg, cat, tmp_path / "cat.out")
            got = [ln for k in range(K) for ln in outs[k].read_bytes().splitlines()]
            ref = (tmp_path / "cat.out").read_bytes().splitlines()
            back, pos = [], 0
            for k in range(K):  # the single call's lines of file k: renamed back, chains renumbered from chain_1
                n_k = len(outs[k].read_bytes().splitlines())
                seg = [re.sub(rb"(^|\t)f%d_" % k, rb"\1", ln) for ln in ref[pos:pos + n_k]]
                back += _renumber(seg)
                pos += n_k
            assert pos == len(ref)
            assert back == got, name
            assert bst.n_kept == sst.n_kept and bst.n_stage1 == sst.n_stage1 and bst.n_chains_kept == sst.n_chains_kept
            assert bst.gpu_launches <= sst.gpu_launches + 8, (K, bst.gpu_launches, sst.gpu_launches)
    finally:
        resource.setrlimit(resource.RLIMIT_NOFILE, limit)


BAD_LINE = b"seq1\t1000\t500\t200\t+\tseq2\t2000\t100\t300\t150\t200\t60\n"  # end < start, passes the retain


def test_split_after_the_newline_scan(ctx, tmp_path, monkeypatch):
    """Files of short lines: a group formed from the 64 B/line estimate needs more device memory than the budget once the
    newline scan has counted its lines, so the union is split (here down to single files).  The bytes and counts stay those
    of the single calls; a range error inside a split union fails the call with the file named, and the context stays
    usable."""
    recs = write_yeast(tmp_path / "recs.paf", 60, 31).read_bytes().splitlines()
    pad = b"#\n" * 20000  # 20000 lines that are no records
    files = []
    for k in range(6):
        p = tmp_path / f"s{k}.paf"
        p.write_bytes(b"\n".join(recs[10 * k:10 * k + 10]) + b"\n" + pad)
        files.append(p)
    bad = tmp_path / "bad.paf"
    bad.write_bytes(BAD_LINE + pad)
    cfg = swg.FilterConfig()
    outs = [tmp_path / f"s{k}.out" for k in range(len(files))]
    want = []
    for src in files:
        st = single(ctx, cfg, src, tmp_path / "single.out")
        want.append(((tmp_path / "single.out").read_bytes(), counts_of(st, (tmp_path / "single.out").read_bytes())))
    _, st0 = ctx.filter_paf_batch(cfg, [str(p) for p in files], [str(o) for o in outs])  # one union
    with monkeypatch.context() as m:
        # room for the estimate of all six files (~3 MB beyond the 1 GiB window), not for the lines of any two (~26 MB)
        m.setenv("SWG_PAF_BATCH_MEMORY", str((1 << 30) + (8 << 20)))
        counts, st = ctx.filter_paf_batch(cfg, [str(p) for p in files], [str(o) for o in outs])
        assert [(o.read_bytes(), counts[k].tolist()) for k, o in enumerate(outs)] == want
        assert st.gpu_launches > st0.gpu_launches, "the union was not split"
        with_bad = [str(p) for p in files[:3]] + [str(bad)] + [str(p) for p in files[3:]]
        with pytest.raises(swg.SwgError) as e:
            ctx.filter_paf_batch(cfg, with_bad, [str(tmp_path / f"b{k}.out") for k in range(len(with_bad))])
        assert e.value.code == swg._lib.ERR_RANGE and "file 3" in str(e.value) and "bad.paf" in str(e.value), str(e.value)
        counts, st = ctx.filter_paf_batch(cfg, [str(p) for p in files], [str(o) for o in outs])
        assert [(o.read_bytes(), counts[k].tolist()) for k, o in enumerate(outs)] == want


def test_groups_and_host_route(ctx, mixed, tmp_path, monkeypatch):
    cfg = swg.FilterConfig.from_cli(scaffold_dist="20k")
    paths = [p for _, p in mixed]
    ref = [tmp_path / f"r{i}.out" for i in range(len(paths))]
    counts0, st0 = ctx.filter_paf_batch(cfg, [str(p) for p in paths], [str(o) for o in ref])
    for env in ({"SWG_PAF_BATCH_BYTES": "1"}, {"SWG_PAF_BATCH_BYTES": "300000"}, {"SWG_PAF_FRONTEND": "host"}):
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            outs = [tmp_path / f"g{i}.out" for i in range(len(paths))]
            counts, st = ctx.filter_paf_batch(cfg, [str(p) for p in paths], [str(o) for o in outs])
        for a, b in zip(ref, outs):
            assert a.read_bytes() == b.read_bytes(), env
        assert np.array_equal(counts, counts0), env
        if "SWG_PAF_BATCH_BYTES" in env:
            assert st.gpu_launches > st0.gpu_launches, "a small SWG_PAF_BATCH_BYTES did not split the call into groups"
        else:
            assert st.ms_tokenize == 0


def test_errors_and_state(ctx, mixed, tmp_path):
    cfg = swg.FilterConfig()
    paths = [str(p) for _, p in mixed][:4]
    outs = [str(tmp_path / f"e{i}.out") for i in range(len(paths))]
    counts, st = ctx.filter_paf_batch(cfg, [], [])
    assert counts.shape == (0, swg.TC_COUNT) and st.n_input == 0
    # two equal output paths
    with pytest.raises(swg.SwgError) as e:
        ctx.filter_paf_batch(cfg, paths[:2], [outs[0], outs[0]])
    assert e.value.code == swg._lib.ERR_ARG and outs[0] in str(e.value)
    # an input that cannot be opened: nothing is created
    missing = str(tmp_path / "missing.paf")
    with pytest.raises(swg.SwgError) as e:
        ctx.filter_paf_batch(cfg, paths[:2] + [missing], outs[:3])
    assert e.value.code == swg._lib.ERR_IO and "missing.paf" in str(e.value) and "file 2" in str(e.value)
    assert not any(os.path.exists(o) for o in outs[:3])
    # an output that cannot be created
    with pytest.raises(swg.SwgError) as e:
        ctx.filter_paf_batch(cfg, paths[:2], [outs[0], str(tmp_path / "no_dir" / "x.out")])
    assert e.value.code == swg._lib.ERR_IO and "no_dir" in str(e.value)
    # a range error in one file fails the call and names it
    bad = tmp_path / "bad.paf"
    bad.write_bytes(BAD_LINE)
    with pytest.raises(swg.SwgError) as e:
        ctx.filter_paf_batch(cfg, paths[:2] + [str(bad)], outs[:3])
    assert e.value.code == swg._lib.ERR_RANGE and "bad.paf" in str(e.value), str(e.value)
    # NULL entries
    import ctypes as C
    arr = (C.c_char_p * 2)(os.fsencode(paths[0]), None)
    oarr = (C.c_char_p * 2)(os.fsencode(outs[0]), os.fsencode(outs[1]))
    cc = cfg.to_c()
    assert swg._lib.lib.swg_filter_paf_batch(ctx._h, C.byref(cc), 2, arr, oarr, None, None) == swg._lib.ERR_ARG
    assert swg._lib.lib.swg_filter_paf_batch(ctx._h, C.byref(cc), 2, None, oarr, None, None) == swg._lib.ERR_ARG
    assert swg._lib.lib.swg_filter_paf_batch(ctx._h, C.byref(cc), 0, None, None, None, None) == 0
    # the context stays usable: a following batch is right, and no last-call chains are reported
    all_paths = [p for _, p in mixed]
    check_batch(ctx, cfg, all_paths, tmp_path, "after errors")
    ctx.filter_paf_batch(cfg, [str(p) for p in all_paths], outs[:1] + [str(tmp_path / f"z{i}") for i in range(1, len(all_paths))])
    assert ctx.last_chain_units()[0].size == 0


def _digest(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        while True:
            b = f.read(64 << 20)
            if not b:
                return h.hexdigest()
            h.update(b)


GiB = 1 << 30


def _write_sized(path, nbytes, block, tag):
    """Repeats of a block of PAF lines up to nbytes; every repeat gets its own sequence names (the R0000 field), so its
    groups stay independent and the work grows linearly."""
    with open(path, "wb") as f:
        pos, r = 0, 0
        while pos + len(block) <= nbytes:
            f.write(block.replace(b"R0000", b"%s%04d" % (tag, r % 10000)))
            pos += len(block)
            r += 1
        rest = block[: nbytes - pos]
        f.write(rest[: rest.rfind(b"\n") + 1])


def test_union_past_4gib(ctx, tmp_path):
    """Three files whose union passes 4 GiB of text: boundaries inside the second 1 GiB window and inside the fourth (the
    last whose offsets fit in u32); every output equals its single call."""
    sizes = [int(1.5 * GiB), int(2.2 * GiB), int(0.7 * GiB)]
    need = int(2.3 * sum(sizes))
    if shutil.disk_usage(tmp_path).free < need:
        pytest.skip(f"{shutil.disk_usage(tmp_path).free / 1e9:.1f} GB free under {tmp_path}, {need / 1e9:.1f} GB needed")
    t = synth.yeast_like(200000, seed=31)
    t.names = [f"R0000_{n}" for n in YEAST_NAMES]
    synth.write_paf_fast(t, str(tmp_path / "block.paf"))
    block = (tmp_path / "block.paf").read_bytes()
    (tmp_path / "block.paf").unlink()
    files = [tmp_path / f"big{i}.paf" for i in range(3)]
    for i, (p, s) in enumerate(zip(files, sizes)):
        _write_sized(str(p), s, block, b"ABC"[i:i + 1])
    assert sum(os.path.getsize(p) for p in files) > 4 * GiB
    cfg = swg.FilterConfig.from_cli(scaffold_dist="50k")
    outs = [tmp_path / f"bo{i}.out" for i in range(3)]
    counts, bst = ctx.filter_paf_batch(cfg, [str(p) for p in files], [str(o) for o in outs])
    assert bst.ms_tokenize > 0
    got = []
    for o in outs:
        got.append(_digest(o))
        o.unlink()
    for i, p in enumerate(files):
        out = tmp_path / "single.out"
        st = single(ctx, cfg, p, out)
        assert _digest(out) == got[i], f"file {i} differs from swg_filter_paf"
        assert counts[i, swg.TC_STAGE1] == st.n_stage1 and counts[i, swg.TC_KEPT] == st.n_kept
        assert counts[i, swg.TC_CHAINS_KEPT] == st.n_chains_kept
        out.unlink()
