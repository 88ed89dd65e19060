#!/usr/bin/env python
"""bench.py — Mmappings/s of the mapping filter (BASELINE.json metric) on N B200s of one node.

A "step" is one pass of the filter (stage-1 retain -> plane sweep -> chaining -> scaffold filter/sweep ->
anchors/inversions [-> rescue]) over one batch of synthetic mappings.
  N = 1 : configs[2]  "synthetic PanSN PAF, 90 haplotypes x 24 chromosomes, 20M mappings, default pipeline"
  N > 1 : configs[3]  ONE unit-structured table of 25 M x N mappings (200 M at 8) with --scaffold-dist 100k, partitioned by
          genome-pair unit with swg_shard_plan_units; every rank builds and filters only its shard (weak scaling).  The timed
          step includes what makes the result global: the (A, count) exchange per unit + chain renumbering on the device
          (chain_N identical to a single-GPU run) and the gather of the 2-bit status planes (the "keep bitmap" gather).
`value`  : device-timed, inputs resident in HBM (CUDA events, max over ranks).
`e2e`    : the same through swg_filter with pinned HOST buffers, H2D and D2H inside the timed region.
`parity` : the GPU result of the timed workload compared with the CPU oracle over the WHOLE table (every rank its shard);
           a mismatch fails the run.
`--impl reference` : the CPU oracle (the Rust reference cannot be built here) on all host threads; this arm imports
          neither the product package nor its library (numpy + workloads/ + tests/oracle_lib.py only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True  # the bench leaves the source tree as it found it (which may be read-only)

import numpy as np

METRIC = "Mmappings/s filtered (sweep+scaffold)"
N_HAP = 90
# --dump-outputs: status (f32) and chain id (f64) of at most this many records over all ranks, 48 MB; the result counts of swg_stats
DUMP_RECORDS = 4_000_000
DUMP_STATS = ("n_input", "n_stage1", "n_after_sweep", "n_chains", "n_chains_after_mass", "n_chains_kept", "n_anchors", "n_rescued",
              "n_kept")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][2]) if self.rows[0][2].isdigit() else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ---- workload (pure numpy: shared by both arms) -----------------------------------------------------------------------
def workload(n_gpus, rank, records):
    """-> (table of this rank, description dict).  N = 1: configs[2] (seed 3).  N > 1: this rank's shard of the ONE
    unit-structured configs[3] table (seed 4; LPT of the planned unit sizes, the rule of swg_shard_plan_units)."""
    from workloads import synth
    if n_gpus == 1:
        n = records or 20_000_000
        table = synth.pansn(n, seed=3)
        return table, {"name": f"configs[2]: synthetic PanSN, 90 haplotypes x 24 chromosomes, {n} mappings, default pipeline",
                       "flags": "defaults", "b_alg": 300, "units": None}
    per = records or 25_000_000
    n_total = per * n_gpus
    pairs, quota = synth.pansn_unit_plan(n_total, N_HAP)
    shard_of_unit = lpt_units(quota, n_gpus)
    mine = np.nonzero(shard_of_unit == rank)[0]
    table, sizes = synth.pansn_units(mine, n_total, 4, N_HAP)
    name = (f"configs[3]: ONE synthetic PanSN table of {n_total} mappings in {len(pairs)} genome-pair units, sharded by unit over "
            f"{n_gpus} GPUs ({per} drawn per GPU), --scaffold-dist 100k")
    return table, {"name": name, "flags": "--scaffold-dist 100k", "b_alg": 520,
                   "units": {"mine": mine, "sizes": sizes, "n_units": len(pairs), "quota": quota}}


def lpt_units(sizes, n_shards):
    """The rule of swg_shard_plan_units (largest first, ties by unit index, least loaded shard, ties by lowest shard) in
    numpy, so that the reference arm shards identically without loading the product library."""
    order = sorted(range(len(sizes)), key=lambda u: (-int(sizes[u]), u))
    load = [0] * n_shards
    out = np.zeros(len(sizes), np.uint32)
    for u in order:
        b = min(range(n_shards), key=lambda s: (load[s], s))
        out[u] = b
        load[b] += int(sizes[u])
    return out


def oracle_config(n_gpus):
    import oracle_lib
    return oracle_lib.Config(scaffold_max_deviation=100_000) if n_gpus > 1 else oracle_lib.Config()


def oracle_mt(cfg, table, threads, want_result=False):
    """The CPU restatement on `threads` host threads: genome-pair units (independent in the reference's algorithm) are
    size-balanced over threads; each thread runs the single-threaded filter on its units (ctypes releases the GIL).
    -> (seconds, (status, chain) merged over the thread shards or None)."""
    import oracle_lib
    from workloads import lpt_shards
    from concurrent.futures import ThreadPoolExecutor
    if threads <= 1:
        t0 = time.perf_counter()
        st, ch, _ = oracle_lib.apply_filters(cfg, table)
        return time.perf_counter() - t0, ((st, ch) if want_result else None)
    shard_of, _ = lpt_shards(table, threads)
    index = [np.nonzero(shard_of == s)[0] for s in range(threads)]
    parts = [table.take(ix) for ix in index]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        res = list(ex.map(lambda p: oracle_lib.apply_filters(cfg, p, with_chain_keys=want_result), parts))
    dt = time.perf_counter() - t0
    if not want_result:
        return dt, None
    # merge the thread shards' chain numbers: runs of equal A (one per genome-pair unit), ordered by the global index of A
    runs = []
    for ix, r in zip(index, res):
        ka = r[3]
        if len(ka):
            first = np.nonzero(np.concatenate(([True], ka[1:] != ka[:-1])))[0]
            runs.append((ix[ka[first]].astype(np.int64), np.diff(np.concatenate((first, [len(ka)]))).astype(np.int64), first))
        else:
            runs.append((np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.int64)))
    a = np.concatenate([r[0] for r in runs])
    cnt = np.concatenate([r[1] for r in runs])
    order = np.argsort(a, kind="stable")
    excl = np.zeros(len(a), np.int64)
    excl[order] = np.cumsum(cnt[order]) - cnt[order]
    status, chain = np.zeros(table.n, np.uint8), np.zeros(table.n, np.uint32)
    off = 0
    for ix, r, (ra, rc, first) in zip(index, res, runs):
        k = len(ra)
        lut = np.zeros(len(r[3]) + 1, np.int64)
        if k:
            lut[1:] = np.arange(1, len(r[3]) + 1) + np.repeat(excl[off:off + k] - first, rc)
        off += k
        status[ix] = r[0]
        chain[ix] = lut[r[1]]
    return dt, (status, chain)


def run_reference(args, n_gpus):
    """The CPU arm: the oracle on all host threads over this rank-0 workload (bounded sample), plus the honest
    single-thread figure (the reference filter itself is single-threaded: SURVEY 0-2)."""
    table, desc = workload(n_gpus, 0, args.records)
    cfg = oracle_config(n_gpus)
    sample = table.take(np.arange(min(table.n, args.cpu_sample)))
    cores = os.cpu_count() or 1
    times = []
    for i in range(args.warmup + args.steps):
        dt, _ = oracle_mt(cfg, sample, cores)
        if i >= args.warmup:
            times.append(dt)
    per = sum(times) / len(times)
    v = sample.n / per / 1e6
    one = table.take(np.arange(min(table.n, args.cpu_sample_1t)))
    dt1, _ = oracle_mt(cfg, one, 1)
    sample_desc = f"first {sample.n} records (whole genome pairs) of the rank-0 workload, filter only, records in memory"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Mmappings/s", "n_gpus": n_gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32/u64/f64", "data": "synthetic",
        "config": {"workload": desc["name"], "records_per_gpu": int(table.n), "flags": desc["flags"]},
        "cpu_baseline": {"value": v, "unit": "Mmappings/s", "cores": cores, "kind": "port", "sample": sample_desc,
                         "note": "C++ oracle (statement-level restatement of the Rust reference, which cannot be built here: no cargo); "
                                 "the reference filter itself is single-threaded, this arm additionally spreads genome pairs over all host threads"},
        "oracle_1t": {"value": one.n / dt1 / 1e6, "unit": "Mmappings/s", "cores": 1,
                      "sample": f"first {one.n} records, single thread (what the reference's own filter does), {dt1:.1f} s"},
        "e2e": {"value": v, "unit": "Mmappings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ---- the B200 arm -----------------------------------------------------------------------------------------------------
class gpu_numa_affinity:
    """While the pinned host buffers of a rank are allocated and filled, the process runs on the cores of the GPU's NUMA node, so
    that first touch places the pages next to the GPU (8 ranks that all allocate on node 0 share that node's memory and PCIe
    root: round 1 measured 0.5 e2e efficiency at 8 GPUs).  The previous affinity is restored on exit: the CPU legs of the bench
    use every core.  Best effort: any failure leaves the affinity alone."""

    def __init__(self, device_index):
        self.info = None
        self.note = None
        self.prev = None
        try:
            import torch
            p = torch.cuda.get_device_properties(device_index)
            bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
            node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
            if node < 0:
                self.note = {"gpu_pci": bdf, "numa_node": node, "bound": False}
                return
            cpus = set()
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
            cpus &= os.sched_getaffinity(0)
            if cpus:
                self.cpus = cpus
                self.info = {"gpu_pci": bdf, "numa_node": node, "cores_of_node_available": len(cpus), "bound": True}
                self.note = self.info
        except Exception as e:
            self.info = None
            self.note = {"bound": False, "why": repr(e)[:120]}

    def __enter__(self):
        if self.info:
            try:
                self.prev = os.sched_getaffinity(0)
                os.sched_setaffinity(0, self.cpus)
            except Exception:
                self.prev = None
        return self

    def __exit__(self, *a):
        if self.prev is not None:
            try:
                os.sched_setaffinity(0, self.prev)
            except Exception:
                pass


def pinned_copy(table, with_identity):
    """Column copies in page-locked memory (torch is only the allocator)."""
    import torch
    import sweepga_b200 as swg

    def pin(a):
        t = torch.empty(max(a.nbytes, 1), dtype=torch.uint8, pin_memory=True)
        v = t.numpy()[: a.nbytes].view(a.dtype)
        v[...] = a
        return v, t
    keep = []
    cols = {}
    for f in ("query_id", "target_id", "query_start", "query_end", "target_start", "target_end", "block_length", "matches", "identity",
              "strand", "seq_genome_id", "seq_genome2_id"):
        if f == "identity" and not with_identity:
            cols[f] = None
            continue
        v, t = pin(getattr(table, f))
        cols[f] = v
        keep.append(t)
    t2 = swg.MappingTable(**cols)
    if table.n_seq <= 65536:  # 16-bit sequence ids on the wire (swg_mappings.query_id16 / target_id16)
        def alloc(a):
            v, t = pin(a)
            keep.append(t)
            return v
        t2 = swg.with_ids16(t2, alloc)
    t2._pins = keep
    st = torch.empty(max(table.n, 1), dtype=torch.uint8, pin_memory=True)
    ch = torch.empty(max(table.n, 1), dtype=torch.int32, pin_memory=True)
    t2._out = (st.numpy()[: table.n], ch.numpy()[: table.n].view(np.uint32), st, ch)
    return t2


def dump_outputs(out_dir, status, chain, stats, world, rank):
    """What the timed step returned to its caller, as out_dir/<name>.npy (out_dir/<name>_rank<r>.npy for each of several ranks):
    status and chain id of every record, or of a fixed seeded sample of DUMP_RECORDS / world records (in record order) when the
    table is larger, and the result counts DUMP_STATS."""
    os.makedirs(out_dir, exist_ok=True)
    n, m = len(status), DUMP_RECORDS // world
    suffix = "" if world == 1 else f"_rank{rank}"
    idx = np.sort(np.random.default_rng(rank).choice(n, m, replace=False)) if n > m else np.arange(n)
    np.save(os.path.join(out_dir, f"status{suffix}.npy"), status[idx].astype(np.float32))
    np.save(os.path.join(out_dir, f"chain_id{suffix}.npy"), chain[idx].astype(np.float64))
    np.save(os.path.join(out_dir, f"stats{suffix}.npy"), np.array([getattr(stats, k) for k in DUMP_STATS], np.float64))


def paf_file_leg(ctx, cfg, n_lines):
    """Extra, informational: PafFilter::filter_paf file to file (text tokenised and tagged output assembled on the GPU,
    swg_filter_paf) and the same call with the host front end, on a synthetic PAF with cg:Z: tags.  Never fails the bench."""
    import shutil
    import tempfile
    import sweepga_b200 as swg
    from sweepga_b200 import synth
    d = tempfile.mkdtemp(prefix="swg_bench_")
    try:
        t = synth.pansn(n_lines, seed=3, n_hap=40, with_names=True)
        src, out = os.path.join(d, "in.paf"), os.path.join(d, "out.paf")
        synth.write_paf_fast(t, src)
        f = swg.PafFilter(cfg)
        f._ctx = ctx
        res = {}
        for key, host in (("device_front_end", False), ("host_front_end", True)):
            f.filter_paf(src, out, host_frontend=host)  # warm-up: page cache, arenas, pinned pieces
            os.unlink(out)                               # a fresh output file (ext4 flushes a re-written truncated file at close)
            t0 = time.time()
            st = f.filter_paf(src, out, host_frontend=host)
            dt = time.time() - t0
            res[key] = {"wall_s": dt, "Mlines_per_s": t.n / dt / 1e6, "ms_upload": st.ms_h2d, "ms_tokenize": st.ms_tokenize,
                        "ms_filter": st.ms_device, "ms_write": st.ms_write, "gpu_launches": int(st.gpu_launches), "kept": int(st.n_kept)}
        res["lines"] = int(t.n)
        res["input_bytes"] = os.path.getsize(src)
        return res
    except Exception as e:  # informational leg only
        return {"error": repr(e)[:200]}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def skew_leg(ctx, cfg, n_pile):
    """Extra, informational: configs[4] (one centromeric pile + 100 k tiny groups) at --skew-pile mappings (default: the full
    50 M); the two strand groups of the pile go through the fixed-point chaining (DESIGN 4a).  The first call runs with
    SWG_FIXPOINT_VERIFY=1 (after the last round every position of the pile is re-evaluated from scratch against the final picks;
    the call fails if one would choose differently) and doubles as the warm-up, the second is timed.  Host buffers, wall clock.
    Never fails the bench."""
    try:
        from sweepga_b200 import synth
        t = synth.skew(n_pile=n_pile, n_tiny_groups=100_000, seed=5)
        os.environ["SWG_FIXPOINT_VERIFY"] = "1"
        try:
            _, _, st0 = ctx.filter(cfg, t)
            verified = True
        finally:
            del os.environ["SWG_FIXPOINT_VERIFY"]
        t0 = time.time()
        s1, c1, st = ctx.filter(cfg, t)
        dt = time.time() - t0
        same = bool(st0.n_kept == st.n_kept and st0.n_chains_kept == st.n_chains_kept)
        return {"workload": f"configs[4]: {n_pile} mappings on one chromosome pair (95 % inside 6 Mbp) + 100000 tiny groups, defaults",
                "records": int(t.n), "wall_s": dt, "ms_device": float(st.ms_device), "Mmappings_per_s": t.n / dt / 1e6,
                "gpu_launches": int(st.gpu_launches), "kept": int(st.n_kept), "chains": int(st.n_chains_kept),
                "fixpoint_verified": verified and same,
                "ms_device_with_verification_pass": float(st0.ms_device)}
    except Exception as e:  # informational leg only
        return {"error": repr(e)[:200]}


def modes_leg(ctx, d_in, d_res, n):
    """Extra, informational: the 1:1 / 1:1 mode (both plane sweeps fully exercised: configs[1]'s flags) on the resident configs[2]
    table, and --num-mappings 1:1 on a configs[4]-shaped pile of 1 M mappings (deep piles take the segment-tree sweep)."""
    try:
        import sweepga_b200 as swg
        from sweepga_b200 import synth
        out = {}
        cfg = swg.FilterConfig.from_cli(num_mappings="1:1", scaffold_filter="1:1")
        ctx.filter_device(cfg, d_in, d_res)
        sts = [ctx.filter_device(cfg, d_in, d_res) for _ in range(3)]
        ms = min(s.ms_device for s in sts)
        peak, _ = peaks()
        out["1:1/1:1 on the 20 M table"] = {"ms_device": ms, "Mmappings_per_s": n / ms / 1e3, "gpu_launches": int(sts[-1].gpu_launches),
                                            "kept": int(sts[-1].n_kept), "pipeline_algorithmic_bytes_per_mapping": 1134,
                                            "pipeline_fraction_of_hbm_roofline": n * 1134 / (ms / 1e3) / 1e9 / peak}
        try:  # the sweep kernels themselves: DRAM fraction and threads per instruction come from an ncu capture, not from this run
            out["roofline_sweep"] = json.load(open(os.path.join(ROOT, "profiles", "sweep_profile.json")))
        except Exception:
            pass
        t = synth.skew(n_pile=1_000_000, n_tiny_groups=100_000, seed=5)
        p_in, p_res = ctx.upload(t)
        cfg = swg.FilterConfig.from_cli(num_mappings="1:1", scaffold_jump="0")
        ctx.filter_device(cfg, p_in, p_res)
        st = ctx.filter_device(cfg, p_in, p_res)
        ctx.release(p_in, p_res)
        out["--num-mappings 1:1 on a 1 M pile + 100000 tiny groups"] = {"records": int(t.n), "ms_device": float(st.ms_device),
                                                                         "gpu_launches": int(st.gpu_launches), "kept": int(st.n_kept)}
        return out
    except Exception as e:
        return {"error": repr(e)[:200]}


def small_leg(ctx):
    """configs[0] / configs[1]: the yeast-shaped table (~30 k records), defaults and 1:1 / 1:1 — latency-bound calls;
    device-resident, CUDA-event time per call, mean of 20 after 3 warm-ups."""
    try:
        import sweepga_b200 as swg
        from sweepga_b200 import synth
        t = synth.yeast_like(30000, seed=1)
        d_in, d_res = ctx.upload(t)
        out = {"records": int(t.n)}
        for key, cfg in (("configs[0] defaults", swg.FilterConfig()),
                         ("configs[1] 1:1/1:1", swg.FilterConfig.from_cli(num_mappings="1:1", scaffold_filter="1:1"))):
            for _ in range(3):
                ctx.filter_device(cfg, d_in, d_res)
            ms, t0 = [], time.perf_counter()
            for _ in range(20):
                st = ctx.filter_device(cfg, d_in, d_res)
                ms.append(st.ms_device)
            wall = (time.perf_counter() - t0) / 20
            out[key] = {"ms_device": sum(ms) / len(ms), "ms_wall": wall * 1e3, "gpu_launches": int(st.gpu_launches), "kept": int(st.n_kept)}
        ctx.release(d_in, d_res)
        return out
    except Exception as e:
        return {"error": repr(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--records", type=int, default=0, help="override the per-GPU record count (debug only)")
    ap.add_argument("--paf-lines", type=int, default=2_000_000,
                    help="N = 1 only: also time swg_filter_paf file to file on a synthetic PAF of this many lines (0 = skip)")
    ap.add_argument("--skew-pile", type=int, default=50_000_000,
                    help="size of the configs[4] pile of the informational skew leg (0 = skip)")
    ap.add_argument("--cpu-sample", type=int, default=20_000_000,
                    help="records of the workload the CPU oracle is timed on (~20 core-seconds at the default)")
    ap.add_argument("--cpu-sample-1t", type=int, default=2_000_000, help="records of the single-thread oracle figure")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-size comparison with the oracle (profiling runs)")
    ap.add_argument("--no-anchor", action="store_true", help="N = 1: skip the configs[3]-shard scaling anchor")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (status and chain id of a fixed seeded sample "
                         "of the records, the result counts) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the result of the b200 arm")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n_gpus = args.gpus

    import __graft_entry__
    if not os.path.exists(__graft_entry__.LIB) or not os.path.exists(__graft_entry__.ORACLE):
        sys.exit("the native libraries are not built: run `python __graft_entry__.py` first")

    if args.impl == "reference":
        if rank == 0:
            run_reference(args, n_gpus)
        return

    import ctypes as C
    import torch
    import torch.distributed as dist
    import sweepga_b200 as swg
    from sweepga_b200.distributed import unit_offsets
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    wtable, desc = workload(n_gpus, rank, args.records)
    table = swg.MappingTable(wtable.query_id, wtable.target_id, wtable.query_start, wtable.query_end, wtable.target_start,
                             wtable.target_end, wtable.block_length, wtable.matches, wtable.identity, wtable.strand,
                             wtable.seq_genome_id, wtable.seq_genome2_id)
    cfg = swg.FilterConfig.from_cli(scaffold_dist="100k") if n_gpus > 1 else swg.FilterConfig()
    n = table.n
    ctx = swg.Context(local_rank)
    # the synthetic tables carry no dv:f: / cg:Z: tags: identity == matches / max(block_length, 1) bit for bit, so both the
    # device-resident table and the e2e call leave the column out (swg_mappings.identity == NULL: the device derives it)
    identity_is_default = bool(np.array_equal(table.identity, table.matches / np.maximum(table.block_length, 1)))
    if identity_is_default:
        import copy
        dtable = copy.copy(table)
        dtable.identity = None
    else:
        dtable = table
    d_in, d_res = ctx.upload(dtable)

    # ---- N > 1: what makes the shard results global ------------------------------------------------------------------
    units = desc["units"]
    if world > 1:
        all_sizes = torch.zeros(units["n_units"], dtype=torch.int64, device=dev)
        all_sizes[torch.from_numpy(units["mine"]).to(dev)] = torch.from_numpy(units["sizes"]).to(dev)
        dist.all_reduce(all_sizes)
        all_sizes = all_sizes.cpu().numpy()
        goff = np.concatenate(([0], np.cumsum(all_sizes)))           # global record index of every unit's first record
        loff = np.concatenate(([0], np.cumsum(units["sizes"])))      # ... inside this shard
        n_words = (n + 15) // 16
        max_words = torch.tensor([n_words], dtype=torch.int64, device=dev)
        dist.all_reduce(max_words, op=dist.ReduceOp.MAX)
        max_words = int(max_words.item())
        status_t = torch.zeros(n, dtype=torch.uint8, device=dev)
        chain_t = torch.zeros(n, dtype=torch.int32, device=dev)
        packed_t = torch.zeros(max_words, dtype=torch.int32, device=dev)
        gathered_t = torch.zeros(max_words * world, dtype=torch.int32, device=dev)
        d_res.status = C.cast(status_t.data_ptr(), C.POINTER(C.c_uint8))
        d_res.chain_id = C.cast(chain_t.data_ptr(), C.POINTER(C.c_uint32))

    if world > 1:
        n_mine = len(units["mine"])
        max_units = torch.tensor([n_mine], dtype=torch.int64, device=dev)
        dist.all_reduce(max_units, op=dist.ReduceOp.MAX)
        max_units = int(max_units.item())
        runs_send = torch.zeros(max_units * 2 + 1, dtype=torch.int64, device=dev)     # [count, A..., n...]
        runs_recv = torch.zeros((max_units * 2 + 1) * world, dtype=torch.int64, device=dev)
        runs_host = torch.zeros(max_units * 2 + 1, dtype=torch.int64, pin_memory=True)

    def make_global(res_chain_ptr, n_ch):
        """chain_N of the shard -> chain_N of the whole table: one (A, count) pair per genome-pair unit is exchanged (one
        fixed-size all-gather of a few thousand integers), sorted by the global index of A, prefix-summed, and every rank adds
        its runs' offsets on the device.  Returns the number of kernels of ours launched here."""
        a_loc, first_k = ctx.last_chain_units(n_mine)
        k = len(a_loc)
        cnt = np.diff(np.concatenate((first_k.astype(np.int64), [n_ch + 1])))
        u = np.searchsorted(loff, a_loc, side="right") - 1
        a_glob = goff[units["mine"][u]] + (a_loc.astype(np.int64) - loff[u])
        h = runs_host.numpy()
        h[0] = k
        h[1:1 + k] = a_glob
        h[1 + max_units:1 + max_units + k] = cnt
        runs_send.copy_(runs_host, non_blocking=True)
        dist.all_gather_into_tensor(runs_recv, runs_send)
        allr = runs_recv.cpu().numpy().reshape(world, -1)
        runs = [(allr[r, 1:1 + int(allr[r, 0])], allr[r, 1 + max_units:1 + max_units + int(allr[r, 0])]) for r in range(world)]
        delta = unit_offsets(runs)[rank]
        ctx.renumber_chains_device(n, res_chain_ptr, first_k, delta)
        return 3

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            e0.record()
        st = ctx.filter_device(cfg, d_in, d_res)
        ms, extra = st.ms_device, 0
        if world > 1:
            extra = make_global(chain_t.data_ptr(), int(st.n_chains_kept))
            ctx.pack_status_device(n, status_t.data_ptr(), packed_t.data_ptr())
            dist.all_gather_into_tensor(gathered_t, packed_t)
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)  # the library calls are synchronous: the two events bracket the whole step
        return ms, st, extra + (1 if world > 1 else 0)

    for _ in range(args.warmup):
        step_device()
    barrier()
    dev_ms, sort_ms, sort_passes, launches, filter_ms, pre_ms = 0.0, 0.0, 0, 0, 0.0, 0.0
    with ClockSampler(local_rank) as clk:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ms, st, extra = step_device()
            dev_ms += ms
            filter_ms += st.ms_device
            sort_ms += st.ms_sort_passes
            pre_ms += st.ms_prefilter
            sort_passes += st.n_sort_passes
            launches += st.gpu_launches + extra
        barrier()
        wall_dev = time.perf_counter() - t0
    stats = st
    if world > 1:
        status_dev, chain_dev = status_t.cpu().numpy(), chain_t.cpu().numpy().view(np.uint32)
    else:
        status_dev, chain_dev = ctx.download(n, d_res)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, status_dev, chain_dev, stats, world, rank)

    # ---- end to end: pinned host buffers in, host result out, copies inside the timed region ---------------------------
    with gpu_numa_affinity(local_rank) as numa:
        pt = pinned_copy(table, with_identity=not identity_is_default)
    out_s, out_c = pt._out[0], pt._out[1]

    def step_e2e():
        _, _, st2 = ctx.filter(cfg, pt, out_s, out_c)
        return st2.ms_h2d + st2.ms_device + st2.ms_d2h, st2

    for _ in range(min(args.warmup, 2)):
        step_e2e()
    barrier()
    with ClockSampler(local_rank) as clk2:  # the e2e loop is the longer timed region: more clock samples under load
        e2e_ms, t0 = 0.0, time.perf_counter()
        for _ in range(args.steps):
            ms, st2 = step_e2e()
            e2e_ms += ms
        barrier()
        wall_e2e = time.perf_counter() - t0
    clk.rows += clk2.rows
    h2d, d2h = int(st2.h2d_bytes), int(st2.d2h_bytes)
    # the same calls as a stream of tables (swg_prefetch): the upload of step k + 1 is started before the filter call of step k,
    # so it overlaps that call's kernels and result download; every step still moves its own bytes in both directions
    pipelined = None
    if world == 1:
        try:
            ctx.prefetch(pt)
            step_e2e()            # consumes the prefetched copy (warm-up of the second staging arena)
            ctx.prefetch(pt)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                ctx.prefetch(pt)  # table k + 1
                _, _, st3 = ctx.filter(cfg, pt, out_s, out_c)  # table k: already on the device
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) / args.steps
            ctx.filter(cfg, pt, out_s, out_c)  # the last prefetched table
            assert np.array_equal(out_s, status_dev) and np.array_equal(out_c, chain_dev), "pipelined e2e result differs"
            pipelined = {"wall_ms_per_step": wall * 1e3, "value": n / wall / 1e6, "unit": "Mmappings/s",
                         "h2d_bytes_per_step": int(st3.h2d_bytes), "d2h_bytes_per_step": int(st3.d2h_bytes),
                         "note": "swg_prefetch(table k+1) before swg_filter(table k): a stream of tables; wall clock over the loop"}
        except Exception as e:
            pipelined = {"error": repr(e)[:200]}
            ctx.prefetch_drop()
    # the same call with PAGEABLE buffers (what a Rust Vec or a plain numpy array is): pinned staging inside the library
    pageable_ms = None
    if world == 1:
        import copy
        tp = copy.copy(table)
        if identity_is_default:
            tp.identity = None
        ps, pc = np.zeros(n, np.uint8), np.zeros(n, np.uint32)
        ctx.filter(cfg, tp, ps, pc)
        t0 = time.perf_counter()
        for _ in range(3):
            ctx.filter(cfg, tp, ps, pc)
        pageable_ms = (time.perf_counter() - t0) / 3 * 1e3
        assert np.array_equal(ps, out_s) and np.array_equal(pc, out_c), "pageable-buffer call differs"
    if world == 1:
        assert np.array_equal(out_s, status_dev) and np.array_equal(out_c, chain_dev), "e2e and device-resident results differ"
    else:  # the e2e call returns shard-local chain numbers; the device-resident step has renumbered them
        assert np.array_equal(out_s, status_dev) and np.array_equal(out_c != 0, chain_dev != 0), "e2e and device-resident results differ"

    # ---- parity with the CPU oracle over the whole (per-rank) table ------------------------------------------------------
    parity = None
    cores = os.cpu_count() or 1
    cpu_dt = None
    if not args.no_parity:
        ocfg = oracle_config(n_gpus)
        cpu_dt, (o_status, o_chain) = oracle_mt(ocfg, wtable, max(1, cores // world), want_result=True)
        if world > 1:  # the oracle numbered this shard alone: compare chain membership through the shard-local numbers
            local_chain = out_c
        else:
            local_chain = chain_dev
        parity = {"records": int(n), "status_mismatch": int((o_status != status_dev).sum()),
                  "chain_mismatch": int((o_chain != local_chain).sum()), "oracle_kept": int((o_status != 0).sum())}
        if world > 1:
            # global numbering: every rank's numbers are a set of disjoint runs that tile 1 .. total
            tot_local = torch.tensor([int(stats.n_chains_kept)], dtype=torch.int64, device=dev)
            dist.all_reduce(tot_local)
            mx = torch.tensor([int(chain_dev.max()) if n else 0], dtype=torch.int64, device=dev)
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            distinct = torch.tensor([len(np.unique(chain_dev[chain_dev != 0]))], dtype=torch.int64, device=dev)
            dist.all_reduce(distinct)
            parity["global_chain_numbers"] = {"total_chains": int(tot_local.item()), "max_number": int(mx.item()),
                                              "distinct_over_ranks": int(distinct.item())}
            pm = torch.tensor([parity["status_mismatch"], parity["chain_mismatch"], parity["records"]], dtype=torch.int64, device=dev)
            dist.all_reduce(pm)
            parity["status_mismatch"], parity["chain_mismatch"], parity["records"] = (int(x) for x in pm.tolist())
            ok_global = parity["global_chain_numbers"]["total_chains"] == parity["global_chain_numbers"]["max_number"] == \
                parity["global_chain_numbers"]["distinct_over_ranks"]
        else:
            ok_global = True
        parity["ok"] = parity["status_mismatch"] == 0 and parity["chain_mismatch"] == 0 and ok_global

    t_dev, t_e2e = dev_ms / 1e3, max(e2e_ms / 1e3, 0.0)
    t_filter = filter_ms / 1e3
    if world > 1:
        tt = torch.tensor([t_dev, t_e2e, wall_dev, wall_e2e, t_filter], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_dev, t_e2e, wall_dev, wall_e2e, t_filter = tt.tolist()
        nn = torch.tensor([n], dtype=torch.int64, device=dev)
        sizes_t = [torch.zeros_like(nn) for _ in range(world)]
        dist.all_gather(sizes_t, nn)
        shard_sizes = [int(x.item()) for x in sizes_t]
        n_total = sum(shard_sizes)
    else:
        n_total, shard_sizes = n, [n]

    if rank == 0:
        peak, peak_src = peaks()
        value = n_total * args.steps / t_dev / 1e6
        e2e_v = n_total * args.steps / t_e2e / 1e6
        # the dominant kernel of the step: the LSD passes of the record sort when they ran (huge groups / very many sequences),
        # otherwise k_prefilter (the record sort is a counting sort by group then: csrc/group_sort.cuh)
        traffic, traffic_note = None, None
        if sort_ms > pre_ms:
            pass_ms = sort_ms / max(sort_passes, 1)
            bpp = int(stats.sort_bytes_per_pair) or 24
            units_per_launch = int(stats.n_sort_pairs)
            launches_timed = int(stats.n_sort_passes)
            kernel = ("rs_onesweep_kernel<RS_PACKED> (record sort pass on packed words, 8 B read + 8 B written per record)"
                      if bpp == 16 else "rs_onesweep_kernel (record sort pass, 12 B read + 12 B written per pair)")
            tfile = "onesweep_traffic.json"
        else:
            pass_ms = pre_ms / args.steps
            bpp = int(stats.prefilter_bytes_per_record)
            units_per_launch = int(n)
            launches_timed = 1
            kernel = (f"k_prefilter (stage-1 retain, range checks, genome-pair first appearance, packed coordinates and sort keys: "
                      f"{bpp} B read + written per record)")
            tfile = "prefilter_traffic.json"
        achieved = units_per_launch * bpp / (pass_ms / 1e3) / 1e9 if pass_ms > 0 else 0.0
        tp = os.path.join(ROOT, "profiles", tfile)
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if int(tj.get("pairs_per_launch", 0)) == units_per_launch and int(tj.get("bytes_per_pair", 24)) == bpp:
                    traffic = tj.get("dram_bytes_per_launch")
                    traffic_note = tj.get("source")
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": "Mmappings/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev * 1e3 / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32/u64/f64", "data": "synthetic",
            "config": {"workload": desc["name"], "records_per_gpu": int(n), "flags": desc["flags"]},
            "detail": {"l2": "inputs (41 B/record) are larger than the 126 MB L2",
                       "timing": ("N = 1: sum of per-step CUDA-event times on the library stream; N > 1: CUDA events around the whole step "
                                  "(filter + unit exchange + renumber + 2-bit status gather), max over ranks"),
                       "wall_ms_per_step": wall_dev * 1e3 / args.steps,
                       "filter_only_ms_per_step": t_filter * 1e3 / args.steps,
                       "shard_records": {"max": max(shard_sizes), "mean": n_total / len(shard_sizes), "min": min(shard_sizes)},
                       "pipeline_algorithmic_bytes_per_mapping": desc["b_alg"],
                       "pipeline_fraction_of_hbm_roofline": (n * desc["b_alg"] / (t_filter / args.steps)) / 1e9 / peak,
                       "log_matches_host": ctx.log_matches_host(),
                       "stats": {k: int(getattr(stats, k)) for k in ("n_stage1", "n_after_sweep", "n_chains", "n_chains_after_mass",
                                                                     "n_chains_kept", "n_anchors", "n_rescued", "n_kept", "exact_rerank", "n_dirty_groups", "n_unsorted_groups")}},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_v, "unit": "Mmappings/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": t_e2e * 1e3 / args.steps, "wall_ms_per_step": wall_e2e * 1e3 / args.steps,
                    "identity_column_uploaded": not identity_is_default, "ids_16bit": bool(table.n_seq <= 65536),
                    "pageable_buffers_wall_ms_per_step": pageable_ms,
                    "h2d_gbs_per_rank": h2d / max(st2.ms_h2d, 1e-9) / 1e6, "stream_of_tables": pipelined,
                    "pinned_buffers_numa": numa.note},
            "gpu_launches": int(launches),
            "roofline": {"kernel": kernel, "bound": "hbm", "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_note,
                         "launch_ms": pass_ms, "records_per_launch": units_per_launch, "bytes_per_record": bpp,
                         "launches_timed_per_step": launches_timed},
            "parity": parity,
        }
        if n_gpus == 1:
            line["modes"] = modes_leg(ctx, d_in, d_res, n)
            line["small"] = small_leg(ctx)
        if n_gpus == 1 and args.paf_lines > 0:
            line["paf_e2e"] = paf_file_leg(ctx, cfg, args.paf_lines)
        if n_gpus == 1 and args.skew_pile > 0:
            line["skew"] = skew_leg(ctx, cfg, args.skew_pile)
        if n_gpus == 1 and not args.no_anchor:
            line["scale_anchor"] = scale_anchor(ctx, args)
        if n_gpus == 1:
            if cpu_dt is None:
                sample = wtable.take(np.arange(min(n, args.cpu_sample)))
                cpu_dt, _ = oracle_mt(oracle_config(1), sample, cores)
                cpu_n = sample.n
            else:
                cpu_n = n
            line["cpu_baseline"] = {"value": cpu_n / cpu_dt / 1e6, "unit": "Mmappings/s", "cores": cores, "kind": "port",
                                    "sample": f"the whole workload ({cpu_n} records, whole genome pairs per thread), filter only, {cpu_dt:.1f} s"}
        print(json.dumps(line))
    if world == 1:
        ctx.release(d_in, d_res)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        sys.exit("parity with the CPU oracle FAILED: " + json.dumps(parity))


def scale_anchor(ctx, args):
    """N = 1 only: the per-GPU workload of the N > 1 runs (shard 0 of the 8-GPU partition of configs[3], --scaffold-dist 100k)
    on this one GPU, so that scaling efficiency can be read like for like (same records per GPU, same pipeline)."""
    try:
        import sweepga_b200 as swg
        wt, desc = workload(8, 0, args.records)
        t = swg.MappingTable(wt.query_id, wt.target_id, wt.query_start, wt.query_end, wt.target_start, wt.target_end, wt.block_length,
                             wt.matches, wt.identity, wt.strand, wt.seq_genome_id, wt.seq_genome2_id)
        cfg = swg.FilterConfig.from_cli(scaffold_dist="100k")
        d_in, d_res = ctx.upload(t)
        for _ in range(2):
            ctx.filter_device(cfg, d_in, d_res)
        sts = [ctx.filter_device(cfg, d_in, d_res) for _ in range(5)]
        ms = [s.ms_device for s in sts]
        ctx.release(d_in, d_res)
        return {"workload": "shard 0 of the 8-GPU partition of configs[3] on one GPU (filter only, no exchange)", "records": int(t.n),
                "ms_per_step": sum(ms) / len(ms), "Mmappings_per_s": t.n / (sum(ms) / len(ms)) / 1e3,
                "lsd_sort_passes": int(sts[-1].n_sort_passes), "groups_ordered_after_scatter": int(sts[-1].n_unsorted_groups),
                "gpu_launches": int(sts[-1].gpu_launches)}
    except Exception as e:
        return {"error": repr(e)[:200]}


if __name__ == "__main__":
    main()
