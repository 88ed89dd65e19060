"""Many small PAF files: a loop of swg_filter_paf against one swg_filter_paf_batch.

For each K in --files (default 10, 100, 1000) the first K of the seeded files yeast_like(26000, seed=k) (dv:f: and cg:Z: tags,
written once into a temporary directory) are filtered file to file both ways after a warm-up, alternating, best of --reps;
both timings are host wall time around calls that return after their output is written.  Every output of the batch must hash
like the loop's.  Prints one JSON line with both times, the batch's phase times and launches, and the card's name and power
limit.

    python tools/bench_paf_batch.py [--files 10,100,1000] [--reps 3]
"""
import argparse
import hashlib
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_batch import gpu_info  # noqa: E402


def digest(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", default="10,100,1000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--records", type=int, default=26000)
    args = ap.parse_args()
    import sweepga_b200 as swg
    from sweepga_b200 import synth

    ks = [int(x) for x in args.files.split(",")]
    names = [f"{g}#{c}" for g in synth.YEAST_GENOMES for c in synth.YEAST_CHROMS]
    d = tempfile.mkdtemp(prefix="swg_paf_batch_")
    try:
        ins = []
        for k in range(max(ks)):
            t = synth.yeast_like(args.records, seed=k)
            t.names = names
            p = os.path.join(d, f"in{k}.paf")
            synth.write_paf(t, p)
            ins.append(p)
        cfg = swg.FilterConfig()
        out = {"workload": f"yeast_like({args.records}, seed=k) as PAF with dv:f: and cg:Z: tags, k < K", "config": "defaults",
               "reps": args.reps, **gpu_info(), "runs": []}
        f = swg.PafFilter(cfg)
        with swg.Context(0) as ctx:
            f._ctx = ctx
            f.filter_paf(ins[0], os.path.join(d, "warm.out"))  # warm-up of both paths: page cache, arenas, pinned pieces
            ctx.filter_paf_batch(cfg, ins[:2], [os.path.join(d, "warm0.out"), os.path.join(d, "warm1.out")])
            for K in ks:
                loop_outs = [os.path.join(d, f"loop{k}.out") for k in range(K)]
                batch_outs = [os.path.join(d, f"batch{k}.out") for k in range(K)]
                loop_ms, batch_ms, bst = [], [], None
                for _ in range(args.reps):
                    for o in loop_outs + batch_outs:  # fresh output files for both
                        if os.path.exists(o):
                            os.unlink(o)
                    t0 = time.perf_counter()
                    for src, o in zip(ins[:K], loop_outs):
                        f.filter_paf(src, o)
                    loop_ms.append((time.perf_counter() - t0) * 1e3)
                    t0 = time.perf_counter()
                    counts, st = ctx.filter_paf_batch(cfg, ins[:K], batch_outs)
                    batch_ms.append((time.perf_counter() - t0) * 1e3)
                    if bst is None or batch_ms[-1] == min(batch_ms):
                        bst = st
                same = all(digest(a) == digest(b) for a, b in zip(loop_outs, batch_outs))
                out["runs"].append({
                    "K": K, "input_bytes": int(sum(os.path.getsize(p) for p in ins[:K])), "kept": int(counts[:, swg.TC_KEPT].sum()),
                    "loop_ms": round(min(loop_ms), 3), "batch_ms": round(min(batch_ms), 3),
                    "speedup": round(min(loop_ms) / min(batch_ms), 2), "identical": bool(same),
                    "batch_ms_h2d": round(bst.ms_h2d, 3), "batch_ms_tokenize": round(bst.ms_tokenize, 3),
                    "batch_ms_device": round(bst.ms_device, 3), "batch_ms_write": round(bst.ms_write, 3),
                    "gpu_launches": int(bst.gpu_launches),
                })
                if not same:
                    print(json.dumps(out))
                    sys.exit("batch and loop outputs differ")
        print(json.dumps(out))
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
