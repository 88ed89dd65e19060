"""Many small tables: a loop of Context.filter against one Context.filter_batch (swg_filter_batch).

For each K in --tables (default 10, 100, 1000) the first K of the seeded tables yeast_like(26000, seed=k) (~23 k records,
136 sequences each, pageable numpy arrays) are filtered both ways after a warm-up; both timings are host wall time around calls
that end in a stream synchronise.  The two sets of outputs must be identical.  Prints one JSON line with both times, the
batch's phase times and counts, and the card's name and power limit.

    python tools/bench_batch.py [--tables 10,100,1000] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    """Name and power limit of the card (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "nvidia_smi": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tables", default="10,100,1000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--records", type=int, default=26000)
    args = ap.parse_args()
    import sweepga_b200 as swg
    from sweepga_b200 import synth

    ks = [int(x) for x in args.tables.split(",")]
    tables = [synth.yeast_like(args.records, seed=k) for k in range(max(ks))]
    cfg = swg.FilterConfig()
    out = {"workload": f"yeast_like({args.records}, seed=k), k < K", "config": "defaults", "reps": args.reps, **gpu_info(), "runs": []}
    with swg.Context(0) as ctx:
        ctx.filter(cfg, tables[0])  # warm-up of both paths
        ctx.filter_batch(cfg, tables[:2])
        for K in ks:
            tk = tables[:K]
            loop_ms, batch_ms = [], []
            for _ in range(args.reps):  # alternating, best of reps
                t0 = time.perf_counter()
                single = [ctx.filter(cfg, t)[:2] for t in tk]
                loop_ms.append((time.perf_counter() - t0) * 1e3)
                t0 = time.perf_counter()
                res, counts, st = ctx.filter_batch(cfg, tk)
                batch_ms.append((time.perf_counter() - t0) * 1e3)
            same = all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(single, res))
            out["runs"].append({
                "K": K, "records": int(sum(t.n for t in tk)), "sequences": int(sum(t.n_seq for t in tk)),
                "loop_ms": round(min(loop_ms), 3), "batch_ms": round(min(batch_ms), 3),
                "speedup": round(min(loop_ms) / min(batch_ms), 2), "identical": bool(same),
                "batch_ms_h2d": round(st.ms_h2d, 3), "batch_ms_device": round(st.ms_device, 3), "batch_ms_d2h": round(st.ms_d2h, 3),
                "gpu_launches": int(st.gpu_launches), "n_sort_passes": int(st.n_sort_passes),
                "sort_bytes_per_pair": int(st.sort_bytes_per_pair), "exact_rerank": int(st.exact_rerank),
                "chains_kept": int(counts[:, swg.TC_CHAINS_KEPT].sum()),
            })
            if not same:
                print(json.dumps(out))
                sys.exit("batch and loop outputs differ")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
