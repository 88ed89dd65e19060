#!/usr/bin/env python
"""Time the chain-level stage and the anchor tail of the flagship step (configs[2]: 20 M synthetic PanSN mappings, defaults).

  python profiles/chain_tail_stages.py [--records N] [--steps K] [--launches OUT.txt]

Stage times come from the stage-timing knob (SWG_STAGE_TIMING: CUDA events at the stage boundaries of every call, printed to
stderr as "[swg stages] name ms ..."); the script runs itself as a child to collect them and prints the median of each stage over
K warmed steps.  The stages of interest: chain_table (chain rows, pass flags, order-key compaction, first sort), chain_order
(t-space, final order, chain numbers), assign+inversion+rescue and stats (the closing counter read).  With --launches, one further
step runs under torch.profiler (CUDA activity) and its kernel list, in launch order with device times, is written to OUT.txt.
"""
import argparse
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(args):
    sys.path.insert(0, ROOT)
    import sweepga_b200 as swg
    from sweepga_b200 import synth
    t = synth.pansn(args.records, seed=3)
    cfg = swg.FilterConfig()
    with swg.Context(0) as ctx:
        d_in, d_res = ctx.upload(t)
        for _ in range(3):
            ctx.filter_device(cfg, d_in, d_res)
        print("[steps begin]", file=sys.stderr, flush=True)
        for _ in range(args.steps):
            st = ctx.filter_device(cfg, d_in, d_res)
        print(f"[launches] {st.gpu_launches}", file=sys.stderr, flush=True)
        if args.launches:
            os.environ.pop("SWG_STAGE_TIMING", None)
            import torch
            from torch.profiler import ProfilerActivity, profile
            torch.cuda.init()
            ctx.filter_device(cfg, d_in, d_res)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                ctx.filter_device(cfg, d_in, d_res)
                torch.cuda.synchronize()
            ev = sorted((e for e in prof.events() if e.device_type.name == "CUDA" and "Memcpy" not in e.name and "Memset" not in e.name),
                        key=lambda e: e.time_range.start)
            with open(args.launches, "w") as f:
                tot = 0.0
                for e in ev:
                    us = e.time_range.end - e.time_range.start
                    tot += us
                    f.write(f"{us:9.1f} {re.sub(r'[(].*', '', e.name.replace('void ', ''))[:70]}\n")
                f.write(f"total us {tot:.1f} launches {len(ev)}\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=20_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--launches", default="")
    ap.add_argument("--child", action="store_true")
    args = ap.parse_args()
    if args.child:
        return child(args)
    env = dict(os.environ, SWG_STAGE_TIMING="1")
    r = subprocess.run([sys.executable, __file__, "--child"] + sys.argv[1:], env=env, stderr=subprocess.PIPE, text=True)
    if r.returncode:
        sys.exit(r.stderr[-4000:])
    lines = r.stderr.splitlines()
    lines = lines[lines.index("[steps begin]") + 1:]
    per = {}
    for ln in lines:
        if ln.startswith("[swg stages]"):
            tok = ln.split()[2:]
            for name, ms in zip(tok[0::2], tok[1::2]):
                per.setdefault(name, []).append(float(ms))
        elif ln.startswith("[launches]"):
            print(ln)
    for name, v in per.items():
        print(f"{name:28s} median {statistics.median(v) * 1e3:9.1f} us   min {min(v) * 1e3:9.1f}   max {max(v) * 1e3:9.1f}   ({len(v)} steps)")


if __name__ == "__main__":
    main()
