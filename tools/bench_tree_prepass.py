"""Time swg_tree_filter_paf (`--sparsify tree:k`) on a two-genome PAF of about 20 M lines, for one or more builds of the
library side by side.

The input is one seeded block of --block distinct lines (genomes A and B, several sequences each, integer matches and
block lengths, some dv:f: tags) written --repeat times into a temporary file.  Every library in --libs runs in a process of
its own (each carries its own static CUDA runtime): a warm-up call, then --reps timed calls, host wall time around calls that
return after the output is written.  The processes alternate, lib by lib, --rounds times; the best time of each library is
reported.  The outputs of all libraries must hash alike.  Prints one JSON line with the times and the card's name and power
limit.  The pair's totals stay near 2 * 10^11, so this times the exact integer sums; --past-2p53 puts a first line with a
block length of 2^53 in front, which sends the call to the sequential f64 sums (one thread walks all the pair's records).

    python tools/bench_tree_prepass.py [--libs sweepga_b200/libsweepga_b200.so,other.so] [--rounds 2] [--reps 3] [--past-2p53]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import random
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_batch import gpu_info  # noqa: E402


def write_input(path, block, repeat, past_2p53=False, seed=1):
    rng = random.Random(seed)
    lines = []
    for i in range(block):
        bl = rng.randrange(100, 20000)
        q, t = ("A", "B") if i % 2 else ("B", "A")
        tag = "\tdv:f:%.4f" % (rng.random() * 0.2) if i % 3 == 0 else ""
        lines.append("%s#1#chr%d\t5000000\t%d\t%d\t+\t%s#1#chr%d\t5000000\t%d\t%d\t%d\t%d\t60%s\n"
                     % (q, i % 16, i, i + bl, t, i % 11, i, i + bl, bl - rng.randrange(0, bl // 4 + 1), bl, tag))
    chunk = "".join(lines).encode()
    with open(path, "wb") as f:
        if past_2p53:
            f.write(b"A#1#chr0\t5000000\t0\t1\t+\tB#1#chr0\t5000000\t0\t1\t%d\t%d\t60\n" % (1 << 52, 1 << 53))
        for _ in range(repeat):
            f.write(chunk)
    return block * repeat + past_2p53


def one(lib_path, src, out, reps):
    """Timed calls of one library in this process -> {"times_s": [...], "kept":, "selected":, "sha256":}"""
    lib = C.CDLL(lib_path)
    lib.swg_create.restype = C.c_void_p
    lib.swg_create.argtypes = [C.c_int]
    lib.swg_destroy.argtypes = [C.c_void_p]
    lib.swg_last_error.restype = C.c_char_p
    lib.swg_last_error.argtypes = [C.c_void_p]
    lib.swg_tree_filter_paf.restype = C.c_int
    lib.swg_tree_filter_paf.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_double,
                                        C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    ctx = lib.swg_create(0)
    if not ctx:
        raise RuntimeError(lib.swg_last_error(None).decode())
    try:
        kept, sel = C.c_uint64(), C.c_uint64()
        times = []
        for r in range(reps + 1):  # the first call warms the page cache, the arenas and the modules
            t0 = time.perf_counter()
            rc = lib.swg_tree_filter_paf(ctx, src.encode(), out.encode(), 1, 0, 0.0, C.byref(kept), C.byref(sel))
            dt = time.perf_counter() - t0
            if rc != 0:
                raise RuntimeError(lib.swg_last_error(ctx).decode())
            if r:
                times.append(dt)
        with open(out, "rb") as f:
            digest = hashlib.sha256(f.read()).hexdigest()
        return {"times_s": times, "kept": kept.value, "selected": sel.value, "sha256": digest}
    finally:
        lib.swg_destroy(ctx)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", default=os.path.join(ROOT, "sweepga_b200", "libsweepga_b200.so"))
    ap.add_argument("--block", type=int, default=1_000_000)
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--past-2p53", action="store_true")
    ap.add_argument("--one", nargs=3, metavar=("LIB", "INPUT", "OUTPUT"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.one:
        print(json.dumps(one(*args.one, args.reps)))
        return
    libs = [os.path.abspath(p) for p in args.libs.split(",")]
    d = tempfile.mkdtemp(prefix="swg_tree_bench_")
    try:
        src = os.path.join(d, "in.paf")
        n = write_input(src, args.block, args.repeat, args.past_2p53)
        res = {lib: [] for lib in libs}
        for _ in range(args.rounds):
            for k, lib in enumerate(libs):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--reps", str(args.reps), "--one", lib, src,
                                    os.path.join(d, f"out{k}.paf")], capture_output=True, text=True)
                if p.returncode != 0:
                    raise RuntimeError(p.stderr)
                res[lib].append(json.loads(p.stdout.strip().splitlines()[-1]))
        digests = {r["sha256"] for rs in res.values() for r in rs}
        print(json.dumps({"workload": f"two genomes, {n} lines ({os.path.getsize(src)} bytes), tree:1"
                          + (", a pair total past 2^53 (sequential f64 sums)" if args.past_2p53 else ", pair totals below 2^53 (exact integer sums)"), **gpu_info(),
                          "same_output": len(digests) == 1,
                          "libs": {os.path.relpath(lib, ROOT): {"best_s": min(t for r in rs for t in r["times_s"]),
                                                               "times_s": [t for r in rs for t in r["times_s"]],
                                                               "kept": rs[0]["kept"], "selected": rs[0]["selected"]}
                                   for lib, rs in res.items()}}))
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
