#!/usr/bin/env python
"""The three device PAF readers (swg_filter_paf, swg_ani_stats, swg_tree_filter_paf) on one synthetic PAF, for one or
more builds of the package, alternating, each run in a fresh process.  Prints one JSON line per run: sha256 of the
filter and tree outputs, the ANI results as f64 bit patterns, ms_tokenize / gpu_launches of the filter, and the wall
time of every call (after one warm-up call each).

The input has cg:Z: and dv:f: tags, '#' lines, lines with fewer than 11 fields, CRLF lines and 20-digit integer
fields (which go through the host patch step), so every path of the readers runs.

Usage: python profiles/bench_paf_readers.py [--n LINES] [--runs R] ROOT [ROOT ...]
  ROOT: a repository tree whose sweepga_b200 package is built."""
import argparse, hashlib, json, os, struct, subprocess, sys, tempfile, time
import numpy as np


def write_paf(path, n, seed=11):
    rng = np.random.default_rng(seed)
    names = np.array([f"HG{h:03d}#{p}#chr{c}" for h in range(40) for p in (1, 2) for c in range(1, 6)])
    m = min(n, 1 << 20)  # one block of distinct lines, repeated: formatting 20 M lines in numpy would take minutes
    q, t = rng.integers(0, len(names), m), rng.integers(0, len(names), m)
    qlen, tlen = rng.integers(1_000_000, 50_000_000, m), rng.integers(1_000_000, 50_000_000, m)
    qs, ts = rng.integers(0, 900_000, m), rng.integers(0, 900_000, m)
    span = rng.integers(1_000, 60_000, m)
    mt = (span * rng.uniform(0.85, 1.0, m)).astype(np.int64)
    qlen_s = qlen.astype(str)
    qlen_s[rng.random(m) < 0.002] = "00000000000012345678"  # 20 digits: the host patch step decides
    cols = [names[q], qlen_s, qs.astype(str), (qs + span).astype(str), np.where(rng.random(m) < 0.5, "+", "-"),
            names[t], tlen.astype(str), ts.astype(str), (ts + span).astype(str), mt.astype(str), span.astype(str),
            np.full(m, "60")]
    line = cols[0]
    for col in cols[1:]:
        line = np.char.add(np.char.add(line, "\t"), col)
    cg = np.char.add(np.char.add("\tcg:Z:", mt.astype(str)), np.char.add("=", np.char.add((span - mt).astype(str), "X")))
    dv = np.char.add("\tdv:f:", np.char.mod("%.4f", rng.uniform(0.0, 0.15, m)))
    r = rng.random(m)
    line = np.where(r < 0.6, np.char.add(line, cg), line)
    line = np.where((r > 0.3) & (r < 0.9), np.char.add(line, dv), line)
    line = np.where(rng.random(m) < 0.001, "#comment line", line)
    line = np.where(rng.random(m) < 0.001, "short\tline", line)
    line = np.where(rng.random(m) < 0.01, np.char.add(line, "\r"), line)
    block = "\n".join(line.tolist()) + "\n"
    with open(path, "w") as f:
        for c0 in range(0, n, m):
            f.write(block if c0 + m <= n else "".join(block.splitlines(True)[: n - c0]))


WORKER = r'''
import hashlib, json, os, struct, sys, time
root, src, d = sys.argv[1:4]
sys.path.insert(0, root)
import sweepga_b200 as swg
def sha(p): return hashlib.sha256(open(p, "rb").read()).hexdigest()
ctx = swg.Context(0)
f = swg.PafFilter(swg.FilterConfig()); f._ctx = ctx
res = {"root": root}
out = os.path.join(d, "filter.paf")
f.filter_paf(src, out); os.unlink(out)
t0 = time.time(); st = f.filter_paf(src, out); res["filter_s"] = time.time() - t0
res["filter_sha"] = sha(out); res["ms_tokenize"] = st.ms_tokenize; res["gpu_launches"] = st.gpu_launches; os.unlink(out)
for m in ("all", "n50"):
    swg.ani_stats(ctx, src, m)
    t0 = time.time(); a = swg.ani_stats(ctx, src, m); res[f"ani_{m}_s"] = time.time() - t0
    res[f"ani_{m}"] = [struct.pack("<d", a[0]).hex(), a[1]]
out = os.path.join(d, "tree.paf")
swg.apply_tree_filter_to_paf(ctx, src, out, 2, 1, 0.05); os.unlink(out)
t0 = time.time(); k = swg.apply_tree_filter_to_paf(ctx, src, out, 2, 1, 0.05); res["tree_s"] = time.time() - t0
res["tree_sha"] = sha(out); res["tree_kept"] = list(k); os.unlink(out)
print(json.dumps(res))
'''


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=20_000_000)
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("roots", nargs="+")
    a = ap.parse_args()
    d = tempfile.mkdtemp()
    src = os.path.join(d, "in.paf")
    t0 = time.time()
    write_paf(src, a.n)
    print(json.dumps({"input_lines": a.n, "input_bytes": os.path.getsize(src), "write_s": round(time.time() - t0, 1)}), flush=True)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        print(json.dumps({"gpu": q.stdout.strip()}), flush=True)
    except OSError:
        pass
    for _ in range(a.runs):
        for root in a.roots:
            r = subprocess.run([sys.executable, "-c", WORKER, os.path.abspath(root), src, d], capture_output=True, text=True)
            res = {**json.loads(r.stdout), "root": root} if r.returncode == 0 else {"root": root, "error": r.stderr[-2000:]}
            print(json.dumps(res), flush=True)
    os.unlink(src)


if __name__ == "__main__":
    main()
