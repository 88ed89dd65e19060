"""ANI pre-pass on the device (swg_ani_stats) against the oracle's restatement of calculate_ani_stats /
calculate_ani_n_percentile (src/main.rs:334-688): the same f64, bit for bit, for the "all", "orthogonal" and
"nX[-length|-identity|-score]" methods ("nX-score" takes ln from the glibc port, the host libm's bits)."""
import random

import numpy as np
import pytest

import oracle_lib
import sweepga_b200 as swg
from sweepga_b200 import synth

from test_host import ANI_PAF

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    with swg.Context(0) as c:
        yield c


def both(ctx, path, method):
    m = swg.parse_ani_method(method)
    return swg.ani_stats(ctx, str(path), method), oracle_lib.ani_stats(str(path), m[0], m[1], m[2])


def test_known_answers(ctx, tmp_path):
    p = tmp_path / "ani.paf"
    p.write_text(ANI_PAF)
    ab, ac = (90.0 + 150.0) / (100.0 + 200.0), ((1.0 - 0.1) * 100.0) / 100.0
    assert swg.ani_stats(ctx, str(p), "all") == ((ab + ac) / 2.0, 2)
    assert swg.ani_stats(ctx, str(p), "n100") == ((ab + ac) / 2.0, 2)
    assert swg.ani_stats(ctx, str(p), "n1") == (0.9, 1)
    assert swg.ani_stats(ctx, str(p), "n1-length") == (0.75, 1)
    assert swg.ani_stats(ctx, str(p), "n3") == ((0.9 + ac) / 2.0, 2)
    (tmp_path / "none.paf").write_text("A#1#x\t1\t0\t1\t+\tA#1#y\t1\t0\t1\t1\t1\t60\n")
    assert swg.ani_stats(ctx, str(tmp_path / "none.paf"), "all") == (0.0, 0)
    (tmp_path / "empty.paf").write_text("")
    assert swg.ani_stats(ctx, str(tmp_path / "empty.paf"), "n50") == (0.0, 0)


def pansn_paf(path, n, seed, dv_every=3, quirks=True):
    """PanSN synthetic alignments with non-integer addends (dv:f: tags) on most lines."""
    t = synth.pansn(n, seed=seed, n_hap=8, with_names=True)
    rng = random.Random(seed)
    with open(path, "w") as f:
        for i in range(t.n):
            q, tt = t.names[t.query_id[i]], t.names[t.target_id[i]]
            line = [q, str(int(t.query_end[i]) + 1000 + (t.query_id[i] % 7) * 1000), str(t.query_start[i]), str(t.query_end[i]),
                    chr(t.strand[i]), tt, str(int(t.target_end[i]) + 5000), str(t.target_start[i]), str(t.target_end[i]),
                    str(t.matches[i]), str(t.block_length[i]), "60"]
            if i % dv_every:
                line += ["tp:A:P", "dv:f:%.*f" % (rng.randrange(2, 9), rng.random() * 0.2)]
            if quirks and i % 97 == 0:
                line += [rng.choice(["dv:f:1e-3", "dv:f:bad\tdv:f:0.05", "dv:f:0.1234567890123456789012", "cg:Z:5=", "dv:f:.5\tdv:f:0.1"])]
            if quirks and i % 211 == 0:
                line[9] = rng.choice(["1e3", "12.5", "x", "+40", "000000000000000000000000077"])
            f.write("\t".join(line) + ("\r\n" if quirks and i % 501 == 0 else "\n"))
            if quirks and i % 1000 == 0:
                f.write(rng.choice(["# header\n", "\n", "too\tshort\n"]))
    return t


@pytest.mark.parametrize("method", ["all", "n100", "n50", "n90-length", "n10-identity", "n0.5-length", "n100-length"])
def test_bit_exact_against_oracle(ctx, tmp_path, method):
    p = tmp_path / "a.paf"
    pansn_paf(str(p), 60000, seed=3)
    got, want = both(ctx, p, method)
    assert want[1] > 10
    assert got == want, method          # the same f64, the same number of genome pairs


def test_score_sort_close(ctx, tmp_path):
    p = tmp_path / "a.paf"
    pansn_paf(str(p), 60000, seed=4)
    assert ctx.log_matches_host()
    for method in ("n50-score", "n100-score"):
        got, want = both(ctx, p, method)
        assert got == want, method


def test_integer_addends_and_two_genomes(ctx, tmp_path):
    """No dv tags: every addend is an integer.  Two genomes only: ONE pair holds every alignment (the longest sequential sum)."""
    p = tmp_path / "i.paf"
    pansn_paf(str(p), 30000, seed=5, dv_every=1, quirks=False)
    for method in ("all", "n50", "n80-length"):
        got, want = both(ctx, p, method)
        assert got == want, method
    rng = random.Random(9)
    with open(tmp_path / "two.paf", "w") as f:
        for i in range(50000):
            b = rng.randrange(100, 20000)
            f.write("g1#1#c%d\t1000000\t%d\t%d\t+\tg2#1#c%d\t2000000\t%d\t%d\t%d\t%d\t60\tdv:f:%.6f\n"
                    % (i % 5, i, i + b, i % 3, i, i + b, b - rng.randrange(0, b // 3 + 1), b, rng.random() * 0.3))
    for method in ("all", "n50", "n100-length"):
        got, want = both(ctx, tmp_path / "two.paf", method)
        assert want[1] == 1
        assert got == want, method


def test_orthogonal(ctx, tmp_path):
    t = synth.yeast_like(20000, seed=6)
    p = tmp_path / "y.paf"
    synth.write_paf(t, str(p))
    got, want = both(ctx, p, "orthogonal")
    assert want[1] > 0
    assert got == want
    got, want = both(ctx, p, "1:1")
    assert got == want


def test_nan_and_errors(ctx, tmp_path):
    p = tmp_path / "nan.paf"
    p.write_text("A#1#c\t10\t0\t5\t+\tB#1#c\t10\t0\t5\t5\t10\t60\tdv:f:nan\nA#1#c\t10\t0\t5\t+\tB#1#c\t10\t0\t5\t5\t10\t60\n")
    with pytest.raises(ValueError):
        oracle_lib.ani_stats(str(p), 2, 50.0, 1)
    with pytest.raises(swg.SwgError):
        swg.ani_stats(ctx, str(p), "n50")
    with pytest.raises(swg.SwgError):
        swg.ani_stats(ctx, str(tmp_path / "missing.paf"), "all")
    # the identity threshold the CLI derives from it (src/main.rs:3590)
    q = tmp_path / "ani.paf"
    q.write_text(ANI_PAF)
    ani, _ = swg.ani_stats(ctx, str(q), "all")
    assert swg.parse_identity_value("ani50-5", ani) == max(ani - 0.05, 0.0)
