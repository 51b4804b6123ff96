"""Differential fuzzing of the classification itself, on the CPU: random read sets built from genome fragments
(chimeras, reverse complements, substitutions, low-complexity repeats, truncated and random reads, pairs) under
random option sets.
  * the oracle's file driver against the unmodified reference binary: classification TSV and report, byte for byte;
  * the product's per-thread logic (cf_logic.h compiled for the host, the code the CUDA kernels run) against the
    oracle, record by record."""
import random

import numpy as np

import util
from util_fuzz import clean_reads

COMP = bytes.maketrans(b"ACGTN", b"TGCAN")


def make_reads(rng, reads):
    out = []
    for i in range(rng.randrange(5, 40)):
        r, a = rng.random(), rng.choice(reads)[1]
        if r < 0.2:
            b = rng.choice(reads)[1]
            s = a[:rng.randrange(20, len(a))] + b[rng.randrange(0, len(b) - 20):]
        elif r < 0.35:
            s = a[::-1].translate(COMP)
        elif r < 0.5:
            s = bytearray(a)
            for _ in range(rng.randrange(1, 6)):
                s[rng.randrange(len(s))] = rng.choice(b"ACGTN")
            s = bytes(s)
        elif r < 0.6:
            s = (rng.choice([b"A", b"AC", b"ACG", b"T"]) * 80)[:rng.randrange(30, 120)]
        elif r < 0.7:
            s = a[:rng.randrange(1, 40)]
        elif r < 0.8:
            s = bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(20, 150)))
        else:
            s = a
        out.append((b"q%d" % i, s))
    return out


CLI_OPTS = [[], ["-k", "1"], ["-k", "3"], ["-k", "50"], ["--min-hitlen", "15"], ["--min-hitlen", "30"], ["--host-taxids", "100,1005"], ["--exclude-taxids", "10"],
            ["--exclude-taxids", "1003,101"], ["--classification-rank", "genus"], ["--classification-rank", "family"], ["--classification-rank", "species"],
            ["--no-traverse"], ["--no-traverse", "-k", "1"], ["-k", "2", "--host-taxids", "11"], ["--min-hitlen", "16", "-k", "1", "--classification-rank", "genus"]]
API_OPTS = [dict(), dict(k=1), dict(k=3), dict(k=50), dict(min_hitlen=15), dict(min_hitlen=30), dict(host=(100, 1005)), dict(excl=(10,)), dict(excl=(1003, 101)),
            dict(rank_slot=2), dict(rank_slot=3), dict(rank_slot=1), dict(traverse=False), dict(traverse=False, k=1), dict(k=2, host=(11,)),
            dict(min_hitlen=16, k=1, rank_slot=2)]


def test_oracle_matches_reference_on_random_reads_and_options(tmp_path):
    util.ensure_oracle()
    base = util.golden_index("adv")
    reads = clean_reads()
    fa = lambda rs: b"".join(b">" + n + b"\n" + s + b"\n" for n, s in rs)
    for case in range(80):
        rng = random.Random(90000 + case)
        rs, opts, paired = make_reads(rng, reads), rng.choice(CLI_OPTS), rng.random() < 0.3
        p1, p2 = str(tmp_path / "a.fa"), str(tmp_path / "b.fa")
        args = ["-f", "-x", base] + opts
        if paired:
            rs2 = make_reads(rng, reads)[:len(rs)]; rs = rs[:len(rs2)]
            with open(p2, "wb") as f:
                f.write(fa(rs2))
            args += ["-1", p1, "-2", p2]
        else:
            args += ["-U", p1]
        with open(p1, "wb") as f:
            f.write(fa(rs))
        a = util.reference_cli(args, tmp_path)
        b = util.run_cli(util.ORACLE_BIN, args, str(tmp_path / "o.tsv"), str(tmp_path / "o.rep"))
        assert a == util.digests(b), (case, opts, paired)


def test_product_logic_matches_oracle_on_random_reads_and_options():
    util.ensure_oracle()
    base = util.golden_index("adv")
    reads = clean_reads()
    o, h = util.Oracle(base), util.HostLogic(base)
    arr = lambda s: np.frombuffer(s, dtype=np.uint8)
    for case in range(400):
        rng = random.Random(70000 + case)
        rs, kw, paired = make_reads(rng, reads), rng.choice(API_OPTS), rng.random() < 0.4
        if paired:
            rs2 = make_reads(rng, reads)[:len(rs)]; rs = rs[:len(rs2)]
            bt = util.Batch([arr(s) for _, s in rs], [arr(s) for _, s in rs2])
        else:
            bt = util.Batch([arr(s) for _, s in rs])
        p = util.make_oparams(**kw)
        on, orec, _ = o.classify(bt, p)
        hn, hrec, _ = h.classify(bt, p)
        assert np.array_equal(on, hn) and np.array_equal(orec, hrec), (case, kw, paired)
    o.close(); h.close()
