"""`centrifuge-promote` equivalent (SURVEY.md 8f rank 4): cfb_promote / `centrifuge-class --promote` against the
reference's own Perl script -- committed goldens (tests/golden/make_promote_golden.py) and differential fuzzing
against recorded runs of the script (tests/golden/reference_runs.json)."""
import ctypes as C
import lzma
import os
import subprocess

import pytest

import util

LEVELS = ["genus", "species", "family", "lca", "phylum"]
CASES = [("default", lv) for lv in LEVELS] + [(c, lv) for c in ("k50", "host", "family") for lv in ("genus", "lca")]


def lib():
    return C.CDLL(util.PRODUCT_LIB)


@pytest.mark.parametrize("case,level", CASES)
def test_promote_matches_reference_script_on_golden_classifications(case, level, tmp_path):
    base = util.golden_index("adv")
    tsv, out = str(tmp_path / "in.tsv"), str(tmp_path / "out.tsv")
    with lzma.open(os.path.join(util.GOLDEN, "adv.%s.tsv.xz" % case)) as f, open(tsv, "wb") as g:
        g.write(f.read())
    assert lib().cfb_promote(base.encode(), tsv.encode(), level.encode(), out.encode()) == 0
    with open(out, "rb") as f, lzma.open(os.path.join(util.GOLDEN, "adv.%s.promote.%s.tsv.xz" % (case, level))) as g:
        assert f.read() == g.read()


@pytest.mark.parametrize("level", LEVELS)
def test_promote_corner_cases_match_reference_script(level, tmp_path):
    base = util.golden_index("adv")
    out = str(tmp_path / "out.tsv")
    assert lib().cfb_promote(base.encode(), os.path.join(util.GOLDEN, "promote_quirks.tsv").encode(), level.encode(), out.encode()) == 0
    with open(out, "rb") as f, open(os.path.join(util.GOLDEN, "promote_quirks.%s.tsv" % level), "rb") as g:
        assert f.read() == g.read()


def test_cli_promote_mode(tmp_path):
    """`centrifuge-class --promote <index> <tsv> <level>` writes the same bytes to stdout (no GPU involved)."""
    from centrifuge_b200 import build
    build.build()
    base = util.golden_index("adv")
    exe = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")
    p = subprocess.run([exe, "--promote", base, os.path.join(util.GOLDEN, "promote_quirks.tsv"), "genus"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
    assert p.returncode == 0
    with open(os.path.join(util.GOLDEN, "promote_quirks.genus.tsv"), "rb") as g:
        assert p.stdout == g.read()


def test_promote_matches_reference_script_on_random_tables(tmp_path):
    """Differential fuzzing against recorded runs of the Perl script: taxIDs at every level of the tree and outside it, dotted
    strain IDs, runs of equal read names, repeated names, unclassified rows, every level."""
    import random
    base = util.golden_index("adv")
    taxa = [0, 1, 10, 11, 100, 101, 102, 103] + list(range(1000, 1020)) + [424242]
    for case in range(60):
        rng = random.Random(77 + case)
        rows = ["readID\tseqID\ttaxID\tscore\t2ndBestScore\thitLength\tqueryLength\tnumMatches"]
        for r in range(rng.randrange(1, 120)):
            name = "r%d" % (r if rng.random() < 0.8 else max(0, r - 1))
            k = rng.choice([1, 1, 1, 2, 3, 5])
            for _ in range(k):
                t = rng.choice(taxa)
                tid = str(t) if (t <= 1 or rng.random() < 0.95) else "%d.%d" % (t, rng.randrange(1, 9))
                sid = "unclassified" if t == 0 else rng.choice(["cid%d" % rng.randrange(20), "species", "genus", "no rank"])
                rows.append("%s\t%s\t%s\t%d\t0\t%d\t100\t%d" % (name, sid, tid, rng.choice([0, 49, 300, 2500, 7225]), rng.choice([0, 22, 39, 40, 85]), k))
        tsv = tmp_path / "t.tsv"
        tsv.write_text("\n".join(rows) + ("\n" if rng.random() < 0.9 else ""))
        level = rng.choice(LEVELS + ["order", "no rank"])
        p = util.reference_run("promote", [base, str(tsv), level])
        out = tmp_path / "o.tsv"
        assert lib().cfb_promote(base.encode(), str(tsv).encode(), level.encode(), str(out).encode()) == 0
        assert util.digest(out.read_bytes()) == p["stdout"], (case, level)
