"""Kraken-style report (SURVEY.md 8f rank 4): `cfb_kreport` / `centrifuge-class --kreport-file` against the
reference's own Perl `centrifuge-kreport` run on the committed golden classification outputs
(tests/golden/make_kreport_golden.py)."""
import ctypes as C
import lzma
import os

import pytest

import util

CASES = [("default", "", (0, 0, 0, 0, 0)), ("default", ".zeros", (1, 0, 0, 0, 0)), ("default", ".minscore", (0, 1, 300, 0, 0)),
         ("default", ".minlen", (0, 0, 0, 1, 40))] + [(c, "", (0, 0, 0, 0, 0)) for c in ("k1", "k50", "minhit15", "host", "excl", "family", "notraverse")]


def lib():
    return C.CDLL(util.PRODUCT_LIB)


@pytest.mark.parametrize("case,suffix,args", CASES)
def test_kreport_from_tsv_matches_reference_script(case, suffix, args, tmp_path):
    base = util.golden_index("adv")
    tsv = str(tmp_path / "in.tsv")
    with lzma.open(os.path.join(util.GOLDEN, "adv.%s.tsv.xz" % case)) as f, open(tsv, "wb") as g:
        g.write(f.read())
    out = str(tmp_path / "k.txt")
    rc = lib().cfb_kreport(base.encode(), tsv.encode(), out.encode(), C.c_int(args[0]), C.c_int(args[1]), C.c_longlong(args[2]), C.c_int(args[3]), C.c_longlong(args[4]))
    assert rc == 0
    with open(out, "rb") as f, open(os.path.join(util.GOLDEN, "adv.%s%s.kreport.txt" % (case, suffix)), "rb") as g:
        assert f.read() == g.read()


@pytest.mark.parametrize("suffix,args", [("", (0, 0, 0, 0, 0)), (".zeros", (1, 0, 0, 0, 0)), (".minscore", (0, 1, 300, 0, 0)), (".minlen", (0, 0, 0, 1, 40))])
def test_kreport_corner_cases_match_reference_script(suffix, args, tmp_path):
    """LCA merging of equal consecutive readIDs, dotted / unknown taxIDs to the root, filtered rows between rows of one read."""
    base = util.golden_index("adv")
    out = str(tmp_path / "k.txt")
    rc = lib().cfb_kreport(base.encode(), os.path.join(util.GOLDEN, "kreport_quirks.tsv").encode(), out.encode(), C.c_int(args[0]), C.c_int(args[1]),
                           C.c_longlong(args[2]), C.c_int(args[3]), C.c_longlong(args[4]))
    assert rc == 0
    with open(out, "rb") as f, open(os.path.join(util.GOLDEN, "kreport_quirks%s.kreport.txt" % suffix), "rb") as g:
        assert f.read() == g.read()


def test_kreport_matches_reference_script_on_random_tables(tmp_path):
    """Differential fuzzing against recorded runs of the Perl script: random classification tables (taxIDs at every level of the
    tree and outside it, dotted strain IDs, runs of equal read names, unclassified rows) with random option sets."""
    import random
    base = util.golden_index("adv")
    taxa = [0, 1, 10, 11, 100, 101, 102, 103] + list(range(1000, 1020)) + [424242]
    for case in range(40):
        rng = random.Random(31 + case)
        rows = ["readID\tseqID\ttaxID\tscore\t2ndBestScore\thitLength\tqueryLength\tnumMatches"]
        for r in range(rng.randrange(1, 120)):
            name = "r%d" % (r if rng.random() < 0.8 else max(0, r - 1))                 # now and then two reads share a name
            for _ in range(rng.choice([1, 1, 1, 2, 3, 5])):
                t = rng.choice(taxa)
                tid = str(t) if (t <= 1 or rng.random() < 0.95) else "%d.%d" % (t, rng.randrange(1, 9))    # strain suffixes only occur on real taxa
                rows.append("%s\tseq\t%s\t%d\t0\t%d\t100\t1" % (name, tid, rng.choice([0, 49, 300, 2500, 7225]), rng.choice([0, 22, 39, 40, 85])))
        tsv = tmp_path / "t.tsv"
        tsv.write_text("\n".join(rows) + "\n")
        args = rng.choice([(0, 0, 0, 0, 0), (1, 0, 0, 0, 0), (0, 1, 300, 0, 0), (0, 0, 0, 1, 40), (1, 1, 49, 1, 22)])
        opts = (["--show-zeros"] if args[0] else []) + (["--min-score", str(args[2])] if args[1] else []) + (["--min-length", str(args[4])] if args[3] else [])
        p = util.reference_run("kreport", ["-x", base] + opts + [str(tsv)])
        out = tmp_path / "k.txt"
        if out.exists():
            out.unlink()
        rc = lib().cfb_kreport(base.encode(), str(tsv).encode(), str(out).encode(), C.c_int(args[0]), C.c_int(args[1]), C.c_longlong(args[2]),
                               C.c_int(args[3]), C.c_longlong(args[4]))
        assert rc == 0
        got = out.read_bytes() if out.exists() else b""
        assert util.digest(got) == (p["stdout"] if p["rc"] == 0 else util.digest(b"")), (case, args)


@pytest.mark.gpu
@pytest.mark.parametrize("reader", ["text", "host"])
@pytest.mark.parametrize("case,opts", [("default", []), ("k1", ["-k", "1"]), ("host", ["--host-taxids", "100,1005", "-k", "2"])])
def test_cli_kreport_file_in_process(case, opts, reader, tmp_path):
    """The classifier writes the same report itself, from rows still in memory, through either reader."""
    import subprocess
    base = util.golden_index("adv")
    reads = str(tmp_path / "reads.fa")
    with lzma.open(os.path.join(util.GOLDEN, "adv.reads.fa.xz")) as f, open(reads, "wb") as g:
        g.write(f.read())
    exe = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")
    out = str(tmp_path / "k.txt")
    subprocess.check_call([exe, "-f", "-x", base, "-U", reads, "-S", str(tmp_path / "o.tsv"), "--report-file", str(tmp_path / "o.rep"), "--kreport-file", out]
                          + opts + (["--host-parse"] if reader == "host" else []), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                          env=dict(os.environ, CFB_TEXT_BLOCK="20000"))
    with open(out, "rb") as f, open(os.path.join(util.GOLDEN, "adv.%s.kreport.txt" % case), "rb") as g:
        assert f.read() == g.read()
