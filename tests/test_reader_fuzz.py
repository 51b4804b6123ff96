"""Differential fuzzing of the readers, on the CPU:
  * the oracle's file driver against the unmodified reference binary, end to end (classification TSV, report, or the
    error message and a failing exit status) on irregular FASTQ / FASTA text;
  * the product's record-level reader (cfb_test_parse: the code `centrifuge-class` falls back to whenever the device
    tokeniser declines a span) against the oracle's reader, read by read (name, bases, seed, filter verdict).
Together they pin the product's reader to the reference on layouts no hand-written case covers."""
import ctypes as C
import os
import random
import subprocess

import pytest

import util
from util_fuzz import clean_reads, mutate_fasta, mutate_fastq

N_CASES = 200


TRIMS = [(0, 0), (0, 0), (3, 0), (0, 5), (4, 7), (90, 0), (0, 200)]


def _case(case, seed0):
    rng = random.Random(seed0 + case)
    sub = rng.sample(clean_reads(), 12)
    fasta = case % 2 == 1
    return fasta, (mutate_fasta(rng, sub) if fasta else mutate_fastq(rng, sub)), TRIMS[rng.randrange(len(TRIMS))]


def test_oracle_file_driver_matches_reference_on_irregular_text(tmp_path):
    util.ensure_oracle()
    base = util.golden_index("adv")

    def run(fmt, path, trims):
        args = [fmt, "-x", base, "-U", path, "-5", str(trims[0]), "-3", str(trims[1])]
        r = util.reference_run("class", args, str(tmp_path / "ref"))
        want = ("fail", r["errors"]) if r["rc"] != 0 else ("ok",) + tuple(r["outputs"])
        tsv, rep = str(tmp_path / "ora.tsv"), str(tmp_path / "ora.rep")
        p = subprocess.run([util.ORACLE_BIN] + args + ["-S", tsv, "--report-file", rep], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
        got = ("fail", util.error_lines(p.stderr)) if p.returncode != 0 else ("ok", util.file_digest(tsv), util.file_digest(rep))
        return want, got

    for case in range(N_CASES):
        fasta, data, trims = _case(case, 1000)
        path = str(tmp_path / "in.txt")
        with open(path, "wb") as f:
            f.write(data)
        fmt = "-f" if fasta else "-q"
        want, got = run(fmt, path, trims)
        assert want == got, (case, fmt, trims)


def test_oracle_file_driver_matches_reference_on_irregular_mate_files(tmp_path):
    """Paired input: independently mutated mate files, including the ones that fall out of step
    ("fewer reads in file specified with -1/-2": same message, failing exit status)."""
    util.ensure_oracle()
    base = util.golden_index("adv")
    reads = clean_reads()

    def run(fmt, p1, p2):
        args = [fmt, "-x", base, "-1", p1, "-2", p2]
        r = util.reference_run("class", args, str(tmp_path / "ref"))
        want = ("fail", r["errors"]) if r["rc"] != 0 else ("ok",) + tuple(r["outputs"])
        tsv, rep = str(tmp_path / "ora.tsv"), str(tmp_path / "ora.rep")
        p = subprocess.run([util.ORACLE_BIN] + args + ["-S", tsv, "--report-file", rep], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
        got = ("fail", util.error_lines(p.stderr)) if p.returncode != 0 else ("ok", util.file_digest(tsv), util.file_digest(rep))
        return want, got

    for case in range(100):
        rng = random.Random(424200 + case)
        sub = rng.sample(reads, rng.randrange(1, 10))
        sub2 = [(n, s[::-1]) for n, s in sub]
        fasta = rng.random() < 0.5
        mut = mutate_fasta if fasta else mutate_fastq
        p1, p2 = str(tmp_path / "a.txt"), str(tmp_path / "b.txt")
        with open(p1, "wb") as f:
            f.write(mut(rng, sub))
        with open(p2, "wb") as f:
            f.write(mut(rng, sub2))
        fmt = "-f" if fasta else "-q"
        want, got = run(fmt, p1, p2)
        assert want == got, (case, fmt)


def test_product_reader_matches_oracle_reader_on_irregular_text(tmp_path):
    util.ensure_oracle()
    base = util.golden_index("adv")
    lib = C.CDLL(util.PRODUCT_LIB)
    for case in range(N_CASES):
        fasta, data, trims = _case(case, 5000)
        path, prod, ora = str(tmp_path / "in.txt"), str(tmp_path / "prod.txt"), str(tmp_path / "ora.txt")
        with open(path, "wb") as f:
            f.write(data)
        rc = lib.cfb_test_parse(path.encode(), C.c_int(1 if fasta else 0), C.c_int(trims[0]), C.c_int(trims[1]), C.c_uint32(0), prod.encode())
        if os.path.exists(ora):
            os.remove(ora)
        p = subprocess.run([util.ORACLE_BIN, "-f" if fasta else "-q", "-x", base, "-U", path, "-S", str(tmp_path / "o.tsv"),
                            "--report-file", str(tmp_path / "o.rep"), "--dump-reads", ora, "-5", str(trims[0]), "-3", str(trims[1])],
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        assert (rc != 0) == (p.returncode != 0), (case, trims)
        if rc == 0:
            with open(prod, "rb") as f, open(ora, "rb") as g:
                assert f.read() == g.read(), (case, trims)
