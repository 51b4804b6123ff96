"""Text-level operator (SURVEY.md 8f rank 1): FASTQ/FASTA bytes -> TSV on the device.

Every case runs the drop-in `centrifuge-class` on the files the unmodified reference binary was run on
(recorded runs, tests/golden/reference_runs.json) and demands identical classification TSV and report bytes, and checks through the
CFB_TEXT_STATS line which reader handled the input: well-formed files must go through the device
tokeniser/formatter entirely, files with irregular layout must switch to the record-level reader
at the span that failed (and still produce the reference's bytes)."""
import os
import re
import subprocess

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

EXE = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")


def run_ours(args, tmp, tag, block=None, extra_env=None):
    env = dict(os.environ, CFB_TEXT_STATS="1")
    if block:
        env["CFB_TEXT_BLOCK"] = str(block)
    env.update(extra_env or {})
    tsv, rep = str(tmp / (tag + ".tsv")), str(tmp / (tag + ".rep"))
    p = subprocess.run([EXE] + list(args) + ["-S", tsv, "--report-file", rep], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=env)
    assert p.returncode == 0, p.stderr.decode()
    m = re.search(r"text operator: (\d+) units in (\d+) spans .* (\d+) fallbacks\); record-level reader: (\d+) units", p.stderr.decode())
    assert m, p.stderr.decode()
    return (util.file_digest(tsv), util.file_digest(rep)), dict(text=int(m.group(1)), spans=int(m.group(2)), fallbacks=int(m.group(3)), host=int(m.group(4)))


def run_ref(args, tmp, tag):
    return util.reference_cli(args, tmp / tag)


@pytest.fixture(scope="module")
def syn():
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    return base, seqs


def decorate(reads, rng):
    """Names and sequence spellings the strict layout still covers."""
    out = []
    for k, (name, a) in enumerate(reads):
        a = a.copy()
        r = k % 11
        if r == 1: name += " extra words"
        if r == 2: name += "/1"
        if r == 3: name += "/3 tail"
        if r == 4: name = "x/y/" + name
        if r == 5: a = np.frombuffer(a.tobytes().lower(), dtype=np.uint8).copy()
        if r == 6 and len(a) > 8: a[3] = ord("."); a[5] = ord("R"); a[7] = ord("y")
        if r == 7: name += "\tTAB"
        if r == 8 and len(a) > 20: a[rng.integers(0, len(a), size=max(1, len(a) // 5))] = ord("N")      # fails the N filter
        out.append((name, a))
    return out


def write_fq(path, reads, rng, tail_newline=True, var_qual=True):
    with open(path, "wb") as f:
        for i, (name, a) in enumerate(reads):
            q = rng.integers(33, 74, size=len(a) + (i % 3 == 0), dtype=np.uint8).tobytes() if var_qual else b"I" * len(a)
            end = b"\n" if (tail_newline or i + 1 < len(reads)) else b""
            f.write(b"@" + name.encode() + b"\n" + a.tobytes() + b"\n+" + (name.encode() if i % 5 == 0 else b"") + b"\n" + q + end)


def test_fastq_se_mixed_lengths_all_on_device(syn, tmp_path):
    base, seqs = syn
    rng = np.random.default_rng(1)
    # short reads first so that the length class grows mid-run (128 -> 320 -> 1024)
    reads = (util.synth.sample_reads(seqs, 2500, 60, seed=11, lens=(1, 120)) + util.synth.sample_reads(seqs, 2500, 150, seed=12, lens=(100, 300))
             + util.synth.sample_reads(seqs, 600, 500, seed=13, lens=(300, 900)))
    reads = decorate(reads, rng)
    fq = str(tmp_path / "r.fq")
    write_fq(fq, reads, rng, tail_newline=False)
    for extra in ([], ["-5", "3", "-3", "7"], ["-k", "1"], ["-k", "9", "--min-hitlen", "15"], ["--seed", "77", "--classification-rank", "genus"]):
        args = ["-q", "-x", base, "-U", fq] + extra
        want = run_ref(args, tmp_path, "ref")
        got, st = run_ours(args, tmp_path, "our", block=100000)
        assert got == want, extra
        assert st["fallbacks"] == 0 and st["host"] == 0 and st["text"] == len(reads) and st["spans"] > 5, st
    # row-buffer overflow inside a span: classification stages re-run, the formatter follows
    got, st = run_ours(["-q", "-x", base, "-U", fq], tmp_path, "rows", block=100000, extra_env={"CFB_ROWS_CAP": "64"})
    assert got == run_ref(["-q", "-x", base, "-U", fq], tmp_path, "ref") and st["fallbacks"] == 0
    # one big span and the forced host reader give the same bytes
    got, st = run_ours(["-q", "-x", base, "-U", fq], tmp_path, "big")
    assert got == run_ref(["-q", "-x", base, "-U", fq], tmp_path, "ref") and st["spans"] == 1
    got2, st2 = run_ours(["-q", "-x", base, "-U", fq, "--host-parse"], tmp_path, "host")
    assert got2 == got and st2["text"] == 0 and st2["host"] == len(reads)


def test_fastq_pe_all_on_device(syn, tmp_path):
    base, seqs = syn
    rng = np.random.default_rng(2)
    prs = util.synth.sample_pairs(seqs, 5000, 125, seed=31)
    r1 = decorate([(n, x) for n, x, _ in prs], rng)
    r2 = [(n + "/2", y[: max(1, len(y) - (i % 40))]) for i, (n, _, y) in enumerate(prs)]      # mates of different lengths
    f1, f2 = str(tmp_path / "p_1.fq"), str(tmp_path / "p_2.fq")
    write_fq(f1, r1, rng); write_fq(f2, r2, rng)
    for extra in ([], ["-3", "100"], ["-k", "2"]):
        args = ["-q", "-x", base, "-1", f1, "-2", f2] + extra
        want = run_ref(args, tmp_path, "ref")
        got, st = run_ours(args, tmp_path, "our", block=150000)
        assert got == want, extra
        assert st["fallbacks"] == 0 and st["host"] == 0 and st["text"] == len(prs), st


def test_fasta_se_and_pe_on_device(syn, tmp_path):
    base, seqs = syn
    rng = np.random.default_rng(3)
    reads = decorate(util.synth.sample_reads(seqs, 4000, 100, seed=5, lens=(20, 200)), rng)
    for i in range(0, len(reads), 13):
        a = reads[i][1].copy(); a[0] = ord("-"); reads[i] = (reads[i][0], a)       # gap characters count as bases in FASTA reads
    reads = [(n, np.frombuffer(a.tobytes().replace(b".", b"N"), dtype=np.uint8)) for n, a in reads]   # '.' is not a FASTA base: keep the layout strict
    fa = str(tmp_path / "r.fa")
    with open(fa, "wb") as f:
        for n, a in reads:
            f.write(b">" + n.encode() + b"\n" + a.tobytes() + b"\n")
    args = ["-f", "-x", base, "-U", fa]
    got, st = run_ours(args, tmp_path, "our", block=50000)
    assert got == run_ref(args, tmp_path, "ref")
    assert st["fallbacks"] == 0 and st["text"] == len(reads), st
    args = ["-f", "-x", base, "-1", fa, "-2", fa, "-5", "2"]
    got, st = run_ours(args, tmp_path, "our2", block=50000)
    assert got == run_ref(args, tmp_path, "ref2")
    assert st["fallbacks"] == 0 and st["text"] == len(reads), st


IRREGULAR = {
    "crlf": lambda rec: rec.replace(b"\n", b"\r\n"),
    "wrapped": lambda rec: (lambda p: p[0] + b"\n" + p[1][:10] + b"\n" + p[1][10:] + b"\n" + b"\n".join(p[2:]))(rec.split(b"\n")),
    "blank_line": lambda rec: b"\n" + rec,
    "empty_read": lambda rec: rec.split(b"\n")[0] + b"\n\n+\n\n",
    "digits_in_seq": lambda rec: (lambda p: p[0] + b"\n" + p[1][:5] + b"12" + p[1][5:] + b"\n" + p[2] + b"\n" + p[3] + b"\n")(rec.split(b"\n")),
}


@pytest.mark.parametrize("kind", sorted(IRREGULAR))
def test_irregular_layout_switches_to_record_reader(kind, syn, tmp_path):
    base, seqs = syn
    rng = np.random.default_rng(4)
    reads = util.synth.sample_reads(seqs, 3000, 100, seed=21, lens=(40, 140))
    fq = str(tmp_path / "r.fq")
    with open(fq, "wb") as f:
        for i, (name, a) in enumerate(reads):
            rec = b"@" + name.encode() + b"\n" + a.tobytes() + b"\n+\n" + b"F" * len(a) + b"\n"
            if i == 2000:
                rec = IRREGULAR[kind](rec)
            f.write(rec)
    args = ["-q", "-x", base, "-U", fq]
    want = run_ref(args, tmp_path, "ref")
    got, st = run_ours(args, tmp_path, "our", block=60000)
    assert got == want
    assert st["fallbacks"] == 1 and st["text"] > 1000 and st["host"] > 900 and st["text"] + st["host"] == len(reads), st


@pytest.mark.parametrize("kind", ["too_many", "too_few", "space", "control"])
def test_quality_string_errors_match_the_reference(kind, syn, tmp_path):
    base, seqs = syn
    reads = util.synth.sample_reads(seqs, 1200, 80, seed=9)
    fq = str(tmp_path / "q.fq")
    with open(fq, "wb") as f:
        for i, (name, a) in enumerate(reads):
            q = b"F" * len(a)
            if i == 900:
                q = {"too_many": q + b"FF", "too_few": q[:-1], "space": q[:10] + b" " + q[11:], "control": q[:10] + b"\x1f" + q[11:]}[kind]
            f.write(b"@" + name.encode() + b"\n" + a.tobytes() + b"\n+\n" + q + b"\n")
    r = util.reference_run("class", ["-q", "-x", base, "-U", fq], str(tmp_path / "ref"))
    assert r["rc"] != 0
    p = subprocess.run([EXE, "-q", "-x", base, "-U", fq, "-S", str(tmp_path / "o.tsv"), "--report-file", str(tmp_path / "o.rep")],
                       stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=dict(os.environ, CFB_TEXT_BLOCK="30000"))
    assert p.returncode != 0
    assert r["errors"] and r["errors"] == util.error_lines(p.stderr)


def test_mate_files_out_of_step_report_the_reference_error(syn, tmp_path):
    base, seqs = syn
    rng = np.random.default_rng(6)
    prs = util.synth.sample_pairs(seqs, 800, 100, seed=3)
    f1, f2 = str(tmp_path / "a_1.fq"), str(tmp_path / "a_2.fq")
    write_fq(f1, [(n, x) for n, x, _ in prs], rng); write_fq(f2, [(n, y) for n, _, y in prs][:700], rng)
    r = util.reference_run("class", ["-q", "-x", base, "-1", f1, "-2", f2], str(tmp_path / "ref"))
    assert r["rc"] != 0 and any("fewer reads in file specified with -2" in l for l in r["errors"]), r
    p = subprocess.run([EXE, "-q", "-x", base, "-1", f1, "-2", f2, "-S", str(tmp_path / "o.tsv"), "--report-file", str(tmp_path / "o.rep")],
                       stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=dict(os.environ, CFB_TEXT_BLOCK="40000"))
    assert p.returncode != 0
    assert b"fewer reads in file specified with -2" in p.stderr


def test_fasta_record_wrapped_across_a_span_cut(syn, tmp_path):
    """A FASTA record runs up to the next '>' (pat.cpp:806-826): when a span cut falls right after the first sequence
    line of a wrapped record, the span must not emit that record from its first line alone.  The cut position depends
    on the span size, so a range of sizes is swept; every one must reproduce the reference's bytes, and the wrapped
    record must end up with the record-level reader."""
    base, seqs = syn
    reads = util.synth.sample_reads(seqs, 1500, 100, seed=41, lens=(60, 140))
    fa = str(tmp_path / "w.fa")
    recs = []
    for i, (name, a) in enumerate(reads):
        s = a.tobytes()
        if i >= 700 and i % 2 == 0:          # from the middle of the file on, every other record is wrapped after 30 bases
            recs.append(b">" + name.encode() + b"\n" + s[:30] + b"\n" + s[30:] + b"\n")
        else:
            recs.append(b">" + name.encode() + b"\n" + s + b"\n")
    with open(fa, "wb") as f:
        f.write(b"".join(recs))
    # a file whose only wrapped record is the one a cut can split: spans are cut where the line count allows, so put
    # the wrapped record at many different byte offsets by sweeping the block size
    args = ["-f", "-x", base, "-U", fa]
    want = run_ref(args, tmp_path, "ref")
    for block in (4096, 5000, 7777, 12345, 20011, 33333):
        got, st = run_ours(args, tmp_path, "our%d" % block, block=block)
        assert got == want, block
        assert st["fallbacks"] == 1 and st["text"] + st["host"] == len(reads), (block, st)
    # single wrapped record exactly at a cut: strict records of fixed size, so the cut position is known
    fixed = [(("r%04d" % i), np.frombuffer(b"ACGT" * 20, dtype=np.uint8)) for i in range(600)]
    for i in range(len(fixed)):
        fixed[i] = (fixed[i][0], reads[i][1][:80] if len(reads[i][1]) >= 80 else fixed[i][1])
    rec_bytes = 1 + 5 + 1 + 80 + 1                       # ">r0000\n" + 80 bases + "\n"
    for split_at in (100, 101):
        body = []
        for i, (n, a) in enumerate(fixed):
            s = a.tobytes()
            body.append(b">" + n.encode() + b"\n" + (s[:40] + b"\n" + s[40:] if i == split_at else s) + b"\n")
        with open(fa, "wb") as f:
            f.write(b"".join(body))
        want = run_ref(args, tmp_path, "ref2")
        # a block that ends inside record `split_at`, after its first sequence line
        block = split_at * rec_bytes + 1 + 5 + 1 + 40 + 1 + 3
        got, st = run_ours(args, tmp_path, "cut%d" % split_at, block=block)
        assert got == want, split_at
        assert st["text"] + st["host"] == len(fixed) and st["host"] >= len(fixed) - split_at - 1, st
