"""CPU suite: pins the oracle (oracle/cf_oracle.cpp) against the reference's outputs, and the
product's host-compilable classification logic against the oracle.  No GPU needed, except where a synthetic
index comes from the product's builder (marked gpu)."""
import ctypes as C
import hashlib
import lzma
import os
import re
import subprocess

import numpy as np
import pytest

import util

GOLDEN_CASES = {
    "default": [], "k1": ["-k", "1"], "k50": ["-k", "50"], "minhit15": ["--min-hitlen", "15"],
    "host": ["--host-taxids", "100,1005", "-k", "2"], "excl": ["--exclude-taxids", "10"],
    "family": ["--classification-rank", "family"], "notraverse": ["--no-traverse"],
}
PARAM_CASES = {
    "default": {}, "k1": dict(k=1), "k50": dict(k=50), "minhit15": dict(min_hitlen=15),
    "host": dict(host=(100, 1005), k=2), "excl": dict(excl=(10,)), "family": dict(rank_slot=3), "notraverse": dict(traverse=False),
}


def _golden(name):
    with lzma.open(os.path.join(util.GOLDEN, "adv.%s.tsv.xz" % name)) as f:
        tsv = f.read()
    with open(os.path.join(util.GOLDEN, "adv.%s.report.tsv" % name), "rb") as f:
        rep = f.read()
    return tsv, rep


@pytest.mark.parametrize("case", sorted(GOLDEN_CASES))
def test_oracle_matches_reference_golden(case, adv_base, adv_reads, tmp_path):
    """Oracle file driver == committed output of the unmodified reference binary (byte for byte)."""
    util.ensure_oracle()
    tsv, rep = util.run_cli(util.ORACLE_BIN, ["-f", "-x", adv_base, "-U", adv_reads] + GOLDEN_CASES[case],
                            str(tmp_path / "o.tsv"), str(tmp_path / "o.rep"))
    gt, gr = _golden(case)
    assert tsv == gt
    assert rep == gr


def test_oracle_matches_manual_example(tmp_path):
    """The reference's only known-answer fixture (MANUAL.markdown:1586-1603)."""
    util.ensure_oracle()
    base, reads = util.golden_index("example"), os.path.join(util.GOLDEN, "example.reads.fa")   # committed copy (tests/golden/make_example_golden.py)
    # the copy is the reference's own bytes: sha256 of its example/index/test.{1,2,3,4}.cf and example/reads/input.fa
    ref_sha256 = {".1.cf": "73894274fbeef3ff3927e50f5d7896693b821b25d84888f2113d019edbc16ad3", ".2.cf": "864df23898e55c42f5a04f23ce85528255dfa0ef51313f9db84ee6e0560e826e",
                  ".3.cf": "65cf2737ded0050ff8f00947322934b1c987c07b31033ba661072cc4b77df032", ".4.cf": "876eff21a39ac41dbd88421eea70dc9c23474e39b7ff338ab5d500e24dc37364"}
    for ext, want in ref_sha256.items():
        with open(base + ext, "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == want, ext
    with open(reads, "rb") as f:
        assert hashlib.sha256(f.read()).hexdigest() == "885b4f7483e0814d2ce9b935465735f9dbcd3f8ed7c0eaee363834b87b93bfb9"
    tsv, rep = util.run_cli(util.ORACLE_BIN, ["-f", "-x", base, "-U", reads], str(tmp_path / "o.tsv"), str(tmp_path / "o.rep"))
    with open(os.path.join(util.GOLDEN, "example.tsv"), "rb") as f:
        assert tsv == f.read()
    with open(os.path.join(util.GOLDEN, "example.report.tsv"), "rb") as f:
        assert rep == f.read()
    # and the table printed in the manual itself (it predates the queryLength column)
    rows = [ln.split("\t") for ln in tsv.decode().strip().split("\n")[1:]]
    assert [r[0] for r in rows[:4]] == ["C_1", "C_1", "C_2", "C_2"]
    assert [r[1] for r in rows[:4]] == ["gi|7", "gi|4", "gi|4", "gi|7"]      # RNG-dependent tie order
    assert all(r[3] == "4225" for r in rows)


@pytest.mark.gpu      # the index comes from the product's builder
@pytest.mark.parametrize("opts", [[], ["-k", "1"], ["--classification-rank", "genus"], ["--min-hitlen", "30", "-k", "3"]])
def test_oracle_matches_live_reference_synthetic(opts, tmp_path):
    """Seeded synthetic genus/species index (SURVEY Appendix C recipe, with strains), SE FASTA + PE FASTQ."""
    util.ensure_oracle()
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    rd = util.synth.sample_reads(seqs, 3000, 100, seed=11, lens=(40, 220))
    fa = str(tmp_path / "r.fa")
    util.synth.write_fasta(fa, rd)
    a = util.reference_cli(["-f", "-x", base, "-U", fa] + opts, tmp_path)
    b = util.run_cli(util.ORACLE_BIN, ["-f", "-x", base, "-U", fa] + opts, str(tmp_path / "b.tsv"), str(tmp_path / "b.rep"))
    assert a == util.digests(b)
    prs = util.synth.sample_pairs(seqs, 1500, 125, seed=12)
    f1, f2 = str(tmp_path / "p_1.fq"), str(tmp_path / "p_2.fq")
    util.synth.write_fastq(f1, [(n, x) for n, x, _ in prs])
    util.synth.write_fastq(f2, [(n, y) for n, _, y in prs], qual=b"5")
    a = util.reference_cli(["-q", "-x", base, "-1", f1, "-2", f2] + opts, tmp_path)
    b = util.run_cli(util.ORACLE_BIN, ["-q", "-x", base, "-1", f1, "-2", f2] + opts, str(tmp_path / "b.tsv"), str(tmp_path / "b.rep"))
    assert a == util.digests(b)


@pytest.mark.parametrize("case", sorted(PARAM_CASES))
def test_product_logic_matches_oracle_adversarial(case, adv_base, adv_reads):
    """cf_logic.h (the per-thread code of the CUDA kernels, compiled for the host by the test)
    produces the same record stream as the oracle, stage counters included."""
    reads = util.parse_reads(adv_reads)
    b = util.Batch([a for _, a in reads])
    o, h = util.Oracle(adv_base), util.HostLogic(adv_base)
    p = util.make_oparams(**PARAM_CASES[case])
    on, orec, ost = o.classify(b, p)
    hn, hrec, hst = h.classify(b, p)
    assert np.array_equal(on, hn)
    assert np.array_equal(orec, hrec)
    # partial searches / ftab probes / sides touched by the search are identical; the product
    # skips resolving rows of hits the reference resolves and then discards (classifier.h:299)
    assert (ost[1], ost[2], ost[6], ost[10]) == (hst[1], hst[2], hst[3], hst[7])
    assert hst[4] <= ost[7] and hst[5] <= ost[8]
    o.close(); h.close()


@pytest.mark.gpu      # the index comes from the product's builder
def test_product_logic_matches_oracle_paired_and_wide_sample():
    """> 65535 sequences (u32 SA sample, boundary rows), paired units with filtered mates."""
    import numpy as np
    d = os.path.join(util.CACHE, "wide")
    base = os.path.join(d, "idx")
    rng = np.random.default_rng(44)
    n, L = 66000, 120
    g = rng.integers(0, 4, size=(n, L), dtype=np.uint8)
    g[33000:] = np.where(rng.random((33000, L)) < 0.03, (g[:33000] + 1) & 3, g[:33000])
    if not os.path.exists(base + ".4.cf"):
        os.makedirs(d, exist_ok=True)
        A = util.synth.ACGT
        with open(os.path.join(d, "g.fa"), "wb") as f:
            for i in range(n):
                f.write(b">c%d\n" % i + A[g[i]].tobytes() + b"\n")
        with open(os.path.join(d, "conv.tsv"), "w") as f:
            for i in range(n):
                f.write("c%d\t%d\n" % (i, 1000 + i % 300))
        with open(os.path.join(d, "nodes.dmp"), "w") as f:
            f.write("1\t|\t1\t|\tno rank\t|\n")
            for t in range(30):
                f.write("%d\t|\t1\t|\tgenus\t|\n" % (100 + t))
            for t in range(300):
                f.write("%d\t|\t%d\t|\tspecies\t|\n" % (1000 + t, 100 + t % 30))
        with open(os.path.join(d, "names.dmp"), "w") as f:
            f.write("1\t|\troot\t|\t\t|\tscientific name\t|\n")
        util.build_fasta_index([os.path.join(d, "g.fa")], os.path.join(d, "conv.tsv"), os.path.join(d, "nodes.dmp"), os.path.join(d, "names.dmp"), base)
    A = util.synth.ACGT
    m1, m2 = [], []
    for k in range(1500):
        i = int(rng.integers(0, n))
        a, b = A[g[i][:90]].copy(), A[(3 - g[i][30:120])[::-1]].copy()
        u = rng.random()
        if u < 0.1:
            b[:] = ord("N")
        elif u < 0.2:
            a[:] = ord("N")
        elif u < 0.25:
            a[:] = ord("N"); b[:] = ord("N")
        elif u < 0.3:
            b = b[:1]
        m1.append(a); m2.append(b)
    bt = util.Batch(m1, m2)
    o, h = util.Oracle(base), util.HostLogic(base)
    for kw in ({}, dict(rank_slot=2), dict(k=1)):
        p = util.make_oparams(**kw)
        on, orec, _ = o.classify(bt, p)
        hn, hrec, _ = h.classify(bt, p)
        assert np.array_equal(on, hn) and np.array_equal(orec, hrec)
    o.close(); h.close()


def test_restated_std_sort_is_libstdcxx_exact():
    """The device's introsort restatement must reproduce std::sort's permutation, ties included."""
    util.ensure_oracle()
    lib = C.CDLL(util.HOSTLOGIC_LIB)
    HIT = np.dtype([("top", "<u8"), ("bot", "<u8"), ("bwoff", "<u4"), ("len", "<u4")])
    rng = np.random.default_rng(0)
    for trial in range(3000):
        n = int(rng.integers(0, 120)) if trial % 3 else int(rng.integers(17, 400))
        a = np.zeros(n, dtype=HIT)
        mode = trial % 5
        if mode == 0:
            lens, sizes = rng.integers(0, 40, n), rng.integers(0, 4, n)
        elif mode == 1:
            lens, sizes = rng.integers(20, 24, n), rng.integers(0, 3, n)
        elif mode == 2:
            lens, sizes = np.sort(rng.integers(0, 100, n)), rng.integers(0, 50, n)
        elif mode == 3:
            lens, sizes = np.sort(rng.integers(0, 30, n))[::-1], np.ones(n, dtype=np.int64)
        else:
            lens, sizes = rng.integers(15, 30, n), rng.integers(0, 2, n) * rng.integers(1, 1000, n)
        a["top"] = rng.integers(0, 1000, n)
        a["bot"] = a["top"] + sizes.astype(np.uint64)
        a["len"] = lens
        a["bwoff"] = np.arange(n)
        b, c = a.copy(), a.copy()
        lib.hl_sort_hits(b.ctypes.data_as(C.c_void_p), C.c_size_t(n))
        lib.hl_std_sort_hits(c.ctypes.data_as(C.c_void_p), C.c_size_t(n))
        assert np.array_equal(b, c)


def test_c_abi_exports_every_declared_symbol():
    """libcfb200.so loads without a GPU and exports every function include/cfb200.h declares."""
    from centrifuge_b200 import build
    build.build()
    lib = C.CDLL(os.path.join(util.ROOT, "centrifuge_b200", "libcfb200.so"))
    with open(os.path.join(util.ROOT, "include", "cfb200.h")) as f:
        hdr = f.read()
    names = sorted(set(re.findall(r"\b(cfb_[a-z_0-9]+)\s*\(", hdr)))
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), n


def test_product_loader_host_only(adv_base):
    """cfb_index_load(device=-1) parses the .cf files; classify entry points refuse without a GPU."""
    from centrifuge_b200 import capi
    ix = capi.Index(adv_base, device=-1)
    assert ix.info.line_rate == 7 and ix.info.ftab_chars == 10 and ix.info.sample_bytes == 2
    assert ix.info.compressed == 1 and ix.info.n_seqs == 20
    assert ix.seq_name(0) == "cid0" and ix.seq_taxid(3) == 1003
    assert ix.tax_node(1003)[0] == 103 and ix.tax_node(99999) is None
    with pytest.raises(capi.CfbError):
        capi.Context(ix)
    ix.close()


@pytest.mark.gpu      # the index comes from the product's builder
@pytest.mark.parametrize("kind", ["too_many", "too_few", "space", "control", "plus_one"])
def test_oracle_reader_rejects_what_the_reference_rejects(kind, tmp_path):
    """FASTQ quality-string rules (pat.cpp:1042-1078): same message and a failing exit status, or the same output."""
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    reads = util.synth.sample_reads(seqs, 300, 80, seed=9)
    fq = str(tmp_path / "q.fq")
    with open(fq, "wb") as f:
        for i, (name, a) in enumerate(reads):
            q = b"F" * len(a)
            if i == 200:
                q = {"too_many": q + b"FF", "too_few": q[:-1], "space": q[:10] + b" " + q[11:], "control": q[:10] + b"\x1f" + q[11:], "plus_one": q + b"F"}[kind]
            f.write(b"@" + name.encode() + b"\n" + a.tobytes() + b"\n+\n" + q + b"\n")
    r = util.reference_run("class", ["-q", "-x", base, "-U", fq], str(tmp_path))
    outs = [(r["rc"] != 0, r["errors"], r["outputs"][0] if r["rc"] == 0 else None)]
    p = subprocess.run([util.ORACLE_BIN, "-q", "-x", base, "-U", fq, "-S", str(tmp_path / "o.tsv"), "--report-file", str(tmp_path / "o.rep")],
                       stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    outs.append((p.returncode != 0, util.error_lines(p.stderr), util.file_digest(tmp_path / "o.tsv") if p.returncode == 0 else None))
    assert outs[0] == outs[1]
    assert outs[0][0] == (kind != "plus_one")
