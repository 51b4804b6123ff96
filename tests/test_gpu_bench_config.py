"""GPU suite, part 2: parity at the configurations BASELINE.json names.

  configs[0]  the reference's own known-answer fixture (example/index + example/reads, MANUAL.markdown:1586-1603)
  configs[1]  the index bench.py measures on -- 9 Gbp / 4.1 GB, "compressed" (cid names), every derived table live
              (K = 15 jump table, resolve table, walk8), SA rows beyond 2^32 -- through the C ABI against the oracle and
              through the drop-in CLI (CFB_FULL_TABLES=1) against the unmodified reference binary
  configs[3]  class: > 65 535 sequences at multi-Gbp scale (u32 SA sample, u32 resolve table)

The big indexes are built on the GPU by the product's own builder (byte-identical to centrifuge-build-bin,
tests/test_gpu_build.py) because nothing else can produce them here; CFB_TEST_SKIP_BIG=1 skips them.
"""
import os
import subprocess

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

EXE = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")
BIG = pytest.mark.skipif(os.environ.get("CFB_TEST_SKIP_BIG") == "1", reason="CFB_TEST_SKIP_BIG=1")


def capi():
    from centrifuge_b200 import capi as m
    return m


def synth_index(tag, genera, species, length, seed=12345, prefix="cid"):
    m = capi()
    d = os.path.join(util.CACHE, "%s_g%d_s%d_l%d_%s" % (tag, genera, species, length, prefix))
    base = os.path.join(d, "idx")
    if not os.path.exists(os.path.join(d, "done")):
        os.makedirs(d, exist_ok=True)
        tax = m.write_synth_taxonomy(d, genera, species, length, prefix=prefix)
        m.build_index(m.build_opts(base, synth=(genera, species, length, seed, 0.03), conversion_table=tax[0], taxonomy_tree=tax[1], name_table=tax[2],
                                   synth_prefix=prefix))
        open(os.path.join(d, "done"), "w").close()
    return base, m.build_opts(None, synth=(genera, species, length, seed, 0.03), synth_prefix=prefix)


def write_fastq(path, codes):
    asc = np.frombuffer(b"ACGTN", dtype=np.uint8)[codes]
    n, L = asc.shape
    rec = np.empty((n, 2 + 9 + 1 + L + 3 + L + 1), dtype=np.uint8)
    rec[:, 0] = ord("@"); rec[:, 1] = ord("r")
    idx = np.arange(n, dtype=np.int64)
    rec[:, 2:11] = (idx[:, None] // (10 ** np.arange(8, -1, -1, dtype=np.int64))[None, :] % 10 + 48).astype(np.uint8)
    rec[:, 11] = 10; rec[:, 12:12 + L] = asc; rec[:, 12 + L] = 10; rec[:, 13 + L] = ord("+"); rec[:, 14 + L] = 10
    rec[:, 15 + L:15 + 2 * L] = ord("I"); rec[:, 15 + 2 * L] = 10
    with open(path, "wb") as f:
        f.write(rec.tobytes())


def abi_vs_oracle(base, codes, expect_tables):
    """records of cfb_classify_batch on the fully-tabled replica == the oracle's, unit by unit"""
    m = capi()
    n, L = codes.shape
    flags = ((codes == 4).sum(axis=1) <= int(0.15 * L)).astype(np.uint8)
    lens = np.full(n, L, dtype=np.uint32); offs = np.arange(n, dtype=np.uint64) * np.uint64(L)
    bases = np.ascontiguousarray(codes.reshape(-1))
    ix = m.Index(base, 0)
    tb = ix.tables()
    for k, want in expect_tables.items():
        assert (tb[k] > 0) == want if isinstance(want, bool) else tb[k] == want, (k, tb)
    ctx = m.Context(ix)
    off, recs = ctx.classify(m.make_batch(bases, offs, lens, None, None, flags))
    ctx.close(); ix.close()
    o = util.Oracle(base)
    b = util.Batch([])
    b.n, b.paired, b.bases, b.off1, b.len1, b.flags = n, False, bases, offs, lens, flags
    b.off2 = np.zeros(n, dtype=np.uint64); b.len2 = np.zeros(n, dtype=np.uint32)
    on, orec, _ = o.classify(b, util.make_oparams())
    o.close()
    assert np.array_equal(np.diff(off.astype(np.int64)), on.astype(np.int64))
    assert len(orec) == len(recs)
    for f in ("taxid", "score", "hitlen", "uid"):
        assert np.array_equal(orec[f], recs[f]), f
    return tb


def test_manual_example_fixture_on_gpu(tmp_path):
    """BASELINE configs[0]: the reference's known-answer fixture through the drop-in CLI and the C ABI."""
    base, reads = util.golden_index("example"), os.path.join(util.GOLDEN, "example.reads.fa")
    for extra in ([], ["--host-parse"]):              # text operator and record-level reader
        tsv, rep = util.run_cli(EXE, ["-f", "-x", base, "-U", reads] + extra, str(tmp_path / "g.tsv"), str(tmp_path / "g.rep"))
        with open(os.path.join(util.GOLDEN, "example.tsv"), "rb") as f:
            assert tsv == f.read()
        with open(os.path.join(util.GOLDEN, "example.report.tsv"), "rb") as f:
            assert rep == f.read()
    m = capi()
    rd = util.parse_reads(reads)
    b = util.Batch([a for _, a in rd])
    ix = m.Index(base, 0); ctx = m.Context(ix)
    off, recs = ctx.classify(m.make_batch(b.bases, b.off1, b.len1, None, None, (b.flags & 1).astype(np.uint8)))
    o = util.Oracle(base)
    on, orec, _ = o.classify(b, util.make_oparams())
    assert np.array_equal(np.diff(off.astype(np.int64)), on.astype(np.int64))
    for f in ("taxid", "score", "hitlen", "uid"):
        assert np.array_equal(orec[f], recs[f]), f
    o.close(); ctx.close(); ix.close()


@BIG
def test_bench_configuration_all_tables_matches_oracle_and_reference(tmp_path):
    """The exact device configuration bench.py times: 9 Gbp compressed index, K = 15, resolve table, walk8, rows > 2^32."""
    m = capi()
    base, so = synth_index("bench", 900, 10, 1000000)
    codes = m.synth_reads(so, 200000, 100, 4242)
    tb = abi_vs_oracle(base, codes, {"ftabk_chars": 15, "resolve_table_bytes": True, "walk8_bytes": True, "resolve_entry_bytes": 2})
    assert tb["walk8_bytes"] > 8 * (1 << 32)                    # entries of rows beyond 2^32 exist (and uniform reads land on them)
    ix = m.Index(base, -1)
    assert ix.info.compressed == 1 and ix.info.len > (1 << 32)
    ix.close()
    fq = str(tmp_path / "r.fq")
    write_fastq(fq, codes)
    ref = util.reference_cli(["-q", "-x", base, "-U", fq, "-p", "16", "--reorder"], tmp_path)
    env = dict(os.environ, CFB_FULL_TABLES="1")
    subprocess.check_call([EXE, "-q", "-x", base, "-U", fq, "-S", str(tmp_path / "b.tsv"), "--report-file", str(tmp_path / "b.rep")],
                          env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    assert util.file_digest(tmp_path / "b.tsv") == ref[0]
    assert util.file_digest(tmp_path / "b.rep") == ref[1]


@BIG
def test_many_sequence_multi_gbp_index_matches_oracle():
    """> 65 535 sequences at 7 Gbp: u32 SA sample and u32 resolve table (bt2_io.h:280), all tables live."""
    m = capi()
    base, so = synth_index("wide", 7000, 10, 100000)
    codes = m.synth_reads(so, 100000, 100, 777)
    abi_vs_oracle(base, codes, {"resolve_table_bytes": True, "walk8_bytes": True, "resolve_entry_bytes": 4})
