"""GPU suite for the index builder: cfb_build_index must write the bytes centrifuge-build-bin writes."""
import os

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu


def capi():
    from centrifuge_b200 import capi as m
    return m


def ref_build(fa, conv, nodes, names, base):
    """digests of the .1-.4.cf files centrifuge-build-bin writes (recorded reference run)"""
    r = util.reference_run("build", ["-p", "4", "--conversion-table", conv, "--taxonomy-tree", nodes, "--name-table", names, fa], base)
    assert r["rc"] == 0, r
    return r["outputs"]


def assert_same_index(want, b):
    """`want`: digests of the reference's .1-.4.cf files.  To see where a file differs, record the run again
    (CFB_RECORD_REFERENCE, tests/util.py): the reference's files are then written beside the product's."""
    for k, w in zip("1234", want):
        f = "%s.%s.cf" % (b, k)
        assert util.file_digest(f) == w, ".%s.cf (%d bytes) differs from the reference's" % (k, os.path.getsize(f))


def test_builder_matches_reference_adversarial(tmp_path):
    m = capi()
    d = str(tmp_path)
    util.synth.write_adversarial(d, seed=33, n_reads=10)
    want = ref_build(d + "/genomes.fa", d + "/conv.tsv", d + "/nodes.dmp", d + "/names.dmp", d + "/ref")
    m.build_index(m.build_opts(d + "/mine", fasta=[d + "/genomes.fa"], conversion_table=d + "/conv.tsv", taxonomy_tree=d + "/nodes.dmp", name_table=d + "/names.dmp"))
    assert_same_index(want, d + "/mine")


def test_builder_matches_reference_gaps_descriptions_multifile(tmp_path):
    """Ns / IUPAC gaps at the start, middle and end of sequences, header descriptions, two FASTA files."""
    m = capi()
    d = str(tmp_path)
    rng = np.random.default_rng(9)
    A = util.synth.ACGT

    def rnd(n):
        return A[rng.integers(0, 4, n)].tobytes().decode()
    with open(d + "/a.fa", "w") as f:
        f.write(">s0 first sequence with description\n" + rnd(3000) + "\n")
        f.write(">gi|123|ref|NC_1| piped name\n" + "NNNNN" + rnd(1500) + "NNNNNNNNNNNNNNNNNNNN" + rnd(2500) + "\n")
        f.write(">s2\n" + rnd(700) + "RYKM" + rnd(900) + "NNN\n")
    with open(d + "/b.fa", "w") as f:
        s = rnd(5000)
        f.write(">s3\n" + "\n".join(s[i:i + 60] for i in range(0, len(s), 60)) + "\n")
        f.write(">s4 x\n" + rnd(40) + "\n")
    with open(d + "/conv.tsv", "w") as f:
        f.write("s0\t1000\ngi|123\t1001\ns2\t1002\ns3\t1003\ns4\t1000\n")
    with open(d + "/nodes.dmp", "w") as f:
        f.write("1\t|\t1\t|\tno rank\t|\n100\t|\t1\t|\tgenus\t|\n")
        for t in range(4):
            f.write("%d\t|\t100\t|\tspecies\t|\n" % (1000 + t))
    with open(d + "/names.dmp", "w") as f:
        f.write("1\t|\troot\t|\t\t|\tscientific name\t|\n100\t|\tSome genus\t|\t\t|\tscientific name\t|\n1001\t|\tSp one two\t|\t\t|\tscientific name\t|\n")
    want = ref_build(d + "/a.fa," + d + "/b.fa", d + "/conv.tsv", d + "/nodes.dmp", d + "/names.dmp", d + "/ref")
    m.build_index(m.build_opts(d + "/mine", fasta=[d + "/a.fa", d + "/b.fa"], conversion_table=d + "/conv.tsv", taxonomy_tree=d + "/nodes.dmp", name_table=d + "/names.dmp"))
    assert_same_index(want, d + "/mine")


def test_builder_synthetic_mode_matches_reference(tmp_path):
    """Counter-based synthetic genomes built on the device == the same genomes as FASTA through the reference."""
    m = capi()
    d = str(tmp_path)
    conv, nodes, names = m.write_synth_taxonomy(d, 4, 5, 30000)
    o = m.build_opts(d + "/mine", synth=(4, 5, 30000, 77, 0.03), conversion_table=conv, taxonomy_tree=nodes, name_table=names)
    m.synth_fasta(o, d + "/g.fa")
    want = ref_build(d + "/g.fa", conv, nodes, names, d + "/ref")
    m.build_index(o)
    assert_same_index(want, d + "/mine")
    # reads sampled from the same generator classify to their source species
    codes = m.synth_reads(o, 2000, 100, 5)
    assert codes.shape == (2000, 100) and codes.max() <= 4


def test_builder_many_sequences_wide_sample(tmp_path):
    m = capi()
    d = str(tmp_path)
    rng = np.random.default_rng(10)
    n, L = 66000, 64
    g = rng.integers(0, 4, size=(n, L), dtype=np.uint8)
    A = util.synth.ACGT
    with open(d + "/g.fa", "wb") as f:
        for i in range(n):
            f.write(b">c%d\n" % i + A[g[i]].tobytes() + b"\n")
    with open(d + "/conv.tsv", "w") as f:
        for i in range(n):
            f.write("c%d\t%d\n" % (i, 1000 + i % 7))
    with open(d + "/nodes.dmp", "w") as f:
        f.write("1\t|\t1\t|\tno rank\t|\n")
        for t in range(7):
            f.write("%d\t|\t1\t|\tspecies\t|\n" % (1000 + t))
    with open(d + "/names.dmp", "w") as f:
        f.write("1\t|\troot\t|\t\t|\tscientific name\t|\n")
    want = ref_build(d + "/g.fa", d + "/conv.tsv", d + "/nodes.dmp", d + "/names.dmp", d + "/ref")
    m.build_index(m.build_opts(d + "/mine", fasta=[d + "/g.fa"], conversion_table=d + "/conv.tsv", taxonomy_tree=d + "/nodes.dmp", name_table=d + "/names.dmp"))
    assert_same_index(want, d + "/mine")


def test_bench_data_path_matches_reference_end_to_end(tmp_path):
    """The exact pipeline bench.py times -- index from cfb_build_index (synthetic mode), reads from
    cfb_synth_reads, classification through the drop-in CLI -- equals the unmodified reference binary
    run on the same index files and reads, byte for byte (TSV and report)."""
    import sys
    sys.path.insert(0, util.ROOT)
    import bench
    m = capi()
    d = str(tmp_path)
    g, s, L = 12, 5, 400000
    tax = m.write_synth_taxonomy(d, g, s, L)
    o = m.build_opts(d + "/idx", synth=(g, s, L, 4242, 0.03), conversion_table=tax[0], taxonomy_tree=tax[1], name_table=tax[2])
    m.build_index(o)
    exe = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")
    # bench.py's three workloads: fixed-length SE, mixed-length SE, paired (its own generator and FASTQ writer)
    for tag, lens, paired in (("se", (100, 100), False), ("mixed", (75, 300), False), ("pe", (150, 150), True)):
        codes, ln = m.synth_reads_ex(o, 20000, 17, lens[0], lens[1], paired=paired)
        rd = bench.Reads(codes, ln)
        files = [d + "/%s_%d.fq" % (tag, k + 1) for k in range(rd.mates)]
        bench.write_fastq_files(rd, files)
        rargs = ["-q", "-x", d + "/idx"] + (["-1", files[0], "-2", files[1]] if paired else ["-U", files[0]])
        a = util.reference_cli(rargs, tmp_path)
        b = util.run_cli(exe, rargs + ["--batch-units", "7000"], d + "/b.tsv", d + "/b.rep")
        assert a[0] == util.digest(b[0]), tag
        assert a[1] == util.digest(b[1]), tag
        rows = b[0].decode().strip().split("\n")[1:]
        assert sum(1 for r in rows if "unclassified" not in r) > 15000, tag      # the synthetic reads do classify
