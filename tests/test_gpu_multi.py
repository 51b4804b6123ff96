"""Per-taxon counters on the device and the path's one collective (SURVEY.md 8e): the NCCL all-reduce of those counters.

One-GPU cases run everywhere (a communicator of size 1 still goes through NCCL); the two-GPU cases need
`gpurun --gpus 2` and skip on a single-GPU box.  All comparisons are exact (integers, bytes)."""
import os
import subprocess

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

EXE = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")


def capi():
    from centrifuge_b200 import capi as m
    return m


def n_devices():
    import ctypes as C
    return int(capi().lib().cfb_device_count())


def fastq_bytes(reads):
    return b"".join(b"@" + n.encode() + b"\n" + a.tobytes() + b"\n+\n" + b"I" * len(a) + b"\n" for n, a in reads)


@pytest.fixture(scope="module")
def syn():
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    reads = [(n, a) for n, a in util.synth.sample_reads(seqs, 20000, 100, seed=61, lens=(40, 160)) if len(a) > 0]
    return base, reads


def text_counts(ctx, reads, slot=0):
    m = capi()
    txt = np.frombuffer(fastq_bytes(reads), dtype=np.uint8).copy()
    ctx.text_submit(slot, txt, None, len(reads))
    r = ctx.text_wait(slot)
    assert not r["irregular"]
    return r


def test_record_path_counters_equal_text_path_counters(syn):
    """k_fold_counts (records of cfb_classify_*) == the counters the text operator keeps (k_fmt_plan) == a host fold."""
    base, reads = syn
    m = capi()
    ix = m.Index(base, 0)
    a = m.Context(ix); b = m.Context(ix)
    text_counts(a, reads)
    want = a.counts_dense()
    bt = util.Batch([x for _, x in reads])
    b.count_records(True)
    off, recs = b.classify(m.make_batch(bt.bases, bt.off1, bt.len1, None, None, (bt.flags & 1).astype(np.uint8)))
    got = b.counts_dense()
    assert np.array_equal(got, want)
    taxids = b.counts_taxids()
    assert np.array_equal(taxids, a.counts_taxids()) and np.all(np.diff(taxids.astype(np.int64)) > 0)
    # host fold of the same records (tests/ restatement of addSpeciesCounts)
    from centrifuge_b200.abundance import taxon_counts
    host = taxon_counts(taxids, off, recs, k=5)
    # (taxid 0 collects the unclassified units on the device; the host fold keeps them in its extra last row)
    cls = taxids != 0
    assert np.array_equal(host[:-1, 0][cls].astype(np.uint64), want[0][cls]) and np.array_equal(host[:-1, 1][cls].astype(np.uint64), want[1][cls])
    assert int(want[0][~cls].sum()) == int((np.diff(off.astype(np.int64)) == 0).sum())
    # a second batch accumulates; reset clears
    b.classify(m.make_batch(bt.bases, bt.off1, bt.len1, None, None, (bt.flags & 1).astype(np.uint8)))
    assert np.array_equal(b.counts_dense(), 2 * want)
    b.counts_reset()
    assert int(b.counts_dense().sum()) == 0
    a.close(); b.close(); ix.close()


def test_allreduce_on_a_communicator_of_one(syn):
    """NCCL is loaded and the collective runs even on one GPU (ncclCommInitAll over one device)."""
    base, reads = syn
    m = capi()
    ix = m.Index(base, 0)
    ctx = m.Context(ix)
    text_counts(ctx, reads[:5000])
    m.comm_init_all([ctx])
    m.counts_allreduce_all([ctx])
    assert np.array_equal(ctx.counts_dense(global_=True), ctx.counts_dense())
    # a context without communicator: the reduced totals are the local ones
    c2 = m.Context(ix)
    text_counts(c2, reads[:5000])
    c2.counts_allreduce()
    assert np.array_equal(c2.counts_dense(global_=True), ctx.counts_dense())
    ctx.close(); c2.close(); ix.close()


def test_read_files_are_separate_pattern_sources(syn, tmp_path):
    """Centrifuge runs its inputs one file (pair) at a time (centrifuge.cpp:3006-3046): unnamed reads of a second -U file
    are numbered from 0 again, the report covers all files, and -1/-2 lists must match file by file."""
    base, reads = syn
    rd = reads[:900]
    fa, fb = str(tmp_path / "a.fq"), str(tmp_path / "b.fq")
    with open(fa, "wb") as f:
        f.write(fastq_bytes(rd[:500]))
    with open(fb, "wb") as f:                                   # unnamed reads: their ids come from the file's own record counter
        f.write(b"".join(b"@\n" + a.tobytes() + b"\n+\n" + b"I" * len(a) + b"\n" for _, a in rd[500:]))
    for extra in ([], ["--host-parse"]):
        args = ["-q", "-x", base, "-U", fa + "," + fb] + extra
        want = util.reference_cli(args[:5], tmp_path)
        got = util.run_cli(EXE, args, str(tmp_path / "o.tsv"), str(tmp_path / "o.rep"))
        assert util.digests(got) == want, extra
    m1 = [(n, a) for n, a in rd[:600]]; m2 = [(n, a[::-1].copy()) for n, a in rd[:600]]
    paths = {}
    for tag, lst, cut in (("a", m1, 250), ("b", m2, 400)):      # the -1 list is cut after 250 records, the -2 list after 400
        for k, part in enumerate((lst[:cut], lst[cut:])):
            paths[tag, k] = str(tmp_path / ("%s%d.fq" % (tag, k)))
            with open(paths[tag, k], "wb") as f:
                f.write(fastq_bytes(part))
    args = ["-q", "-x", base, "-1", paths["a", 0] + "," + paths["a", 1], "-2", paths["b", 0] + "," + paths["b", 1]]
    r = util.reference_run("class", args, str(tmp_path / "ref"))
    assert r["rc"] != 0 and any("fewer reads in file specified with -1" in l for l in r["errors"]), r
    p = subprocess.run([EXE] + args + ["-S", str(tmp_path / "x.tsv"), "--report-file", str(tmp_path / "x.rep")], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    assert p.returncode != 0 and b"fewer reads in file specified with -1" in p.stderr
    # equal cuts: two file pairs, one after the other
    for tag, lst in (("c", m1), ("d", m2)):
        for k, part in enumerate((lst[:300], lst[300:])):
            paths[tag, k] = str(tmp_path / ("%s%d.fq" % (tag, k)))
            with open(paths[tag, k], "wb") as f:
                f.write(fastq_bytes(part))
    args = ["-q", "-x", base, "-1", paths["c", 0] + "," + paths["c", 1], "-2", paths["d", 0] + "," + paths["d", 1], "-U", fb]
    want = util.reference_cli(args, tmp_path)
    got = util.run_cli(EXE, args, str(tmp_path / "o2.tsv"), str(tmp_path / "o2.rep"))
    assert util.digests(got) == want


@pytest.mark.skipif(n_devices() < 2, reason="needs two GPUs (gpurun --gpus 2)")
def test_two_gpu_cli_output_is_byte_identical_to_one_gpu(syn, tmp_path):
    """`centrifuge-class --devices 0,1`: spans dealt round-robin, rows in input order, counters reduced over NCCL:
    classification TSV, report TSV (abundance EM included) and Kraken-style report equal the one-GPU run's bytes."""
    base, reads = syn
    fq = str(tmp_path / "r.fq")
    with open(fq, "wb") as f:
        f.write(fastq_bytes(reads))
    outs = []
    for tag, extra in (("one", ["--device", "0"]), ("two", ["--devices", "0,1"]), ("swap", ["--devices", "1,0"])):
        env = dict(os.environ, CFB_TEXT_BLOCK="100000", CFB_TEXT_STATS="1")
        p = subprocess.run([EXE, "-q", "-x", base, "-U", fq, "-S", str(tmp_path / (tag + ".tsv")), "--report-file", str(tmp_path / (tag + ".rep")),
                            "--kreport-file", str(tmp_path / (tag + ".kr"))] + extra, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
        assert p.returncode == 0, p.stderr.decode()
        if tag != "one":
            assert b"devices, per-taxon counters reduced with NCCL" in p.stderr
        outs.append(tuple(open(str(tmp_path / (tag + ext)), "rb").read() for ext in (".tsv", ".rep", ".kr")))
    assert outs[0] == outs[1] == outs[2]
    assert util.digests(outs[1][:2]) == util.reference_cli(["-q", "-x", base, "-U", fq], tmp_path)


@pytest.mark.skipif(n_devices() < 2, reason="needs two GPUs (gpurun --gpus 2)")
def test_two_gpu_allreduce_sums_the_shards(syn):
    base, reads = syn
    m = capi()
    ixs = [m.Index(base, d) for d in (0, 1)]
    ctxs = [m.Context(ix) for ix in ixs]
    half = len(reads) // 2
    text_counts(ctxs[0], reads[:half]); text_counts(ctxs[1], reads[half:])
    loc = [c.counts_dense() for c in ctxs]
    m.comm_init_all(ctxs)
    m.counts_allreduce_all(ctxs)
    for c in ctxs:
        assert np.array_equal(c.counts_dense(global_=True), loc[0] + loc[1])
    whole = m.Context(ixs[0])
    text_counts(whole, reads)
    assert np.array_equal(whole.counts_dense(), loc[0] + loc[1])
    for c in ctxs + [whole]:
        c.close()
    for ix in ixs:
        ix.close()
