"""GPU suite (-m gpu): every call goes through the C ABI of libcfb200.so; the oracle is the checker."""
import lzma
import os
import subprocess

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

PARAM_CASES = {
    "default": {}, "k1": dict(k=1), "k50": dict(k=50), "minhit15": dict(min_hitlen=15),
    "host": dict(host=(100, 1005), k=2), "excl": dict(excl=(10,)), "family": dict(rank_slot=3), "notraverse": dict(traverse=False),
}
GOLDEN_CLI = {
    "default": [], "k1": ["-k", "1"], "host": ["--host-taxids", "100,1005", "-k", "2"],
    "family": ["--classification-rank", "family"], "minhit15": ["--min-hitlen", "15"],
}


def capi():
    from centrifuge_b200 import capi as m
    return m


def to_cbatch(b):
    m = capi()
    if b.paired:
        fl = (b.flags & 3).astype(np.uint8)
        return m.make_batch(b.bases, b.off1, b.len1, b.off2, b.len2, fl)
    return m.make_batch(b.bases, b.off1, b.len1, None, None, (b.flags & 1).astype(np.uint8))


def gpu_classify(base, batch, **kw):
    m = capi()
    ix = m.Index(base, 0)
    ctx = m.Context(ix, m.make_params(**kw))
    off, recs = ctx.classify(to_cbatch(batch))
    ctx.close(); ix.close()
    return np.diff(off.astype(np.int64)).astype(np.uint32), recs


def assert_same(on, orec, gn, grec):
    assert np.array_equal(on, gn), "per-unit record counts differ at units %s" % np.nonzero(on != gn)[0][:10]
    assert len(orec) == len(grec)
    for f in ("taxid", "score", "hitlen", "uid"):
        assert np.array_equal(orec[f], grec[f]), f


def test_cooperative_lf_and_resolve_primitives(adv_base):
    """8-lane side fetch + popcount rank + shuffle reduce == scalar LF of the oracle on random rows."""
    import ctypes as C
    m = capi()
    ix = m.Index(adv_base, 0)
    o = util.Oracle(adv_base)
    n_rows = int(ix.info.len) + 1
    rng = np.random.default_rng(1)
    rows = rng.integers(0, n_rows, size=20000).astype(np.uint64)
    rows[:400] = np.arange(400)                               # first side, incl. side boundaries
    rows[400:800] = np.arange(n_rows - 400, n_rows)           # last side
    chars = rng.integers(0, 5, size=len(rows)).astype(np.uint8)   # 4 => use BWT[row]
    got = m.test_lf(ix, rows, chars)
    o.lib.cfo_lf.restype = C.c_uint64
    o.lib.cfo_bwt_char.restype = C.c_int
    for i in range(len(rows)):
        c = int(chars[i])
        if c > 3:
            c = o.lib.cfo_bwt_char(C.c_void_p(o.h), C.c_uint64(int(rows[i])))
        exp = o.lib.cfo_lf(C.c_void_p(o.h), C.c_uint64(int(rows[i])), C.c_int(c))
        assert int(got[i]) == exp, (i, int(rows[i]), c)
    o.lib.cfo_resolve.restype = C.c_uint64
    got = m.test_resolve(ix, rows[:6000])
    for i in range(6000):
        assert int(got[i]) == o.lib.cfo_resolve(C.c_void_p(o.h), C.c_uint64(int(rows[i])), None), i
    o.close(); ix.close()


@pytest.mark.parametrize("case", sorted(PARAM_CASES))
def test_classify_matches_oracle_adversarial(case, adv_base, adv_reads):
    reads = util.parse_reads(adv_reads)
    b = util.Batch([a for _, a in reads])
    o = util.Oracle(adv_base)
    on, orec, _ = o.classify(b, util.make_oparams(**PARAM_CASES[case]))
    gn, grec = gpu_classify(adv_base, b, **PARAM_CASES[case])
    assert_same(on, orec, gn, grec)
    o.close()


LAYOUT_VARIANTS = {
    "no_walk8": {"CFB_WALK8": "0"},
    "no_ftabd": {"CFB_FTABD": "0"},
    "ftabd_over_ftabk12": {"CFB_FTABK": "12"},
    "half_walk8": {"CFB_WALK8_ROWS": "300000"},
    "range_jump_w1": {"CFB_JUMP_W": "1"},
    "every_hit_stored": {"CFB_KEEP_SHORT": "1"},
    "tiny_regeneration_buffer": {"CFB_REGEN_SLOTS": "8"},      # both-strand reads overflow the side buffer: grow and re-run
    "range_jump_w8_half_walk8": {"CFB_JUMP_W": "8", "CFB_WALK8_ROWS": "300000"},
    "no_tables": {"CFB_WALK8": "0", "CFB_RESOLVE_TABLE": "0", "CFB_FTABK": "10", "CFB_FTABD": "0"},
    "ftabk11": {"CFB_FTABK": "11"},
    "ftabk12_walk_resolve": {"CFB_FTABK": "12", "CFB_RESOLVE_TABLE": "0"},
    "coop8": {"CFB_GROUP": "8", "CFB_LEGACY_LAYOUTS": "1"},
    "tiny_row_buffer": {"CFB_ROWS_CAP": "64"},          # every batch overflows the row buffer once and re-runs from the row stage
}


@pytest.mark.parametrize("variant", sorted(LAYOUT_VARIANTS))
def test_every_device_layout_gives_the_same_records(variant, adv_base, adv_reads, monkeypatch):
    """The derived tables (K-mer jump table, resolve table, walk8) and the kernel variants are pure
    accelerations: with any of them switched off the records are the oracle's as well."""
    for k, v in LAYOUT_VARIANTS[variant].items():
        monkeypatch.setenv(k, v)
    reads = util.parse_reads(adv_reads)
    b = util.Batch([a for _, a in reads])
    o = util.Oracle(adv_base)
    on, orec, _ = o.classify(b, util.make_oparams())
    gn, grec = gpu_classify(adv_base, b)
    assert_same(on, orec, gn, grec)
    o.close()
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    o = util.Oracle(base)
    rd = util.synth.sample_reads(seqs, 6000, 100, seed=77, lens=(30, 300))
    b = util.Batch([a for _, a in rd])
    on, orec, _ = o.classify(b, util.make_oparams())
    gn, grec = gpu_classify(base, b)
    assert_same(on, orec, gn, grec)
    o.close()


@pytest.mark.parametrize("lens", [(100, 128), (129, 160), (150, 150), (161, 320), (300, 700)])
def test_every_read_length_class_matches_oracle(lens):
    """The search kernel is instantiated per read-length class (register words holding the packed read)."""
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    o = util.Oracle(base)
    rd = util.synth.sample_reads(seqs, 5000, lens[0], seed=lens[0] + lens[1], lens=lens)
    b = util.Batch([a for _, a in rd])
    on, orec, _ = o.classify(b, util.make_oparams())
    gn, grec = gpu_classify(base, b)
    assert_same(on, orec, gn, grec)
    o.close()


def test_classify_matches_oracle_synthetic_se_pe_mixed():
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    o = util.Oracle(base)
    rd = util.synth.sample_reads(seqs, 20000, 100, seed=21, lens=(30, 300))
    b = util.Batch([a for _, a in rd])
    for kw in ({}, dict(k=1), dict(rank_slot=2)):
        on, orec, _ = o.classify(b, util.make_oparams(**kw))
        gn, grec = gpu_classify(base, b, **kw)
        assert_same(on, orec, gn, grec)
    prs = util.synth.sample_pairs(seqs, 8000, 150, seed=22)
    m1 = [x for _, x, _ in prs]; m2 = [y for _, _, y in prs]
    for i in range(0, len(m2), 7):                          # filtered / very short mates
        m2[i] = np.full(len(m2[i]), ord("N"), dtype=np.uint8)
    for i in range(3, len(m1), 11):
        m1[i] = np.full(len(m1[i]), ord("N"), dtype=np.uint8)
    for i in range(5, len(m2), 13):
        m2[i] = m2[i][:1]
    bp = util.Batch(m1, m2)
    for kw in ({}, dict(k=2)):
        on, orec, _ = o.classify(bp, util.make_oparams(**kw))
        gn, grec = gpu_classify(base, bp, **kw)
        assert_same(on, orec, gn, grec)
    o.close()


def test_counters_match_host_logic(adv_base, adv_reads, monkeypatch):
    """Algorithmic-operation counters of the kernels == the same counters of the scalar logic."""
    monkeypatch.setenv("CFB_COUNT", "1")
    m = capi()
    reads = util.parse_reads(adv_reads)
    b = util.Batch([a for _, a in reads])
    h = util.HostLogic(adv_base)
    _, _, hst = h.classify(b, util.make_oparams())
    ix = m.Index(adv_base, 0); ctx = m.Context(ix, m.make_params())
    ctx.classify(to_cbatch(b))
    c = ctx.counters()
    assert c["partial_searches"] == hst[1] and c["ftab_probes"] == hst[2] and c["sides_search"] == hst[3]
    assert c["walk_steps"] == hst[4] and c["rows_resolved"] == hst[5] and c["ext_searches"] == hst[7]
    ctx.close(); ix.close(); h.close()


def test_pipelined_and_resident_paths_agree(adv_base, adv_reads):
    m = capi()
    reads = util.parse_reads(adv_reads)
    b = util.Batch([a for _, a in reads])
    cb = to_cbatch(b)
    ix = m.Index(adv_base, 0); ctx = m.Context(ix, m.make_params())
    off0, rec0 = ctx.classify(cb)
    for s in range(ctx.n_slots):
        ctx.submit(s, cb)
    for s in range(ctx.n_slots):
        off, rec = ctx.wait(s)
        assert np.array_equal(off, off0) and np.array_equal(rec, rec0)
    d = ctx.upload(cb)
    for _ in range(2):
        ms, nrec = ctx.classify_resident(d)
        assert nrec == len(rec0) and ms[4] > 0
    off, rec = ctx.resident_result()
    assert np.array_equal(off, off0) and np.array_equal(rec, rec0)
    assert ctx.launches() > 0
    ctx.close(); ix.close()


def test_empty_and_degenerate_batches(adv_base):
    m = capi()
    ix = m.Index(adv_base, 0); ctx = m.Context(ix, m.make_params())
    z = util.Batch([])
    off, rec = ctx.classify(m.make_batch(np.zeros(1, dtype=np.uint8), z.off1, z.len1, None, None, None))
    assert len(rec) == 0
    one = util.Batch([np.frombuffer(b"ACGT", dtype=np.uint8)])       # shorter than the ftab
    off, rec = ctx.classify(to_cbatch(one))
    assert list(off) == [0, 0]
    allf = util.Batch([np.frombuffer(b"N" * 60, dtype=np.uint8), np.frombuffer(b"A", dtype=np.uint8)])
    off, rec = ctx.classify(to_cbatch(allf))
    assert list(off) == [0, 0, 0]
    ctx.close(); ix.close()


@pytest.mark.parametrize("case", sorted(GOLDEN_CLI))
def test_cli_tsv_and_report_match_reference_golden(case, adv_base, adv_reads, tmp_path):
    """Drop-in check: the `centrifuge-class` replacement writes the reference's bytes."""
    exe = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")
    tsv, rep = util.run_cli(exe, ["-f", "-x", adv_base, "-U", adv_reads, "--batch-units", "700"] + GOLDEN_CLI[case],
                            str(tmp_path / "g.tsv"), str(tmp_path / "g.rep"))
    with lzma.open(os.path.join(util.GOLDEN, "adv.%s.tsv.xz" % case)) as f:
        assert tsv == f.read()
    with open(os.path.join(util.GOLDEN, "adv.%s.report.tsv" % case), "rb") as f:
        assert rep == f.read()


def test_cli_matches_live_reference_paired_fastq(tmp_path):
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    prs = util.synth.sample_pairs(seqs, 6000, 125, seed=31)
    f1, f2 = str(tmp_path / "p_1.fq"), str(tmp_path / "p_2.fq")
    util.synth.write_fastq(f1, [(n, x) for n, x, _ in prs])
    util.synth.write_fastq(f2, [(n, y) for n, _, y in prs], qual=b"5")
    exe = os.path.join(util.ROOT, "centrifuge_b200", "centrifuge-class")
    a = util.reference_cli(["-q", "-x", base, "-1", f1, "-2", f2], tmp_path)
    b = util.run_cli(exe, ["-q", "-x", base, "-1", f1, "-2", f2, "--batch-units", "1000"], str(tmp_path / "b.tsv"), str(tmp_path / "b.rep"))
    assert a == util.digests(b)


def test_large_batch_properties():
    """Size-independent properties at a size the oracle cannot sweep in seconds: results do not
    depend on batch composition (split / permutation invariance) and a random sample of units
    equals the oracle."""
    base = util.build_index("syn_big", 10, 10, 300000, seed=3)
    seqs = util.synth.make_genomes(10, 10, 300000, 3)
    rng = np.random.default_rng(5)
    n = 400000
    # vectorised read sampler (100 bp, 1% substitutions, random strand, 5% random reads)
    G = np.stack(seqs)
    si = rng.integers(0, len(seqs), n); pos = rng.integers(0, 300000 - 100, n)
    idx = pos[:, None] + np.arange(100)[None, :]
    R = G[si[:, None], idx]
    sub = rng.random((n, 100)) < 0.01
    R = np.where(sub, (R + 1) & 3, R).astype(np.uint8)
    rc = rng.random(n) < 0.5
    R[rc] = (3 - R[rc])[:, ::-1]
    rnd = rng.random(n) < 0.05
    R[rnd] = rng.integers(0, 4, size=(int(rnd.sum()), 100), dtype=np.uint8)
    bases = np.ascontiguousarray(R.reshape(-1))
    lens = np.full(n, 100, dtype=np.uint32); offs = (np.arange(n, dtype=np.uint64) * np.uint64(100))
    m = capi()
    ix = m.Index(base, 0); ctx = m.Context(ix, m.make_params())
    off_all, rec_all = ctx.classify(m.make_batch(bases, offs, lens))
    cnt_all = np.diff(off_all.astype(np.int64))
    # split invariance
    h = n // 2
    off_a, rec_a = ctx.classify(m.make_batch(bases[:h * 100].copy(), offs[:h].copy(), lens[:h].copy()))
    off_b, rec_b = ctx.classify(m.make_batch(bases[h * 100:].copy(), offs[:n - h].copy(), lens[h:].copy()))
    assert np.array_equal(np.concatenate([rec_a, rec_b]), rec_all)
    # permutation invariance (units permuted through the offset table only)
    perm = rng.permutation(n)
    off_p, rec_p = ctx.classify(m.make_batch(bases, offs[perm].copy(), lens[perm].copy()))
    cnt_p = np.diff(off_p.astype(np.int64))
    assert np.array_equal(cnt_p, cnt_all[perm])
    chk = np.zeros(n, dtype=np.uint64); chk_p = np.zeros(n, dtype=np.uint64)
    key = rec_all["taxid"] * np.uint64(1000003) + rec_all["score"].astype(np.uint64) * np.uint64(7) + rec_all["uid"].astype(np.uint64)
    np.add.at(chk, np.repeat(np.arange(n), cnt_all), key)
    key_p = rec_p["taxid"] * np.uint64(1000003) + rec_p["score"].astype(np.uint64) * np.uint64(7) + rec_p["uid"].astype(np.uint64)
    np.add.at(chk_p, np.repeat(np.arange(n), cnt_p), key_p)
    assert np.array_equal(chk_p, chk[perm])
    # oracle on a sample
    samp = np.sort(rng.choice(n, 5000, replace=False))
    sb = util.Batch([util.synth.ACGT[R[i]] for i in samp])
    o = util.Oracle(base)
    on, orec, _ = o.classify(sb, util.make_oparams())
    assert np.array_equal(on.astype(np.int64), cnt_all[samp])
    got = np.concatenate([rec_all[off_all[i]:off_all[i + 1]] for i in samp]) if len(orec) else rec_all[:0]
    for f in ("taxid", "score", "hitlen", "uid"):
        assert np.array_equal(orec[f], got[f]), f
    o.close(); ctx.close(); ix.close()


def test_packed_input_gives_the_same_records():
    """cfb_classify_submit_packed (2-bit words + N list + lengths) == cfb_classify_batch (1 byte per base), SE and PE,
    ragged lengths incl. empty reads, reads that are all N, lengths on and off the 32-base word boundary."""
    m = capi()
    base = util.build_index("syn_a", 5, 4, 60000, seed=7, strains=True)
    seqs = util.synth.make_genomes(5, 4, 60000, 7)
    rd = [a for _, a in util.synth.sample_reads(seqs, 9000, 100, seed=71, lens=(1, 300), nrate=0.01)]
    rd[5] = rd[5][:0]; rd[6] = np.full(64, ord("N"), dtype=np.uint8); rd[7] = rd[7][:32] if len(rd[7]) >= 32 else rd[7]; rd[8] = np.full(33, ord("N"), dtype=np.uint8)
    ix = m.Index(base, 0); ctx = m.Context(ix)
    b = util.Batch(rd)
    cb = to_cbatch(b)
    off0, rec0 = ctx.classify(cb)
    words, npos = m.pack_batch(cb)
    assert len(words) == int(((b.len1.astype(np.int64) + 31) // 32).sum()) and len(npos) == int((b.bases > 3).sum())
    ctx.submit_packed(1, m.make_batch_packed(words, b.len1, None, npos, (b.flags & 1).astype(np.uint8)))
    off1, rec1 = ctx.wait(1)
    assert np.array_equal(off0, off1) and np.array_equal(rec0, rec1)
    prs = util.synth.sample_pairs(seqs, 4000, 150, seed=72)
    m1 = [x for _, x, _ in prs]; m2 = [y[: max(0, len(y) - (i % 50))] for i, (_, _, y) in enumerate(prs)]
    bp = util.Batch(m1, m2)
    cbp = to_cbatch(bp)
    off0, rec0 = ctx.classify(cbp)
    words, npos = m.pack_batch(cbp)
    ctx.submit_packed(2, m.make_batch_packed(words, bp.len1, bp.len2, npos, (bp.flags & 3).astype(np.uint8)))
    off1, rec1 = ctx.wait(2)
    assert np.array_equal(off0, off1) and np.array_equal(rec0, rec1)
    # malformed: n_words must follow from the lengths
    with pytest.raises(m.CfbError):
        ctx.submit_packed(3, m.make_batch_packed(words[:-1].copy(), bp.len1, bp.len2, npos, None))
    ctx.close(); ix.close()
