"""The host side of `centrifuge-class`'s record-level path, end to end on the CPU: the product's reader, seeds,
filters, tie selection with the per-read generator, TSV rows, per-taxon metrics, EM, report and Kraken-style
report run through the cfb_test_host_path hook around classification records taken from the oracle, and must
reproduce the bytes the unmodified reference binary writes for the same files and options."""
import ctypes as C
import os
import random

import numpy as np

import util
from test_classify_fuzz import API_OPTS, CLI_OPTS, make_reads
from util_fuzz import clean_reads

def dump_reads(lib, path, fasta, trims, tmp):
    out = str(tmp / "dump.txt")
    assert lib.cfb_test_parse(path.encode(), C.c_int(1 if fasta else 0), C.c_int(trims[0]), C.c_int(trims[1]), C.c_uint32(0), out.encode()) == 0
    seqs = []
    with open(out, "rb") as f:
        for line in f.read().split(b"\n")[:-1]:
            seqs.append(np.frombuffer(line.rsplit(b"\t", 3)[1], dtype=np.uint8))
    return seqs


def write_reads(path, rs, fasta, rng):
    with open(path, "wb") as f:
        for i, (n, s) in enumerate(rs):
            name = n + (b" desc" if i % 7 == 3 else b"") + (b"/1" if i % 5 == 2 else b"")
            if fasta:
                f.write(b">" + name + b"\n" + s + b"\n")
            else:
                f.write(b"@" + name + b"\n" + s + b"\n+\n" + bytes(rng.randrange(33, 74) for _ in s) + b"\n")


def test_host_side_reproduces_reference_bytes_around_oracle_records(tmp_path):
    util.ensure_oracle()
    base = util.golden_index("adv")
    lib = C.CDLL(util.PRODUCT_LIB)
    reads = clean_reads()
    o = util.Oracle(base)
    for case in range(200):
        rng = random.Random(33000 + case)
        oi = rng.randrange(len(API_OPTS))
        kw, cli = API_OPTS[oi], CLI_OPTS[oi]
        fasta, paired = rng.random() < 0.5, rng.random() < 0.35
        trims = rng.choice([(0, 0), (0, 0), (2, 0), (0, 4), (3, 5)])
        seed = rng.choice([0, 0, 7, 12345])
        rs = make_reads(rng, reads)
        p1, p2 = str(tmp_path / "a.txt"), str(tmp_path / "b.txt")
        if paired:
            rs2 = make_reads(rng, reads)[:len(rs)]; rs = rs[:len(rs2)]
            write_reads(p2, rs2, fasta, rng)
        write_reads(p1, rs, fasta, rng)
        m1 = dump_reads(lib, p1, fasta, trims, tmp_path)
        bt = util.Batch(m1, dump_reads(lib, p2, fasta, trims, tmp_path)) if paired else util.Batch(m1)
        on, orec, _ = o.classify(bt, util.make_oparams(**kw))
        rec_off = np.concatenate([[0], np.cumsum(on)]).astype(np.uint32)
        recs = np.ascontiguousarray(orec)
        tsv, rep, kr = str(tmp_path / "p.tsv"), str(tmp_path / "p.rep"), str(tmp_path / "p.kr")
        rc = lib.cfb_test_host_path(base.encode(), p1.encode(), p2.encode() if paired else None, C.c_int(1 if fasta else 0), C.c_int(kw.get("k", 5)),
                                    C.c_uint32(seed), C.c_int(trims[0]), C.c_int(trims[1]), rec_off.ctypes.data_as(C.POINTER(C.c_uint32)),
                                    recs.ctypes.data_as(C.c_void_p), C.c_uint64(len(on)), tsv.encode(), rep.encode(), kr.encode())
        assert rc == 0, (case, rc)
        args = ["-f" if fasta else "-q", "-x", base, "--seed", str(seed), "-5", str(trims[0]), "-3", str(trims[1])] + cli + (["-1", p1, "-2", p2] if paired else ["-U", p1])
        want_tsv, want_rep = util.reference_cli(args, tmp_path)
        assert util.file_digest(tsv) == want_tsv, (case, kw, fasta, paired, trims, seed)
        assert util.file_digest(rep) == want_rep, (case, kw, fasta, paired, trims, seed)
        # the in-process Kraken-style report equals the stand-alone one on the reference's TSV (the bytes of p.tsv, just
        # checked; the stand-alone report is itself pinned to the Perl script)
        want_kr = str(tmp_path / "r.kr")
        assert lib.cfb_kreport(base.encode(), tsv.encode(), want_kr.encode(), 0, 0, C.c_longlong(0), 0, C.c_longlong(0)) == 0
        got = open(kr, "rb").read() if os.path.exists(kr) else b""
        exp = open(want_kr, "rb").read() if os.path.exists(want_kr) else b""
        assert got == exp, case
        for fpath in (kr, want_kr):
            if os.path.exists(fpath):
                os.remove(fpath)
    o.close()
