"""Shared helpers for the test-suite: fixture building, read packing, ctypes bindings of the
oracle (oracle/_ref/libcforacle.so, test infrastructure) and of the host-compiled product
logic (tests/native/hostlogic.cpp)."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import synth  # noqa: E402

REFDIR = os.path.join(ROOT, "oracle", "_ref")
REF_CLASS = os.path.join(REFDIR, "centrifuge-class")
REF_BUILD = os.path.join(REFDIR, "centrifuge-build-bin")
ORACLE_BIN = os.path.join(REFDIR, "cf_oracle")
ORACLE_LIB = os.path.join(REFDIR, "libcforacle.so")
HOSTLOGIC_LIB = os.environ.get("CFB_HOSTLOGIC_LIB", os.path.join(REFDIR, "libhostlogic.so"))   # override: a sanitizer build of the shim
PRODUCT_LIB = os.environ.get("CFB_PRODUCT_LIB", os.path.join(ROOT, "centrifuge_b200", "libcfb200.so"))   # override: sanitizer build of the host side (tests/native/host_stub.cpp)
GOLDEN = os.path.join(ROOT, "tests", "golden")
CACHE = os.environ.get("CFB_TEST_CACHE", os.path.join(tempfile.gettempdir(), "cfb200_test_cache"))

ASC2DNA = np.zeros(256, dtype=np.uint8)
for ch, v in (("A", 0), ("C", 1), ("G", 2), ("T", 3), ("N", 4)):
    ASC2DNA[ord(ch)] = v
    ASC2DNA[ord(ch.lower())] = v


# ----------------------------------------------------------------------------- recorded reference runs
# The tests compare with what the unmodified reference did for the same call.  Those results are stored in
# tests/golden/reference_runs.json, keyed by the tool, its arguments and the contents of every input file and
# index they name, so the suite needs neither the reference sources nor its binaries.  With CFB_RECORD_REFERENCE
# set to a file name, every call runs the real binary (oracle/_ref, built from the reference sources by
# `make -C oracle ref`) and appends its result there; tests/golden/merge_reference_runs.py folds such files in.
# A test that skips while recording (one that needs two GPUs, say) makes no calls, so its runs are recorded on a
# machine where it runs, or by making the same calls from a script (the reference's binaries need no GPU).
REFERENCE_RUNS = os.path.join(GOLDEN, "reference_runs.json")
RECORD = os.environ.get("CFB_RECORD_REFERENCE")
_runs = None


def digest(data):
    return hashlib.sha256(data).hexdigest()[:32]


def file_digest(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()[:32]


def _key_token(arg):
    """An argument as it enters the key: input files and index bases by content, other words as they are."""
    parts = []
    for p in str(arg).split(","):
        if os.path.isfile(p):
            parts.append("file:" + file_digest(p))
        elif os.path.isfile(p + ".1.cf"):
            parts.append("index:" + "".join(file_digest("%s.%s.cf" % (p, k)) for k in "1234"))
        else:
            assert not os.path.isabs(p), "reference call names a path that does not exist: %s" % p
            parts.append(p)
    return ",".join(parts)


def error_lines(stderr):
    return [l for l in stderr.decode(errors="replace").splitlines() if l.startswith("Error") or l.startswith("Saw ASCII")]


def reference_run(tool, args, out=None):
    """What the reference's `tool` ("class", "build", "kreport" or "promote") did when run with `args`:
    dict(rc=exit status, errors=its 'Error' / 'Saw ASCII' lines on stderr, outputs=digests of what it wrote, None
    where it wrote nothing) and, for the Perl scripts, whose result is what they print, stdout=digest of stdout.  `out` (not part of the key): for "class" a directory for the
    TSV and report (-S / --report-file), for "build" the index base the .1-.4.cf files go to."""
    global _runs
    key = digest(json.dumps([tool] + [_key_token(a) for a in args]).encode())
    if RECORD:
        res = _run_reference(tool, list(args), out)
        with open(RECORD, "a") as f:
            f.write(json.dumps({key: res}) + "\n")
        return res
    if _runs is None:
        with open(REFERENCE_RUNS) as f:
            _runs = json.load(f)
    if key not in _runs:
        raise KeyError("no recorded reference run for %s %s: record one with CFB_RECORD_REFERENCE (tests/util.py)" % (tool, list(args)))
    return _runs[key]


def _run_reference(tool, args, out):
    """Runs the reference binary; what the binaries print on stdout (paths, timings) is not part of the result."""
    if tool in ("kreport", "promote"):
        return _run_reference_script(tool, args)
    if tool == "class":
        os.makedirs(out, exist_ok=True)
        outputs = [os.path.join(out, "ref.tsv"), os.path.join(out, "ref.rep")]
        cmd = [REF_CLASS] + args + ["-S", outputs[0], "--report-file", outputs[1]]
    else:
        outputs = ["%s.%s.cf" % (out, k) for k in "1234"]
        cmd = [REF_BUILD] + args + [out]
    for o in outputs:
        if os.path.exists(o):
            os.remove(o)
    p = subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    return dict(rc=p.returncode, errors=error_lines(p.stderr), outputs=[file_digest(o) if os.path.exists(o) else None for o in outputs])


def _run_reference_script(tool, args):
    import shutil
    import stat
    with tempfile.TemporaryDirectory() as stage:      # the Perl scripts look for centrifuge-inspect beside themselves
        script = os.path.join(stage, "centrifuge-" + tool)
        shutil.copy(os.path.join(os.environ["CFB_REFERENCE_SRC"], "centrifuge-" + tool), script)
        shim = os.path.join(stage, "centrifuge-inspect")
        with open(shim, "w") as f:
            f.write("#!/bin/sh\nexec %s \"$@\"\n" % os.path.join(REFDIR, "centrifuge-inspect-bin"))
        os.chmod(shim, os.stat(shim).st_mode | stat.S_IEXEC)
        p = subprocess.run(["perl", script] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return dict(rc=p.returncode, errors=error_lines(p.stderr), stdout=digest(p.stdout), outputs=[])


def reference_cli(args, tmp):
    """Digests of the classification TSV and report the reference's centrifuge-class writes for `args`
    (it must succeed); compare with `digests(run_cli(...))`."""
    r = reference_run("class", args, os.path.join(str(tmp), "reference"))
    assert r["rc"] == 0, r
    return tuple(r["outputs"])


def digests(outputs):
    return tuple(digest(x) for x in outputs)


def ensure_oracle():
    """Build the CPU restatement (and the host-logic shim) if missing.  Never touches /root/reference."""
    if not (os.path.exists(ORACLE_LIB) and os.path.exists(ORACLE_BIN)
            and os.path.getmtime(ORACLE_LIB) >= os.path.getmtime(os.path.join(ROOT, "oracle", "cf_oracle.cpp"))):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "port"], stdout=subprocess.DEVNULL)
    srcs = [os.path.join(ROOT, "tests", "native", "hostlogic.cpp"),
            os.path.join(ROOT, "centrifuge_b200", "csrc", "cf_index.cpp"),
            os.path.join(ROOT, "centrifuge_b200", "csrc", "cf_index.h"),
            os.path.join(ROOT, "centrifuge_b200", "csrc", "cf_logic.h")]
    if not os.path.exists(HOSTLOGIC_LIB) or any(os.path.getmtime(s) > os.path.getmtime(HOSTLOGIC_LIB) for s in srcs):
        os.makedirs(REFDIR, exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", HOSTLOGIC_LIB, srcs[0], srcs[1]])


# ----------------------------------------------------------------------------- fixtures
def build_index(tag, genera, species, length, seed, div=0.03, cid=False, strains=False):
    """Synthetic genomes -> .cf index through the product's builder (needs a GPU), checked against the reference's
    centrifuge-build-bin on the same files.  Cached."""
    key = hashlib.md5(repr((tag, genera, species, length, seed, div, cid, strains, ())).encode()).hexdigest()[:12]
    d = os.path.join(CACHE, "%s_%s" % (tag, key))
    base = os.path.join(d, "idx")
    if not os.path.exists(base + ".4.cf"):
        os.makedirs(d, exist_ok=True)
        synth.write_genomes(d, genera, species, length, seed, div, cid, strains)
        build_fasta_index([os.path.join(d, "genomes.fa")], os.path.join(d, "conv.tsv"), os.path.join(d, "nodes.dmp"), os.path.join(d, "names.dmp"), base)
    return base


def build_fasta_index(fasta, conv, nodes, names, base):
    """cfb_build_index over FASTA files; the .1-.4.cf files must be the bytes centrifuge-build-bin -p 4 writes
    (recorded reference run), else they are removed and the call fails."""
    from centrifuge_b200 import capi
    want = reference_run("build", ["-p", "4", "--conversion-table", conv, "--taxonomy-tree", nodes, "--name-table", names, ",".join(fasta)], base + "_reference")
    capi.build_index(capi.build_opts(base, fasta=list(fasta), conversion_table=conv, taxonomy_tree=nodes, name_table=names))
    files = ["%s.%s.cf" % (base, k) for k in "1234"]
    bad = [f for f, w in zip(files, want["outputs"]) if file_digest(f) != w]
    if bad:
        for f in files:
            os.remove(f)
        raise AssertionError("the product's builder does not write the reference's bytes: %s" % ", ".join(os.path.basename(f) for f in bad))
    return base


def golden_index(name):
    """Decompress a committed golden index (tests/golden/<name>.{1,2,3,4}.cf.xz) into the cache."""
    import lzma
    d = os.path.join(CACHE, "golden")
    os.makedirs(d, exist_ok=True)
    base = os.path.join(d, name)
    for k in "1234":
        dst = "%s.%s.cf" % (base, k)
        src = os.path.join(GOLDEN, "%s.%s.cf.xz" % (name, k))
        if not os.path.exists(dst) or os.path.getmtime(dst) < os.path.getmtime(src):
            with lzma.open(src) as f, open(dst + ".tmp", "wb") as g:
                g.write(f.read())
            os.replace(dst + ".tmp", dst)
    return base


def parse_reads(path):
    """Minimal FASTA/FASTQ reader for tests -> list of (name, uint8 ascii array)."""
    out = []
    with open(path, "rb") as f:
        data = f.read().split(b"\n")
    if not data or not data[0]:
        return out
    if data[0][:1] == b">":
        name, seq = None, []
        for ln in data:
            if ln[:1] == b">":
                if name is not None:
                    out.append((name, np.frombuffer(b"".join(seq), dtype=np.uint8)))
                name, seq = ln[1:].decode(), []
            elif ln:
                seq.append(ln.strip())
        if name is not None:
            out.append((name, np.frombuffer(b"".join(seq), dtype=np.uint8)))
    else:
        for i in range(0, len(data) - 3, 4):
            if data[i][:1] != b"@":
                break
            out.append((data[i][1:].decode(), np.frombuffer(data[i + 1].strip(), dtype=np.uint8)))
    return out


def n_filter_ok(codes):
    """Scoring::nFilter with NCEIL=L,0,0.15 plus the length filter (centrifuge.cpp:2559-2584)."""
    n = len(codes)
    return n >= 2 and int((codes == 4).sum()) <= int(0.15 * n)


class Batch:
    """Packed batch in the C-ABI layout (1 byte/base, 0..4)."""

    def __init__(self, mates1, mates2=None):
        n = len(mates1)
        self.n = n
        self.paired = mates2 is not None
        seqs = [ASC2DNA[a] for a in mates1]
        if self.paired:
            seqs2 = [ASC2DNA[a] for a in mates2]
        self.len1 = np.array([len(s) for s in seqs], dtype=np.uint32)
        self.off1 = np.zeros(n, dtype=np.uint64)
        if n:
            self.off1[1:] = np.cumsum(self.len1[:-1], dtype=np.uint64)
        tot1 = int(self.len1.sum())
        flags = np.array([1 if n_filter_ok(s) else 0 for s in seqs], dtype=np.uint8)
        if self.paired:
            self.len2 = np.array([len(s) for s in seqs2], dtype=np.uint32)
            self.off2 = np.zeros(n, dtype=np.uint64)
            if n:
                self.off2[1:] = np.cumsum(self.len2[:-1], dtype=np.uint64)
            self.off2 += np.uint64(tot1)
            flags |= np.array([2 if n_filter_ok(s) else 0 for s in seqs2], dtype=np.uint8)
            flags |= np.array([4 if len(s) > 0 else 0 for s in seqs2], dtype=np.uint8)   # oracle: bit2 = unit is a pair
            self.bases = np.concatenate(seqs + seqs2) if n else np.zeros(0, dtype=np.uint8)
        else:
            self.len2 = np.zeros(n, dtype=np.uint32)
            self.off2 = np.zeros(n, dtype=np.uint64)
            self.bases = np.concatenate(seqs) if n else np.zeros(0, dtype=np.uint8)
        self.bases = np.ascontiguousarray(self.bases, dtype=np.uint8)
        self.flags = flags


REC = np.dtype([("taxid", "<u8"), ("score", "<u4"), ("hitlen", "<u4"), ("uid", "<u4"), ("pad", "<u4")])


class OParams(C.Structure):
    _fields_ = [("khits", C.c_int), ("min_hitlen", C.c_int), ("tree_traverse", C.c_int), ("class_rank_slot", C.c_int),
                ("host", C.POINTER(C.c_uint64)), ("n_host", C.c_size_t), ("excl", C.POINTER(C.c_uint64)), ("n_excl", C.c_size_t)]


def make_oparams(k=5, min_hitlen=22, traverse=True, rank_slot=0, host=(), excl=()):
    p = OParams()
    p.khits, p.min_hitlen, p.tree_traverse, p.class_rank_slot = k, min_hitlen, 1 if traverse else 0, rank_slot
    p._h = (C.c_uint64 * max(1, len(host)))(*host)
    p._e = (C.c_uint64 * max(1, len(excl)))(*excl)
    p.host, p.n_host = C.cast(p._h, C.POINTER(C.c_uint64)), len(host)
    p.excl, p.n_excl = C.cast(p._e, C.POINTER(C.c_uint64)), len(excl)
    return p


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class _Classifier:
    """Common driver for the oracle and the host-logic shim (identical call signature)."""

    def __init__(self, lib, load, free, classify, base):
        self.lib, self._free, self._classify = lib, free, classify
        err = C.create_string_buffer(256)
        load.restype = C.c_void_p
        self.h = load(base.encode(), err, 256)
        if not self.h:
            raise RuntimeError(err.value.decode())
        classify.restype = C.c_longlong

    def close(self):
        if self.h:
            self._free(C.c_void_p(self.h))
            self.h = None

    def classify(self, batch, params, counters=False):
        n = batch.n
        out_n = np.zeros(n, dtype=np.uint32)
        cap = max(1024, n * 64)
        while True:
            out = np.zeros(cap, dtype=REC)
            ctr = (C.c_uint64 * 16)()
            r = self._classify(C.c_void_p(self.h), C.byref(params), _ptr(batch.bases, C.c_uint8), _ptr(batch.off1, C.c_uint64),
                               _ptr(batch.len1, C.c_uint32), _ptr(batch.off2, C.c_uint64), _ptr(batch.len2, C.c_uint32),
                               _ptr(batch.flags, C.c_uint8), C.c_size_t(n), _ptr(out_n, C.c_uint32),
                               out.ctypes.data_as(C.c_void_p), C.c_size_t(cap), ctr)
            if r == -1:
                cap *= 4
                continue
            if r < 0:
                raise RuntimeError("classify failed: %d" % r)
            return out_n, out[:r], list(ctr)


def Oracle(base):
    ensure_oracle()
    lib = C.CDLL(ORACLE_LIB)
    return _Classifier(lib, lib.cfo_index_load, lib.cfo_index_free, lib.cfo_classify, base)


def HostLogic(base):
    ensure_oracle()
    lib = C.CDLL(HOSTLOGIC_LIB)
    return _Classifier(lib, lib.hl_load, lib.hl_free, lib.hl_classify, base)


ORACLE_STATS = ["reads", "partial_searches", "ftab_probes", "lf_range_steps", "lf_range_same_side", "lf_single_steps",
                "sides_search", "walk_steps", "rows_resolved", "hits_resolved", "ext_searches"]


def run_cli(binary, args, out_tsv, report):
    subprocess.check_call([binary] + list(args) + ["-S", out_tsv, "--report-file", report],
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    with open(out_tsv, "rb") as f:
        a = f.read()
    with open(report, "rb") as f:
        b = f.read()
    return a, b
