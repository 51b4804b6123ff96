#!/usr/bin/env python3
"""bench.py -- reads/s of the classification hot path on B200 (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of DISTINCT synthetic reads (default: BASELINE.json configs[1],
10 M x 100 bp single-end reads per GPU) against a synthetic genus/species index (SURVEY.md Appendix C recipe, sequences
named cid<i> so that the index is a "compressed" one like p_compressed) replicated in each GPU's HBM.

  value      units/s with the step's reads already resident in HBM: kernels only, in windows of --chunk units, every step's
             own per-taxon counters folded on the device and all-reduced (cfb_counts_allreduce: NCCL) at the end of the step
  e2e        the same through cfb_classify_submit_packed/wait with HOST buffers (2-bit packed reads in pinned memory in, result
             records out): every step's H2D and D2H copies are inside the timed region; sub-batches stream over the
             context's slots
  e2e_byteform   the same with the 1-byte-per-base cfb_batch form (cfb_classify_submit)
  e2e_text   FASTQ bytes in -> classification TSV bytes out through the text-level operator (cfb_text_submit/wait): the
             like-for-like of what the reference arm times
  roofline   the FM-walk kernel: its own load requests (counted by the kernel in this run) x 32-byte DRAM sector / its
             CUDA-event time against the measured HBM copy peak, and against the random-gather ceiling measured in this
             process over the replica's own arrays; the reference algorithm's bytes (SURVEY 8d) kept as a separate figure
  parity_check   un-timed: a sample of this run's own reads, same context, against the unmodified reference binary
  cpu_baseline   the unmodified reference binary (oracle/_ref/centrifuge-class -p <cores>) on a bounded sample

`--impl reference` times that reference binary instead (best thread count, bounded sample per step).
Other BASELINE configs: --paired --rdlen 150 (configs[2]), --index-gbp 26 (configs[3]), --lens 75-300 (configs[4]).
Multi-GPU: one process per GPU (torchrun), reads sharded, index replicated; the only exchange is the product's own
collective (cfb_comm_init_rank + cfb_counts_allreduce); torch.distributed carries the barrier and the 128-byte NCCL id.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

REF_CLASS = os.path.join(ROOT, "oracle", "_ref", "centrifuge-class")
CACHE = os.environ.get("CFB_BENCH_CACHE", "/tmp/cfb200_bench")
PREFIX = "cid"      # sequence names cid<i>: >= 10 of them make the index a "compressed" one (ihits = 20, bt2_idx.h:648-663), as p_compressed is
HEADER = b"readID\tseqID\ttaxID\tscore\t2ndBestScore\thitLength\tqueryLength\tnumMatches\n"


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------ workload
def synth_opts(a, base=None, device=0, tax=None):
    from centrifuge_b200 import capi
    kw = dict(conversion_table=tax[0], taxonomy_tree=tax[1], name_table=tax[2]) if tax else {}
    return capi.build_opts(base, synth=(a.genera, a.species, a.genome_len, 12345, 0.03), device=device, synth_prefix=PREFIX, **kw)


def get_index(a, device=0):
    """Synthetic index on local disk, built once per box by the GPU builder (centrifuge_b200/csrc/cf_build.cu;
    byte-identical to centrifuge-build-bin, tests/test_gpu_build.py)."""
    from centrifuge_b200 import capi
    tag = "%s_g%d_s%d_l%d_seed%d" % (PREFIX, a.genera, a.species, a.genome_len, 12345)
    d = os.path.join(CACHE, tag)
    base = os.path.join(d, "idx")
    if os.path.exists(os.path.join(d, "done")):
        return base, d
    os.makedirs(d, exist_ok=True)
    t0 = time.time()
    tax = capi.write_synth_taxonomy(d, a.genera, a.species, a.genome_len, prefix=PREFIX)
    capi.build_index(synth_opts(a, base, device, tax))
    open(os.path.join(d, "done"), "w").close()
    log("index %s built on the GPU in %.1f s" % (tag, time.time() - t0))
    return base, d


class Reads:
    """n units of 1 or 2 mates: codes[m] (n, Lmax) uint8 in 0..4 (rows padded), lens[m] (n,) uint32."""

    def __init__(self, codes, lens):
        self.codes, self.lens = codes, lens
        self.n, self.mates, self.lmax = codes.shape[1], codes.shape[0], codes.shape[2]

    def sub(self, lo, hi):
        return Reads(self.codes[:, lo:hi], self.lens[:, lo:hi])

    def flags(self):
        f = np.zeros(self.n, dtype=np.uint8)
        for m in range(self.mates):
            L = self.lens[m].astype(np.int64)
            ns = ((self.codes[m] == 4) & (np.arange(self.lmax)[None, :] < L[:, None])).sum(axis=1)
            f |= (((L >= 2) & (ns <= (0.15 * L).astype(np.int64))).astype(np.uint8) << m)      # nFilter NCEIL=L,0,0.15 + lenfilt
        return f

    def byte_form(self, pin):
        """arrays of a cfb_batch (mate 1 of all units, then mate 2), in pinned memory"""
        tot = int(self.lens.sum())
        bases = pin((tot,), np.uint8)
        offs, pos = [], 0
        for m in range(self.mates):
            L = self.lens[m].astype(np.int64)
            mask = np.arange(self.lmax)[None, :] < L[:, None]
            k = int(L.sum())
            bases[pos:pos + k] = self.codes[m][mask]
            o = pin((self.n,), np.uint64); o[:] = (pos + np.concatenate([[0], np.cumsum(L[:-1])])).astype(np.uint64) if self.n else 0
            offs.append(o); pos += k
        lens = [pin((self.n,), np.uint32) for _ in range(self.mates)]
        for m in range(self.mates):
            lens[m][:] = self.lens[m]
        fl = pin((self.n,), np.uint8); fl[:] = self.flags()
        return bases, offs, lens, fl

    def packed_form(self, pin):
        """arrays of a cfb_batch_packed: 2-bit words (mate 1 of all units, then mate 2), N positions"""
        words, npos, wbase = [], [], 0
        W = (self.lmax + 31) // 32
        for m in range(self.mates):
            L = self.lens[m].astype(np.int64)
            valid = np.arange(self.lmax)[None, :] < L[:, None]
            isn = (self.codes[m] > 3) & valid
            pad = np.zeros((self.n, W * 32), dtype=np.uint8)
            pad[:, :self.lmax] = np.where(isn | ~valid, 0, self.codes[m])
            q = pad.reshape(self.n, W * 8, 4)                     # four bases per byte, base j of a word at bits 2j (little-endian words)
            w = (q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)).view("<u8")
            wl = (L + 31) // 32
            keep = np.arange(W)[None, :] < wl[:, None]
            words.append(w[keep])
            wstart = wbase + np.concatenate([[0], np.cumsum(wl[:-1])]) if self.n else np.zeros(0, dtype=np.int64)
            r, j = np.nonzero(isn)
            npos.append(((wstart[r] + j // 32).astype(np.uint64) << np.uint64(5)) | (j % 32).astype(np.uint64))
            wbase += int(wl.sum())
        wcat, ncat = np.concatenate(words), np.concatenate(npos)
        pw = pin((max(1, wcat.size),), np.uint64)[:wcat.size]; pw[:] = wcat
        pn = pin((max(1, ncat.size),), np.uint64)[:ncat.size]; pn[:] = ncat
        lens = [pin((self.n,), np.uint32) for _ in range(self.mates)]
        for m in range(self.mates):
            lens[m][:] = self.lens[m]
        fl = pin((self.n,), np.uint8); fl[:] = self.flags()
        return pw, pn, lens, fl

    def fastq(self, m, start=0, suffix=b"", force_general=False):
        """FASTQ text of mate m: "@r%09d<suffix>", bases, "+", qualities 'I' (vectorised, variable lengths)"""
        n = self.n
        L = self.lens[m].astype(np.int64)
        hl = 11 + len(suffix)                                   # "@r%09d" + suffix
        rec = hl + 1 + L + 3 + L + 1
        off = np.concatenate([[0], np.cumsum(rec[:-1])]) if n else np.zeros(0, dtype=np.int64)
        out = np.full(int(rec.sum()), ord("I"), dtype=np.uint8)
        hdr = np.empty((n, hl + 1), dtype=np.uint8)
        hdr[:, 0] = ord("@"); hdr[:, 1] = ord("r")
        v = np.arange(start, start + n, dtype=np.int64).astype(np.uint32)
        for k in range(8, -1, -1):                              # nine decimal digits, last first
            q = v // 10
            hdr[:, 2 + k] = (v - q * 10 + 48).astype(np.uint8); v = q
        if suffix:
            hdr[:, 11:11 + len(suffix)] = np.frombuffer(suffix, dtype=np.uint8)[None, :]
        hdr[:, hl] = 10
        if n and not force_general and int(L.min()) == int(L.max()):          # one length: the records are the rows of a 2-D array
            l = int(L[0])
            rows = out.reshape(n, int(rec[0]))
            rows[:, :hl + 1] = hdr
            rows[:, hl + 1:hl + 1 + l] = np.frombuffer(b"ACGTN", dtype=np.uint8)[self.codes[m][:, :l]]
            rows[:, hl + 1 + l:hl + 4 + l] = np.array([10, 43, 10], dtype=np.uint8)[None, :]
            rows[:, -1] = 10
            return out
        out[(off[:, None] + np.arange(hl + 1)[None, :]).reshape(-1)] = hdr.reshape(-1)
        mask = np.arange(self.lmax)[None, :] < L[:, None]
        pos = (off + hl + 1)[:, None] + np.arange(self.lmax)[None, :]
        out[pos[mask]] = np.frombuffer(b"ACGTN", dtype=np.uint8)[self.codes[m]][mask]
        tail = (off + hl + 1 + L)[:, None] + np.arange(3)[None, :]
        out[tail.reshape(-1)] = np.tile(np.array([10, 43, 10], dtype=np.uint8), n)
        out[off + rec - 1] = 10
        return out


def make_reads(a, n, seed, device=0):
    from centrifuge_b200 import capi
    so = synth_opts(a, device=device)
    lo, hi = a.lens
    out_c, out_l = [], []
    for s in range(0, n, 2000000):                             # generated on the device in slabs
        k = min(2000000, n - s)
        c, l = capi.synth_reads_ex(so, k, seed * 1000003 + s, lo, hi, paired=a.paired)
        out_c.append(c); out_l.append(l)
    return Reads(np.concatenate(out_c, axis=1), np.concatenate(out_l, axis=1))


def write_fastq_files(rd, paths):
    for m, p in enumerate(paths):
        with open(p, "wb") as f:
            for s in range(0, rd.n, 200000):
                f.write(rd.sub(s, min(rd.n, s + 200000)).fastq(m, start=s).tobytes())


def bind_to_gpu_numa_node(dev):
    """Run this rank on the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers it allocates
    (first touch) and the threads that fill them are local to that GPU's PCIe root.  Best effort."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(dev)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                   # sysfs uses 4-digit domains
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:  # noqa: BLE001
        pass
    return None


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed regions, via NVML in-process (no nvidia-smi forks, which
    contend for the driver lock with the CUDA calls being timed)."""

    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev, self.samples, self.reasons, self.stop_flag, self.maxmhz = dev, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.dev)
            self.maxmhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else nv.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0)),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0)),
                    "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0))}
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop_flag:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(h))
                for nm, b in bits.items():
                    if b and (r & b):
                        self.reasons.add(nm)
                time.sleep(0.05)
        except Exception as e:  # noqa: BLE001
            self.reasons.add("nvml_unavailable: %s" % e)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.maxmhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.maxmhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def ref_cmd(a, base, files, threads, out="/dev/null", extra=()):
    rd = ["-1", files[0], "-2", files[1]] if a.paired else ["-U", files[0]]
    return [REF_CLASS, "-q", "-x", base] + rd + ["-p", str(threads), "-S", out, "--report-file", "/dev/null"] + list(extra)


def ref_seconds(a, base, files, threads):
    t0 = time.time()
    subprocess.check_call(ref_cmd(a, base, files, threads), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return time.time() - t0


class RefArm:
    """The unmodified reference binary on the host cores.  Index load is excluded by differencing two
    sample sizes; the thread count is the best of a short sweep (the reference's one-read-per-mutex
    input loop, pat.h:786-811, stops scaling well before 128 threads)."""

    def __init__(self, a, base, d, device=0):
        self.a, self.base = a, base
        self.n_small, self.n = 20000, a.cpu_sample
        tag = "%s_%d_%d%s" % ("pe" if a.paired else "se", a.lens[0], a.lens[1], "")
        rd = None
        self.files = {}
        for n in (self.n_small, self.n):
            fs = [os.path.join(d, "sample_%s_%d_%d.fq" % (tag, n, m + 1)) for m in range(2 if a.paired else 1)]
            if not all(os.path.exists(f) for f in fs):
                if rd is None:
                    rd = make_reads(a, self.n, 999, device)
                write_fastq_files(rd.sub(0, n), fs)
            self.files[n] = fs
        ncores = os.cpu_count() or 1
        best = None
        for p in sorted(set(min(x, ncores) for x in (8, 16, 24, 32, 64, ncores))):
            t1 = ref_seconds(a, base, self.files[self.n_small], p)
            t2 = ref_seconds(a, base, self.files[self.n], p)
            rate = (self.n - self.n_small) / max(t2 - t1, 1e-6)
            log("reference -p %d: %.0f units/s (%.1f s for %d, %.1f s for %d)" % (p, rate, t2, self.n, t1, self.n_small))
            if best is None or rate > best[1]:
                best = (p, rate)
            elif rate < 0.5 * best[1]:
                break
        self.threads, self.sweep_rate = best

    def step(self):
        """seconds of classification work for self.n - self.n_small units (index load differenced out)"""
        t2 = ref_seconds(self.a, self.base, self.files[self.n], self.threads)
        t1 = ref_seconds(self.a, self.base, self.files[self.n_small], self.threads)
        return max(t2 - t1, 1e-6), self.n - self.n_small


def parity_check(a, ctx, ix, base, d, rd, nsample):
    """Un-timed: the first `nsample` units of this run's own reads, classified by the *same* context the timed loops
    use (every derived table that was built is live), against the unmodified reference binary on the same index and
    the same FASTQ: (1) the TSV the text operator returns must equal the reference's bytes, (2) the records the C ABI
    returns (byte form and packed form) must be the rows of that TSV (per unit: the records with the best score <->
    the rows, taxID / score / hitLength)."""
    from centrifuge_b200 import capi
    import pandas as pd
    tb = ix.tables()
    tables = {"ftabk": tb["ftabk_chars"], "ftabd": tb["ftabd_chars"], "rtab": 8 * tb["resolve_entry_bytes"], "walk8": tb["walk8_bytes"] > 0, "walk8_row_coverage": tb["walk8_rows"] / float(ix.info.len + 1),
              "compressed": bool(ix.info.compressed), "rows_beyond_2^32": bool(ix.info.len >= (1 << 32))}
    if not os.path.exists(REF_CLASS):
        return {"reads": 0, "identical": None, "tables": tables, "skipped": "oracle/_ref/centrifuge-class not shipped"}
    sub = rd.sub(0, nsample)
    n = sub.n
    texts = [sub.fastq(m, suffix=(b"/%d" % (m + 1)) if a.paired else b"") for m in range(sub.mates)]
    files = [os.path.join(d, "parity_%d_%d.fq" % (os.getpid(), m)) for m in range(sub.mates)]
    ref_tsv = os.path.join(d, "parity_%d.tsv" % os.getpid())
    for f, t in zip(files, texts):
        with open(f, "wb") as g:
            g.write(t.tobytes())
    p = min(16, os.cpu_count() or 1)
    t0 = time.time()
    subprocess.check_call(ref_cmd(a, base, files, p, out=ref_tsv, extra=["--reorder"]), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    with open(ref_tsv, "rb") as f:
        want = f.read()
    t_ref = time.time() - t0
    pts = []
    for t in texts:
        pt = capi.pinned_array((t.size,), np.uint8); pt[:] = t
        pts.append(pt)
    ctx.text_submit(0, pts[0], pts[1] if a.paired else None, n, maxlen_hint=sub.lmax)
    r = ctx.text_wait(0, discard=True)
    tsv_ok = (not r["irregular"]) and HEADER + r["tsv"] == want
    # records of the C ABI (byte form, then packed form) against the reference's rows
    pin = lambda shape, dt: np.zeros(shape, dtype=dt)          # noqa: E731  (pageable is fine here)
    bases, offs, lens, fl = sub.byte_form(pin)
    off, recs = ctx.classify(capi.make_batch(bases, offs[0], lens[0], offs[1] if a.paired else None, lens[1] if a.paired else None, fl))
    pw, pn, plens, pfl = sub.packed_form(pin)
    ctx.submit_packed(1, capi.make_batch_packed(pw, plens[0], plens[1] if a.paired else None, pn, pfl))
    off2, recs2 = ctx.wait(1)
    packed_ok = bool(np.array_equal(off, off2) and np.array_equal(recs, recs2))
    df = pd.read_csv(ref_tsv, sep="\t", dtype={"readID": str, "seqID": str})
    rid = df["readID"].str[1:10].astype(np.int64).to_numpy()
    cls = (df["seqID"] != "unclassified").to_numpy()
    rows = np.stack([rid[cls], df["taxID"].to_numpy(np.int64)[cls], df["score"].to_numpy(np.int64)[cls], df["hitLength"].to_numpy(np.int64)[cls]], axis=1)
    cnt = np.diff(off.astype(np.int64))
    unit = np.repeat(np.arange(n), cnt)
    best = np.zeros(n, dtype=np.int64)
    np.maximum.at(best, unit, recs["score"].astype(np.int64))
    top = recs["score"].astype(np.int64) == best[unit]
    mine = np.stack([unit[top], recs["taxid"][top].astype(np.int64), recs["score"][top].astype(np.int64), recs["hitlen"][top].astype(np.int64)], axis=1)
    key = lambda x: x[np.lexsort((x[:, 3], x[:, 2], x[:, 1], x[:, 0]))]       # noqa: E731
    rec_ok = mine.shape == rows.shape and bool(np.array_equal(key(mine), key(rows)))
    uncl_ok = bool(np.array_equal(np.sort(rid[~cls]), np.nonzero(cnt == 0)[0]))
    for f in files + [ref_tsv]:
        os.unlink(f)
    return {"reads": int(n), "identical": bool(tsv_ok and rec_ok and uncl_ok and packed_ok), "tsv_bytes_identical": bool(tsv_ok),
            "abi_records_match_rows": bool(rec_ok and uncl_ok), "packed_form_equals_byte_form": packed_ok, "tables": tables, "rows": int(len(df)),
            "reference": "oracle/_ref/centrifuge-class -p %d --reorder, same index, same FASTQ (%.1f s)" % (p, t_ref)}


DUMP_UNITS = 1 << 17


def dump_outputs(out_dir, ctx, first, taxids, counts):
    """The last timed step's outputs, as a caller of the resident path receives them: the step's per-taxon counters
    (cfb_counts_dense after the all-reduce) and the records of its last window (cfb_resident_result holds that window
    only), of which a fixed sample of units is kept.  float64 holds every value exactly (counts and taxIDs < 2^53)."""
    os.makedirs(out_dir, exist_ok=True)
    off, recs = ctx.resident_result()
    off = off.astype(np.int64)
    n = len(off) - 1
    units = np.sort(np.random.default_rng(20240601).choice(n, min(n, DUMP_UNITS), replace=False))
    cnt = off[units + 1] - off[units]
    idx = np.repeat(off[units], cnt) + np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    out = {"counts_taxid": taxids, "counts": counts, "sample_unit": first + units, "sample_records_per_unit": cnt}
    for f in ("taxid", "score", "hitlen", "uid"):
        out["sample_record_" + f] = recs[f][idx]
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))
    log("outputs of the last timed step written to %s (%s)" % (out_dir, ", ".join(sorted(out))))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------ main
def main():
    # stdout carries exactly one JSON line: route everything else that native libraries print to fd 1
    # (e.g. NCCL's version banner) to stderr, and keep a private handle for the result line
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)
    result = os.fdopen(result_fd, "w")
    try:
        return _main(result)
    finally:
        result.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cfb200", choices=["cfb200", "reference"])
    ap.add_argument("--genera", type=int, default=int(os.environ.get("CFB_BENCH_GENERA", 0)))
    ap.add_argument("--species", type=int, default=int(os.environ.get("CFB_BENCH_SPECIES", 10)))
    ap.add_argument("--genome-len", type=int, default=int(os.environ.get("CFB_BENCH_GENOME_LEN", 1000000)))
    ap.add_argument("--index-gbp", type=float, default=float(os.environ.get("CFB_BENCH_INDEX_GBP", 9)), help="joined reference length in Gbp (9 = p_compressed-class 4.1 GB, 17 = 8 GB class, 26 = 12 GB class)")
    ap.add_argument("--reads", type=int, default=int(os.environ.get("CFB_BENCH_READS", 0)), help="units (reads or pairs) per step per GPU; default 10 M reads / 5 M pairs")
    ap.add_argument("--chunk", type=int, default=int(os.environ.get("CFB_BENCH_CHUNK", 2000000)), help="units per resident window / kernel launch")
    ap.add_argument("--sub", type=int, default=int(os.environ.get("CFB_BENCH_SUB", 500000)), help="units per e2e sub-batch")
    ap.add_argument("--rdlen", type=int, default=100)
    ap.add_argument("--lens", default=None, help="LO-HI: uniform mixed read lengths (BASELINE configs[4]: 75-300)")
    ap.add_argument("--paired", action="store_true", help="2 x rdlen paired-end units, insert 200-500 (BASELINE configs[2])")
    ap.add_argument("--cpu-sample", type=int, default=int(os.environ.get("CFB_BENCH_CPU_SAMPLE", 400000)))
    ap.add_argument("--parity-reads", type=int, default=int(os.environ.get("CFB_BENCH_PARITY_READS", 200000)), help="units of the step batch checked against the reference binary (un-timed)")
    ap.add_argument("--skip-arms", default=os.environ.get("CFB_BENCH_SKIP", ""), help="comma list of e2e_byteform,e2e_text,cpu_baseline,gather to leave out (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64): "
                    "its all-reduced per-taxon counters, and the records of a fixed, seeded sample of %d units of its last window" % DUMP_UNITS)
    a = ap.parse_args()
    if a.genera == 0:
        a.genera = max(1, int(round(a.index_gbp * 1e9 / (a.species * a.genome_len))))
    a.lens = tuple(int(x) for x in a.lens.split("-")) if a.lens else (a.rdlen, a.rdlen)
    if a.reads == 0:
        a.reads = 5000000 if (a.paired or a.lens[1] > 160) else 10000000
    a.chunk = min(a.chunk, a.reads); a.sub = min(a.sub, a.reads)
    a.skip = set(x for x in a.skip_arms.split(",") if x)
    return a


def describe(a):
    shape = "%d-%d bp" % a.lens if a.lens[0] != a.lens[1] else "%d bp" % a.lens[0]
    kind = "2 x %s PE pairs (insert 200-500, mate 2 reverse-complemented)" % shape if a.paired else "%s SE reads" % shape
    return ("synthetic %d genera x %d species x %d bp index (%.0f Mbp, %s names), %d DISTINCT %s per step per GPU"
            % (a.genera, a.species, a.genome_len, a.genera * a.species * a.genome_len / 1e6, PREFIX, a.reads, kind))


def metric_name(a):
    shape = "%d-%d" % a.lens if a.lens[0] != a.lens[1] else "%d" % a.lens[0]
    return "%s/sec (%s bp %s classification)" % ("pairs" if a.paired else "reads", shape, "PE" if a.paired else "SE")


def _main(result):
    a = parse_args()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    ncores = os.cpu_count() or 1
    unit = "pairs/s" if a.paired else "reads/s"
    workload = describe(a)

    if a.impl == "reference":
        if rank != 0:
            return 0
        base, d = get_index(a)
        arm = RefArm(a, base, d)
        for _ in range(min(a.warmup, 1)):
            arm.step()
        tot, nreads = 0.0, 0
        for _ in range(a.steps):
            t, n = arm.step()
            tot += t; nreads += n
        val = nreads / tot
        sample = "%d units per step (bounded sample of the same generator), centrifuge-class -p %d (best of a thread sweep up to %d), FASTQ in, TSV to /dev/null, index load differenced out" % (
            nreads // a.steps, arm.threads, ncores)
        print(json.dumps({"metric": metric_name(a), "value": val, "unit": unit, "n_gpus": a.gpus, "steps": a.steps,
                          "warmup": min(a.warmup, 1), "ms_per_step": 1000 * tot / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "u64", "data": "synthetic", "impl": "reference",
                          "config": {"workload": workload, "sample": sample},
                          "cpu_baseline": {"value": val, "unit": unit, "cores": arm.threads, "kind": "reference", "sample": sample},
                          "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), file=result, flush=True)
        return 0

    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    import torch
    from centrifuge_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the cfb200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        get_index(a, local)
    if dist:
        dist.barrier()
    base, d = get_index(a, local)
    t0 = time.time()
    rd = make_reads(a, a.reads, 1000 + rank, local)
    n = rd.n
    bases_per_unit = float(rd.lens.sum()) / n
    log("rank %d: %d units generated in %.1f s (%.1f bases per unit)" % (rank, n, time.time() - t0, bases_per_unit))
    pin = capi.pinned_array

    # HBM head-room the batch buffers of this run need (the derived tables take what is left, cfb_index_tables): sized by the
    # longest read -- hit lists (maxlen/4+8 records of 24 B per strand), packed strands, ~12 rows per unit of scoring scratch
    E2E_SLOTS = 8
    lc = 128 if rd.lmax <= 128 else (160 if rd.lmax <= 160 else (320 if rd.lmax <= 320 else ((rd.lmax + 1023) // 1024) * 1024))    # the text operator sizes by length class
    per_unit = rd.mates * ((lc // 22 + 2) * 48 + (lc / 4 + 8) * 48 / 32 + (lc // 32 + 1) * 24 + 3.5 * lc + 64) + 1776 + 160     # long hits only + 1/32 regenerated lists
    headroom_gb = max(24.0, ((E2E_SLOTS * a.sub + a.chunk) * per_unit * 1.3 + float(rd.lens.sum()) + 8.0 * n * rd.mates * 2 + (3 << 30)) / 2 ** 30)
    os.environ.setdefault("CFB_HBM_HEADROOM_GB", "%.1f" % headroom_gb)
    t0 = time.time()
    ix = capi.Index(base, local)
    tb = ix.tables()
    log("rank %d: index in HBM: %.2f GB in %.1f s (K-mer table K=%d, resolve table %d-bit, walk8 %s; %.1f GB free)" % (
        rank, ix.info.device_bytes / 1e9, time.time() - t0, tb["ftabk_chars"], 8 * tb["resolve_entry_bytes"],
        ("%.0f%% of the rows" % (100.0 * tb["walk8_rows"] / (ix.info.len + 1))) if tb["walk8_bytes"] else "no", tb["free_bytes_after_load"] / 1e9))
    ctx = capi.Context(ix)
    ctx.count_records(True)                                  # every batch's per-taxon counters are folded on the device
    if dist:                                                 # the product's own communicator: rank 0's NCCL id travels over torch.distributed
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(capi.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        ctx.comm_init_rank(world, rank, bytes(uid.cpu().numpy().tobytes()))
    n_tax = len(ctx.counts_taxids())

    def sync_all():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn):
        """fn() between synchronize+barrier brackets; seconds by CUDA events and by the wall clock, max over ranks"""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); w0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        e1.record(); w = time.perf_counter() - w0
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1) / 1000.0, w], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return out, float(t[0]), float(t[1])

    # ---------------- host-side forms of the step's reads (built before any timing)
    t0 = time.time()
    nsub = (n + a.sub - 1) // a.sub
    subs = [rd.sub(i * a.sub, min(n, (i + 1) * a.sub)) for i in range(nsub)]
    whole = rd.byte_form(pin)
    batch = capi.make_batch(whole[0], whole[1][0], whole[2][0], whole[1][1] if a.paired else None, whole[2][1] if a.paired else None, whole[3])
    packed, byteform, texts = [], [], []
    for i, sb in enumerate(subs):
        pw, pn, pl, pf = sb.packed_form(pin)
        packed.append(capi.make_batch_packed(pw, pl[0], pl[1] if a.paired else None, pn, pf))
        if "e2e_byteform" not in a.skip:
            b_, o_, l_, f_ = sb.byte_form(pin)
            byteform.append(capi.make_batch(b_, o_[0], l_[0], o_[1] if a.paired else None, l_[1] if a.paired else None, f_))
        if "e2e_text" not in a.skip:
            tt = []
            for m in range(sb.mates):
                t = sb.fastq(m, start=i * a.sub, suffix=(b"/%d" % (m + 1)) if a.paired else b"")
                pt = pin((t.size,), np.uint8); pt[:] = t
                tt.append(pt)
            texts.append(tt)
    h2d_packed = sum(int(p.n_words) * 8 + int(p.n_n) * 8 + int(p.n_units) * (4 * rd.mates + 1) for p in packed)
    h2d_bytes = int(whole[0].nbytes + sum(o.nbytes for o in whole[1]) + sum(l.nbytes for l in whole[2]) + whole[3].nbytes)
    h2d_text = sum(sum(int(t.nbytes) for t in tt) for tt in texts)
    log("rank %d: host forms ready in %.1f s (packed %.1f B/unit, byte form %.1f B/unit)" % (rank, time.time() - t0, h2d_packed / n, h2d_bytes / n))

    # ---------------- un-timed parity check of the configuration being timed (rank 0; the other ranks wait at the barrier)
    parity = None
    if rank == 0:
        parity = parity_check(a, ctx, ix, base, d, rd, min(a.parity_reads, n))
        log("parity check: %s" % json.dumps(parity))
    ctx.counts_reset()

    # ---------------- un-timed counter passes over one window of this exact batch:
    # (1) the reference algorithm's operations (SURVEY 8d), (2) the product's own load requests
    win = min(a.chunk, n)
    wsub = rd.sub(0, win).byte_form(lambda s, t: np.zeros(s, dtype=t))
    wbatch = capi.make_batch(wsub[0], wsub[1][0], wsub[2][0], wsub[1][1] if a.paired else None, wsub[2][1] if a.paired else None, wsub[3])
    os.environ["CFB_COUNT"] = "1"
    cctx = capi.Context(ix)
    cctx.classify(wbatch); ctr = cctx.counters(); cctx.close()
    os.environ["CFB_COUNT"] = "2"
    cctx = capi.Context(ix)
    cctx.classify(wbatch); req = cctx.requests(); cctx.close()
    del os.environ["CFB_COUNT"]
    scale = n / win
    sample_w = ix.info.sample_bytes
    ref_bytes_search = (128 * ctr["sides_search"] + 16 * ctr["ftab_probes"]) * scale
    ref_bytes_walk = (128 * ctr["walk_steps"] + sample_w * ctr["rows_resolved"]) * scale
    req_total = sum(req.values()) * scale

    # ---------------- the random-gather ceiling of this device over the replica's own arrays (same process, same footprint)
    ceil = {}
    if "gather" not in a.skip:
        for name, t in (("rank16", 0), ("ftabk", 1), ("walk8", 2), ("ftabd", 4)):
            have = {"rank16": tb["rank16_bytes"], "ftabk": tb["ftabk_bytes"], "walk8": tb["walk8_bytes"], "ftabd": tb["ftabd_bytes"]}[name]
            if have:
                ceil[name] = capi.gather_ceiling(ix, t, 1 << 31)[0]
        ceil["ftab2"] = None                                  # 16 MB: lives in L2, not a DRAM gather
        log("rank %d: random-gather ceilings (G requests/s): %s" % (rank, json.dumps(ceil)))

    # ---------------- value: the step's reads resident in HBM, kernels only; counters of the step reduced at its end
    dbatch = ctx.upload(batch)
    windows = [(s, min(a.chunk, n - s)) for s in range(0, n, a.chunk)]
    kms = np.zeros(5)

    def value_steps(k):
        for _ in range(k):
            ctx.counts_reset()
            for (s, c) in windows:
                ms, _ = ctx.classify_resident(dbatch, s, c)    # per-stage CUDA-event times on the kernels' own stream
                kms[:] += np.array(ms)
            ctx.counts_allreduce()                             # NCCL all-reduce (sum, u64) of this step's per-taxon counters
        return ctx.launches()

    value_steps(a.warmup)
    sampler = ClockSampler(local); sampler.start()
    kms[:] = 0
    l0 = ctx.launches()
    l1, dev_s, wall_s = timed(lambda: value_steps(a.steps))
    launches_value = l1 - l0
    value = world * n * a.steps / dev_s
    # the last step's counters: the product's all-reduce (NCCL through cfb_counts_allreduce) against the sum of the ranks' local
    # vectors carried by torch.distributed; numReads counts reported assignments (a unit with a 2-way tie counts twice)
    step_counts = ctx.counts_dense(global_=True, n=n_tax)
    local_counts = torch.from_numpy(ctx.counts_dense(global_=False, n=n_tax).astype(np.int64)).cuda()
    if dist:
        dist.all_reduce(local_counts)
    counts_check = {"taxon_vector_len": int(3 * n_tax), "assignments_counted_global": int(step_counts[0].sum()), "unclassified_units_global": int(step_counts[0][0]),
                    "unique_units_global": int(step_counts[1].sum()), "units_global": int(world * n),
                    "equals_sum_of_local_vectors": bool(np.array_equal(local_counts.cpu().numpy().astype(np.uint64), step_counts))}
    kms_step = kms / a.steps
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, ctx, windows[-1][0], ctx.counts_taxids()[:n_tax], step_counts)

    # ---------------- e2e arms: host buffers in, host results out, sub-batches streaming over the context's slots
    nslots = min(ctx.n_slots, E2E_SLOTS)

    host_s = {"submit": 0.0, "wait": 0.0}

    def stream(steps, submit, wait, per_step):
        got, q, pending = 0, 0, [None] * nslots
        for st in range(steps):
            for i in range(nsub):
                sl = q % nslots; q += 1
                if pending[sl] is not None:
                    t_ = time.perf_counter(); got += wait(sl); host_s["wait"] += time.perf_counter() - t_
                t_ = time.perf_counter(); submit(sl, i); host_s["submit"] += time.perf_counter() - t_
                pending[sl] = i
            if per_step:
                per_step()
        for k in range(nslots):                                  # drain in submission order
            sl = (q + k) % nslots
            if pending[sl] is not None:
                got += wait(sl); pending[sl] = None
        per_step()
        return got

    def e2e_arm(forms, submit_fn):
        ctx.counts_reset()
        run = lambda steps: stream(steps, lambda sl, i: submit_fn(sl, forms[i]), lambda sl: ctx.wait(sl, copy=False)[1], ctx.counts_allreduce)   # noqa: E731
        run(max(1, min(a.warmup, 2)))                             # every slot allocates its buffers before the timed region
        ctx.counts_reset()
        host_s["submit"] = host_s["wait"] = 0.0
        nrec, ds, ws = timed(lambda: run(a.steps))
        return world * n * a.steps / ds, nrec, ds, ws, {k: 1000 * v / a.steps for k, v in host_s.items()}

    e2e, nrec_e2e, e2e_dev_s, e2e_wall_s, e2e_host = e2e_arm(packed, ctx.submit_packed)
    d2h = nrec_e2e * 24 // a.steps + (n + nsub) * 4
    e2e_counts = int(ctx.counts_dense(global_=True, n=n_tax)[0].sum())
    out_e2e = {"value": e2e, "unit": unit, "h2d_bytes_per_step": int(h2d_packed), "d2h_bytes_per_step": int(d2h),
               "what": "cfb_classify_submit_packed/wait: 2-bit packed reads + lengths + N list in pinned host memory -> result records in host memory; %d sub-batches of %d units per step streaming over %d slots; per-taxon counters folded on the device and all-reduced once per step" % (nsub, a.sub, nslots),
               "assignments_counted_global": e2e_counts, "host_ms_per_step_in_calls": e2e_host}
    out_bf = None
    if "e2e_byteform" not in a.skip:
        v, nr, _, _, bf_host = e2e_arm(byteform, ctx.submit)
        out_bf = {"value": v, "unit": unit, "host_ms_per_step_in_calls": bf_host, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(nr * 24 // a.steps + (n + nsub) * 4),
                  "what": "cfb_classify_submit/wait with the 1-byte-per-base cfb_batch form"}
    out_text = None
    if "e2e_text" not in a.skip:
        def text_wait(sl):
            r = ctx.text_wait(sl, copy=False)
            if r["irregular"]:
                raise RuntimeError("text operator rejected the synthetic FASTQ")
            return r["tsv_bytes"] + r["n_multi"] * 8 * 6
        trun = lambda steps: stream(steps, lambda sl, i: ctx.text_submit(sl, texts[i][0], texts[i][1] if a.paired else None, subs[i].n, maxlen_hint=rd.lmax), text_wait, ctx.counts_allreduce)   # noqa: E731
        ctx.counts_reset(); trun(max(1, min(a.warmup, 2))); ctx.counts_reset()
        tsv_bytes, ds, _ = timed(lambda: trun(a.steps))
        out_text = {"value": world * n * a.steps / ds, "unit": unit, "what": "FASTQ text in pinned host memory -> TSV rows in host memory (cfb_text_submit/wait); the like-for-like of the reference arm",
                    "h2d_bytes_per_step": int(h2d_text), "d2h_bytes_per_step": int(tsv_bytes // a.steps)}
    sampler.stop_flag = True; sampler.join(timeout=2)

    # ---------------- roofline of the FM-walk kernel (k_search_t)
    peak, peak_src = measured_peak()
    search_s = kms_step[0] / 1000.0                                # per step (all windows), CUDA events around k_pack + k_search_t
    sector_bytes = 32.0 * req_total                                # every request of the kernel is one 32-byte DRAM sector (16-byte rank16 / table entries, 8-byte walk8 entries)
    achieved = sector_bytes / search_s / 1e9
    gather = None
    if ceil:
        per_table = {k: req[k] * scale for k in req}
        t_min = sum(per_table[k] / (ceil[k] * 1e9) for k in per_table if ceil.get(k))     # time the DRAM-resident gathers alone would take at their ceilings
        gather = {"what": "independent random gathers over the replica's own arrays, measured in this process before the timed loops (cfb_gather_ceiling)",
                  "ceiling_grequests_s": ceil, "requests_per_step": {k: int(v) for k, v in per_table.items()},
                  "achieved_grequests_s": req_total / search_s / 1e9, "frac": t_min / search_s}
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        if tj.get("workload_key") == "%d_%d_%d_%s" % (a.lens[0], a.lens[1], int(a.paired), a.genera):
            traffic = tj["dram_bytes_per_unit"] * win
            per_launch_s = search_s / len(windows)
            traffic_src = {"what": "ncu --set full capture of k_search_t on this workload (%s), scaled to a %d-unit launch; NOT measured in this run" % (tj.get("file", "profiles/"), win),
                           "dram_frac_of_hbm_peak": traffic / per_launch_s / 1e9 / peak,
                           "dram_read_gsectors_s": tj["dram_bytes_read"] / 32.0 / tj["units_in_capture"] * win / per_launch_s / 1e9,
                           "random_sector_ceiling_gsectors_s": 34.5, "ceiling_source": "tools/gather_bench.cu on this part, profiles/r02_gather_bench.txt (32 / 64 / 128-byte gathers all top out at ~1.1 TB/s)"}
    roof = {"bound": "hbm", "kernel": "k_search_t", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src, "kernel_ms_per_launch": 1000 * search_s / len(windows), "launches_per_step": len(windows),
            "bytes_definition": "the product's own algorithmic bytes: load requests counted by the kernel (CFB_COUNT=2 pass over one window of this batch) x one 32-byte DRAM sector each",
            "requests_per_unit": req_total / n, "random_gather": gather,
            "reference_algorithm": {"what": "bytes the reference's algorithm touches for the same reads (SURVEY 8d: 128 B per side + 16 B per ftab probe), counted with the jump tables off; the K-mer table and walk8 skip most of them, so this is a speed-up figure, not a roofline fraction",
                                    "bytes_per_step": int(ref_bytes_search), "bytes_per_unit": ref_bytes_search / n, "gb_s_equivalent": ref_bytes_search / search_s / 1e9,
                                    "algorithmic_speedup_vs_reference_bytes": ref_bytes_search / search_s / 1e9 / peak, "sides_per_unit": ctr["sides_search"] / max(ctr["units"], 1),
                                    "walk_bytes_per_step": int(ref_bytes_walk)}}
    out = {
        "metric": metric_name(a), "value": value, "unit": unit, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1000 * dev_s / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload, "index_bytes_hbm": int(ix.info.device_bytes), "tables": tb,
                   "hbm_headroom_gb": float(os.environ["CFB_HBM_HEADROOM_GB"]),
                   "l2": "every step walks %d distinct reads; index replica %.0f MB vs 126 MB L2" % (n, ix.info.device_bytes / 1e6),
                   "parallelism": "reads sharded over %d GPU(s), index replicated, one NCCL all-reduce (cfb_counts_allreduce) of the step's per-taxon counters per step" % world,
                   "timing": "K steps between synchronize+barrier brackets, CUDA events on the device, max over ranks (wall clock of the same region: %.4f s)" % wall_s},
        "e2e": out_e2e, "e2e_byteform": out_bf, "e2e_text": out_text,
        "gpu_launches": int(launches_value),
        "roofline": roof,
        "kernel_ms": {"search": kms_step[0], "prep_rows": kms_step[1], "resolve": kms_step[2], "score_compact": kms_step[3], "sum_of_stages": kms_step[4],
                      "what": "per step, summed over its %d launches of %d units" % (len(windows), a.chunk)},
        "clocks": sampler.summary(),
        "counts_allreduce": counts_check,
        "parity_check": parity,
    }
    if numa is not None:
        out["config"]["numa_node"] = numa
    if rank == 0 and world > 1:
        out["cpu_baseline"] = {"value": None, "unit": unit, "cores": 0, "kind": "reference", "sample": "reported by the N=1 run only"}
        print(json.dumps(out), file=result, flush=True)
    elif rank == 0:
        # bounded CPU baseline: the unmodified reference binary on the host cores
        if "cpu_baseline" in a.skip:
            out["cpu_baseline"] = {"value": None, "unit": unit, "cores": 0, "kind": "reference", "sample": "skipped (--skip-arms)"}
        else:
            try:
                arm = RefArm(a, base, d, local)
                tt, nn = arm.step()
                out["cpu_baseline"] = {"value": nn / tt, "unit": unit, "cores": arm.threads, "kind": "reference",
                                       "sample": "%d units, centrifuge-class -p %d (best of a sweep up to %d threads), FASTQ in, TSV to /dev/null, index load differenced out" % (nn, arm.threads, ncores)}
            except Exception as e:  # noqa: BLE001
                out["cpu_baseline"] = {"value": None, "unit": unit, "cores": ncores, "kind": "reference", "sample": "failed: %s" % e}
        print(json.dumps(out), file=result, flush=True)
    ok_counts = counts_check["equals_sum_of_local_vectors"] and counts_check["assignments_counted_global"] >= counts_check["units_global"] >= counts_check["unique_units_global"]
    ctx.close(); ix.close()
    if dist:
        dist.destroy_process_group()
    if rank == 0 and parity is not None and parity.get("identical") is False:
        log("PARITY CHECK FAILED: the timed configuration does not reproduce the reference's output")
        return 3
    if rank == 0 and not ok_counts:
        log("COUNTS CHECK FAILED: the all-reduced per-taxon counters are not the sum of the ranks' counters")
        return 4
    return 0


if __name__ == "__main__":
    sys.exit(main())
