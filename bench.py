#!/usr/bin/env python
"""bench.py — throughput of the `speedseq align` hot path on B200: reads/s ALIGNED + DUP-MARKED (BASELINE.json's metric).

One STEP = one run of `bwa mem | samblaster` (/root/reference/bin/speedseq:438-439) over the whole workload: every batch goes
through seeding, SA look-up, chaining, seed extension, sort/dedup/patch, insert-size statistics, mate rescue, pairing, MAPQ,
CIGAR/NM/MD, samblaster's signature / discordant / splitter tests, first-seen-wins duplicate marking against all earlier batches
of the step, and the three SAM record streams are written (main with 0x400 + MC/MQ, splitters, discordants) — the C-ABI call
ssq_aligner_* of include/ssq.h, which is what the `bwa` shim drives.

Workload ("config.workload"): synthetic 2x150 bp paired-end reads (wgsim-like: 0.5 % substitution errors, 0.085 % SNPs, ~2 % of
reads with a 1-3 bp indel, insert 500+-50; 10 % of the pairs are exact duplicates of earlier pairs under new names, 1 % are
chimeric: the mate comes from elsewhere) against a seeded synthetic reference with planted repeat families (no real genome
exists on the box), in batches of 2 M reads (bwa's batch rule at -t 30: 10 Mbp x threads).

  value : reads/s with every batch's FASTQ fields already resident in HBM when the timed region starts; the timed region ends when
          the last batch's SAM text is complete in HBM (CUDA events on the launching streams, max over ranks).
  e2e   : the same metric through the same C-ABI with HOST (pinned) buffers: every batch's names / bases / qualities are copied
          host->device and its three SAM streams device->host inside the timed region.
  Inputs + scratch per step exceed the 126 MB L2 many times over (config.l2).
  roofline : the kernel with the largest share of the step among those with a defined byte count (seeding: rank-block bytes
          dereferenced, counted on the device; SA look-up; text: bytes written + FASTQ bytes read; dup-set: 25 B/pair).
  cpu_baseline : the oracle (scalar C restatement of bwa mem + samblaster, oracle/) on all host cores over a bounded sample of
          the same reads ("port": the reference's bwa/samblaster sources are not vendored in /root/reference).
  parity : the GPU streams of that same sample (run as its own batch) compared byte for byte with the oracle's.

`--impl reference` runs ONLY the CPU arm (rank 0), K steps of a bounded sample each.
Multi-GPU: batches are dealt to ranks (weak scaling: every rank runs the same number of batches on its own reads), the index is
replicated; see DESIGN.md §6 for the dup-signature exchange.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from speedseq_b200 import capi  # noqa: E402  (ctypes bindings of the product's C-ABI; no compute)

GENOME_LEN = 1000000000  # the largest round size the GPU index builder handles (2 x 10^9 suffixes < 2^31); chr20-sized: --genome-len 63025520
READ_LEN = 150
SB = dict(exclude_dups=1, add_mate_tags=1, max_split_count=2, min_non_overlap=20)  # bin/speedseq:439 with its defaults (:241-243)
SB_ARGS = ["--excludeDups", "--addMateTags", "--maxSplitCount", "2", "--minNonOverlap", "20"]
CONTIGS = ["chrS%d" % (i + 1) for i in range(8)]
DUMP_PAIRS = 65536  # read pairs whose main-stream records --dump-outputs writes: ~11 MB at the default workload
DUMP_SIDE_RECORDS = 131072  # splitter / discordant records beyond this many are sampled (90 k discordants at the default workload)
DUMP_MAX_BYTES = 64 << 20


# ------------------------------------------------------------------------------------ data ----
def synth_genome(n, seed, repeat_frac=0.08):
    """seeded synthetic genome with planted diverged repeats so that seeds are not all unique (same generator as the tests)"""
    rng = np.random.default_rng(seed)
    g = rng.choice(4, size=n, p=[0.295, 0.205, 0.205, 0.295]).astype(np.uint8)
    fam = rng.integers(0, 4, 300, dtype=np.uint8)
    n_rep = int(n * repeat_frac / 300)
    pos = rng.integers(0, max(1, n - 300), n_rep)
    for p in pos:
        c = fam.copy()
        m = rng.random(300) < 0.08
        c[m] = rng.integers(0, 4, int(m.sum()), dtype=np.uint8)
        g[p:p + 300] = c
    if n > 5000:
        g[2000:2400] = g[1000:1400]
        g[3000:3060] = np.tile(np.array([0, 1], np.uint8), 30)
    return g


def write_fasta(path, g, names, bounds):
    acgt = np.frombuffer(b"ACGT", np.uint8)
    with open(path, "wb") as f:
        for i, nm in enumerate(names):
            f.write((">%s\n" % nm).encode())
            s = acgt[g[bounds[i]:bounds[i + 1]]]
            w = 1 << 16  # long lines: the parser does not care and Python writes far fewer of them
            for j in range(0, len(s), w):
                f.write(s[j:j + w].tobytes()); f.write(b"\n")


def fast_pairs(g, n_pairs, read_len, seed, ins_mean=500, ins_sd=50, dup_frac=0.10, chim_frac=0.01, dup_pool=None):
    """vectorised wgsim-like simulator -> base codes [2*n_pairs, read_len]; 10 % exact duplicate pairs (re-emitted earlier pairs,
    half of them from `dup_pool` = an earlier batch), 1 % chimeric pairs (mate drawn from another fragment)"""
    rng = np.random.default_rng(seed)
    comp = np.array([3, 2, 1, 0, 4], np.uint8)
    n = len(g)
    ins = np.clip(rng.normal(ins_mean, ins_sd, n_pairs).astype(np.int64), read_len + 10, None)
    p = (rng.random(n_pairs) * (n - ins - 8)).astype(np.int64)
    ar = np.arange(read_len, dtype=np.int64)
    r1 = g[p[:, None] + ar]
    r2 = comp[g[(p + ins - 1)[:, None] - ar]]
    for r in (r1, r2):
        m = rng.random(r.shape) < 0.00585
        r[m] = (r[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) & 3
        who = np.nonzero(rng.random(n_pairs) < 0.0225)[0]
        for i in who:  # small indels
            at, l = int(rng.integers(10, read_len - 10)), int(rng.integers(1, 4))
            if rng.random() < 0.5:
                r[i, at + l:] = r[i, at:read_len - l].copy()
                r[i, at:at + l] = rng.integers(0, 4, l, dtype=np.uint8)
            else:
                r[i, at:read_len - l] = r[i, at + l:].copy()
                r[i, read_len - l:] = rng.integers(0, 4, l, dtype=np.uint8)
    sw = rng.random(n_pairs) < 0.5
    out = np.empty((2 * n_pairs, read_len), np.uint8)
    out[0::2] = np.where(sw[:, None], r2, r1)
    out[1::2] = np.where(sw[:, None], r1, r2)
    ch = np.nonzero(rng.random(n_pairs) < chim_frac)[0]  # chimeric: the second end comes from another pair
    out[2 * ch + 1] = out[2 * ((ch + n_pairs // 2) % n_pairs) + 1]
    nd = int(n_pairs * dup_frac)
    dst = rng.choice(np.arange(n_pairs // 4, n_pairs), nd, replace=False)  # duplicates sit in the later 3/4 of the batch
    src = (rng.random(nd) * (n_pairs // 4)).astype(np.int64)                 # ... and copy pairs of its first quarter
    out[2 * dst] = out[2 * src]; out[2 * dst + 1] = out[2 * src + 1]
    if dup_pool is not None:  # half of them copy pairs of an earlier batch instead
        k = nd // 2
        out[2 * dst[:k]] = dup_pool[2 * src[:k]]; out[2 * dst[:k] + 1] = dup_pool[2 * src[:k] + 1]
    return out


class Batch:
    """one batch of reads as the FASTQ fields ssq_aligner_upload() takes, in pinned host memory"""
    def __init__(self, torch, codes, first_pair, pin=True):
        n, rl = codes.shape
        acgt = np.frombuffer(b"ACGT", np.uint8)
        mk = (lambda a: torch.from_numpy(a).pin_memory()) if pin else (lambda a: torch.from_numpy(a))
        self.n = n
        self.seq = mk(acgt[codes].reshape(-1))
        self.qual = mk(np.full(n * rl, ord("I"), np.uint8))
        self.seq_off = mk((np.arange(n + 1, dtype=np.int64) * rl))
        ids = first_pair + np.arange(n) // 2
        nm = np.char.add("p", np.char.zfill(ids.astype("U10"), 9)).astype("S10")
        self.names = [x.decode() for x in nm] if n <= 400000 else None  # python strings only for the parity sample
        self.name = mk(np.frombuffer(nm.tobytes(), np.uint8).copy())
        self.name_off = mk((np.arange(n + 1, dtype=np.int64) * 10).astype(np.uint32))
        r = capi.Reads()
        r.n_reads, r.paired, r.n_processed = n, 1, 2 * first_pair
        r.seq, r.seq_off, r.qual, r.name, r.name_off = self.seq.data_ptr(), self.seq_off.data_ptr(), self.qual.data_ptr(), self.name.data_ptr(), self.name_off.data_ptr()
        self.reads = r
        self.h2d = int(self.seq.numel()) * 2 + (n + 1) * 12 + int(self.name.numel())


def ensure_reference(cache, genome_len, builder):
    """seeded synthetic genome (8 contigs) + index under `cache`; builder(fasta) makes the five index files"""
    os.makedirs(cache, exist_ok=True)
    fa = os.path.join(cache, "syn_%d.fa" % genome_len)
    gnpy = fa + ".npy"
    t0 = time.time()
    if not os.path.exists(gnpy):
        g = synth_genome(genome_len, 20)
        bounds = np.linspace(0, genome_len, 9).astype(np.int64)
        write_fasta(fa, g, CONTIGS, bounds)
        np.save(gnpy, g)
        sys.stderr.write("[bench] synthetic genome of %d bp written in %.1f s\n" % (genome_len, time.time() - t0))
    if not all(os.path.exists(fa + e) for e in (".bwt", ".sa", ".pac", ".ann", ".amb")):
        t0 = time.time()
        builder(fa)
        sys.stderr.write("[bench] index built in %.1f s\n" % (time.time() - t0))
    return fa, np.load(gnpy)


def usable_cores():
    """host cores this process may actually use: affinity mask capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(p))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = max(1, min(n, q // p))
        except Exception:
            pass
    return n


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm = sorted(int(r[1]) for r in rows if len(r) > 8 and r[1].isdigit())
        reasons = set()
        for r in rows:
            if len(r) > 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip() == "Active":
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(rows[0][2]) if rows and rows[0][2].isdigit() else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class OutputDump:
    """--dump-outputs: the SAM text of one step as float64 arrays, so that two builds can be compared output for output.
    The three streams (0 main, 1 splitters, 2 discordants) are taken over all batches in input order:
      summary.npy  [3, 3]: per stream [records, bytes, CRC-32 of the text]
      records.npy  [n, 11]: one row per record: stream, pair id, FLAG, RNAME, POS, MAPQ, CRC-32 of CIGAR, RNEXT, PNEXT, TLEN,
                   CRC-32 of the whole line (contigs numbered from 0, '*' = -1).  Main stream: every record of a fixed, seeded
                   sample of DUMP_PAIRS read pairs.  Side streams: every record (they are small; a few per million reads are
                   splitters, which no pair sample would reliably hit), a fixed, seeded sample of DUMP_SIDE_RECORDS beyond that."""

    def __init__(self, pair_ids):
        rng = np.random.default_rng(7)
        self.keep = np.sort(rng.choice(pair_ids, min(DUMP_PAIRS, len(pair_ids)), replace=False))
        self.summary = np.zeros((3, 3))
        self.rows = [[] for _ in range(3)]
        self.ctg = {c.encode(): i for i, c in enumerate(CONTIGS)}
        self.ctg[b"*"] = -1

    def add(self, k, text):
        """text: one batch's stream k, any buffer (read in place, not copied)"""
        buf = np.frombuffer(text, np.uint8)
        ends = np.flatnonzero(buf == 10)
        starts = np.concatenate(([0], ends[:-1] + 1)) if len(ends) else ends
        self.summary[k] += [len(ends), len(buf), 0]
        self.summary[k, 2] = zlib.crc32(buf, int(self.summary[k, 2]))
        if k == 0:
            ids = (buf[starts[:, None] + np.arange(1, 10)].astype(np.int64) - 48) @ 10 ** np.arange(8, -1, -1, dtype=np.int64)  # QNAME p%09d
            sel = np.isin(ids, self.keep)
            starts, ends = starts[sel], ends[sel]
        for s, e in zip(starts, ends):
            line = buf[s:e].tobytes()
            f = line.split(b"\t")
            rname = self.ctg[f[2]]
            self.rows[k].append((k, int(f[0][1:]), int(f[1]), rname, int(f[3]), int(f[4]), zlib.crc32(f[5]), rname if f[6] == b"=" else self.ctg[f[6]],
                                 int(f[7]), int(f[8]), zlib.crc32(line)))

    def write(self, d):
        rows = [np.array(r, np.float64).reshape(-1, 11) for r in self.rows]
        for k in (1, 2):
            if len(rows[k]) > DUMP_SIDE_RECORDS:
                rows[k] = rows[k][np.sort(np.random.default_rng(7 + k).choice(len(rows[k]), DUMP_SIDE_RECORDS, replace=False))]
        arrays = {"summary": self.summary, "records": np.concatenate(rows)}
        total = sum(a.nbytes for a in arrays.values())
        if total > DUMP_MAX_BYTES:
            raise SystemExit("bench.py: --dump-outputs would write %d bytes, more than %d" % (total, DUMP_MAX_BYTES))
        os.makedirs(d, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(d, name + ".npy"), a)


# ---------------------------------------------------------------------------------- CPU arm ----
def oracle_lib():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ssq_testlib as T  # the oracle's ctypes bindings live with the tests (test infrastructure)
    return T


def cpu_arm(T, o, oidx, fa, batch, n, threads):
    """oracle `bwa mem` (threads) piped through the oracle's samblaster on the first n reads of `batch`;
    returns (reads/s, seconds, (main, splitters, discordants) record text)"""
    rl = READ_LEN
    seqs = [bytes(batch.seq.numpy()[i * rl:(i + 1) * rl]).decode() for i in range(n)]
    names = batch.names[:n]
    quals = ["I" * rl] * n
    t0 = time.time()
    body = o.mem_pe(oidx, names, seqs, quals, 0, threads, b"bench")
    t_mem = time.time() - t0
    hdr = "".join("@SQ\tSN:%s\tLN:%d\n" % (l.split()[1], int(m.split()[1])) for l, m in zip(*[iter(open(fa + ".ann").read().splitlines()[1:])] * 2))
    with tempfile.TemporaryDirectory() as d:
        spl, disc = os.path.join(d, "s"), os.path.join(d, "d")
        t0 = time.time()
        out = subprocess.run([T.ORACLE_BIN, "samblaster"] + SB_ARGS + ["--splitterFile", spl, "--discordantFile", disc], input=(hdr + body).encode(), check=True,
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL).stdout
        t_sb = time.time() - t0
        rec = lambda b: b"".join(l for l in b.splitlines(True) if not l.startswith(b"@"))
        streams = (rec(out), rec(open(spl, "rb").read()), rec(open(disc, "rb").read()))
    dt = t_mem + t_sb
    return n / dt, dt, streams, (t_mem, t_sb)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--batch", type=int, default=2_000_000)
    ap.add_argument("--genome-len", type=int, default=int(os.environ.get("SSQ_BENCH_GENOME", GENOME_LEN)))
    ap.add_argument("--cache", default=os.environ.get("SSQ_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "ssq_bench_cache_%d" % os.getuid())),
                    help="directory for the synthetic reference and its index (reused by later runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the SAM records of the last step as .npy arrays (class OutputDump)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads in the CPU-arm sample (0: sized for ~15 s)")
    ap.add_argument("--streams", type=int, default=int(os.environ.get("SSQ_BENCH_STREAMS", "5")), help="host threads / CUDA streams that drive batches concurrently")
    a = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ncores = usable_cores()
    nb = max(1, a.reads // a.batch)
    workload = "%dM synthetic 2x%dbp PE reads (10%% duplicate pairs, 1%% chimeric) vs synthetic %d bp reference (8 contigs, planted repeats), full `bwa mem | samblaster` path: align + pair + CIGAR + dup-mark + discordant/splitter streams + SAM text" % (nb * a.batch // 1_000_000, READ_LEN, a.genome_len)
    metric = "150bp PE reads/sec aligned+dupmarked"
    import torch

    if a.impl == "reference":
        if rank != 0:
            return 0
        T = oracle_lib()
        o = T.Oracle()

        def build(f):  # index construction is set-up, not the timed path: the GPU builder when a GPU is present (the oracle's SA-IS takes minutes beyond 100 Mbp)
            if torch.cuda.is_available():
                capi.SSQ().index_build(f, None, local)
            else:
                o.index_build(f)
        fa, g = ensure_reference(a.cache, a.genome_len, build)
        oidx = o.load(fa)
        n_s = a.cpu_sample or 400000
        b0 = Batch(torch, fast_pairs(g, n_s // 2, READ_LEN, 1000), 0, pin=False)
        rates, desc = [], ""
        n_try = min(n_s, 40000)
        r, dt, _, _ = cpu_arm(T, o, oidx, fa, b0, n_try, ncores)
        n_run = int(min(n_s, max(n_try, r * 8.0))) & ~1  # ~8 s per step
        for s in range(a.warmup + a.steps):
            n = n_run if s >= a.warmup else min(n_run, 20000)
            r, dt, streams, parts = cpu_arm(T, o, oidx, fa, b0, n, ncores)
            if s >= a.warmup:
                rates.append(r)
                desc = "%d reads per step (a batch of the same generator as the workload), bwa-mem port on %d threads %.1f s + samblaster port (1 thread, like the reference) %.1f s" % (n, ncores, parts[0], parts[1])
        if a.dump_outputs:
            dump = OutputDump(np.arange(n // 2))
            for k in range(3):
                dump.add(k, streams[k])
            dump.write(a.dump_outputs)
        v = float(np.mean(rates))
        print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": "reads/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                          "ms_per_step": 1000.0 * n_run / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                          "config": {"workload": workload, "note": "CPU arm: oracle port of bwa mem | samblaster (their sources are not vendored in the reference tree); each step = the bounded sample in cpu_baseline.sample, ms_per_step is that sample's time"},
                          "cpu_baseline": {"value": v, "unit": "reads/s", "cores": ncores, "kind": "port", "sample": desc},
                          "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    s = capi.SSQ()
    L = s.lib
    if rank == 0:
        fa, g = ensure_reference(a.cache, a.genome_len, lambda f: s.index_build(f, None, local))
    if world > 1:
        dist.barrier()
    if rank != 0:
        fa, g = ensure_reference(a.cache, a.genome_len, lambda f: s.index_build(f, None, local))
    t0 = time.time()
    idx = s.index_load(fa, local)
    t_load = time.time() - t0
    # batches: pinned host copies + one aligner object (own stream, own scratch) per batch, all sharing one dup-set
    nstreams = max(1, min(a.streams, nb, max(1, ncores // max(1, world))))
    L.ssq_dupset_create.argtypes = [C.c_int, C.c_void_p]
    L.ssq_comm_dupset.restype = C.c_void_p
    L.ssq_comm_dupset.argtypes = [C.c_void_p]
    L.ssq_comm_counter.restype = C.c_uint64
    L.ssq_comm_counter.argtypes = [C.c_void_p, C.c_int]
    dset, comm = C.c_void_p(), None
    if world > 1:  # the duplicate stage of every batch is one round of libssq's NCCL exchange (csrc/ssq_dist.cu): rank 0 makes the id, torch carries it
        idb = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = (C.c_uint8 * 128)()
            s.ck(L.ssq_comm_unique_id(buf), "ssq_comm_unique_id")
            idb = torch.tensor(list(buf), dtype=torch.uint8)
        idb = idb.cuda()
        dist.broadcast(idb, 0)
        comm = C.c_void_p()
        s.ck(L.ssq_comm_create(bytes(idb.cpu().tolist()), C.c_int(rank), C.c_int(world), C.c_int(local), C.byref(comm)), "ssq_comm_create")
        dset = C.c_void_p(L.ssq_comm_dupset(comm))
    else:
        s.ck(L.ssq_dupset_create(local, C.byref(dset)), "ssq_dupset_create")
    L.ssq_aligner_set_turn.argtypes = [C.c_void_p, C.c_longlong]
    batches, aligners = [], []
    pool0 = None
    for b in range(nb):
        codes = fast_pairs(g, a.batch // 2, READ_LEN, 1000 + rank * 100 + b, dup_pool=pool0)
        if b == 0:
            pool0 = codes[: a.batch // 4 + 2].copy()
        batches.append(Batch(torch, codes, (b * world + rank) * (a.batch // 2)))  # round b: rank r holds global batch b * world + r
        al = s.aligner_create(idx, SB, b"bench")
        if comm is not None:
            s.ck(L.ssq_aligner_set_comm(al, comm), "ssq_aligner_set_comm")
        else:
            s.ck(L.ssq_aligner_share_dupset(al, dset), "ssq_aligner_share_dupset")
        aligners.append(al)
    exts = [torch.cuda.ExternalStream(L.ssq_aligner_stream(al)) for al in aligners]
    for al, bt in zip(aligners, batches):
        s.ck(L.ssq_aligner_upload(al, C.byref(bt.reads)), "ssq_aligner_upload")
    n_reads_step = nb * a.batch
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(nstreams)

    def lanes(fn):
        for f in [pool.submit(fn, k) for k in range(nstreams)]:
            f.result()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        s.ck(L.ssq_dupset_reset(dset), "ssq_dupset_reset")

        def one(k):
            torch.cuda.set_device(local)
            for b in range(k, nb, nstreams):
                L.ssq_aligner_set_turn(aligners[b], b)
                s.ck(L.ssq_aligner_compute(aligners[b], None, 0), "ssq_aligner_compute")
        lanes(one)

    def span_ms(ev):
        return max(ev[i][0].elapsed_time(ev[j][1]) for i in range(nb) for j in range(nb))

    # ---- value: HBM-resident ----
    for _ in range(a.warmup):
        step_resident()
    barrier()
    clk = ClockSampler(local)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nb)]
    for k in range(nb):
        ev[k][0].record(exts[k])
    for _ in range(a.steps):
        step_resident()
    for k in range(nb):
        ev[k][1].record(exts[k])
    barrier()
    ms_total = span_ms(ev)
    clocks = clk.stop()
    if a.dump_outputs and rank == 0:  # what the last timed step left in each aligner: rank 0's batches
        dump = OutputDump(np.concatenate([(b * world + rank) * (a.batch // 2) + np.arange(a.batch // 2) for b in range(nb)]))
        sam = capi.Sam()
        for al in aligners:
            s.ck(L.ssq_aligner_fetch(al, C.byref(sam)), "ssq_aligner_fetch")
            for k in range(3):
                dump.add(k, (C.c_char * sam.len[k]).from_address(sam.text[k]))
        dump.write(a.dump_outputs)
    # ---- per-stage statistics: one extra step, batches one after the other so that stage durations are not stretched by overlap ----
    STAGES = ["upload", "seed_chain_extend", "sort_dedup_patch", "insert_size_stats", "mate_rescue", "pair_mapq_plan", "cigar_nm_md", "samblaster_dupset", "sam_text", "fetch",
              "k_smem", "k_sa", "k_chain", "k_extend", "k_select"]
    stage_ms = np.zeros(len(STAGES))
    counters = np.zeros(12)
    n_tasks = text_bytes = n_rescue = n_gapped = n_swl = swl_cells = 0
    bwd_blocks = bwd_us = 0
    out = capi.Sam()
    s.ck(L.ssq_dupset_reset(dset), "reset")
    for b, al in enumerate(aligners):
        L.ssq_aligner_set_turn(al, b)
        s.ck(L.ssq_aligner_compute(al, None, 0), "compute")
        s.ck(L.ssq_aligner_fetch(al, C.byref(out)), "fetch")
        stage_ms += [L.ssq_aligner_stage_ms(al, i) for i in range(len(STAGES))]
        counters += [L.ssq_aligner_counter(al, i) for i in range(12)]
        n_tasks += L.ssq_aligner_counter(al, 100)
        text_bytes += sum(L.ssq_aligner_counter(al, 101 + k) for k in range(3))
        n_rescue += L.ssq_aligner_counter(al, 105)
        n_gapped += L.ssq_aligner_counter(al, 106)
        bwd_blocks += L.ssq_aligner_counter(al, 25)
        bwd_us += L.ssq_aligner_counter(al, 26)
        n_swl += L.ssq_aligner_counter(al, 107)
        swl_cells += L.ssq_aligner_counter(al, 108)
    dup_frac_seen = None
    # ---- e2e: host buffers through the C-ABI (upload + compute + fetch per batch) ----
    d2h_step = [0]

    def step_e2e():
        s.ck(L.ssq_dupset_reset(dset), "ssq_dupset_reset")
        tot = [0] * nstreams

        def one(k):
            torch.cuda.set_device(local)
            o = capi.Sam()
            for b in range(k, nb, nstreams):
                L.ssq_aligner_set_turn(aligners[b], b)
                s.ck(L.ssq_aligner_upload(aligners[b], C.byref(batches[b].reads)), "upload")
                s.ck(L.ssq_aligner_compute(aligners[b], None, 0), "compute")
                s.ck(L.ssq_aligner_fetch(aligners[b], C.byref(o)), "fetch")
                tot[k] += int(o.len[0]) + int(o.len[1]) + int(o.len[2]) + (a.batch + 1) * 8
        lanes(one)
        d2h_step[0] = sum(tot)
    step_e2e()
    barrier()
    ee = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nb)]
    for k in range(nb):
        ee[k][0].record(exts[k])
    for _ in range(a.steps):
        step_e2e()
    for k in range(nb):
        ee[k][1].record(exts[k])
    barrier()
    ms_e2e = span_ms(ee)
    h2d = sum(bt.h2d for bt in batches)
    tmax = torch.tensor([ms_total, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = float(tmax[0]), float(tmax[1])
    value = world * n_reads_step * a.steps / (ms_total / 1000.0)
    e2e_v = world * n_reads_step * a.steps / (ms_e2e / 1000.0)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        blk = float(L.ssq_index_info(idx, 7))
        st = dict(zip(STAGES, (stage_ms / nb).tolist()))
        fq_bytes = sum(bt.h2d for bt in batches) / nb
        kern = {
            "k_smem (seeding, all passes)": {"ms": st["k_smem"], "bytes": blk * counters[0] / nb},
            "k_smem_bwd (backward sweeps, 2 launches)": {"ms": bwd_us / 1000.0 / nb, "bytes": blk * bwd_blocks / nb, "part_of": "k_smem"},
            "k_sa (SA look-up)": {"ms": st["k_sa"], "bytes": (blk * counters[1] + float(L.ssq_index_info(idx, 8)) * counters[2]) / nb},
            "k_chain": {"ms": st["k_chain"], "bytes": None},
            "k_extend (ksw_extend2)": {"ms": st["k_extend"], "bytes": counters[5] / nb, "gcups": counters[4] / nb / (st["k_extend"] * 1e6) if st["k_extend"] else None,
                                       # ALU roofline: ~16 integer lane-operations per DP cell (SASS of k_ext_run's inner loop) against 148 SMs x 128 lanes x clock
                                       "roofline": {"bound": "alu", "unit": "G lane-ops/s", "ops_per_cell": 16, "achieved": 16 * counters[4] / nb / (st["k_extend"] * 1e6) if st["k_extend"] else None,
                                                    "peak": 148 * 128 * 1.965, "frac": (16 * counters[4] / nb / (st["k_extend"] * 1e6)) / (148 * 128 * 1.965) if st["k_extend"] else None}},
            "k_select": {"ms": st["k_select"], "bytes": None},
            "k_dedup (sort/dedup/patch)": {"ms": st["sort_dedup_patch"], "bytes": None},
            "k_pestat + host reduction": {"ms": st["insert_size_stats"], "bytes": None},
            "k_rescue (mate rescue, ksw_align2)": {"ms": st["mate_rescue"], "bytes": None, "gcups": swl_cells / nb / (st["mate_rescue"] * 1e6) if st["mate_rescue"] else None},
            "k_plan (primary/pair/MAPQ)": {"ms": st["pair_mapq_plan"], "bytes": None},
            "k_cigar (ksw_global2 + traceback)": {"ms": st["cigar_nm_md"], "bytes": None},
            "k_sb + dup-set (radix sort + mark)": {"ms": st["samblaster_dupset"], "bytes": 25.0 * a.batch / 2},
            "k_text (SAM records, 3 streams)": {"ms": st["sam_text"], "bytes": 2.0 * text_bytes / nb + fq_bytes},
        }
        tot_ms = sum(k["ms"] for k in kern.values() if "part_of" not in k)
        for k in kern.values():
            k["share_of_step"] = k["ms"] / tot_ms if tot_ms else None
            k["achieved_GBps"] = (k["bytes"] / (k["ms"] * 1e-3) / 1e9) if k["bytes"] and k["ms"] else None
        # the single dominant kernel: the backward sweeps of the seeding when the split seeding ran (their own events / block counter), else the stage
        cand = [k for k in kern if kern[k]["bytes"] is not None and not (k == "k_smem (seeding, all passes)" and bwd_us)]
        dom = max(cand, key=lambda k: kern[k]["ms"])
        traffic = None
        try:  # DRAM bytes of the same kernel from the committed `ncu --set full` capture (same batch size and reference)
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            if dom in tj and a.batch == tj["batch_reads"] and a.genome_len == tj["genome_bp"]:
                traffic = tj[dom]["dram_bytes_read"] + tj[dom]["dram_bytes_write"]
        except Exception:
            pass
        ach = kern[dom]["achieved_GBps"] or 0.0
        rnd = None
        try:  # what this device serves when the reads are dependent random 32-byte sectors over a table of the rank structure's size (measured, profiles/)
            rj = json.load(open(os.path.join(ROOT, "profiles", "r02_random_sector.json")))
            tab_gb = a.genome_len * 2 * 32 / 64 / 2**30  # 32 bytes per 64 BWT symbols, both strands
            key = min(rj["table_GB"], key=lambda k: abs(float(k) - tab_gb))
            if "k_smem" in dom and abs(float(key) - tab_gb) < 0.25 * tab_gb:
                rnd = {"GBps": rj["table_GB"][key], "table_GB": float(key), "frac_of_ceiling": ach / rj["table_GB"][key], "source": "profiles/r02_random_sector.log (tools/random_sector_bench.cu)"}
        except Exception:
            pass
        res = {"metric": metric, "value": value, "unit": "reads/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_total / a.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
               "config": {"workload": workload, "batch_reads": a.batch, "batches_per_step": nb, "streams": nstreams, "genome_bp": a.genome_len,
                          "l2": "inputs + scratch per step exceed L2 (%.1f GB of FASTQ fields, %.1f GB of SAM text per step)" % (h2d / 1e9, text_bytes / 1e9),
                          "index": "replicated per GPU, %.0f MB on the device, loaded in %.1f s" % (L.ssq_index_info(idx, 6) / 1e6, t_load),
                          "parallelism": ("batches dealt round-robin to %d ranks, index replicated; duplicate stage = one NCCL exchange per round (signatures to owner rank hash mod N, 16 B/pair out, 1 B/pair back): rank 0 sent %.1f MB / received back %.1f MB per step" % (world, L.ssq_comm_counter(comm, 0) / 1e6 / max(1, L.ssq_comm_counter(comm, 2) // nb), L.ssq_comm_counter(comm, 1) / 1e6 / max(1, L.ssq_comm_counter(comm, 2) // nb))) if comm is not None else "single GPU: no collective",
                          "samblaster": " ".join(SB_ARGS)},
               "clocks": clocks, "gpu_launches": int(counters[6]) * a.steps + 16 * nb * a.steps,  # seed..extend launches counted by the library + the 16 pipeline kernels of a batch (k_dedup .. k_text; CUB scans / sorts not counted)
               "e2e": {"value": e2e_v, "unit": "reads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_step[0], "ms_per_step": ms_e2e / a.steps},
               "roofline": {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                            "peak_source": peak_src, "algorithmic_bytes_per_launch": kern[dom]["bytes"], "launch_ms": kern[dom]["ms"], "rank_block_bytes": blk,
                            "access_pattern": "dependent random 32-byte sector reads (one or two rank blocks per FM-index extension)", "random_sector_ceiling": rnd},
               "kernels": kern,
               "work_per_step": {"occ_blocks_smem": counters[0], "occ_blocks_sa": counters[1], "sa_samples": counters[2], "sw_calls": counters[3], "sw_cells": counters[4], "seeds": counters[7],
                                 "alignments_written": n_tasks, "sam_bytes": text_bytes, "pairs_through_mate_rescue": n_rescue, "alignments_with_banded_dp": n_gapped, "rescue_sw_passes": n_swl, "rescue_sw_cells": swl_cells},
               "kernel_stats_note": "kernels{} come from one extra step after the timed region with the batches run one after the other (stage boundaries by CUDA events on each batch's stream)"}
        if world == 1 and not a.no_cpu_baseline:
            T = oracle_lib()
            o = T.Oracle()
            oidx = o.load(fa)
            n_try = 20000
            smp = Batch(torch, fast_pairs(g, 200000, READ_LEN, 999), 0, pin=False)  # a 400 k-read sample from the same generator as the batches
            r, dt, _, _ = cpu_arm(T, o, oidx, fa, smp, n_try, ncores)
            n = a.cpu_sample or int(min(400000, max(n_try, r * 15.0))) & ~1
            v, dt, ref, parts = cpu_arm(T, o, oidx, fa, smp, n, ncores)
            res["cpu_baseline"] = {"value": v, "unit": "reads/s", "cores": ncores, "kind": "port",
                                   "sample": "%d reads (a batch of the same generator as the workload), bwa-mem port on %d threads %.1f s + samblaster port (1 thread) %.1f s" % (n, ncores, parts[0], parts[1])}
            # parity at bench scale: the same sample as its own batch through the product
            al = s.aligner_create(idx, SB, b"bench")
            rd, keep = capi.pack_reads(smp.names[:n], [bytes(smp.seq.numpy()[i * READ_LEN:(i + 1) * READ_LEN]) for i in range(n)], ["I" * READ_LEN] * n, None, 1, 0)
            got, info = s.aligner_run(al, rd)
            s.aligner_free(al)
            same = [got[k] == ref[k] for k in range(3)]
            res["parity"] = {"reads_checked": n, "identical": all(same), "streams": dict(zip(("main", "splitters", "discordants"), same)),
                             "sam_bytes_compared": sum(len(x) for x in ref), "dup_pairs_in_sample": info["n_dup"]}
            if not all(same):
                print(json.dumps(res))
                raise SystemExit("bench.py: GPU output differs from the oracle on the CPU-baseline sample")
        print(json.dumps(res))
    for al in aligners:
        s.aligner_free(al)
    if comm is not None:
        L.ssq_comm_free(comm)
    else:
        L.ssq_dupset_free(dset)
    s.index_free(idx)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
