"""Shared helpers for the test-suite: ctypes bindings of the oracle (oracle/libssqo.so), of the product's C-ABI
(speedseq_b200/libssq.so) and of the test-only host harness (tests/hostsim/libhostsim.so), plus seeded read/genome
generators.  Nothing here reads /root/reference at run time."""
import ctypes as C
import gzip
import os
import subprocess
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
ORACLE_SO = os.path.join(ROOT, "oracle", "libssqo.so")
ORACLE_BIN = os.path.join(ROOT, "oracle", "ssqo")
HOSTSIM_SO = os.path.join(ROOT, "tests", "hostsim", "libhostsim.so")
SSQ_SO = os.path.join(ROOT, "speedseq_b200", "libssq.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")

from speedseq_b200.capi import SMEM_DT, SEED_DT, SWTASK_DT, SWRES_DT, REG_DT, DUPSIG_DT, SSQ, pack_reads  # noqa: E402,F401  (the product's own bindings)
ODUPSIG_DT = np.dtype([("pos1", "<u8"), ("pos2", "<u8"), ("strand1", "u1"), ("strand2", "u1"), ("valid", "u1")], align=True)


def gpu_visible():
    """a CUDA device is usable from this process, as the CUDA runtime sees it (a process's GPU need not be /dev/nvidia0)"""
    import torch
    return torch.cuda.is_available()


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])


def build_hostsim():
    d = os.path.join(ROOT, "tests", "hostsim")
    src, out = os.path.join(d, "hostsim.cpp"), HOSTSIM_SO
    hdrs = [os.path.join(ROOT, "speedseq_b200", "csrc", f) for f in ("ssq_dev.cuh", "ssq_dev2.cuh", "ssq_dev3.cuh", "ssq_pipe_host.h")]
    if not os.path.exists(out) or os.path.getmtime(out) < max([os.path.getmtime(src), os.path.getmtime(ORACLE_SO)] + [os.path.getmtime(h) for h in hdrs]):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-w", "-pthread", "-o", out, src, "-L" + os.path.join(ROOT, "oracle"), "-lssqo",
                               "-Wl,-rpath," + os.path.join(ROOT, "oracle")])


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    def __init__(self):
        build_oracle()
        self.lib = C.CDLL(ORACLE_SO)
        L = self.lib
        L.ssqo_idx_load.restype = C.c_void_p
        L.ssqo_idx_load.argtypes = [C.c_char_p]
        L.ssqo_idx_destroy.argtypes = [C.c_void_p]
        L.ssqo_index_build.argtypes = [C.c_char_p, C.c_char_p]
        L.ssqo_api_idx_info.restype = C.c_uint64
        L.ssqo_api_idx_info.argtypes = [C.c_void_p, C.c_int]
        for f in ("ssqo_api_smem_batch", "ssqo_api_chain_batch", "ssqo_api_align_batch"):
            getattr(L, f).restype = C.c_int64
        L.ssqo_api_mem_pe.restype = C.c_void_p
        L.ssqo_api_free.argtypes = [C.c_void_p]

    def index_build(self, fasta, prefix=None):
        rc = self.lib.ssqo_index_build(fasta.encode(), (prefix or fasta).encode())
        assert rc == 0, rc

    def load(self, prefix):
        h = self.lib.ssqo_idx_load(prefix.encode())
        assert h, "oracle failed to load " + prefix
        return h

    def info(self, idx, what):
        return int(self.lib.ssqo_api_idx_info(C.c_void_p(idx), what))

    def smem_batch(self, idx, seq, off, lib=None, fn="ssqo_api_smem_batch"):
        L = lib or self.lib
        n = len(off) - 1
        cap = max(1024, 64 * n)
        while True:
            out = np.zeros(cap, SMEM_DT)
            ooff = np.zeros(n + 1, np.uint64)
            f = getattr(L, fn)
            f.restype = C.c_int64
            r = f(C.c_void_p(idx), C.c_int(n), _ptr(seq), _ptr(off), _ptr(out), C.c_uint64(cap), _ptr(ooff))
            if r >= 0:
                return out[:r], ooff
            cap *= 4

    def sa_batch(self, idx, rows):
        pos = np.zeros(len(rows), np.uint64)
        self.lib.ssqo_api_sa_batch(C.c_void_p(idx), C.c_uint64(len(rows)), _ptr(rows), _ptr(pos))
        return pos

    def sw_extend_batch(self, tasks, qbuf, tbuf, lib=None, fn="ssqo_api_sw_extend_batch"):
        L = lib or self.lib
        res = np.zeros(len(tasks), SWRES_DT)
        getattr(L, fn)(C.c_uint64(len(tasks)), _ptr(tasks), _ptr(qbuf), _ptr(tbuf), _ptr(res))
        return res

    def chain_batch(self, idx, seq, off, lib=None, fn="ssqo_api_chain_batch"):
        L = lib or self.lib
        n = len(off) - 1
        scap, ccap = max(4096, 256 * n), max(1024, 64 * n)
        while True:
            seeds = np.zeros(scap, SEED_DT)
            cso = np.zeros(ccap + 1, np.uint64)
            rco = np.zeros(n + 1, np.uint64)
            f = getattr(L, fn)
            f.restype = C.c_int64
            r = f(C.c_void_p(idx), C.c_int(n), _ptr(seq), _ptr(off), _ptr(seeds), C.c_uint64(scap), _ptr(cso), C.c_uint64(ccap), _ptr(rco))
            if r >= 0:
                return seeds[: int(cso[r])], cso[: r + 1], rco
            scap *= 4
            ccap *= 4

    def align_batch(self, idx, seq, off, stage=0, threads=8):
        n = len(off) - 1
        cap = max(1024, 16 * n)
        while True:
            out = np.zeros(cap, REG_DT)
            ooff = np.zeros(n + 1, np.uint64)
            r = self.lib.ssqo_api_align_batch(C.c_void_p(idx), C.c_int(n), _ptr(seq), _ptr(off), C.c_int(stage), _ptr(out), C.c_uint64(cap), _ptr(ooff), C.c_int(threads))
            if r <= cap:
                return out[:r], ooff
            cap = int(r) + 16

    def mem_pe(self, idx, names, seqs, quals, n_processed=0, threads=8, rg_id=b""):
        n = len(names)
        arr = lambda xs: (C.c_char_p * n)(*[x if isinstance(x, bytes) else x.encode() for x in xs])
        p = self.lib.ssqo_api_mem_pe(C.c_void_p(idx), C.c_int(n), arr(names), arr(seqs), arr(quals), C.c_int64(n_processed), C.c_int(threads), rg_id)
        s = C.string_at(p).decode()
        self.lib.ssqo_api_free(C.c_void_p(p))
        return s

    def dupmark(self, sig):
        o = np.zeros(len(sig), ODUPSIG_DT)
        for k in ("pos1", "pos2", "strand1", "strand2", "valid"):
            o[k] = sig[k]
        d = np.zeros(len(sig), np.uint8)
        self.lib.ssqo_dupmark(C.c_size_t(len(sig)), _ptr(o), _ptr(d))
        return d


class HostSim:
    """test-only host build of the kernels' routines (see tests/hostsim/hostsim.cpp)"""
    def __init__(self, oracle):
        build_hostsim()
        self.o = oracle
        self.lib = C.CDLL(HOSTSIM_SO)

    def smem_batch(self, idx, seq, off):
        return self.o.smem_batch(idx, seq, off, lib=self.lib, fn="hostsim_smem_batch")

    def chain_batch(self, idx, seq, off):
        return self.o.chain_batch(idx, seq, off, lib=self.lib, fn="hostsim_chain_batch")

    def sw_extend_batch(self, tasks, qbuf, tbuf):
        return self.o.sw_extend_batch(tasks, qbuf, tbuf, lib=self.lib, fn="hostsim_sw_extend_batch")

    def mem_pe(self, idx, names, seqs, quals, n_processed=0, rg_id=b"", paired=1):
        n = len(names)
        arr = lambda xs: (C.c_char_p * n)(*[x if isinstance(x, bytes) else x.encode() for x in xs])
        self.lib.hostsim_mem_pe.restype = C.c_void_p
        p = self.lib.hostsim_mem_pe(C.c_void_p(idx), C.c_int(n), arr(names), arr(seqs), arr(quals), C.c_int64(n_processed), rg_id, C.c_int(paired))
        assert p, "hostsim_mem_pe failed"
        s = C.string_at(p).decode()
        self.o.lib.ssqo_api_free(C.c_void_p(p))
        return s

    def pipe(self, idx, names, seqs, quals, n_processed=0, rg_id=b"", paired=1, sb=(1, 1, 2, 20, 0), reset=1, comments=None, pes=None):
        """the fused `bwa mem | samblaster` pipeline (bodies of ssq_pipe.cu's kernels run on the host) -> (main, splitters, discordants)
        sb = (excludeDups, addMateTags, maxSplitCount, minNonOverlap, removeDups); pes = 4 x (low, high, failed, avg, std) for -I"""
        n = len(names)
        arr = lambda xs: (C.c_char_p * n)(*[x if isinstance(x, bytes) else x.encode() for x in xs])
        outs = [C.c_void_p() for _ in range(3)]
        sbv = (C.c_int * 5)(*sb)
        pv = (C.c_double * 20)(*[float(x) for row in pes for x in row]) if pes is not None else None
        rc = self.lib.hostsim_pipe(C.c_void_p(idx), C.c_int(n), arr(names), arr(seqs), arr(quals) if quals is not None else None, arr(comments) if comments is not None else None,
                                   C.c_int64(n_processed), rg_id, C.c_int(paired), sbv, C.c_int(reset), pv, C.byref(outs[0]), C.byref(outs[1]), C.byref(outs[2]))
        assert rc == 0, "hostsim_pipe failed: flags 0x%x" % rc
        res = []
        for o in outs:
            res.append(C.string_at(o).decode())
            self.o.lib.ssqo_api_free(o)
        return tuple(res)

    def pipe_bam(self, *a, blank_side=1, **kw):
        """like pipe(), additionally the coordinate-sorted BAM records of the three streams (bytes)"""
        self.lib.hostsim_pipe_want_bam(C.c_int(1), C.c_int(blank_side))
        try:
            txt = self.pipe(*a, **kw)
        finally:
            self.lib.hostsim_pipe_want_bam(C.c_int(0), C.c_int(1))
        self.lib.hostsim_pipe_bam.restype = C.c_uint64
        bams = []
        for k in range(3):
            n = int(self.lib.hostsim_pipe_bam(C.c_int(k), None, C.c_uint64(0)))
            buf = C.create_string_buffer(max(n, 1))
            self.lib.hostsim_pipe_bam(C.c_int(k), buf, C.c_uint64(n))
            bams.append(buf.raw[:n])
        return txt, tuple(bams)

    def align_batch(self, idx, seq, off):
        n = len(off) - 1
        cap = max(1024, 16 * n)
        self.lib.hostsim_align_batch.restype = C.c_int64
        while True:
            out = np.zeros(cap, REG_DT)
            ooff = np.zeros(n + 1, np.uint64)
            r = self.lib.hostsim_align_batch(C.c_void_p(idx), C.c_int(n), _ptr(seq), _ptr(off), _ptr(out), C.c_uint64(cap), _ptr(ooff))
            if r >= 0:
                return out[:r], ooff
            cap *= 4


# ------------------------------------------------------------------------------------ data ----
_NT4 = np.full(256, 4, np.uint8)
for _i, _c in enumerate("ACGT"):
    _NT4[ord(_c)] = _i
    _NT4[ord(_c.lower())] = _i


def encode_reads(seqs):
    """list of ASCII strings -> (concatenated nt4 codes, offsets)"""
    off = np.zeros(len(seqs) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    buf = np.frombuffer("".join(seqs).encode(), np.uint8)
    return _NT4[buf].copy(), off


def synth_genome(n, seed, n_contigs=1, repeat_frac=0.08):
    """seeded synthetic genome with planted diverged repeats so that seeds are not all unique"""
    rng = np.random.default_rng(seed)
    g = rng.choice(4, size=n, p=[0.295, 0.205, 0.205, 0.295]).astype(np.uint8)
    fam = rng.integers(0, 4, 300, dtype=np.uint8)
    n_rep = int(n * repeat_frac / 300)
    for _ in range(n_rep):
        p = int(rng.integers(0, max(1, n - 300)))
        c = fam.copy()
        m = rng.random(300) < 0.08
        c[m] = rng.integers(0, 4, int(m.sum()), dtype=np.uint8)
        g[p:p + 300] = c[: len(g[p:p + 300])]
    if n > 5000:  # one exact tandem duplication and one microsatellite
        g[2000:2400] = g[1000:1400]
        g[3000:3060] = np.tile(np.array([0, 1], np.uint8), 30)
    bounds = np.linspace(0, n, n_contigs + 1).astype(int)
    return g, bounds


def write_fasta(path, g, bounds, names=None):
    acgt = np.frombuffer(b"ACGT", np.uint8)
    with open(path, "w") as f:
        for i in range(len(bounds) - 1):
            f.write(">%s\n" % (names[i] if names else "ctg%d" % (i + 1)))
            s = acgt[g[bounds[i]:bounds[i + 1]]].tobytes().decode()
            for j in range(0, len(s), 60):
                f.write(s[j:j + 60] + "\n")


def simulate_pairs(g, bounds, n_pairs, read_len, seed, ins_mean=400, ins_sd=40, err=0.005, indel=0.0005, n_frac=0.001):
    """wgsim-like paired reads: FR orientation, substitutions, small indels, a few Ns. returns (names, seqs, quals) interleaved"""
    rng = np.random.default_rng(seed)
    comp = np.array([3, 2, 1, 0, 4], np.uint8)
    acgtn = np.frombuffer(b"ACGTN", np.uint8)
    names, seqs, quals = [], [], []
    nc = len(bounds) - 1

    def mutate(x):
        x = x.copy()
        m = rng.random(len(x)) < err
        x[m] = (x[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) % 4
        if rng.random() < indel * len(x):
            p = int(rng.integers(5, len(x) - 5))
            l = int(rng.integers(1, 4))
            if rng.random() < 0.5:
                x = np.concatenate([x[:p], rng.integers(0, 4, l, dtype=np.uint8), x[p:]])[: len(x)]
            else:
                x = np.concatenate([x[:p], x[p + l:], rng.integers(0, 4, l, dtype=np.uint8)])
        m = rng.random(len(x)) < n_frac
        x[m] = 4
        return x

    for i in range(n_pairs):
        c = int(rng.integers(0, nc))
        lo, hi = int(bounds[c]), int(bounds[c + 1])
        ins = max(read_len + 10, int(rng.normal(ins_mean, ins_sd)))
        if hi - lo <= ins + 2:
            ins = hi - lo - 2
        p = int(rng.integers(lo, hi - ins))
        frag = g[p:p + ins]
        r1 = mutate(frag[:read_len])
        r2 = mutate(comp[frag[::-1][:read_len]])
        if rng.random() < 0.5:
            r1, r2 = r2, r1
        nm = "r%d_%d_%d" % (i, c, p - lo)
        for r in (r1, r2):
            names.append(nm)
            seqs.append(acgtn[r].tobytes().decode())
            quals.append("I" * len(r))
    return names, seqs, quals


def write_fastq(path, names, seqs, quals, interleaved_suffix=True):
    op = gzip.open if path.endswith(".gz") else open
    with op(path, "wt") as f:
        for i, (n, s, q) in enumerate(zip(names, seqs, quals)):
            f.write("@%s/%d\n%s\n+\n%s\n" % (n, 1 + (i & 1), s, q))


def extension_tasks(rng, n, qmax=150):
    """random ksw_extend2 problems: related query/target with substitutions and indels, varied h0/band"""
    tasks = np.zeros(n, SWTASK_DT)
    qs, ts = [], []
    qo = to = 0
    for i in range(n):
        ql = int(rng.integers(1, qmax + 1))
        q = rng.integers(0, 4, ql, dtype=np.uint8)
        t = list(q)
        k = rng.random()
        if k < 0.7:  # diverged copy
            j = 0
            out = []
            while j < len(t):
                u = rng.random()
                if u < 0.03:
                    out.append(int(rng.integers(0, 4)))
                    j += 1
                elif u < 0.04:
                    j += int(rng.integers(1, 6))
                elif u < 0.05:
                    out.extend(rng.integers(0, 4, int(rng.integers(1, 6))).tolist())
                else:
                    out.append(int(t[j]))
                    j += 1
            t = out
        else:
            t = rng.integers(0, 4, ql + 20).tolist()
        t = t + rng.integers(0, 4, int(rng.integers(0, 60))).tolist()
        if not t:
            t = [0]
        t = np.array(t, np.uint8)
        if rng.random() < 0.1:
            q[rng.integers(0, ql)] = 4
        if rng.random() < 0.1:
            t[rng.integers(0, len(t))] = 4
        tasks[i] = (qo, to, ql, len(t), int(rng.integers(1, 151)), 100 if rng.random() < 0.8 else int(rng.integers(1, 201)), 5, 100)
        qs.append(q)
        ts.append(t)
        qo += ql
        to += len(t)
    return tasks, np.concatenate(qs), np.concatenate(ts)
