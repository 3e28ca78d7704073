"""GPU parity: every C-ABI entry point of libssq.so against the oracle on the same seeded inputs (bit-exact), at sizes the
oracle finishes in seconds, plus size-independent properties at larger sizes."""
import gzip
import os

import numpy as np
import pytest

import ssq_testlib as T

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu_ex(ssq, ex_index):
    h = ssq.index_load(ex_index)
    yield h
    ssq.index_free(h)


@pytest.fixture(scope="module")
def gpu_syn(ssq, syn_index):
    h = ssq.index_load(syn_index[0])
    yield h
    ssq.index_free(h)


def test_index_upload_matches_files(ssq, oracle, ex_index, gpu_ex):
    idx = oracle.load(ex_index)
    for what in range(6):
        assert int(ssq.lib.ssq_index_info(gpu_ex, what)) == oracle.info(idx, what), what


def test_sa_lookup(ssq, oracle, ex_index, gpu_ex):
    idx = oracle.load(ex_index)
    n = oracle.info(idx, 1)
    rows = np.concatenate([np.arange(0, 3000, dtype=np.uint64), np.random.default_rng(1).integers(0, n + 1, 50000).astype(np.uint64),
                           np.array([oracle.info(idx, 2), n, n - 1], np.uint64)])
    assert np.array_equal(ssq.sa_lookup_batch(gpu_ex, rows), oracle.sa_batch(idx, rows))


def test_sa_lookup_is_a_permutation(ssq, oracle, ex_index, gpu_ex):
    idx = oracle.load(ex_index)
    n = oracle.info(idx, 1)
    pos = ssq.sa_lookup_batch(gpu_ex, np.arange(1, n + 1, dtype=np.uint64))
    assert np.array_equal(np.sort(pos), np.arange(0, n, dtype=np.uint64))


def test_smem_example_reads(ssq, oracle, ex_index, ex_reads, gpu_ex):
    idx = oracle.load(ex_index)
    seq, off = T.encode_reads(ex_reads[1])
    a, ao = oracle.smem_batch(idx, seq, off)
    b, bo = ssq.smem_batch(gpu_ex, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)


def test_smem_edge_cases(ssq, oracle, syn_index, gpu_syn):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    acgt = "ACGT"
    ref = "".join(acgt[x] for x in g[5000:5400])
    seqs = ["", "A", "N" * 30, "ACGT" * 4, ref[:18], ref[:19], ref[:20], ref[:150], "N" + ref[1:150], ref[:75] + "N" + ref[76:150], "AC" * 60,
            ref[:60] + ref[200:290], "".join(acgt[x] for x in g[int(bounds[1]) - 70:int(bounds[1]) + 80]), "T" * 100, ref[:255]]
    seq, off = T.encode_reads(seqs)
    a, ao = oracle.smem_batch(idx, seq, off)
    b, bo = ssq.smem_batch(gpu_syn, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)
    # empty batch
    b, bo = ssq.smem_batch(gpu_syn, np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    assert len(b) == 0


def test_interval_rich_reads(ssq, oracle, syn_index, gpu_syn):
    """low-complexity reads produce more seed intervals than a seeding lane's scratch holds (768): they must be redone by the
    overflow pass, not fail the batch"""
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = T.simulate_pairs(g, bounds, 100, 150, 31, err=0.01)
    seqs = seqs[:60] + ["AC" * 70, "A" * 150, "ACGT" * 37, "AAC" * 50, "AC" * 75] + seqs[60:]
    seq, off = T.encode_reads(seqs)
    a, ao = oracle.smem_batch(idx, seq, off)
    assert int(np.diff(ao).max()) > 768
    b, bo = ssq.smem_batch(gpu_syn, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)
    a, ao = oracle.align_batch(idx, seq, off)
    b, bo = ssq.align_batch(gpu_syn, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)


def test_read_too_long_is_rejected(ssq, gpu_syn):
    seq, off = T.encode_reads(["A" * 256])
    with pytest.raises(RuntimeError, match="rc=-7"):
        ssq.smem_batch(gpu_syn, seq, off)


def test_sw_extend(ssq, oracle):
    rng = np.random.default_rng(5)
    tasks, q, t = T.extension_tasks(rng, 20000, qmax=255)
    assert np.array_equal(ssq.sw_extend_batch(tasks, q, t), oracle.sw_extend_batch(tasks, q, t))
    tasks, q, t = T.extension_tasks(rng, 3000, qmax=20)
    assert np.array_equal(ssq.sw_extend_batch(tasks, q, t), oracle.sw_extend_batch(tasks, q, t))


@pytest.mark.parametrize("rl,seed", [(75, 1), (101, 4), (150, 2), (250, 3)])
def test_chain_and_regions_synthetic(ssq, oracle, syn_index, gpu_syn, rl, seed):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = T.simulate_pairs(g, bounds, 1500, rl, seed, err=0.01, indel=0.002, n_frac=0.003)
    seq, off = T.encode_reads(seqs)
    a = oracle.chain_batch(idx, seq, off)
    b = ssq.chain_batch(gpu_syn, seq, off)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    a, ao = oracle.align_batch(idx, seq, off)
    b, bo = ssq.align_batch(gpu_syn, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)


@pytest.mark.parametrize("heavy_seeds,heavy_tasks", [(2, 1), (8, 4)])
def test_heavy_read_tiers(ssq, oracle, syn_index, gpu_syn, monkeypatch, heavy_seeds, heavy_tasks):
    """Reads with many seeds / many extension tasks are handled by warp-per-read kernels (k_chain_heavy, k_select_heavy).
    Lower their thresholds so that nearly every read takes that route, and a repeat-family batch so chains are plentiful."""
    monkeypatch.setenv("SSQ_HEAVY_SEEDS", str(heavy_seeds))
    monkeypatch.setenv("SSQ_HEAVY_TASKS", str(heavy_tasks))
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = T.simulate_pairs(g, bounds, 1200, 150, 11, err=0.01, indel=0.002, n_frac=0.002)
    rng = np.random.default_rng(5)
    # reads drawn from inside the planted repeat family: find its copies by their shared 40-mer
    gs = "".join("ACGT"[b] for b in g[:200000])
    reps = [seqs[i] for i in range(len(seqs))]
    kmer_hits = {}
    for i in range(0, len(gs) - 32, 7):
        kmer_hits.setdefault(gs[i:i + 24], []).append(i)
    hot = [v for v in kmer_hits.values() if len(v) >= 4]
    for v in hot[:300]:
        p0 = max(0, v[int(rng.integers(0, len(v)))] - int(rng.integers(0, 100)))
        reps.append(gs[p0:p0 + 150])
    reps = [r for r in reps if len(r) >= 40]
    seq, off = T.encode_reads(reps)
    a = oracle.chain_batch(idx, seq, off)
    b = ssq.chain_batch(gpu_syn, seq, off)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    a, ao = oracle.align_batch(idx, seq, off)
    b, bo = ssq.align_batch(gpu_syn, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)


def test_regions_example_reads(ssq, oracle, ex_index, ex_reads, gpu_ex):
    idx = oracle.load(ex_index)
    seq, off = T.encode_reads(ex_reads[1])
    a, ao = oracle.align_batch(idx, seq, off)
    b, bo = ssq.align_batch(gpu_ex, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)
    assert len(a) >= 3900


def test_regions_large_batch_properties(ssq, oracle, syn_index, gpu_syn):
    """60k reads: too slow to compare everything with the scalar oracle in the CPU budget, so check a 2k sample exactly and
    the whole batch through properties: simulated origin recovered, coordinates inside one contig/strand, batch-split invariance"""
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = T.simulate_pairs(g, bounds, 30000, 150, 9)
    seq, off = T.encode_reads(seqs)
    regs, roff = ssq.align_batch(gpu_syn, seq, off)
    l_pac = len(g)
    assert (regs["rb"] < regs["re"]).all() and (regs["qb"] < regs["qe"]).all()
    assert ((regs["re"] <= l_pac) | (regs["rb"] >= l_pac)).all()
    hit = 0
    for i in range(0, len(seqs), 2):
        c, p = int(names[i].split("_")[1]), int(names[i].split("_")[2])
        r = regs[int(roff[i]):int(roff[i + 1])]
        if len(r):
            best = r[np.argmax(r["score"])]
            f = best["rb"] if best["rb"] < l_pac else 2 * l_pac - best["re"]
            hit += abs(int(f) - (int(bounds[c]) + p)) < 700
    assert hit > 0.97 * (len(seqs) // 2)
    # the same reads in two halves give the same regions (no cross-read state)
    h = len(seqs) // 2
    s1, o1 = T.encode_reads(seqs[:h]); s2, o2 = T.encode_reads(seqs[h:])
    r1, _ = ssq.align_batch(gpu_syn, s1, o1); r2, _ = ssq.align_batch(gpu_syn, s2, o2)
    r2 = r2.copy(); r2["read_id"] += h
    assert np.array_equal(np.concatenate([r1, r2]), regs)
    # exact comparison on a sample
    sub = seqs[:2000]
    s, o = T.encode_reads(sub)
    a, ao = oracle.align_batch(idx, s, o)
    assert np.array_equal(a, regs[: int(roff[2000])])


def test_dupmark(ssq, oracle):
    rng = np.random.default_rng(8)
    n = 200000
    sig = np.zeros(n, T.DUPSIG_DT)
    sig["pos1"] = rng.integers(0, 5000, n); sig["pos2"] = rng.integers(0, 50, n) + sig["pos1"]
    sig["strand1"] = rng.integers(0, 2, n); sig["strand2"] = rng.integers(0, 2, n)
    sig["valid"] = rng.random(n) > 0.02
    sig["pos1"][::1000] = (1 << 40) + 5  # large coordinates
    d = ssq.dupmark_batch(sig)
    assert np.array_equal(d, oracle.dupmark(sig))
    assert d[sig["valid"] == 0].sum() == 0 and 0 < d.sum() < n
    # order-independence of the SET of survivors: exactly one survivor per distinct valid signature
    v = sig[sig["valid"] == 1]
    keys = set(zip(v["pos1"].tolist(), v["pos2"].tolist(), v["strand1"].tolist(), v["strand2"].tolist()))
    assert int((d == 0)[sig["valid"] == 1].sum()) == len(keys)
    assert len(ssq.dupmark_batch(np.zeros(0, T.DUPSIG_DT))) == 0


def test_sw_local_striped_order(ssq, oracle):
    """ksw_align2 problems (mate rescue): one warp per problem with the SSE lanes on warp lanes vs the oracle's scalar restatement of
    the striped kernel — byte mode (saturating, 16 lanes) and word mode (8 lanes), sub-optimal score, start coordinates"""
    import ctypes as C
    rng = np.random.default_rng(17)
    SWL_T = np.dtype([("q_off", "<u8"), ("t_off", "<u8"), ("qlen", "<i4"), ("tlen", "<i4"), ("xtra", "<i4"), ("pad", "<i4")])
    SWL_R = np.dtype([("score", "<i4"), ("te", "<i4"), ("qe", "<i4"), ("score2", "<i4"), ("te2", "<i4"), ("tb", "<i4"), ("qb", "<i4")])
    n = 1500
    tasks = np.zeros(n, SWL_T)
    qs, ts = [], []
    qo = to = 0
    for i in range(n):
        ql = int(rng.integers(20, 256)) if i % 7 else int(rng.integers(1, 20))
        q = rng.integers(0, 4, ql, dtype=np.uint8)
        tl = int(rng.integers(ql, ql + 700))
        t = rng.integers(0, 4, tl, dtype=np.uint8)
        kind = i % 5
        if kind < 3:  # plant a diverged copy of the query (sometimes two: sub-optimal hit)
            for rep in range(1 + (kind == 2)):
                c = q.copy()
                m = rng.random(ql) < (0.03 if kind else 0.0)
                c[m] = rng.integers(0, 4, int(m.sum()), dtype=np.uint8)
                if kind == 1 and ql > 30:
                    p = int(rng.integers(5, ql - 5)); c = np.concatenate([c[:p], c[p + int(rng.integers(1, 4)):]])
                at = int(rng.integers(0, tl - len(c) + 1))
                t[at:at + len(c)] = c
        if rng.random() < 0.1:
            q[rng.integers(0, ql)] = 4
        if rng.random() < 0.05:
            t[rng.integers(0, tl)] = 4
        minsc = 19
        xtra = 0x40000 | 0x80000 | (0x10000 if ql < 250 and i % 11 else 0) | minsc
        if i % 13 == 0:
            xtra &= ~0x80000  # no start coordinates wanted
        tasks[i] = (qo, to, ql, tl, xtra, 0)
        qs.append(q); ts.append(t)
        qo += ql; to += tl
    qbuf, tbuf = np.concatenate(qs), np.concatenate(ts)
    got = np.zeros(n, SWL_R)
    ssq.ck(ssq.lib.ssq_sw_local_batch(ssq.opts, C.c_int(0), C.c_uint64(n), tasks.ctypes.data_as(C.c_void_p), qbuf.ctypes.data_as(C.c_void_p), C.c_uint64(len(qbuf)),
                                      tbuf.ctypes.data_as(C.c_void_p), C.c_uint64(len(tbuf)), got.ctypes.data_as(C.c_void_p)), "ssq_sw_local_batch")
    mat = np.array([1 if i == j else -4 for i in range(4) for j in range(5)] , np.int8)
    mat = np.zeros(25, np.int8)
    for i in range(5):
        for j in range(5):
            mat[i * 5 + j] = -1 if (i == 4 or j == 4) else (1 if i == j else -4)

    class KR(C.Structure):
        _fields_ = [(k, C.c_int) for k in ("score", "te", "qe", "score2", "te2", "tb", "qb")]
    oracle.lib.ssqo_ksw_align2.restype = KR
    ref = np.zeros(n, SWL_R)
    for i in range(n):
        q = qs[i].copy(); t = ts[i].copy()
        r = oracle.lib.ssqo_ksw_align2(C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), C.c_int(5), mat.ctypes.data_as(C.c_void_p),
                                       C.c_int(6), C.c_int(1), C.c_int(6), C.c_int(1), C.c_int(int(tasks["xtra"][i])))
        ref[i] = (r.score, r.te, r.qe, r.score2, r.te2, r.tb, r.qb)
    bad = np.nonzero(got != ref)[0]
    assert len(bad) == 0, (bad[:5], got[bad[:5]], ref[bad[:5]], tasks[bad[:5]])
    assert (ref["score"] >= 19).sum() > 500 and (ref["score2"] >= 19).sum() > 50
    # both modes found hits, byte mode up to scores near its 255 ceiling (saturation itself: test_gpu_edges.py::test_sw_local_grid)
    byte = (tasks["xtra"] & 0x10000) != 0
    assert (byte & (ref["score"] >= 19)).sum() > 600 and (byte & (ref["score"] >= 200)).sum() > 50 and (~byte & (ref["score"] >= 19)).sum() > 50
    assert (ref["tb"] >= 0).sum() > 600
