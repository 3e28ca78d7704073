"""GPU parity on the reads the simulator never produces (corpora of tests/test_hostsim_edges.py): large indels, two indels per
read, clipped ends, contig and genome edges, the planted exact repeats, N runs and rescue-heavy pairs, compared bit for bit with
the oracle as regions, as plain `bwa mem` records and as the fused `bwa mem | samblaster` streams.  Each test asserts a coverage
floor, so that a change of the corpus cannot quietly stop reaching the path it is there for: the extension rerun with a doubled
band (k_ext_retry), banded global DP over four or more 32-column chunks (sw_global_warp), mate rescue computed inside the warp
replay (SSQ_RESCUE_SPEC=0) and in the 16-lane register form (SSQ_RESCUE_SPLIT=0).  Below them, grids of the two DP entry
points: ssq_sw_extend_batch against ksw_extend2 (both packings of the DP row, and the h0 limit of that row) and
ssq_sw_local_batch against ksw_align2 (byte mode saturating at 255, word mode, register and split forms)."""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import ssq_testlib as T
from test_hostsim_edges import CATEGORIES, SB_SPEEDSEQ_ARGS, edge_pairs, sw_extend_grid
from test_hostsim_pipe import oracle_streams, sq_header

pytestmark = pytest.mark.gpu
SB_SPEEDSEQ = dict(exclude_dups=1, add_mate_tags=1, max_split_count=2, min_non_overlap=20)
N_PAIRS = 320


@pytest.fixture(scope="module")
def gpu_syn(ssq, syn_index):
    h = ssq.index_load(syn_index[0])
    yield h
    ssq.index_free(h)


@pytest.fixture(scope="module")
def corpora(syn_index):
    fa, g, bounds = syn_index
    return {c: edge_pairs(g, bounds, c, N_PAIRS, 5 + i) for i, c in enumerate(CATEGORIES)}


def _split_restore(ssq, gpu_syn):
    """ssq_rescue_split is a device global that outlives the aligner which set it: put the default form back"""
    import os
    os.environ["SSQ_RESCUE_SPLIT"] = "1"
    try:
        ssq.aligner_free(ssq.aligner_create(gpu_syn, None, b""))
    finally:
        del os.environ["SSQ_RESCUE_SPLIT"]


@pytest.fixture(params=["default", "spec0", "split0"])
def rescue_form(request, ssq, gpu_syn, monkeypatch):
    """default: rescue alignments computed ahead of the replay by the split local SW; spec0: every one computed inside the
    warp replay (mate_rescue_warp's own branch); split0: the 16-lane register form for every query length"""
    if request.param == "spec0":
        monkeypatch.setenv("SSQ_RESCUE_SPEC", "0")
    elif request.param == "split0":
        monkeypatch.setenv("SSQ_RESCUE_SPLIT", "0")
    yield request.param
    if request.param == "split0":
        monkeypatch.delenv("SSQ_RESCUE_SPLIT")
        _split_restore(ssq, gpu_syn)


def _run(ssq, h, names, seqs, quals, n_processed=0, rg=b"", sb=None, al=None):
    """-> (texts, info, counters 105 / 106 / 107 of the run)"""
    own = al is None
    if own:
        al = ssq.aligner_create(h, sb, rg)
    rd, keep = T.pack_reads(names, seqs, quals, None, 1, n_processed)
    txt, info = ssq.aligner_run(al, rd)
    cnt = {k: int(ssq.lib.ssq_aligner_counter(al, k)) for k in (105, 106, 107)}
    if own:
        ssq.aligner_free(al)
    return [t.decode() for t in txt], info, cnt


def _longest_gap(sam):
    return max([int(x) for l in sam.splitlines() for x, op in re.findall(r"(\d+)([ID])", l.split("\t")[5])] + [0])


# ------------------------------------------------------------------------------------------------ regions ----
@pytest.mark.parametrize("env", [{}, {"SSQ_EXT_ALL": "1"}, {"SSQ_EXT_FORCE_ROUND": "0"}, {"SSQ_EXT_FORCE_ROUND": "1"}], ids=["lazy", "ext_all", "force0", "force1"])
@pytest.mark.parametrize("cat", CATEGORIES)
def test_regions(ssq, oracle, syn_index, gpu_syn, corpora, monkeypatch, cat, env):
    """chains and regions; every extension schedule (eager, forced from round 0 / 1, the default lazy one) gives the same regions"""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    seq, off = T.encode_reads(corpora[cat][1])
    a = oracle.chain_batch(idx, seq, off)
    b = ssq.chain_batch(gpu_syn, seq, off)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    a, ao = oracle.align_batch(idx, seq, off)
    b, bo = ssq.align_batch(gpu_syn, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)
    if cat == "large_del":  # the GPU's own output: the rerun with the doubled band ran
        assert (b["w"] == 2 * ssq.opts[9]).sum() >= 300


# ------------------------------------------------------------------------------------------------ records ----
# Coverage floors.  Every record with an I or D came from the banded global DP, and a pair with one end mapped and the other
# unmapped went through mate rescue, so the records themselves bound counters 106 and 105 from below; the stated minimums are
# what this seeded corpus gives the oracle (gapped records) and a conservative share of its rescue work.
MIN_GAPPED = {"large_del": 500, "two_indels": 400}
MIN_RESCUED = {"clipped": 20, "contig_edges": 20, "repeats": 20, "rescue": 20}


def _n_gapped_records(sam):
    return sum(1 for l in sam.splitlines() if re.search(r"\d[ID]", l.split("\t")[5]))


def _n_half_mapped_pairs(sam):
    return len(set(l.split("\t")[0] for l in sam.splitlines() if int(l.split("\t")[1]) & 0xc in (4, 8)))


@pytest.mark.parametrize("cat", CATEGORIES)
def test_plain_records(ssq, oracle, syn_index, gpu_syn, corpora, rescue_form, cat):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = corpora[cat]
    txt, info, cnt = _run(ssq, gpu_syn, names, seqs, quals, 0, b"e")
    assert txt[0] == oracle.mem_pe(idx, names, seqs, quals, 0, 8, b"e")
    if cat == "large_del":
        assert _longest_gap(txt[0]) >= 48  # a band of 97+ columns: four or more 32-column chunks
    assert cnt[106] >= max(_n_gapped_records(txt[0]), MIN_GAPPED.get(cat, 0)), cnt
    assert cnt[105] >= max(_n_half_mapped_pairs(txt[0]), MIN_RESCUED.get(cat, 0)), cnt
    if rescue_form == "spec0" and cat in MIN_RESCUED:  # the replay aligned them itself
        assert cnt[107] > 0, cnt


@pytest.mark.parametrize("cat", CATEGORIES)
def test_fused_streams(ssq, oracle, syn_index, gpu_syn, corpora, tmp_path, cat):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = corpora[cat]
    _, o_main, o_spl, o_disc = oracle_streams(oracle, idx, sq_header(oracle, idx, fa), names, seqs, quals, 0, b"e", SB_SPEEDSEQ_ARGS, tmp_path)
    txt, info, cnt = _run(ssq, gpu_syn, names, seqs, quals, 0, b"e", SB_SPEEDSEQ)
    assert txt[0] == o_main
    assert txt[1] == o_spl
    assert txt[2] == o_disc


@pytest.mark.parametrize("cat", ["large_del", "clipped", "contig_edges", "rescue"])
def test_fused_streams_three_batches(ssq, oracle, syn_index, gpu_syn, corpora, tmp_path, cat):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = corpora[cat]
    n = len(names)
    cuts = [0, (n // 3) & ~1, (2 * n // 3) & ~1, n]
    body = "".join(oracle.mem_pe(idx, names[a:b], seqs[a:b], quals[a:b], a, 8, b"r") for a, b in zip(cuts, cuts[1:]))
    spl, disc = str(tmp_path / "o.spl"), str(tmp_path / "o.disc")
    out = subprocess.run([T.ORACLE_BIN, "samblaster"] + SB_SPEEDSEQ_ARGS + ["--splitterFile", spl, "--discordantFile", disc],
                         input=(sq_header(oracle, idx, fa) + body).encode(), check=True, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL).stdout.decode()
    rec = lambda t: "".join(l for l in t.splitlines(True) if not l.startswith("@"))
    al = ssq.aligner_create(gpu_syn, SB_SPEEDSEQ, b"r")
    got = ["", "", ""]
    try:
        for a, b in zip(cuts, cuts[1:]):
            txt, _, _ = _run(ssq, gpu_syn, names[a:b], seqs[a:b], quals[a:b], a, al=al)
            for i in range(3):
                got[i] += txt[i]
    finally:
        ssq.aligner_free(al)
    assert got[0] == rec(out)
    assert got[1] == rec(open(spl).read())
    assert got[2] == rec(open(disc).read())


# ----------------------------------------------------------------------------------------- sw_extend grid ----
def test_sw_extend_grid(ssq, oracle):
    tasks, q, t = sw_extend_grid(3)
    ref = oracle.sw_extend_batch(tasks, q, t)
    got = ssq.sw_extend_batch(tasks, q, t)
    bad = np.nonzero(got != ref)[0]
    assert len(bad) == 0, (tasks[bad[:5]], got[bad[:5]], ref[bad[:5]])
    big = tasks["h0"] + tasks["qlen"] >= 8192  # the unpacked DP row (sw_extend_impl<false>) ran for these
    assert 1000 < big.sum() < len(tasks) - 1000
    assert (ref["score"] > tasks["h0"]).sum() > 1000 and (ref["gscore"] > 0).sum() > 1000


def test_sw_extend_rejects_scores_the_row_cannot_hold(ssq, oracle):
    """H and E are 16 bits each in the DP row: h0 + qlen * a > 65535 must fail the call, not return wrong results"""
    tasks, q, t = sw_extend_grid(4, h0_kind="over")
    for i in range(0, len(tasks), 97):
        one = tasks[i:i + 1].copy()
        with pytest.raises(RuntimeError, match="rc=-4"):
            ssq.sw_extend_batch(one, q, t)
    # the largest h0 the row holds still gives the oracle's result
    tasks["h0"] = 65535 - tasks["qlen"]
    assert np.array_equal(ssq.sw_extend_batch(tasks, q, t), oracle.sw_extend_batch(tasks, q, t))


# ------------------------------------------------------------------------------------------ sw_local grid ----
SWL_T = np.dtype([("q_off", "<u8"), ("t_off", "<u8"), ("qlen", "<i4"), ("tlen", "<i4"), ("xtra", "<i4"), ("pad", "<i4")])
SWL_R = np.dtype([("score", "<i4"), ("te", "<i4"), ("qe", "<i4"), ("score2", "<i4"), ("te2", "<i4"), ("tb", "<i4"), ("qb", "<i4")])
XBYTE, XSUBO, XSTART = 0x10000, 0x40000, 0x80000


def _sw_local_grid(seed):
    """ksw_align2 problems: byte mode with qlen 251-255 against an exact copy (the score saturates at 255), byte and word mode for
    qlen 1-16 (register form) and 17-255 (split form), targets shorter than the query and of one base, with and without
    XSUBO / XSTART"""
    rng = np.random.default_rng(seed)
    tasks, qs, ts = [], [], []
    qo = to = 0

    def add(q, t, xtra):
        nonlocal qo, to
        tasks.append((qo, to, len(q), len(t), xtra, 0)); qs.append(q); ts.append(t)
        qo += len(q); to += len(t)

    for i in range(200):  # saturation: an exact copy of a 251-255 bp query
        ql = 251 + i % 5
        q = rng.integers(0, 4, ql, dtype=np.uint8)
        fl = rng.integers(0, 4, int(rng.integers(0, 300)), dtype=np.uint8)
        at = int(rng.integers(0, len(fl) + 1))
        t = np.concatenate([fl[:at], q, fl[at:]])
        add(q, t, XBYTE | (XSUBO if i & 1 else 0) | (XSTART if i & 2 else 0) | 19)
    for i in range(2400):
        ql = int(rng.integers(1, 17)) if i % 3 == 0 else int(rng.integers(17, 256))
        q = rng.integers(0, 4, ql, dtype=np.uint8)
        tk = i % 6
        tl = 1 if tk == 0 else int(rng.integers(1, ql + 1)) if tk == 1 else int(rng.integers(ql, ql + 500))
        t = rng.integers(0, 4, tl, dtype=np.uint8)
        kind = (i // 6) % 4
        if kind < 3:  # a copy (exact / diverged with an indel / two diverged copies), clipped to the target
            for _ in range(1 + (kind == 2)):
                c = q.copy()
                if kind:
                    m = rng.random(ql) < 0.04
                    c[m] = rng.integers(0, 4, int(m.sum()), dtype=np.uint8)
                    if ql > 30:
                        p = int(rng.integers(5, ql - 5)); l = int(rng.integers(1, 12))
                        c = np.concatenate([c[:p], c[p + l:]]) if rng.random() < 0.5 else np.concatenate([c[:p], rng.integers(0, 4, l, dtype=np.uint8), c[p:]])
                c = c[:tl]
                at = int(rng.integers(0, tl - len(c) + 1))
                t[at:at + len(c)] = c
        if rng.random() < 0.05:
            t[rng.integers(0, tl)] = 4
        byte = (i // 24) % 2 == 0 and ql * 1 < 250
        add(q, t, (XBYTE if byte else 0) | (XSUBO if (i // 2) % 2 else 0) | (XSTART if (i // 4) % 3 else 0) | int(rng.integers(10, 40)))
    arr = np.zeros(len(tasks), SWL_T)
    for i, x in enumerate(tasks):
        arr[i] = x
    return arr, qs, ts


def _sw_local_oracle(oracle, tasks, qs, ts):
    mat = np.zeros(25, np.int8)
    for i in range(5):
        for j in range(5):
            mat[i * 5 + j] = -1 if (i == 4 or j == 4) else (1 if i == j else -4)

    class KR(C.Structure):
        _fields_ = [(k, C.c_int) for k in ("score", "te", "qe", "score2", "te2", "tb", "qb")]
    oracle.lib.ssqo_ksw_align2.restype = KR
    ref = np.zeros(len(tasks), SWL_R)
    for i in range(len(tasks)):
        q, t = qs[i].copy(), ts[i].copy()
        r = oracle.lib.ssqo_ksw_align2(C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), C.c_int(5),
                                       mat.ctypes.data_as(C.c_void_p), C.c_int(6), C.c_int(1), C.c_int(6), C.c_int(1), C.c_int(int(tasks["xtra"][i])))
        ref[i] = (r.score, r.te, r.qe, r.score2, r.te2, r.tb, r.qb)
    return ref


def _sw_local_gpu(ssq, tasks, qs, ts):
    qbuf, tbuf = np.concatenate(qs), np.concatenate(ts)
    got = np.zeros(len(tasks), SWL_R)
    ssq.ck(ssq.lib.ssq_sw_local_batch(ssq.opts, C.c_int(0), C.c_uint64(len(tasks)), tasks.ctypes.data_as(C.c_void_p), qbuf.ctypes.data_as(C.c_void_p), C.c_uint64(len(qbuf)),
                                      tbuf.ctypes.data_as(C.c_void_p), C.c_uint64(len(tbuf)), got.ctypes.data_as(C.c_void_p)), "ssq_sw_local_batch")
    return got


@pytest.mark.parametrize("form", ["split", "register"])
def test_sw_local_grid(ssq, oracle, gpu_syn, monkeypatch, form):
    tasks, qs, ts = _sw_local_grid(23)
    ref = _sw_local_oracle(oracle, tasks, qs, ts)
    if form == "register":  # an aligner created with SSQ_RESCUE_SPLIT=0 switches the device to the 16-lane form
        monkeypatch.setenv("SSQ_RESCUE_SPLIT", "0")
        ssq.aligner_free(ssq.aligner_create(gpu_syn, None, b""))
        monkeypatch.delenv("SSQ_RESCUE_SPLIT")
    try:
        got = _sw_local_gpu(ssq, tasks, qs, ts)
    finally:
        if form == "register":
            _split_restore(ssq, gpu_syn)
    bad = np.nonzero(got != ref)[0]
    assert len(bad) == 0, (bad[:5], got[bad[:5]], ref[bad[:5]], tasks[bad[:5]])
    byte = (tasks["xtra"] & XBYTE) != 0
    assert (byte & (ref["score"] == 255)).sum() >= 150  # saturated byte-mode scores
    assert (byte & (ref["score"] >= 19) & (ref["score"] < 255) & (tasks["qlen"] > 16)).sum() > 300
    assert (byte & (ref["score"] >= 8) & (tasks["qlen"] <= 16)).sum() > 50
    assert (~byte & (ref["score"] >= 19)).sum() > 300 and (~byte & (ref["score"] >= 200)).sum() > 20
    assert (ref["tb"] >= 0).sum() > 500 and (ref["score2"] > 0).sum() > 50
    assert (tasks["tlen"] < tasks["qlen"]).sum() > 300 and (tasks["tlen"] == 1).sum() > 300
