"""Reads the simulator never produces, through the host build of the kernels' routines (tests/hostsim) against the oracle.

simulate_pairs / stress_reads make reads with at most one 1-3 bp indel, 0.5-2 % errors and mates 400 +- 40 bp apart, so
several code paths of the aligner never see an input that reaches them: the extension rerun with a doubled band (an indel of
75 bp or more), banded global DP over many 32-column chunks, z-drop and clipping choices, the ends of the concatenated
reference, the planted exact repeats, N runs, and mate rescue of badly diverged mates.  edge_pairs() makes one seeded corpus
per category; tests/test_gpu_edges.py runs the same corpora through the GPU.  The sw_extend grid below walks the remainders
of the four-column loop, band widths around a warp's width, the z-drop and end-bonus settings and both packings of the DP
row (h0 + qlen * a below and above 8192)."""
import numpy as np
import pytest

import ssq_testlib as T
from test_hostsim_pipe import oracle_streams, sq_header

CATEGORIES = ("large_del", "two_indels", "clipped", "contig_edges", "repeats", "n_runs", "rescue")
SB_SPEEDSEQ_ARGS = ["--excludeDups", "--addMateTags", "--maxSplitCount", "2", "--minNonOverlap", "20"]
_COMP = np.array([3, 2, 1, 0, 4], np.uint8)
_ACGTN = np.frombuffer(b"ACGTN", np.uint8)


def _rc(x):
    return _COMP[x[::-1]]


def _subst(rng, x, err):
    x = x.copy()
    m = rng.random(len(x)) < err
    x[m] = (x[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) % 4
    return x


def _big_del(rng, src, rl, lo, hi):
    """rl bases of src (which holds at least rl + hi bases) with a lo..hi bp deletion starting at 40-60 % of the read"""
    d = int(rng.integers(lo, hi + 1))
    s = int(rng.integers(int(0.4 * rl), int(0.6 * rl) + 1))
    return np.concatenate([src[:s], src[s + d:s + d + rl - s]])


def _big_ins(rng, src, rl, lo, hi):
    d = int(rng.integers(lo, hi + 1))
    s = int(rng.integers(int(0.4 * rl), int(0.6 * rl) + 1))
    return np.concatenate([src[:s], rng.integers(0, 4, d, dtype=np.uint8), src[s:]])[:rl]


def _two_indels(rng, src, rl):
    """two 5-30 bp indels, one in each half of the read"""
    out, at = [], 0
    for lo_f, hi_f in ((0.15, 0.35), (0.55, 0.8)):
        p = int(rng.integers(int(lo_f * rl), int(hi_f * rl)))
        l = int(rng.integers(5, 31))
        out.append(src[at:p])
        if rng.random() < 0.5:
            out.append(rng.integers(0, 4, l, dtype=np.uint8)); at = p
        else:
            at = p + l
    out.append(src[at:])
    return np.concatenate(out)[:rl]


def _clip(rng, g, x):
    """a random 3' tail or 5' head of 15-100 bp: random bases, or bases from elsewhere in the genome (supplementary, SA)"""
    l = int(rng.integers(15, 101))
    if rng.random() < 0.5:
        p = int(rng.integers(0, len(g) - l))
        junk = g[p:p + l] if rng.random() < 0.5 else _rc(g[p:p + l])
    else:
        junk = rng.integers(0, 4, l, dtype=np.uint8)
    x = x.copy()
    if rng.random() < 0.5:
        x[len(x) - l:] = junk
    else:
        x[:l] = junk
    return x


def _n_run(rng, x):
    x = x.copy()
    l = int(rng.integers(10, 41))
    p = int(rng.integers(1, len(x) - l))
    x[p:p + l] = 4
    return x


def edge_pairs(g, bounds, cat, n_pairs, seed):
    """seeded read pairs of one edge-case category (see CATEGORIES), followed by n_pairs // 4 plain pairs so that the batch's
    insert-size statistics stay those of a real library.  Returns (names, seqs, quals), mates interleaved"""
    rng = np.random.default_rng(seed)
    n = len(g)
    pad = 700
    G = np.concatenate([rng.integers(0, 4, pad, dtype=np.uint8), g, rng.integers(0, 4, pad, dtype=np.uint8)])  # random bases past both genome ends
    names, seqs = [], []

    def frag_at(p, ins):
        """the fragment [p, p + ins) of the genome (coordinates may run past its ends into random bases)"""
        return G[pad + p:pad + p + ins]

    def add(tag, r1, r2, swap=None):
        if swap if swap is not None else rng.random() < 0.5:
            r1, r2 = r2, r1
        nm = "%s%d" % (tag, len(names) // 2)
        for r in (r1, r2):
            names.append(nm)
            seqs.append(_ACGTN[r].tobytes().decode())

    def ins_draw():
        return int(rng.normal(400, 40))

    def rand_pos(span):
        return int(rng.integers(0, n - span))

    for i in range(n_pairs):
        if cat == "large_del":
            k = i % 8
            if k < 6:  # 250 bp mates, each with a 76-99 bp deletion: the first extension's band is too narrow, the rerun doubles it
                rl, ins = 250, max(600, ins_draw())
                p = rand_pos(ins + 200)
                f = frag_at(p, ins + 200)
                r1 = _subst(rng, _big_del(rng, f, rl, 76, 99), 0.005)
                r2 = _subst(rng, _big_del(rng, _rc(f), rl, 76, 99), 0.005)
            elif k == 6:  # insertions of the same size (they end up clipped), and of 40-60 bp (kept as I: wide CIGAR bands)
                rl, ins = 250, max(300, ins_draw())
                p = rand_pos(ins)
                f = frag_at(p, ins)
                lo, hi = (76, 99) if i % 16 == 6 else (40, 60)
                r1, r2 = _big_ins(rng, f, rl, lo, hi), _subst(rng, _rc(f)[:rl], 0.005)
            else:  # 150 bp reads with 40-70 bp deletions
                rl, ins = 150, max(300, ins_draw())
                p = rand_pos(ins + 100)
                f = frag_at(p, ins + 100)
                r1, r2 = _big_del(rng, f, rl, 40, 70), _big_del(rng, _rc(f), rl, 40, 70)
            add("del", r1, r2)
        elif cat == "two_indels":
            rl = 150 if i % 2 else 250
            ins = max(rl + 20, ins_draw())
            p = rand_pos(ins + 80)
            f = frag_at(p, ins + 80)
            r1 = _subst(rng, _two_indels(rng, f, rl), 0.005)
            r2 = _subst(rng, _two_indels(rng, _rc(f), rl), 0.005) if i % 3 == 0 else _subst(rng, _rc(f)[:rl], 0.005)
            add("ind", r1, r2)
        elif cat == "clipped":
            rl, ins = 150, max(170, ins_draw())
            p = rand_pos(ins)
            f = frag_at(p, ins)
            r1, r2 = _subst(rng, f[:rl], 0.005), _subst(rng, _rc(f)[:rl], 0.005)
            r1 = _clip(rng, g, r1)
            if i % 3 == 0:
                r2 = _clip(rng, g, r2)
            add("clp", r1, r2)
        elif cat == "contig_edges":
            # a fragment that straddles the first / last base of a contig or of the genome: one or both mates overhang the
            # edge, or the mate lies wholly past it (random bases past the genome's ends, the next contig inside it)
            rl = 150 if i % 3 else 101
            ins = max(rl + 10, ins_draw())
            e = int(bounds[i % len(bounds)])
            p = e - int(rng.integers(1, ins + 60))
            f = frag_at(p, ins)
            r1, r2 = _subst(rng, f[:rl], 0.005), _subst(rng, _rc(f)[:rl], 0.005)
            add("edg", r1, r2, swap=bool(i & 4))
        elif cat == "repeats":
            # reads from the exact tandem copy g[1000:1400] == g[2000:2400] and across the (AC)30 at 3000
            rl = 150 if i % 2 else 101
            ins = max(rl + 10, ins_draw())
            k = i % 3
            if k == 0:
                s = int(rng.integers(1000, 1400 - rl)) + (1000 if rng.random() < 0.5 else 0)
            elif k == 1:
                s = int(rng.integers(3060 - rl + 10, 3000))
            else:  # the mate in the repeat, this end outside
                s = int(rng.integers(1000, 1400 - rl)) + 1000 * int(rng.integers(0, 2)) - ins + rl
                s = max(s, 0)
            f = frag_at(s, ins)
            r1, r2 = _subst(rng, f[:rl], 0.003), _subst(rng, _rc(f)[:rl], 0.003)
            add("rep", r1, r2, swap=k == 2)
        elif cat == "n_runs":
            rl, ins = 150, max(170, ins_draw())
            p = rand_pos(ins)
            f = frag_at(p, ins)
            r1, r2 = _n_run(rng, _subst(rng, f[:rl], 0.005)), _subst(rng, _rc(f)[:rl], 0.005)
            if i % 3 == 0:
                r2 = _n_run(rng, r2)
            add("nrn", r1, r2)
        elif cat == "rescue":
            # one clean end; its mate diverged (6-12 % substitutions) and carrying a large deletion or a clipped end, so that
            # seeding often misses it and mate rescue aligns it across the whole window; some inserts at +-3 sigma
            rl = 150
            ins = 400 + (120 if i % 4 == 0 else -120 if i % 4 == 1 else int(rng.normal(0, 40)))
            ins += int(rng.integers(-5, 6))
            p = rand_pos(ins)
            f = frag_at(p, ins)
            r1 = _subst(rng, f[:rl], 0.003)
            r2 = _big_del(rng, _rc(f), rl, 76, 99) if i % 2 else _clip(rng, g, _rc(f)[:rl])
            r2 = _subst(rng, r2, 0.06 + 0.06 * rng.random())
            add("res", r1, r2)
        else:
            raise ValueError(cat)
    pn, ps, _ = T.simulate_pairs(g, bounds, n_pairs // 4, 150, seed + 1000)
    names += ["pl" + x for x in pn]
    seqs += ps
    return names, seqs, ["I" * len(s) for s in seqs]


def sw_extend_grid(seed, h0_kind="in_range", a=1):
    """ksw_extend2 problems across the axes where a row-sequential banded DP goes wrong: qlen around the four-column loop's
    remainders, tlen 0 / 1 / qlen / qlen + w / long, band widths around 32, z-drop 0 / 1 / 10 / 100, end bonus 0 / 5 / 60, identical /
    diverged / unrelated / all-N sequences, and h0 from 1 up to 65535 - qlen * a (on both sides of the 8192 - qlen * a switch
    between the packed and the unpacked DP row).  h0_kind="over": every task has h0 + qlen * a > 65535.
    Returns (tasks, qbuf, tbuf)"""
    rng = np.random.default_rng(seed)
    qlens = list(range(1, 9)) + list(range(29, 36)) + [63, 64, 65, 127, 128, 129, 253, 254, 255]
    ws = (0, 1, 2, 3, 31, 32, 33, 100, 200)
    tasks, qs, ts = [], [], []
    qo = to = 0
    k = 0
    for ql in qlens:
        h0s = [1, 19, 255, 8191 - ql * a, 8192 - ql * a, 40000, 65535 - ql * a] if h0_kind == "in_range" else [65536 - ql * a, 70000, 1 << 30]
        for w in ws:
            for kind in range(4):
                for tsel in range(5):
                    tl = (0, 1, ql, ql + w, int(rng.integers(ql + w + 1, 2001)))[tsel]
                    q = rng.integers(0, 4, ql, dtype=np.uint8)
                    if kind == 0:  # identical, then random bases
                        t = np.concatenate([q, rng.integers(0, 4, max(0, tl - ql), dtype=np.uint8)])[:tl]
                    elif kind == 1:  # diverged: substitutions and indels
                        c = list(_subst(rng, q, 0.06))
                        for _ in range(int(rng.integers(0, 3))):
                            p = int(rng.integers(0, len(c) + 1))
                            l = int(rng.integers(33, 61)) if rng.random() < 0.3 else int(rng.integers(1, 9))
                            if rng.random() < 0.5:
                                c[p:p] = rng.integers(0, 4, l).tolist()
                            else:
                                del c[p:p + l]
                        t = np.concatenate([np.array(c, np.uint8), rng.integers(0, 4, max(0, tl), dtype=np.uint8)])[:tl]
                    elif kind == 2:  # unrelated
                        t = rng.integers(0, 4, tl, dtype=np.uint8)
                    else:  # all N (query or target)
                        t = rng.integers(0, 4, tl, dtype=np.uint8)
                        if k & 1:
                            q[:] = 4
                        else:
                            t[:] = 4
                    h0 = h0s[k % len(h0s)]
                    zdrop = (0, 1, 10, 100)[(k // 7) % 4]
                    eb = (0, 5, 60)[(k // 3) % 3]
                    tasks.append((qo, to, ql, tl, h0, w, eb, zdrop))
                    qs.append(q); ts.append(t.astype(np.uint8))
                    qo += ql; to += tl
                    k += 1
    arr = np.zeros(len(tasks), T.SWTASK_DT)
    for i, x in enumerate(tasks):
        arr[i] = x
    return arr, np.concatenate(qs), np.concatenate(ts + [np.zeros(1, np.uint8)])


# --------------------------------------------------------------------------------------------------- tests ----
@pytest.fixture(scope="module")
def corpora(syn_index):
    fa, g, bounds = syn_index
    return {c: edge_pairs(g, bounds, c, 240, 5 + i) for i, c in enumerate(CATEGORIES)}


@pytest.mark.parametrize("cat", CATEGORIES)
def test_regions(oracle, hostsim, syn_index, corpora, cat):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    seq, off = T.encode_reads(corpora[cat][1])
    a, ao = oracle.align_batch(idx, seq, off)
    b, bo = hostsim.align_batch(idx, seq, off)
    assert np.array_equal(ao, bo) and np.array_equal(a, b)
    if cat == "large_del":  # the doubled band was taken
        assert (a["w"] == 200).sum() >= 250


@pytest.mark.parametrize("cat", CATEGORIES)
def test_plain_records(oracle, hostsim, syn_index, corpora, cat):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = corpora[cat]
    assert hostsim.mem_pe(idx, names, seqs, quals, 0, b"e") == oracle.mem_pe(idx, names, seqs, quals, 0, 4, b"e")


@pytest.mark.parametrize("cat", CATEGORIES)
def test_fused_streams(oracle, hostsim, syn_index, corpora, tmp_path, cat):
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = corpora[cat]
    _, o_main, o_spl, o_disc = oracle_streams(oracle, idx, sq_header(oracle, idx, fa), names, seqs, quals, 0, b"e", SB_SPEEDSEQ_ARGS, tmp_path)
    h_main, h_spl, h_disc = hostsim.pipe(idx, names, seqs, quals, 0, b"e", 1, (1, 1, 2, 20, 0))
    assert h_main == o_main
    assert h_spl == o_spl
    assert h_disc == o_disc


@pytest.mark.parametrize("env", [{"HOSTSIM_RESCUE_SPEC": "0"}, {"HOSTSIM_RESCUE_DROP": "2"}])
@pytest.mark.parametrize("cat", ["rescue", "large_del", "clipped"])
def test_rescue_in_the_replay(oracle, hostsim, syn_index, corpora, monkeypatch, env, cat):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    fa, g, bounds = syn_index
    idx = oracle.load(fa)
    names, seqs, quals = corpora[cat]
    assert hostsim.mem_pe(idx, names, seqs, quals, 0, b"e") == oracle.mem_pe(idx, names, seqs, quals, 0, 4, b"e")


def test_sw_extend_grid(oracle, hostsim):
    tasks, q, t = sw_extend_grid(3)
    ref = oracle.sw_extend_batch(tasks, q, t)
    got = hostsim.sw_extend_batch(tasks, q, t)
    bad = np.nonzero(got != ref)[0]
    assert len(bad) == 0, (tasks[bad[:5]], got[bad[:5]], ref[bad[:5]])
    big = tasks["h0"] + tasks["qlen"] >= 8192
    assert 1000 < big.sum() < len(tasks) - 1000  # both forms of the DP row ran
    assert (ref["score"] > tasks["h0"]).sum() > 1000 and (ref["gscore"] > 0).sum() > 1000 and (ref["max_off"] > 0).sum() > 30
