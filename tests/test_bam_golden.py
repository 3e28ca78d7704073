"""f1 (SURVEY.md §8): the BAM records the pipeline encodes straight from its structured alignment records, coordinate-sorted per batch,
against what the REFERENCE'S OWN TOOL makes of the oracle's SAM text: tests/golden/ex_bam_*.records.gz were written by
/root/reference/src/sambamba v0.5.9 (`view -S -f bam -l 0 | sort`, the commands of bin/speedseq:440-448) — see
tests/golden/make_bam_golden.py.  CPU: the encoder bodies through tests/hostsim.  GPU: the kernels through ssq_aligner_fetch_bam."""
import gzip
import hashlib
import json
import os

import pytest

import ssq_testlib as T

SB = dict(exclude_dups=1, add_mate_tags=1, max_split_count=2, min_non_overlap=20)


def golden(tag, prefix="ex"):
    return gzip.open(os.path.join(T.GOLDEN, "%s_bam_%s.records.gz" % (prefix, tag))).read()


def syn_reads(syn_index):
    from test_hostsim_pipe import stress_reads
    fa, g, bounds = syn_index  # the same seeded genome and reads tests/golden/make_bam_golden.py used
    return stress_reads(g, bounds, 700, 150, 5, err=0.01, indel=0.002)


def split_records(b):
    import struct
    out, p = [], 0
    while p < len(b):
        n = struct.unpack("<i", b[p:p + 4])[0]
        out.append(b[p:p + 4 + n]); p += 4 + n
    return out


def test_bam_records_match_sambamba_cpu(oracle, hostsim, ex_index, ex_reads):
    idx = oracle.load(ex_index)
    names, seqs, quals = ex_reads
    txt, bams = hostsim.pipe_bam(idx, names, seqs, quals, 0, b"NA12878", 1, (1, 1, 2, 20, 0))
    for k, tag in enumerate(("main", "spl", "disc")):
        want, got = golden(tag), bams[k]
        if got != want:
            a, b = split_records(want), split_records(got)
            first = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
            raise AssertionError("%s: %d vs %d records, first difference at record %d:\n%r\n%r" % (tag, len(a), len(b), first, a[first:first + 1], b[first:first + 1]))
    assert len(split_records(bams[0])) == txt[0].count("\n") > 4000


def test_bam_records_match_sambamba_synthetic_stress_cpu(oracle, hostsim, syn_index):
    """duplicates, splitters with SA tags, discordants, XA hits, junk pairs and orphans over three contigs"""
    idx = oracle.load(syn_index[0])
    names, seqs, quals = syn_reads(syn_index)
    txt, bams = hostsim.pipe_bam(idx, names, seqs, quals, 0, b"NA12878", 1, (1, 1, 2, 20, 0))
    for k, tag in enumerate(("main", "spl", "disc")):
        assert bams[k] == golden(tag, "syn"), tag
    assert len(split_records(bams[1])) > 20 and len(split_records(bams[2])) > 50


def test_merged_runs_of_three_batches_match_sambamba_sort(ssq_lib_cpu, oracle, hostsim, syn_index):
    """a run of three batches: every batch's coordinate-sorted records (hostsim bodies) merged by ssq_bam_merge_runs must equal what the
    reference's sambamba makes of the whole run's SAM (golden syn3: per-batch insert-size statistics, duplicates across batches)"""
    import ctypes as C
    idx = oracle.load(syn_index[0])
    names, seqs, quals = syn_reads(syn_index)
    cuts = [0, 1000, 2100, len(names)]
    runs = []
    for k, (a, b) in enumerate(zip(cuts, cuts[1:])):
        txt, bams = hostsim.pipe_bam(idx, names[a:b], seqs[a:b], quals[a:b], a, b"NA12878", 1, (1, 1, 2, 20, 0), reset=1 if k == 0 else 0)
        runs.append(bams[0])
    L = ssq_lib_cpu
    arr = (C.c_char_p * 3)(*runs); lens = (C.c_size_t * 3)(*[len(r) for r in runs])
    out, n = C.c_void_p(), C.c_size_t(0)
    L.ssq_bam_merge_runs.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    assert L.ssq_bam_merge_runs(3, arr, lens, C.byref(out), C.byref(n)) == 0
    merged = C.string_at(out, n.value)
    L.ssq_free(out)
    assert merged == golden("main", "syn3")


@pytest.mark.gpu
def test_bam_records_match_sambamba_synthetic_stress_gpu(ssq, syn_index):
    import ctypes as C
    h = ssq.index_load(syn_index[0])
    names, seqs, quals = syn_reads(syn_index)
    al = ssq.aligner_create(h, SB, b"NA12878")
    ssq.ck(ssq.lib.ssq_aligner_set_bam(al, C.c_int(1), C.c_int(1)), "ssq_aligner_set_bam")
    rd, keep = T.pack_reads(names, seqs, quals, None, 1, 0)
    ssq.aligner_run(al, rd)
    for k, tag in enumerate(("main", "spl", "disc")):
        p, n = C.c_void_p(), C.c_size_t(0)
        ssq.ck(ssq.lib.ssq_aligner_fetch_bam(al, C.c_int(k), C.byref(p), C.byref(n)), "ssq_aligner_fetch_bam")
        assert C.string_at(p, n.value) == golden(tag, "syn"), tag
    ssq.aligner_free(al)
    ssq.index_free(h)


@pytest.mark.gpu
def test_bam_records_match_sambamba_gpu(ssq, ex_index, ex_reads):
    import ctypes as C
    h = ssq.index_load(ex_index)
    names, seqs, quals = ex_reads
    al = ssq.aligner_create(h, SB, b"NA12878")
    ssq.ck(ssq.lib.ssq_aligner_set_bam(al, C.c_int(1), C.c_int(1)), "ssq_aligner_set_bam")
    rd, keep = T.pack_reads(names, seqs, quals, None, 1, 0)
    txt, info = ssq.aligner_run(al, rd)
    for k, tag in enumerate(("main", "spl", "disc")):
        p, n = C.c_void_p(), C.c_size_t(0)
        ssq.ck(ssq.lib.ssq_aligner_fetch_bam(al, C.c_int(k), C.byref(p), C.byref(n)), "ssq_aligner_fetch_bam")
        got = C.string_at(p, n.value)
        assert got == golden(tag), tag
    ssq.aligner_free(al)
    ssq.index_free(h)


def sambamba_golden(name):
    """what the reference's sambamba v0.5.9 made of a BAM file a test writes (tests/golden/make_sambamba_golden.py)"""
    return json.load(open(os.path.join(T.GOLDEN, "sambamba_reads.json")))[name]


def sha256(b):
    return hashlib.sha256(b).hexdigest()


def example_bam(oracle, hostsim, ex_index, ex_reads):
    """(uncompressed BAM of the example reads' main records, the oracle pipeline's SAM text of them)"""
    import struct
    idx = oracle.load(ex_index)
    names, seqs, quals = ex_reads
    txt, bams = hostsim.pipe_bam(idx, names, seqs, quals, 0, b"NA12878", 1, (1, 1, 2, 20, 0))
    hdr_text = b"@HD\tVN:1.3\tSO:coordinate\n@SQ\tSN:20_slice\tLN:321635\n@RG\tID:NA12878\tSM:NA12878\tLB:lib1\n"
    return b"BAM\x01" + struct.pack("<i", len(hdr_text)) + hdr_text + struct.pack("<i", 1) + struct.pack("<i", 9) + b"20_slice\x00" + struct.pack("<i", 321635) + bams[0], txt[0]


def test_bgzf_framing_roundtrip_and_sambamba_reads_it(ssq_lib_cpu, oracle, hostsim, ex_index, ex_reads):
    """ssq_bgzf_compress (host, zlib): members of at most 64 KiB with the BC extra field and the EOF marker; python's gzip reads the
    resulting .bam back, and the reference's sambamba read the same BAM as the oracle pipeline's records (golden)"""
    import ctypes as C
    import struct
    L = ssq_lib_cpu
    raw, main_text = example_bam(oracle, hostsim, ex_index, ex_reads)
    for level in (0, 1, 6):
        out, n = C.c_void_p(), C.c_size_t(0)
        assert L.ssq_bgzf_compress(raw, C.c_size_t(len(raw)), C.c_int(level), C.c_int(1), C.byref(out), C.byref(n)) == 0
        comp = C.string_at(out, n.value)
        L.ssq_free(out)
        assert gzip.decompress(comp) == raw
        p, nb = 0, 0
        while p < len(comp):  # every member: gzip magic, FEXTRA, "BC", BSIZE
            assert comp[p:p + 4] == b"\x1f\x8b\x08\x04" and comp[p + 12:p + 14] == b"BC"
            bsize = struct.unpack("<H", comp[p + 16:p + 18])[0] + 1
            assert struct.unpack("<I", comp[p + bsize - 4:p + bsize])[0] <= 0xff00
            p += bsize; nb += 1
        assert p == len(comp) and nb == (len(raw) + 0xff00 - 1) // 0xff00 + 1
        assert comp.endswith(bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0]))
    # sambamba's text of these bytes == the oracle pipeline's SAM records, re-ordered by coordinate (stable)
    want = sambamba_golden("bgzf_example")
    assert sha256(raw) == want["bam_sha256"]
    key = lambda l: (1 << 40 if l.split("\t")[2] == "*" else 0, int(l.split("\t")[3]), (int(l.split("\t")[1]) >> 4) & 1)
    view = sorted(main_text.splitlines(), key=key)
    assert len(view) == want["view_lines"] and sha256("".join(l + "\n" for l in view).encode()) == want["view_sha256"]


def test_header_rewrite_matches_sambamba(ssq_lib_cpu):
    """@HD SO:coordinate first, @RG / @PG tags in sambamba's field order: the header text of the golden BAM from the SAM header it was made of"""
    import ctypes as C
    L = ssq_lib_cpu
    src = open(os.path.join(T.GOLDEN, "ex_sam_header.txt"), "rb").read()
    out = C.c_void_p()
    L.ssq_bam_header_text.argtypes = [C.c_char_p, C.c_int, C.c_void_p]
    L.ssq_bam_header_text.restype = C.c_int
    assert L.ssq_bam_header_text(src, 1, C.byref(out)) == 0
    got = C.string_at(out)
    L.ssq_free(out)
    assert got == open(os.path.join(T.GOLDEN, "ex_bam_header.txt"), "rb").read()


def contigs_of(syn_index):
    fa, g, bounds = syn_index
    return [(b"ctg%d" % (i + 1), int(bounds[i + 1] - bounds[i])) for i in range(len(bounds) - 1)]


def _bam_file(path):
    """(header text, number of references, records) of a BGZF file; every block must be a well-formed BGZF member"""
    import struct
    raw = open(path, "rb").read()
    assert raw[-28:] == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")  # the end-of-file block
    p = 0
    while p < len(raw):
        assert raw[p:p + 4] == b"\x1f\x8b\x08\x04" and raw[p + 12:p + 16] == b"BC\x02\x00"
        p += struct.unpack("<H", raw[p + 16:p + 18])[0] + 1
    assert p == len(raw)
    d = gzip.decompress(raw)
    assert d[:4] == b"BAM\x01"
    l_text = struct.unpack("<i", d[4:8])[0]
    text = d[8:8 + l_text]
    q = 8 + l_text
    n_ref = struct.unpack("<i", d[q:q + 4])[0]
    q += 4
    refs = []
    for _ in range(n_ref):
        l = struct.unpack("<i", d[q:q + 4])[0]
        refs.append((d[q + 4:q + 4 + l - 1], struct.unpack("<i", d[q + 4 + l:q + 8 + l])[0]))
        q += 8 + l
    return text, refs, d[q:]


def shim_run_stream(oracle, hostsim, syn_index):
    """(SAM header, what the `bwa` shim writes in BAM mode for the synthetic reads as a run of three batches: header, marker, frames)"""
    import struct
    idx = oracle.load(syn_index[0])
    names, seqs, quals = syn_reads(syn_index)
    cuts = [0, 1000, 2100, len(names)]
    hdr = b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (n, l) for n, l in contigs_of(syn_index)) + b"@RG\tID:NA12878\tSM:NA12878\tLB:lib1\n@PG\tID:bwa\tPN:bwa\tVN:0.7.12-r1039\tCL:bwa mem x\n" \
        + b"@PG\tID:SAMBLASTER\tVN:0.1.22\tCL:samblaster -i stdin -o stdout\n"
    stream = hdr + b"@CO\tssq-bam-runs-v1\n"
    for k, (a, b) in enumerate(zip(cuts, cuts[1:])):
        txt, bams = hostsim.pipe_bam(idx, names[a:b], seqs[a:b], quals[a:b], a, b"NA12878", 1, (1, 1, 2, 20, 0), reset=1 if k == 0 else 0)
        stream += b"SSQFRAME" + struct.pack("<QQ", 3, len(bams[0])) + bams[0]
    return hdr, stream


def test_sambamba_shim_merges_the_run_stream(ssq_lib_cpu, oracle, hostsim, syn_index, tmp_path):
    """BAM mode of the shims (ssq_fuse.h): header text + marker + one frame per batch through `sambamba view -S -f bam -l 0 /dev/stdin |
    sambamba sort ... -o out.bam /dev/stdin` as speedseq:440-441 calls them.  The file's records must be the reference sambamba's
    (golden syn3), its header the rewritten one, with and without spilling to --tmpdir, for any thread count."""
    import ctypes as C
    import subprocess
    shim = os.path.join(T.ROOT, "speedseq_b200", "bin", "sambamba")
    hdr, stream = shim_run_stream(oracle, hostsim, syn_index)
    L = ssq_lib_cpu
    L.ssq_bam_header_text.argtypes = [C.c_char_p, C.c_int, C.c_void_p]
    out = C.c_void_p()
    assert L.ssq_bam_header_text(hdr, 1, C.byref(out)) == 0
    want_text = C.string_at(out)
    L.ssq_free(out)
    files = []
    for tag, env, t in (("plain", {}, 4), ("spill", {"SSQ_SORT_SPILL_BYTES": "200000"}, 1)):
        viewed = subprocess.run([shim, "view", "-S", "-f", "bam", "-l", "0", "/dev/stdin"], input=stream, stdout=subprocess.PIPE, check=True, timeout=60).stdout
        assert viewed == stream
        o = str(tmp_path / (tag + ".bam"))
        subprocess.run([shim, "sort", "-t", str(t), "-m", "1G", "--tmpdir=" + str(tmp_path), "-o", o, "/dev/stdin"], input=viewed, check=True, timeout=60, env=dict(os.environ, **env))
        text, refs, recs = _bam_file(o)
        assert text == want_text and text.startswith(b"@HD\tVN:1.3\tSO:coordinate\n")
        assert refs == list(contigs_of(syn_index))
        assert recs == golden("main", "syn3"), tag
        files.append(open(o, "rb").read())
    assert files[0] == files[1]  # block boundaries do not depend on threads or spills
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".run")]
    # the reference's sambamba read the file's BAM content and counted every record (golden)
    want = sambamba_golden("shim_sort")
    assert sha256(gzip.decompress(files[0])) == want["bam_sha256"] and want["records"] == len(split_records(golden("main", "syn3")))
    # foreign input goes through the shim to the real sambamba unchanged: arguments and bytes, seen by a stand-in that echoes both
    real = tmp_path / "sambamba.real"
    real.write_text('#!/bin/sh\nprintf "%s\\n" "$*"\nexec cat\n')
    real.chmod(0o755)
    sam = hdr + b"r1\t4\t*\t0\t0\t*\t*\t0\t0\tACGT\tIIII\n"
    for argv in (["view", "-S", "-f", "bam", "-l", "0", "/dev/stdin"], ["sort", "-t", "2", "-m", "1G", "--tmpdir=" + str(tmp_path), "-o", str(tmp_path / "foreign.bam"), "/dev/stdin"]):
        b = subprocess.run([shim] + argv, input=sam, stdout=subprocess.PIPE, check=True, timeout=60, env=dict(os.environ, SSQ_SAMBAMBA_REAL=str(real))).stdout
        assert b == (" ".join(argv) + "\n").encode() + sam, argv


def test_bam_mode_chain_of_the_three_shims_cpu(oracle, hostsim, ex_index, ex_reads, tmp_path):
    """`bwa mem | samblaster | sambamba view | sambamba sort` in BAM mode with the device stage played by tests/hostsim (same bodies):
    what `bwa` would write (header, marker, frames: main records as one BAM run, side streams as text) through the real samblaster and
    sambamba shims.  out.bam must hold the reference sambamba's records of the example reads; the side files the oracle's text."""
    import struct
    import subprocess
    bin_ = os.path.join(T.ROOT, "speedseq_b200", "bin")
    idx = oracle.load(ex_index)
    names, seqs, quals = ex_reads
    txt, bams = hostsim.pipe_bam(idx, names, seqs, quals, 0, b"NA12878", 1, (1, 1, 2, 20, 0))
    hdr = b"@SQ\tSN:20_slice\tLN:321635\n@RG\tID:NA12878\tSM:NA12878\tLB:lib1\n@PG\tID:bwa\tPN:bwa\tVN:0.7.12-r1039\tCL:bwa mem -p ref reads\n"
    opts = b"excludeDups=1 addMateTags=1 removeDups=0 maxSplitCount=2 minNonOverlap=20 minIndelSize=50 maxUnmappedBases=50"
    frame = lambda s, b: b"SSQFRAME" + struct.pack("<QQ", s, len(b)) + b if b else b""
    side = [t.encode() if isinstance(t, str) else t for t in txt]
    stream = hdr + b"@CO\tssq-fused-v1\t" + opts + b"\tbam\n" + frame(3, bams[0]) + frame(1, side[1]) + frame(2, side[2])
    spl, disc, out = str(tmp_path / "spl.sam"), str(tmp_path / "disc.sam"), str(tmp_path / "out.bam")
    p1 = subprocess.run([os.path.join(bin_, "samblaster"), "--excludeDups", "--addMateTags", "--maxSplitCount", "2", "--minNonOverlap", "20", "--splitterFile", spl, "--discordantFile", disc],
                        input=stream, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert p1.returncode == 0, p1.stderr
    assert b"routed %d records" % len(split_records(bams[0])) in p1.stderr
    p2 = subprocess.run([os.path.join(bin_, "sambamba"), "view", "-S", "-f", "bam", "-l", "0", "/dev/stdin"], input=p1.stdout, stdout=subprocess.PIPE, check=True, timeout=60)
    subprocess.run([os.path.join(bin_, "sambamba"), "sort", "-t", "4", "-m", "1G", "--tmpdir=" + str(tmp_path), "-o", out, "/dev/stdin"], input=p2.stdout, check=True, timeout=60)
    text, refs, recs = _bam_file(out)
    assert recs == golden("main")
    assert refs == [(b"20_slice", 321635)]
    want = open(os.path.join(T.GOLDEN, "ex_bam_header.txt"), "rb").read().split(b"\n")
    got = text.split(b"\n")
    assert got[:3] == want[:3]  # @HD, @SQ, @RG (tags re-ordered) as sambamba writes them
    assert got[3].startswith(b"@PG\tID:bwa\tPN:bwa\tCL:") and got[3].endswith(b"\tVN:0.7.12-r1039") and got[4].startswith(b"@PG\tID:SAMBLASTER\tCL:samblaster ")
    assert b"ssq-" not in text
    for fn, k in ((spl, 1), (disc, 2)):  # header + the oracle-identical text of the side stream
        lines = open(fn, "rb").read().split(b"\n")
        body = b"\n".join(l for l in lines if not l.startswith(b"@"))
        assert body == side[k] and lines[0] == b"@SQ\tSN:20_slice\tLN:321635" and any(l.startswith(b"@PG\tID:SAMBLASTER") for l in lines)
    # a samblaster command line that asks for something else than the stream was made under is refused
    p3 = subprocess.run([os.path.join(bin_, "samblaster"), "--addMateTags"], input=stream, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert p3.returncode != 0 and b"other options" in p3.stderr


def test_sambamba_shim_edge_cases(tmp_path):
    """no runs at all -> a valid BAM without records; a truncated or corrupt run stream -> an error, not a short file that looks
    complete; anything that is not a run stream needs the real sambamba and says so"""
    import struct
    import subprocess
    shim = os.path.join(T.ROOT, "speedseq_b200", "bin", "sambamba")
    hdr = b"@SQ\tSN:c1\tLN:1000\n@PG\tID:bwa\tPN:bwa\tVN:x\tCL:y\n"
    env = {k: v for k, v in os.environ.items() if k != "SSQ_SAMBAMBA_REAL"}
    out = str(tmp_path / "empty.bam")
    subprocess.run([shim, "sort", "-t", "2", "-m", "1G", "--tmpdir=" + str(tmp_path), "-o", out, "/dev/stdin"], input=hdr + b"@CO\tssq-bam-runs-v1\n", check=True, timeout=60, env=env)
    text, refs, recs = _bam_file(out)
    assert recs == b"" and refs == [(b"c1", 1000)] and text.startswith(b"@HD\tVN:1.3\tSO:coordinate\n@SQ\tSN:c1\tLN:1000\n")
    rec = struct.pack("<iiiBBHHHiiii", 32 + 2 + 1 + 1, 0, 5, 2, 0, 4680, 0, 4, 1, -1, -1, 0) + b"r\0" + b"\x10" + b"\xff"  # one unmapped-looking record placed at c1:6
    good = hdr + b"@CO\tssq-bam-runs-v1\n" + b"SSQFRAME" + struct.pack("<QQ", 3, len(rec)) + rec
    subprocess.run([shim, "sort", "-o", out, "/dev/stdin"], input=good, check=True, timeout=60, env=env)
    assert _bam_file(out)[2] == rec
    for bad in (good[:-3], good.replace(b"SSQFRAME", b"SSQFRAMX"), hdr + b"@CO\tssq-bam-runs-v1\n" + b"SSQFRAME" + struct.pack("<QQ", 3, 7) + b"1234567"):
        p = subprocess.run([shim, "sort", "-o", str(tmp_path / "bad.bam"), "/dev/stdin"], input=bad, stderr=subprocess.PIPE, timeout=60, env=env)
        assert p.returncode != 0 and b"B200 shim" in p.stderr, bad[-20:]
    for argv in (["view", "-S", "-f", "bam", "-l", "0", "/dev/stdin"], ["sort", "-o", str(tmp_path / "x.bam"), "/dev/stdin"], ["index", "x.bam"]):
        p = subprocess.run([shim] + argv, input=hdr + b"r1\t4\t*\t0\t0\t*\t*\t0\t0\tA\tI\n", stderr=subprocess.PIPE, stdout=subprocess.PIPE, timeout=60, env=env)
        assert p.returncode != 0 and b"needs the real sambamba" in p.stderr
