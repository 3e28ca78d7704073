"""Generates tests/golden/sambamba_reads.json: what the reference's sambamba (v0.5.9) makes of two BAM files the tests write, so
that the tests keep the comparison without the binary.
  bgzf_example : the example reads' main records compressed by ssq_bgzf_compress (test_bgzf_framing_roundtrip_and_sambamba_reads_it);
                 `sambamba view` of the file: its line count and the SHA-256 of its text
  shim_sort    : the `sambamba` shim's sorted BAM of the synthetic run of three batches (test_sambamba_shim_merges_the_run_stream);
                 `sambamba view -c` of the file
with the SHA-256 of each file's decompressed BAM content.  usage: python tests/golden/make_sambamba_golden.py <sambamba v0.5.9>"""
import ctypes as C
import gzip
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import ssq_testlib as T  # noqa: E402
import test_bam_golden as B  # noqa: E402

sb = sys.argv[1]
out = {}
with tempfile.TemporaryDirectory() as d:
    o = T.Oracle()
    h = T.HostSim(o)
    L = C.CDLL(T.SSQ_SO)
    L.ssq_bgzf_compress.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    fa = os.path.join(d, "ex.fa")
    open(fa, "wb").write(gzip.open(os.path.join(T.GOLDEN, "ex_ref.fa.gz")).read())
    o.index_build(fa)
    names, seqs, quals = [], [], []
    with gzip.open(os.path.join(T.GOLDEN, "ex_reads_2k.fq.gz"), "rt") as f:  # as tests/conftest.py's ex_reads
        for i, l in enumerate(f):
            l = l.rstrip("\n")
            if i % 4 == 0:
                names.append(l[1:].split()[0][:-2])
            elif i % 4 == 1:
                seqs.append(l)
            elif i % 4 == 3:
                quals.append(l)
    raw, _ = B.example_bam(o, h, fa, (names, seqs, quals))
    p, n = C.c_void_p(), C.c_size_t(0)
    assert L.ssq_bgzf_compress(raw, C.c_size_t(len(raw)), C.c_int(6), C.c_int(1), C.byref(p), C.byref(n)) == 0
    bam = os.path.join(d, "x.bam")
    open(bam, "wb").write(C.string_at(p, n.value))
    view = subprocess.run([sb, "view", bam], check=True, stdout=subprocess.PIPE).stdout.splitlines()
    out["bgzf_example"] = {"bam_sha256": hashlib.sha256(raw).hexdigest(), "view_lines": len(view),
                           "view_sha256": hashlib.sha256(b"".join(l + b"\n" for l in view)).hexdigest()}

    g, bounds = T.synth_genome(400000, 7, n_contigs=3)  # as tests/conftest.py's syn_index
    fa2 = os.path.join(d, "syn.fa")
    T.write_fasta(fa2, g, bounds)
    o.index_build(fa2)
    hdr, stream = B.shim_run_stream(o, h, (fa2, g, bounds))
    shim = os.path.join(T.ROOT, "speedseq_b200", "bin", "sambamba")
    bam = os.path.join(d, "plain.bam")
    subprocess.run([shim, "sort", "-t", "4", "-m", "1G", "--tmpdir=" + d, "-o", bam, "/dev/stdin"], input=stream, check=True)
    out["shim_sort"] = {"bam_sha256": hashlib.sha256(gzip.decompress(open(bam, "rb").read())).hexdigest(),
                        "records": int(subprocess.run([sb, "view", "-c", bam], check=True, stdout=subprocess.PIPE).stdout)}
json.dump(out, open(os.path.join(HERE, "sambamba_reads.json"), "w"), indent=1)
print(out)
