"""`ssq_index_build` beyond the device sort's 2^31 - 2 suffixes builds the suffix array on the host (induced sorting, 64-bit indices,
csrc/ssq_sais.h) and writes the same five files; no GPU is touched.  SSQ_INDEX_HOST forces that path for any size (1: narrowest entry
type, 40: the 5-byte entries a whole genome gets, 64: 8-byte entries), so it is pinned here, on the CPU, on the reference's own golden index
(/root/reference/example/data/*.fasta.{amb,ann,pac,bwt,sa}) and against the oracle's builder on synthetic multi-contig genomes."""
import ctypes as C
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

import ssq_testlib as T


def _build(lib, fasta, prefix=None):
    lib.ssq_index_build.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
    lib.ssq_last_error.restype = C.c_char_p
    rc = lib.ssq_index_build(fasta.encode(), prefix.encode() if prefix else None, 0)
    assert rc == 0, lib.ssq_last_error()


@pytest.mark.parametrize("mode", ["1", "40", "64"])
def test_host_index_matches_reference_goldens(ssq_lib_cpu, tmp_path, monkeypatch, mode):
    monkeypatch.setenv("SSQ_INDEX_HOST", mode)
    fa = str(tmp_path / "ex.fa")
    open(fa, "wb").write(gzip.open(os.path.join(T.GOLDEN, "ex_ref.fa.gz")).read())
    _build(ssq_lib_cpu, fa)
    gold = json.load(open(os.path.join(T.GOLDEN, "ex_index.sha256.json")))
    for ext, g in gold.items():
        data = open(fa + "." + ext, "rb").read()
        assert len(data) == g["size"], ext
        assert hashlib.sha256(data).hexdigest() == g["sha256"], ext


@pytest.mark.parametrize("n,nc,seed,mode", [(1000, 1, 1, "64"), (4097, 3, 2, "1"), (250000, 5, 3, "40"), (1 << 20, 2, 4, "40"), (1 << 20, 2, 4, "64"), (3, 1, 5, "40")])
def test_host_index_equals_oracle_on_synthetic_genomes(ssq_lib_cpu, oracle, tmp_path, monkeypatch, n, nc, seed, mode):
    """multi-contig genomes with N runs (hole table + lrand48 replacement), long exact repeats and l_pac % 4 in {0,1,2,3}"""
    monkeypatch.setenv("SSQ_INDEX_HOST", mode)
    g, bounds = T.synth_genome(n, seed, n_contigs=nc)
    a, b = str(tmp_path / "a.fa"), str(tmp_path / "b.fa")
    T.write_fasta(a, g, bounds)
    txt = open(a).read().split("\n")
    rng = np.random.default_rng(seed)
    for k in rng.integers(1, max(2, len(txt) - 1), 6):
        if txt[k] and not txt[k].startswith(">") and len(txt[k]) > 20:
            txt[k] = txt[k][:5] + "NNNNnnRY" + txt[k][13:]
    open(a, "w").write("\n".join(txt))
    open(b, "w").write("\n".join(txt))
    oracle.index_build(a)
    _build(ssq_lib_cpu, b)
    for ext in ("amb", "ann", "pac", "bwt", "sa"):
        assert open(a + "." + ext, "rb").read() == open(b + "." + ext, "rb").read(), ext


def test_small_reference_still_needs_the_gpu(ssq_lib_cpu, tmp_path, monkeypatch):
    """without the knob a reference the device sort holds goes to the device: on a box without a GPU that is an error, not a silent CPU build"""
    if T.gpu_visible():
        pytest.skip("a GPU is present")
    monkeypatch.delenv("SSQ_INDEX_HOST", raising=False)
    fa = str(tmp_path / "ex.fa")
    open(fa, "wb").write(gzip.open(os.path.join(T.GOLDEN, "ex_ref.fa.gz")).read())
    ssq_lib_cpu.ssq_index_build.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
    assert ssq_lib_cpu.ssq_index_build(fa.encode(), None, 0) != 0
    assert not os.path.exists(fa + ".bwt") and not os.path.exists(fa + ".ann")


def test_bwa_shim_index_on_the_host_path(tmp_path):
    """`$BWA index $REF` (speedseq:389) with the shim, host path forced: the five golden files, no GPU in this container"""
    import subprocess
    fa = str(tmp_path / "ex.fa")
    open(fa, "wb").write(gzip.open(os.path.join(T.GOLDEN, "ex_ref.fa.gz")).read())
    subprocess.run([os.path.join(T.ROOT, "speedseq_b200", "bin", "bwa"), "index", fa], check=True, env=dict(os.environ, SSQ_INDEX_HOST="64"), timeout=120, stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL)
    gold = json.load(open(os.path.join(T.GOLDEN, "ex_index.sha256.json")))
    for ext, g in gold.items():
        assert hashlib.sha256(open(fa + "." + ext, "rb").read()).hexdigest() == g["sha256"], ext
