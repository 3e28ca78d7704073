"""GPU parity of the seeding paths that are not the default: the lean backward kernel (SSQ_SMEM_VARIANT=4), the k-mer jump-start
table (SSQ_KMER_K) and the split path's pool-overflow retry."""
import numpy as np
import pytest

import ssq_testlib as T

pytestmark = pytest.mark.gpu


def _reads(syn_index, n=1500, seed=41):
    fa, g, bounds = syn_index
    names, seqs, quals = T.simulate_pairs(g, bounds, n, 150, seed, err=0.01, indel=0.002, n_frac=0.003)
    return seqs + ["", "A", "N" * 30, "AC" * 70, "A" * 150, "ACGT" * 37, "T" * 100]


@pytest.mark.parametrize("variant,kmer", [("3", None), ("4", None), ("3", "8"), ("4", "8"), ("4", "10"), ("2", "10")])
def test_seeding_variants(ssq, oracle, syn_index, monkeypatch, variant, kmer):
    monkeypatch.setenv("SSQ_SMEM_VARIANT", variant)
    if kmer:
        monkeypatch.setenv("SSQ_KMER_K", kmer)  # read by ssq_index_load
    fa = syn_index[0]
    idx = oracle.load(fa)
    h = ssq.index_load(fa)
    try:
        seq, off = T.encode_reads(_reads(syn_index))
        a, ao = oracle.smem_batch(idx, seq, off)
        b, bo = ssq.smem_batch(h, seq, off)
        assert np.array_equal(ao, bo) and np.array_equal(a, b)
        a, ao = oracle.align_batch(idx, seq, off)
        b, bo = ssq.align_batch(h, seq, off)
        assert np.array_equal(ao, bo) and np.array_equal(a, b)
    finally:
        ssq.index_free(h)


def test_split_pool_overflow_retry(ssq, oracle, syn_index, monkeypatch):
    """tiny initial pools: the split path must grow them and run the stage again"""
    monkeypatch.setenv("SSQ_SMEM_VARIANT", "3")
    monkeypatch.setenv("SSQ_SPLIT_TINY_POOLS", "1")
    fa = syn_index[0]
    idx = oracle.load(fa)
    h = ssq.index_load(fa)
    try:
        seq, off = T.encode_reads(_reads(syn_index, 800, 43))
        a, ao = oracle.smem_batch(idx, seq, off)
        b, bo = ssq.smem_batch(h, seq, off)
        assert np.array_equal(ao, bo) and np.array_equal(a, b)
    finally:
        ssq.index_free(h)
