"""The C-ABI library loads without a GPU, exports every symbol include/ssq.h declares, and refuses to compute on a box
without an sm_100 device (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import ssq_testlib as T


def _declared():
    h = open(os.path.join(T.ROOT, "include", "ssq.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return sorted(set(re.findall(r"\b(ssq_[a-z0-9_]+)\s*\(", h)))


def test_exports_every_declared_symbol():
    assert os.path.exists(T.SSQ_SO), "run __graft_entry__.build() first"
    lib = C.CDLL(T.SSQ_SO)
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n


def test_default_options_match_oracle(oracle):
    s = T.SSQ()
    o = np.frombuffer(bytes(s.opts), np.int32)
    f = np.frombuffer(bytes(s.opts), np.float32)
    # a b o_del e_del o_ins e_ins pen_unpaired clip5 clip3 w zdrop T min_seed split_width max_occ max_chain_gap max_mem_intv
    assert o[:17].tolist() == [1, 4, 6, 1, 6, 1, 17, 5, 5, 100, 100, 30, 19, 10, 500, 10000, 20]
    assert o[17:22].tolist() == [0, 1 << 30, 10000, 50, 5]
    assert np.allclose(f[22:27], [1.5, 0.5, 0.5, 0.8, 0.95])
    assert o[27:30].tolist() == [50, 3, 1]
    assert C.sizeof(s.opts) == 30 * 4


@pytest.mark.skipif(T.gpu_visible(), reason="box has a GPU")
def test_no_cpu_fallback_without_gpu(ex_index):
    s = T.SSQ()
    h = C.c_void_p()
    rc = s.lib.ssq_index_load(ex_index.encode(), 0, C.byref(h))
    assert rc == -1 and "no CPU path" in s.err()
    d = np.zeros(4, np.uint8)
    sig = np.zeros(4, T.DUPSIG_DT)
    assert s.lib.ssq_dupmark_batch(0, C.c_uint64(4), sig.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p)) == -1
