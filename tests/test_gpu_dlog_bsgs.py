"""`-m gpu`: baby-step giant-step discrete-log tables and eg_dlog_lookup_batch on the CUDA library -- the boundary ranges of
the CPU harness tests, ranges no table can hold ([0, 2^40), [0, 2^48) with 2^24 - 1 baby steps, [2^64 - 2^52, 2^64 - 1) with
2^20 and J = 2^32 giant steps), tallies past 2^28 through eg_combine_decrypt_batch, batch shapes up to ~10^5 and multi-GPU
contexts (dlog_bsgs_common.py)."""
import functools

import pytest

import dlog_bsgs_common as B
import edge_common as EC
from tests.test_gpu_decrypt import counts
from tests.test_gpu_edges import TorchBuffers

pytestmark = pytest.mark.gpu

M = 256                          # the boundary ranges hold every value (up to 37 m + 1), so they take small baby-step counts


@functools.lru_cache(maxsize=None)
def corpus(m):
    return EC.TableCorpus(B.boundary_ranges(m))


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def shares(e):
    return EC.library_shares(e, corpus(M))


def test_equal_to_range_table(e, shares):
    B.check_equal_to_range_table(e, corpus(M), M, shares, TorchBuffers())


@pytest.mark.parametrize("lo,hi,m,misses", [
    (0, 2**40, 2**24 - 1, 4),
    (0, 2**48, 2**24 - 1, 4),
    (2**64 - 2**52, 2**64 - 1, 2**20, 1),         # J = 2^32: every miss walks 2^32 giant steps
    (0, 2**36, 2**16 - 1, 4),
])
def test_large_range(e, lo, hi, m, misses):
    B.check_large_range(e, lo, hi, m, samples=32, misses=misses)


def test_large_tally(e):
    B.check_large_tally(e, [2**28, 2**28 + 1, 2**30 + 12345, 10**9], 0, 2**32, 2**24 - 1)


@pytest.mark.parametrize("n", [1, 5, 257, 100_003])
def test_shapes(e, n):
    B.check_shapes(e, 0, 2**36, 2**16 - 1, [n], walks=min(1000, max(1, n // 3)), misses=min(4, n // 4))


def test_shapes_chunked_and_constant_time(e):
    B.check_shapes(e, 12345, 12345 + 2**34, 2**20 - 1, [257], walks=40, misses=3, chunk=7, ct_mode=True)


@pytest.mark.parametrize("n_dev", counts())
def test_multi_gpu(shares, n_dev):
    from elastic_elgamal_b200 import Engine
    m = Engine(devices=list(range(n_dev)))
    try:
        B.check_equal_to_range_table(m, corpus(M), M, shares, None)
        B.check_large_range(m, 0, 2**40, 2**24 - 1, samples=16, misses=2)
    finally:
        m.close()


def test_argument_errors(e):
    from elastic_elgamal_b200 import Engine
    other = Engine(device=0)
    try:
        B.check_argument_errors(e, other, M)
    finally:
        other.close()
