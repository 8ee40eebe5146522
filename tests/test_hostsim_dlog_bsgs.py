"""Baby-step giant-step discrete-log tables and eg_dlog_lookup_batch on the CPU-compiled library (TEST HARNESS ONLY,
tests/hostsim): small baby-step counts (256 - 1023) and ranges up to about 2^16 values, on single and multi-device contexts
(dlog_bsgs_common.py)."""
import functools

import pytest

import dlog_bsgs_common as B
import edge_common as EC
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build
from test_hostsim_edges import HostBuffers

M = 256


@functools.lru_cache(maxsize=None)
def corpus(m):
    return EC.TableCorpus(B.boundary_ranges(m))


@pytest.fixture(scope="module")
def e():
    eng = Engine(lib_path=build())
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def shares(e):
    return EC.library_shares(e, corpus(M))


def test_equal_to_range_table(e, shares):
    B.check_equal_to_range_table(e, corpus(M), M, shares, HostBuffers())


@pytest.mark.parametrize("lo,hi,m", [(0, 2**16, 256), (0, 2**16, 257), (2**64 - 2**17, 2**64 - 1, 1023)])
def test_large_range(e, lo, hi, m):
    B.check_large_range(e, lo, hi, m, samples=16, misses=2)


def test_large_tally(e):
    B.check_large_tally(e, [2**12, 2**12 + 1, 2**14 + 12345, 60000], 0, 2**16, 1023)


@pytest.mark.parametrize("n", [1, 5, 257, 100_000])
def test_shapes(e, n):
    B.check_shapes(e, 0, 2**16, 256, [n], walks=min(64, max(1, n // 3)), misses=min(4, n // 4), decrypt=n < 100_000)


def test_shapes_chunked_and_constant_time(e):
    B.check_shapes(e, 1000, 1000 + 2**14, 300, [257], walks=40, misses=3, chunk=7, ct_mode=True)


@pytest.mark.parametrize("children", [1, 3])
def test_multi_context(e, shares, children):
    m = Engine(lib_path=build(), devices=[0] * children)
    try:
        B.check_equal_to_range_table(m, corpus(M), M, shares, None)
    finally:
        m.close()


def test_argument_errors(e):
    other = Engine(lib_path=build())
    try:
        B.check_argument_errors(e, other, M)
    finally:
        other.close()
