"""Edge values of the decryption side on the CPU-compiled library (TEST HARNESS ONLY, tests/hostsim): discrete-log tables over
u64 ranges up to 2^64 - 1 through eg_decrypt_batch and both forms of eg_combine_decrypt_batch, on single and multi-device
contexts; u64 plaintexts at the ends of their range; secret keys and nonces on the digit limits of the decryption kernels."""
import numpy as np
import pytest

import edge_common as EC
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build


class HostBuffers:
    """Device buffers of the CPU harness, whose device memory is host memory: numpy arrays stand in."""

    def up(self, a):
        return np.ascontiguousarray(a).copy()

    def empty(self, n, dtype):
        return np.zeros(n, dtype)

    def ptr(self, a):
        return a.ctypes.data

    def down(self, a):
        return a


@pytest.fixture(scope="module")
def e():
    eng = Engine(lib_path=build())
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def shares(e):
    return EC.library_shares(e, EC.table_corpus())


@pytest.fixture(params=[False, True], ids=["default", "constant_time"])
def mode(request, e):
    e.set_prover_mode(request.param)
    yield request.param
    e.set_prover_mode(False)


def test_table_ranges_decrypt(e):
    EC.check_tables_decrypt(e, EC.table_corpus())


def test_table_ranges_combine_decrypt(e, shares):
    EC.check_tables_combine(e, EC.table_corpus(), shares)
    EC.check_tables_combine_dev(e, EC.table_corpus(), shares, HostBuffers())


@pytest.mark.parametrize("children", [1, 3])
def test_table_ranges_multi_context(shares, children):
    m = Engine(lib_path=build(), devices=[0] * children)
    try:
        EC.check_tables_decrypt(m, EC.table_corpus())
        EC.check_tables_combine(m, EC.table_corpus(), shares)
    finally:
        m.close()


def test_table_argument_errors(e):
    EC.check_table_argument_errors(e, EC.table_corpus())


def test_u64_plaintexts(e, mode):
    EC.check_u64_plaintexts(e)


def test_recodings_hit_their_edges():
    EC.check_recodings_hit_their_edges()


def test_edge_keys_decrypt(e):
    EC.check_edge_keys_decrypt(e)


def test_edge_keys_and_nonces_prove_decryption(e):
    EC.check_edge_keys_and_nonces_prove(e)


def test_wide_window_nonces_prove_decryption(e):
    EC.check_wide_window_nonces_prove(e)
