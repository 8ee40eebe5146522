"""`-m gpu`: edge values of the decryption side on the CUDA library -- discrete-log tables over u64 ranges up to 2^64 - 1
(incl. a 2^20-value table whose top build slices sit next to the wrap) through eg_decrypt_batch and both forms of
eg_combine_decrypt_batch, on one GPU and sharded over 1, 2, 4 and 8; u64 plaintexts at the ends of their range; secret keys
and nonces on the digit limits of the device's PTX field arithmetic and masked selects (edge_common.py)."""
import numpy as np
import pytest

import edge_common as EC
from tests.test_gpu_decrypt import counts

pytestmark = pytest.mark.gpu


class TorchBuffers:
    """Device buffers on cuda:0 (the engine's device); synchronised so that the library's own stream sees them filled."""

    def up(self, a):
        import torch
        t = torch.from_numpy(np.ascontiguousarray(a).copy()).cuda()
        torch.cuda.synchronize()
        return t

    def empty(self, n, dtype):
        import torch
        t = torch.zeros(n, dtype=getattr(torch, dtype), device="cuda")
        torch.cuda.synchronize()
        return t

    def ptr(self, t):
        return t.data_ptr()

    def down(self, t):
        return t.cpu().numpy()


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
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
    EC.check_tables_combine_dev(e, EC.table_corpus(), shares, TorchBuffers())


@pytest.mark.parametrize("n_dev", counts())
def test_table_ranges_multi_gpu(shares, n_dev):
    from elastic_elgamal_b200 import Engine
    m = Engine(devices=list(range(n_dev)))
    try:
        EC.check_tables_decrypt(m, EC.table_corpus())
        EC.check_tables_combine(m, EC.table_corpus(), shares)
    finally:
        m.close()


def test_table_argument_errors(e):
    EC.check_table_argument_errors(e, EC.table_corpus())


def test_top_table_2_20(e):
    EC.check_top_table_2_20(e, TorchBuffers())


def test_u64_plaintexts(e, mode):
    EC.check_u64_plaintexts(e)


def test_edge_keys_decrypt(e):
    EC.check_edge_keys_decrypt(e)


def test_edge_keys_and_nonces_prove_decryption(e):
    EC.check_edge_keys_and_nonces_prove(e)


def test_wide_window_nonces_prove_decryption(e):
    EC.check_wide_window_nonces_prove(e)
