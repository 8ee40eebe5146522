"""`-m gpu`: eg_ciphertexts_weighted_sum on the CUDA library -- the CPU harness checks at device sizes (every window width of
the device policy, chosen at 2^8 .. 2^17 items), 2^20 + 77 items of five ciphertexts checked algebraically, a weighted tally
of 10^5 ballots decrypted end to end with a baby-step giant-step table, and multi-GPU contexts (weighted_sum_common.py)."""
import random

import numpy as np
import pytest

import decrypt_common as D
import edge_common as EC
import oracle as O
import weighted_sum_common as WS
import workloads as W
from tests.test_gpu_decrypt import counts
from tests.test_gpu_edges import TorchBuffers

pytestmark = pytest.mark.gpu

L = W.L


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
    yield eng
    eng.close()


@pytest.mark.parametrize("n,n_cts", [(1, 1), (2, 2), (31, 5), (257, 2), (3000, 5), (2, 64), (500, 64)])
@pytest.mark.parametrize("kind", ["mixed", "u64", "full"])
def test_parity(e, n, n_cts, kind):
    WS.check_parity(e, n, n_cts, kind)


@pytest.mark.parametrize("c", range(4, 14))
def test_widths(e, c):
    WS.check_width(e, 2 ** (c + 4) + 3, c, n_cts=1)


def test_thresholds(e):
    WS.check_thresholds(e, [s for k in range(8, 18) for s in (2**k - 1, 2**k)])


@pytest.mark.parametrize("n,n_cts", [(1, 1), (33, 2), (3000, 5), (70000, 1)])
def test_skew(e, n, n_cts):
    WS.check_skew(e, n, n_cts)


def test_choice_mask(e):
    WS.check_choice_mask(e, n=2000)


def test_qv_mask(e):
    WS.check_qv_mask(e, n=300)


def test_validation(e):
    WS.check_validation(e)


@pytest.mark.parametrize("n,n_cts", [(300, 1), (3000, 5)])
def test_chunks(e, n, n_cts):
    WS.check_chunks(e, n, n_cts)


@pytest.mark.parametrize("chunk", [0, 7, 1000])
def test_dev(e, chunk):
    WS.check_dev(e, TorchBuffers(), n=3000, chunk=chunk)


def test_argument_errors(e):
    WS.check_argument_errors(e)


@pytest.mark.parametrize("n_dev", counts())
def test_multi_gpu(e, n_dev):
    from elastic_elgamal_b200 import Engine
    m = Engine(devices=list(range(n_dev)))
    try:
        WS.check_multi(m, e, n=3000)
        WS.check_argument_errors(m, multi=m)
    finally:
        m.close()


def _known_ciphertexts(e, n, n_cts, key, seed):
    """n x n_cts ciphertexts under `key` of values v with randomness r, both known: (cts, r, v)."""
    rng = np.random.default_rng(seed)
    e.set_receiver(key)
    v = rng.integers(0, 2**20, n * n_cts, dtype=np.uint64)
    wide = rng.integers(0, 256, (n * n_cts, 64), dtype=np.uint8)
    cts = e.encrypt(v, wide).reshape(n, n_cts, 64)
    r = e.scalars_from_wide(wide)
    r = [int.from_bytes(bytes(x), "little") for x in r]
    return cts, r, [int(x) for x in v]


@pytest.mark.parametrize("kind", ["u64", "full"])
def test_at_size_algebraic(e, kind):
    """2^20 + 77 items of 5 ciphertexts: column j totals ([sum k_i r_ij]G, [sum k_i v_ij]G + [sum k_i r_ij]K)."""
    n, n_cts = 2**20 + 77, 5
    sk, pk = W.receiver()
    cts, r, v = _known_ciphertexts(e, n, n_cts, pk, 11)
    rnd = random.Random(13)
    ks = [rnd.randrange(2**64) for _ in range(n)] if kind == "u64" else [rnd.randrange(L) for _ in range(n)]
    out, ok = e.weighted_sum(cts, WS.scalar_rows(ks))
    assert ok
    for j in range(n_cts):
        sr = sum(ks[i] * r[i * n_cts + j] for i in range(n)) % L
        sv = sum(ks[i] * v[i * n_cts + j] for i in range(n)) % L
        want_r = O.point_mul_generator(WS.sc(sr))
        want_b = O.point_add(O.point_mul_generator(WS.sc(sv)), O.point_mul(WS.sc(sr), bytes(pk)))
        assert bytes(out[j, :32]) == want_r and bytes(out[j, 32:]) == want_b, f"column {j}"


def test_weighted_tally_decrypts(e):
    """10^5 ballots of value 0 / 1 with weights up to 2^24: the weighted total, threshold-decrypted with a baby-step
    giant-step table over [0, 2^42), is sum w_i v_i exactly."""
    n = 10**5
    ks, eks, secrets = D.keyset()
    rng = np.random.default_rng(17)
    values = rng.integers(0, 2, n, dtype=np.uint64)
    weights = rng.integers(0, 2**24 + 1, n, dtype=np.uint64)
    e.set_receiver(bytes(ks.shared_key))
    cts = e.encrypt(values, seed=bytes([0x44] * 32))
    total, ok = e.weighted_sum(cts.reshape(n, 1, 64), weights)
    assert ok
    shares = np.zeros((1, len(EC.USED), 32), np.uint8)
    for j, idx in enumerate(EC.USED):
        sh, _, sok = e.decrypt_share(eks, idx, secrets[idx], total, seed=D.SEED)
        assert sok.all()
        shares[:, j] = sh
    t = e.dlog_table(0, 2**42, 2**24 - 1)
    try:
        vals, found = e.combine_decrypt(list(EC.USED), total, shares, t)
    finally:
        t.close()
    want = int((values.astype(object) * weights.astype(object)).sum())
    assert found[0] == 1 and int(vals[0]) == want
