"""`-m gpu`: eg_ciphertexts_group_sum on the CUDA library -- the CPU harness checks at device sizes (32-entry runs over several
levels, 256-entry scan segments, the 2^22 cell limit, several chunks), 2^20 + 77 items of five ciphertexts in 2^16 Zipf
groups checked algebraically, a per-precinct election decrypted end to end, and multi-GPU contexts (group_sum_common.py)."""
import random

import numpy as np
import pytest

import decrypt_common as D
import group_sum_common as GS
import oracle as O
import weighted_sum_common as WS
import workloads as W
from tests.test_gpu_decrypt import counts
from tests.test_gpu_edges import TorchBuffers
from tests.test_gpu_weighted_sum import _known_ciphertexts

pytestmark = pytest.mark.gpu

L = W.L


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
    yield eng
    eng.close()


@pytest.mark.parametrize("n,n_cts", [(0, 1), (1, 1), (2, 2), (31, 5), (257, 2), (2000, 5), (2, 64), (257, 64)])
@pytest.mark.parametrize("groups", ["1", "2", "7", "1000", "n+5"])
def test_parity(e, n, n_cts, groups):
    GS.check_parity(e, n, n_cts, n + 5 if groups == "n+5" else int(groups))


@pytest.mark.parametrize("kind", GS.DISTRIBUTIONS)
@pytest.mark.parametrize("n,n_cts", [(3000, 2), (70000, 1)])
def test_distributions(e, n, n_cts, kind):
    """70 000 items in one group: runs of 32 entries reduced over four levels."""
    GS.check_distribution(e, n, n_cts, kind)


@pytest.mark.parametrize("n_groups", [255, 256, 257, 513, 65537])
def test_scan_segments(e, n_groups):
    """Group counts on both sides of the 256-entry scan segments."""
    GS.check_parity(e, 3000, 1, n_groups, "uniform")


def test_cell_limit(e):
    """n_groups * n_cts = 2^22 exactly is accepted (2^22 + 1 is refused: check_argument_errors)."""
    n = 1000
    cts, logs = WS.corpus(n, 1)
    ng = GS.MAX_CELLS
    groups = GS.group_ids(n, ng, "uniform", seed=8)
    groups[-1] = ng - 1
    out, ok = e.group_sum(cts, groups, ng)
    want, _ = GS.expected(cts, logs, groups, ng)
    assert ok.all() and (out == want).all()
    cts2, logs2 = WS.corpus(200, 64)
    g2 = GS.group_ids(200, ng // 64, "zipf", seed=9)
    out, ok = e.group_sum(cts2, g2, ng // 64)
    want, _ = GS.expected(cts2, logs2, g2, ng // 64)
    assert ok.all() and (out == want).all()


@pytest.mark.parametrize("n,n_cts", [(1, 1), (3000, 5)])
def test_single_group_is_weighted_sum(e, n, n_cts):
    GS.check_single_group_is_weighted_sum(e, n, n_cts)


def test_choice_mask(e):
    GS.check_choice_mask(e, n=2000, n_groups=37)


def test_qv_mask(e):
    GS.check_qv_mask(e, n=300, n_groups=11)


def test_bad_items(e):
    GS.check_bad_items(e)


@pytest.mark.parametrize("n,n_cts,n_groups", [(300, 1, 1), (3000, 5, 40), (3000, 2, 5000)])
def test_chunks(e, n, n_cts, n_groups):
    GS.check_chunks(e, n, n_cts, n_groups, chunks=(7, 0, 1000))


@pytest.mark.parametrize("chunk", [0, 7, 1000])
def test_dev(e, chunk):
    GS.check_dev(e, TorchBuffers(), n=3000, n_groups=300, chunk=chunk)


def test_argument_errors(e):
    GS.check_argument_errors(e)


@pytest.mark.parametrize("n_dev", counts())
def test_multi_gpu(e, n_dev):
    from elastic_elgamal_b200 import Engine
    m = Engine(devices=list(range(n_dev)))
    try:
        GS.check_multi(m, e, n=3000, n_groups=500)
        GS.check_argument_errors(m, multi=m)
    finally:
        m.close()


def _check_algebraic(out, groups, r, v, n_cts, pk, sample):
    """Group g's column j is ([sum r]G, [sum v]G + [sum r]K) over its items."""
    order = np.argsort(groups, kind="stable")
    bounds = np.searchsorted(groups[order], np.arange(int(groups.max()) + 2))
    for g in sample:
        items = order[bounds[g]:bounds[g + 1]]
        for j in range(n_cts):
            sr = sum(r[int(i) * n_cts + j] for i in items) % L
            sv = sum(v[int(i) * n_cts + j] for i in items) % L
            want_r = O.point_mul_generator(WS.sc(sr))
            want_b = O.point_add(O.point_mul_generator(WS.sc(sv)), O.point_mul(WS.sc(sr), bytes(pk)))
            assert bytes(out[g, j, :32]) == want_r and bytes(out[g, j, 32:]) == want_b, f"group {g} column {j}"


def test_at_size_algebraic(e):
    """2^20 + 77 items of 5 ciphertexts (several chunks) in 2^16 Zipf groups, checked on a seeded sample of 1000 groups plus
    the 24 largest (empty ones in the sample must be the identity); then every group of a 2^14-group run (its few empty groups the identity)."""
    n, n_cts = 2**20 + 77, 5
    sk, pk = W.receiver()
    cts, r, v = _known_ciphertexts(e, n, n_cts, pk, 19)
    ng = 2**16
    groups = GS.group_ids(n, ng, "zipf", seed=10)
    out, ok = e.group_sum(cts, groups, ng)
    assert ok.all()
    sizes = np.bincount(groups, minlength=ng)
    rnd = random.Random(21)
    sample = sorted(set(rnd.sample(range(ng), 1000)) | set(np.argsort(sizes)[-24:].tolist()))
    assert sizes[sample].max() > 10**4
    for g in sample:
        if sizes[g] == 0:
            assert not out[g].any()
    _check_algebraic(out, groups, r, v, n_cts, pk, [g for g in sample if sizes[g]])
    m, ng = 2**17, 2**14
    groups = GS.group_ids(m, ng, "uniform", seed=11)
    out, ok = e.group_sum(cts[:m], groups, ng)
    sizes = np.bincount(groups, minlength=ng)
    assert ok.all() and not out[sizes == 0].any()
    _check_algebraic(out, groups, r, v, n_cts, pk, np.flatnonzero(sizes))


def test_precincts_end_to_end(e):
    """10^5 five-option ballots under the shared key of a 3-of-5 key set, in 1000 precincts of Zipf sizes, 1 % tampered:
    verify_choice, group_sum under the verdicts, five participants' decryption shares (one with tampered proofs),
    verify_shares and combine_decrypt_accepted give each precinct's option counts over the accepted ballots."""
    n, m, ng = 10**5, 5, 1000
    ks, eks, secrets = D.keyset()
    e.set_receiver(bytes(ks.shared_key))
    rng = np.random.default_rng(23)
    choice = rng.integers(0, m, n)
    values = np.zeros((n, m), np.uint8)
    values[np.arange(n), choice] = 1
    cts, rings, sums = e.encrypt_choice(m, values, seed=bytes([0x5a] * 32))
    cts, rings, sums = cts.copy(), rings.copy(), sums.copy()
    W.tamper_choice(cts, rings, sums, random.Random(24), frac=0.01)
    v, tally = e.verify_choice(m, cts, rings, sums)
    assert 0 < int((v != 0).sum()) <= n // 100
    groups = GS.group_ids(n, ng, "zipf", seed=12)
    out, ok = e.group_sum(cts, groups, ng, v)
    assert ok.all()
    total, sok = e.ciphertexts_sum(out)
    assert sok and (total == tally).all()
    flat = out.reshape(ng * m, 64)
    indexes = [0, 1, 2, 3, 4]
    shares, proofs = np.zeros((ng * m, 5, 32), np.uint8), np.zeros((ng * m, 5, 64), np.uint8)
    for j in indexes:
        sh, pr, sok = e.decrypt_share(eks, j, secrets[j], flat, seed=D.SEED)
        assert sok.all()
        shares[:, j], proofs[:, j] = sh, pr
    proofs[:, 1, 40] ^= 1                                # participant 1's proofs are tampered everywhere
    sv = e.verify_shares(eks, indexes, flat, shares, proofs)
    assert (sv[:, 1] != 0).all() and (sv[:, [0, 2, 3, 4]] == 0).all()
    t = e.dlog_table(0, n + 1)
    try:
        vals, found = e.combine_decrypt_accepted(3, indexes, flat, shares, sv, t)
    finally:
        t.close()
    assert (found == 1).all()
    want = np.zeros((ng, m), np.uint64)
    acc = v == 0
    np.add.at(want, (groups[acc], choice[acc]), 1)
    assert (vals.reshape(ng, m) == want).all(), "per-precinct counts differ from the accepted ballots' plaintexts"
