"""`-m gpu`: the decryption side on the CUDA library -- oracle parity in both prover modes, the whole threshold decryption with
unique items at 262 144 + 13 ciphertexts (encrypt -> three participants' shares -> verify_shares -> combine_decrypt), the
device-pointer form, chunking invariance, SecretKey::decrypt at the same size, and multi-GPU sharding giving the bytes of one
GPU."""
import random

import numpy as np
import pytest

import decrypt_common as D
import oracle as O
import workloads as W

pytestmark = pytest.mark.gpu
N = (1 << 18) + 13
USED = (0, 2, 4)


def gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def counts():
    """Device counts 1, 2, 4 and 8; a count above what the machine has skips."""
    n = gpu_count()
    return [c if c <= max(n, 1) else pytest.param(c, marks=pytest.mark.skip(reason=f"needs {c} GPUs, {n} visible"))
            for c in (1, 2, 4, 8)]


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
    yield eng
    eng.close()


@pytest.fixture(params=[False, True], ids=["default", "constant_time"])
def mode(request, e):
    e.set_prover_mode(request.param)
    yield request.param
    e.set_prover_mode(False)


def participant_seed(idx):
    return bytes([0x40 + idx] * 32)


@pytest.fixture(scope="module")
def election(e):
    """N unique ciphertexts of values in [0, 2^20) under the key set's shared key, made on the GPU."""
    ks, eks, secrets = D.keyset()
    values = (np.arange(N, dtype=np.uint64) * 40503 + 11) % (1 << 20)
    e.set_receiver(bytes(ks.shared_key))
    cts = e.encrypt(values, seed=bytes(range(32)))
    return ks, eks, secrets, values, cts


def test_parity_with_oracle(e, mode):
    D.check_share_parity(e)
    D.check_prove_decryption_parity(e)
    D.check_plain_decrypt(e)


def test_undecodable_and_errors(e):
    D.check_undecodable_items(e)
    D.check_errors_leave_context_usable(e)


def test_threshold_decryption_unique_262k(e, election):
    ks, eks, secrets, values, cts = election
    n = cts.shape[0]
    shares, proofs = np.empty((n, len(USED), 32), np.uint8), np.empty((n, len(USED), 64), np.uint8)
    for j, idx in enumerate(USED):
        sh, pr, ok = e.decrypt_share(eks, idx, secrets[idx], cts, seed=participant_seed(idx))
        assert ok.all()
        shares[:, j], proofs[:, j] = sh, pr
        for i in range(16):
            osh, opr = O.decrypt_share(ks, idx, secrets[idx], bytes(cts[i]), O.rng_from_seed(participant_seed(idx), first_block=i << 20))
            assert bytes(sh[i]) == osh and bytes(pr[i]) == opr
    assert (e.verify_shares(eks, list(USED), cts, shares, proofs) == 0).all()
    rnd = random.Random(8)
    rows = sorted(rnd.sample(range(n - 1), 4))
    bad = proofs.copy()
    for i in rows:                                              # swap the proofs of two tallies: 8 proofs in all
        bad[i, 1], bad[i + 1, 1] = proofs[i + 1, 1], proofs[i, 1]
    v = e.verify_shares(eks, list(USED), cts, shares, bad)
    wrong = {(int(i), int(j)) for i, j in zip(*np.nonzero(v))}
    assert wrong == {(i, 1) for i in rows} | {(i + 1, 1) for i in rows}
    assert all(v[i, 1] == O.CHALLENGE_MISMATCH for i in rows)
    table = e.dlog_table(0, 1 << 20)
    try:
        vals, found = e.combine_decrypt(list(USED), cts, shares, table)
    finally:
        table.close()
    assert (found == 1).all() and (vals == values).all()


def test_dev_form_and_chunking(e, election):
    import torch
    ks, eks, secrets, values, cts = election
    n = 20011
    cts = np.ascontiguousarray(cts[:n])
    sh, pr, ok = e.decrypt_share(eks, 2, secrets[2], cts, seed=participant_seed(2), counter_base=3)
    d_cts = torch.from_numpy(cts).cuda()
    d_sh, d_pr = torch.empty((n, 32), dtype=torch.uint8, device="cuda"), torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    d_ok = torch.empty(n, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    e.decrypt_share_dev(eks, 2, secrets[2], n, d_cts.data_ptr(), d_sh.data_ptr(), d_pr.data_ptr(), d_ok.data_ptr(),
                        seed=participant_seed(2), counter_base=3)
    assert (d_sh.cpu().numpy() == sh).all() and (d_pr.cpu().numpy() == pr).all() and (d_ok.cpu().numpy() == 1).all()
    wide = np.frombuffer(np.random.default_rng(3).bytes(n * 64), np.uint8).reshape(n, 64)
    sh_w, pr_w, _ = e.decrypt_share(eks, 2, secrets[2], cts, wide)
    d_wide = torch.from_numpy(wide.copy()).cuda()
    e.decrypt_share_dev(eks, 2, secrets[2], n, d_cts.data_ptr(), d_sh.data_ptr(), d_pr.data_ptr(), d_ok.data_ptr(), d_wide_rand=d_wide.data_ptr())
    assert (d_sh.cpu().numpy() == sh_w).all() and (d_pr.cpu().numpy() == pr_w).all()
    sk, pk = W.receiver()
    dh, dpr, _ = e.prove_decryption(D.LABEL, sk, cts, seed=D.SEED)
    e.set_chunk_items(5000)
    try:
        sh_c, pr_c, _ = e.decrypt_share(eks, 2, secrets[2], cts, seed=participant_seed(2), counter_base=3)
        dh_c, dpr_c, _ = e.prove_decryption(D.LABEL, sk, cts, seed=D.SEED)
    finally:
        e.set_chunk_items(0)
    assert (sh_c == sh).all() and (pr_c == pr).all() and (dh_c == dh).all() and (dpr_c == dpr).all()
    assert (e.verify_decryption(D.LABEL, pk, cts, dh, dpr) == 0).all()


def test_decrypt_at_size(e):
    sk, pk = W.receiver()
    values = (np.arange(N, dtype=np.uint64) * 7919 + 5) % (1 << 20)
    values[7] = (1 << 20) + 5                                    # outside the table
    e.set_receiver(pk)
    cts = e.encrypt(values, seed=bytes([0x33] * 32))
    table = e.dlog_table(0, 1 << 20)
    try:
        el, vals, found = e.decrypt(sk, cts, table)
    finally:
        table.close()
    inside = np.ones(N, bool)
    inside[7] = False
    assert (found[inside] == 1).all() and (vals[inside] == values[inside]).all() and found[7] == 0
    for i in range(0, 64):
        assert bytes(el[i]) == O.decrypt_to_element(sk, bytes(cts[i]))


@pytest.mark.parametrize("n_dev", counts())
def test_multi_gpu_matches_single_gpu(e, election, n_dev):
    from elastic_elgamal_b200 import Engine
    ks, eks, secrets, values, cts = election
    cts = np.ascontiguousarray(cts[:50003])
    ref = D.all_outputs(e) + list(e.decrypt_share(eks, 4, secrets[4], cts, seed=participant_seed(4)))
    m = Engine(devices=list(range(n_dev)))
    try:
        got = D.all_outputs(m) + list(m.decrypt_share(eks, 4, secrets[4], cts, seed=participant_seed(4)))
    finally:
        m.close()
    assert all((a == b).all() for a, b in zip(ref, got))
