"""Checks of the decryption side (eg_decrypt_batch, eg_decrypt_share_batch*, eg_prove_decryption_batch*) shared by the CPU
harness tests (test_hostsim_decrypt.py) and the `-m gpu` tests (test_gpu_decrypt.py): byte parity with the oracle's
eo_decrypt_to_element / eo_decrypt_share / eo_decryption_prove on the same per-item ChaCha20 streams, and acceptance by the
library's own verifiers."""
import numpy as np

import oracle as O
import parity_common as PC
import workloads as W

SEED = bytes([0x21] * 32)
LABEL = "custom_key_decryption"
IDENTITY_CT = bytes(64)          # (identity, identity): e.g. the tally of a batch in which no ballot was accepted


def keyset(shares=5, threshold=3):
    rng = O.rng_from_seed(bytes([9] * 32))
    ks, secrets = O.dealer_new(shares, threshold, rng)
    return ks, PC.as_engine_keyset(ks), secrets


def ciphertexts(key, values, identity_at=()):
    """Encryptions of `values` under `key` (oracle), with (identity, identity) at the given positions."""
    rng = O.rng_from_seed(bytes([3] * 32))
    cts = [IDENTITY_CT if i in identity_at else O.encrypt(key, int(v), rng) for i, v in enumerate(values)]
    return np.frombuffer(b"".join(cts), np.uint8).reshape(len(values), 64).copy()


def item_rng(index):
    return O.rng_from_seed(SEED, first_block=index << 20)


def wide(first, n):
    return np.frombuffer(b"".join(PC.item_blocks(SEED, first + i, 1) for i in range(n)), np.uint8).reshape(n, 64).copy()


def oracle_shares(ks, index, secret, cts, first):
    rows = [O.decrypt_share(ks, index, secret, bytes(cts[i]), item_rng(first + i)) for i in range(cts.shape[0])]
    return (np.frombuffer(b"".join(r[0] for r in rows), np.uint8).reshape(-1, 32),
            np.frombuffer(b"".join(r[1] for r in rows), np.uint8).reshape(-1, 64))


def oracle_decryption_proofs(secret, cts, first):
    rows = [O.decryption_prove(secret, LABEL, bytes(cts[i]), item_rng(first + i)) for i in range(cts.shape[0])]
    return (np.frombuffer(b"".join(r[0] for r in rows), np.uint8).reshape(-1, 32),
            np.frombuffer(b"".join(r[1] for r in rows), np.uint8).reshape(-1, 64))


def check_share_parity(e, n=7, first=5, used=(0, 2, 4)):
    """Both randomness forms equal the oracle byte for byte; the shares verify and combine to the encrypted values."""
    ks, eks, secrets = keyset()
    values = [(37 * i + 1) % 50 for i in range(n)]
    values[1] = 0
    cts = ciphertexts(bytes(ks.shared_key), values, identity_at=(2,))
    values[2] = 0
    shares, proofs = np.zeros((n, len(used), 32), np.uint8), np.zeros((n, len(used), 64), np.uint8)
    for j, idx in enumerate(used):
        osh, opr = oracle_shares(ks, idx, secrets[idx], cts, first)
        sh, pr, ok = e.decrypt_share(eks, idx, secrets[idx], cts, seed=SEED, counter_base=first << 20)
        assert ok.all() and (sh == osh).all() and (pr == opr).all()
        sh2, pr2, ok2 = e.decrypt_share(eks, idx, secrets[idx], cts, wide(first, n))
        assert ok2.all() and (sh2 == sh).all() and (pr2 == pr).all()
        shares[:, j], proofs[:, j] = sh, pr
    assert (shares[2] == 0).all()                               # identity R: identity dh
    assert (e.verify_shares(eks, list(used), cts, shares, proofs) == 0).all()
    table = e.dlog_table(0, 64)
    try:
        vals, found = e.combine_decrypt(list(used), cts, shares, table)
    finally:
        table.close()
    assert found.tolist() == [1] * n and vals.tolist() == values


def check_prove_decryption_parity(e, n=6, first=2):
    sk, pk = W.receiver()
    cts = ciphertexts(pk, [3 * i for i in range(n)], identity_at=(n - 1,))
    odh, opr = oracle_decryption_proofs(sk, cts, first)
    dh, pr, ok = e.prove_decryption(LABEL, sk, cts, seed=SEED, counter_base=first << 20)
    assert ok.all() and (dh == odh).all() and (pr == opr).all()
    dh2, pr2, ok2 = e.prove_decryption(LABEL, sk, cts, wide(first, n))
    assert ok2.all() and (dh2 == dh).all() and (pr2 == pr).all()
    assert (dh[n - 1] == 0).all()
    assert (e.verify_decryption(LABEL, pk, cts, dh, pr) == 0).all()
    assert (e.verify_decryption("another label", pk, cts, dh, pr) == O.CHALLENGE_MISMATCH).all()


def check_plain_decrypt(e, table_hi=40):
    sk, pk = W.receiver()
    values = [0, 1, table_hi - 1, table_hi, 12345, 7, 0]
    cts = ciphertexts(pk, values, identity_at=(6,))
    expected = [O.decrypt_to_element(sk, bytes(c)) for c in cts]
    elements, vals, found = e.decrypt(sk, cts)
    assert vals is None and found.tolist() == [1] * len(values)
    assert [bytes(x) for x in elements] == expected
    table = e.dlog_table(0, table_hi)
    try:
        elements2, vals, found = e.decrypt(sk, cts, table)
    finally:
        table.close()
    assert (elements2 == elements).all()
    otable = O.DlogTable(0, table_hi)
    for i, el in enumerate(expected):
        ov = otable.get(el)
        assert found[i] == (0 if ov is None else 1) and int(vals[i]) == (ov or 0)
    assert found.tolist() == [1, 1, 1, 0, 0, 1, 1] and vals.tolist() == [0, 1, table_hi - 1, 0, 0, 7, 0]


def check_undecodable_items(e):
    """A ciphertext that does not decode gives ok = 0 / found = 2 and zeroed outputs; the other items are unaffected."""
    ks, eks, secrets = keyset()
    sk, pk = W.receiver()
    n = 5
    cts = ciphertexts(bytes(ks.shared_key), list(range(n)))
    bad = cts.copy()
    bad[1, :32] = np.frombuffer(W.BAD_POINT, np.uint8)
    bad[3, :32] = np.frombuffer(W.BAD_POINT2, np.uint8)
    good = [0, 2, 4]
    sh, pr, ok = e.decrypt_share(eks, 1, secrets[1], cts, seed=SEED)
    sh_b, pr_b, ok_b = e.decrypt_share(eks, 1, secrets[1], bad, seed=SEED)
    assert ok_b.tolist() == [True, False, True, False, True]
    assert (sh_b[[1, 3]] == 0).all() and (pr_b[[1, 3]] == 0).all()
    assert (sh_b[good] == sh[good]).all() and (pr_b[good] == pr[good]).all()
    dh, pr, ok = e.prove_decryption(LABEL, sk, bad, seed=SEED)
    assert ok.tolist() == [True, False, True, False, True] and (dh[[1, 3]] == 0).all() and (pr[[1, 3]] == 0).all()
    assert (e.verify_decryption(LABEL, pk, bad[good], dh[good], pr[good]) == 0).all()
    cts = ciphertexts(pk, list(range(n)))
    bad = cts.copy()
    bad[2, 32:] = np.frombuffer(W.BAD_POINT2, np.uint8)          # B does not decode
    bad[4, :32] = np.frombuffer(W.BAD_POINT, np.uint8)
    table = e.dlog_table(0, 16)
    try:
        el, vals, found = e.decrypt(sk, bad, table)
    finally:
        table.close()
    assert found.tolist() == [1, 1, 2, 1, 2] and vals.tolist() == [0, 1, 0, 3, 0] and (el[[2, 4]] == 0).all()


def check_errors_leave_context_usable(e):
    """Every argument error is reported as the header says and the next call on the same context is unaffected."""
    import ctypes as C
    from elastic_elgamal_b200 import EngineError, _ffi
    ks, eks, secrets = keyset()
    sk, pk = W.receiver()
    cts = ciphertexts(bytes(ks.shared_key), [1, 2, 3])
    ref = e.decrypt_share(eks, 2, secrets[2], cts, seed=SEED)
    ref_dh = e.prove_decryption(LABEL, sk, cts, seed=SEED)

    def status(fn):
        try:
            fn()
        except EngineError as err:
            return err.status
        return _ffi.SUCCESS

    bad_keys = PC.as_engine_keyset(ks)
    bad_keys.participant_keys[2][:] = list(W.BAD_POINT2)
    id_keys = PC.as_engine_keyset(ks)
    id_keys.participant_keys[2][:] = [0] * 32
    cases = [
        (lambda: e.decrypt_share(eks, 2, W.BAD_SCALAR, cts, seed=SEED), _ffi.ERR_INVALID_ARG),          # non-canonical secret
        (lambda: e.prove_decryption(LABEL, W.BAD_SCALAR2, cts, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.decrypt(W.BAD_SCALAR, cts), _ffi.ERR_INVALID_ARG),
        (lambda: e.decrypt_share(eks, 2, secrets[1], cts, seed=SEED), _ffi.ERR_INVALID_ARG),            # wrong secret for the index
        (lambda: e.decrypt_share(eks, 5, secrets[2], cts, seed=SEED), _ffi.ERR_INVALID_ARG),            # index out of range
        (lambda: e.decrypt_share(bad_keys, 2, secrets[2], cts, seed=SEED), _ffi.ERR_INVALID_ELEMENT),   # invalid participant key
        (lambda: e.decrypt_share(id_keys, 2, secrets[2], cts, seed=SEED), _ffi.ERR_INVALID_ELEMENT),    # identity participant key
    ]
    for fn, want in cases:
        assert status(fn) == want
        sh, pr, ok = e.decrypt_share(eks, 2, secrets[2], cts, seed=SEED)
        assert ok.all() and (sh == ref[0]).all() and (pr == ref[1]).all()
        dh, pr, ok = e.prove_decryption(LABEL, sk, cts, seed=SEED)
        assert ok.all() and (dh == ref_dh[0]).all() and (pr == ref_dh[1]).all()
    assert status(lambda: e.decrypt_share(eks, 2, secrets[1], cts, seed=SEED)) == _ffi.ERR_INVALID_ARG
    assert "participant" in e.lib.eg_last_error(e.h).decode()
    # n = 0 is a successful no-op, null buffers included
    sec = np.frombuffer(bytes(secrets[2]), np.uint8).copy()
    seed = np.frombuffer(SEED, np.uint8).copy()
    assert e.lib.eg_decrypt_share_batch_seeded(e.h, C.byref(eks), 2, sec.ctypes.data, 0, None, seed.ctypes.data, 0, None, None, None) == 0
    assert e.lib.eg_decrypt_share_batch(e.h, C.byref(eks), 2, sec.ctypes.data, 0, None, None, None, None, None) == 0
    assert e.lib.eg_prove_decryption_batch(e.h, LABEL.encode(), sec.ctypes.data, 0, None, None, None, None, None) == 0
    assert e.lib.eg_decrypt_batch(e.h, sec.ctypes.data, 0, None, None, None, None, None) == 0


def all_outputs(e, n=8):
    """Every output of the three operations on one seeded workload (for comparisons across contexts / chunkings)."""
    ks, eks, secrets = keyset()
    sk, pk = W.receiver()
    cts = ciphertexts(bytes(ks.shared_key), [5 * i for i in range(n)], identity_at=(3,))
    out = list(e.decrypt_share(eks, 4, secrets[4], cts, seed=SEED, counter_base=1 << 20))
    out += list(e.decrypt_share(eks, 0, secrets[0], cts, wide(0, n)))
    out += list(e.prove_decryption(LABEL, secrets[0], cts, seed=SEED))
    table = e.dlog_table(0, 64)
    try:
        el, vals, found = e.decrypt(sk, ciphertexts(pk, [7 * i for i in range(n)]), table)
    finally:
        table.close()
    return out + [el, vals, found]
