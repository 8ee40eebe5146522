"""Known-answer and behaviour tests for the CPU oracle, mirroring the reference's own unit tests
(SURVEY.md 8(c)): decomposition KATs range.rs:591-662,689-706, doc table range.rs:56-65, Lagrange KATs
sharing/mod.rs:334-369, isqrt property quadratic_voting.rs:398-417, negative encodings
serde.rs:402-404,427-429, Merlin/STROBE KAT, Keccak vs hashlib, tamper behaviours basic.rs:35-75,
choice.rs:457-474, quadratic_voting.rs:433-464, range.rs:732-794, sharing round trip sharing.rs:108-173.
"""
import base64
import hashlib
import json
import pathlib
import random

import pytest

import oracle as O

L = 2**252 + 27742317777372353535851937790883648493
P = 2**255 - 19
G_ENC = bytes.fromhex("e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76")


def sc(x):
    return (x % L).to_bytes(32, "little")


def b64(s):
    return base64.urlsafe_b64decode(s + "=" * (-len(s) % 4))


def test_keccak_matches_hashlib_sha3_256():
    # one-block SHA3-256 built on the oracle's permutation
    for msg in (b"", b"abc", bytes(range(100))):
        st = bytearray(200)
        st[:len(msg)] = msg
        st[len(msg)] ^= 0x06
        st[135] ^= 0x80
        assert O.keccak_f1600(st)[:32] == hashlib.sha3_256(msg).digest()


def test_merlin_kat():
    # merlin's own `equivalence_simple` vector (SURVEY.md A.1)
    t = O.MerlinTranscript("test protocol")
    t.append_message("some label", b"some data")
    assert t.challenge_bytes("challenge", 32).hex() == \
        "d5a21972d0d5fe320c0d263fac7fffb8145aa640af6e9bca177c03c7efcf0615"


def test_chacha_rfc8439_block():
    # RFC 8439 2.3.2 keystream uses a 32-bit counter + 96-bit nonce; with nonce = 0 and counter = 1 the layouts coincide
    key = bytes(range(32))
    rng = O.rng_from_seed(key, 1)
    block = O.rng_block(rng)
    import struct
    # independent python ChaCha20 block
    def rotl(x, n): return ((x << n) & 0xffffffff) | (x >> (32 - n))
    def qr(s, a, b, c, d):
        s[a] = (s[a] + s[b]) & 0xffffffff; s[d] = rotl(s[d] ^ s[a], 16)
        s[c] = (s[c] + s[d]) & 0xffffffff; s[b] = rotl(s[b] ^ s[c], 12)
        s[a] = (s[a] + s[b]) & 0xffffffff; s[d] = rotl(s[d] ^ s[a], 8)
        s[c] = (s[c] + s[d]) & 0xffffffff; s[b] = rotl(s[b] ^ s[c], 7)
    init = [0x61707865, 0x3320646e, 0x79622d32, 0x6b206574] + list(struct.unpack("<8I", key)) + [1, 0, 0, 0]
    s = init[:]
    for _ in range(10):
        qr(s, 0, 4, 8, 12); qr(s, 1, 5, 9, 13); qr(s, 2, 6, 10, 14); qr(s, 3, 7, 11, 15)
        qr(s, 0, 5, 10, 15); qr(s, 1, 6, 11, 12); qr(s, 2, 7, 8, 13); qr(s, 3, 4, 9, 14)
    assert block == struct.pack("<16I", *[(a + b) & 0xffffffff for a, b in zip(s, init)])


def test_generator_and_identity_encodings():
    assert O.point_mul_generator(sc(1)) == G_ENC
    assert O.point_mul_generator(sc(0)) == bytes(32)
    assert O.point_valid(G_ENC) and O.point_valid(bytes(32))
    assert O.point_sub(G_ENC, G_ENC) == bytes(32)


def test_rfc9496_small_multiples():
    # RFC 9496 A.1: multiples 0..3 of the generator (first 4 of the published vectors)
    expected = [
        "0000000000000000000000000000000000000000000000000000000000000000",
        "e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76",
        "6a493210f7499cd17fecb510ae0cea23a110e8d5b901f8acadd3095c73a3b919",
        "94741f5d5d52755ece4f23f044ee27d5d1ea1e2bd196b462166b16152a9d0259",
    ]
    for i, e in enumerate(expected):
        assert O.point_mul_generator(sc(i)).hex() == e


def test_rfc9496_invalid_encodings():
    bad = [
        # non-canonical field encodings
        "00ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff",
        "ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
        "f3ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
        "edffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
        # negative field elements
        "0100000000000000000000000000000000000000000000000000000000000000",
        "01ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
        # non-square x^2
        "26948d35ca62e643e26a83177332e6b6afeb9d08e4268b650f1f5bbd8d81d371",
        "4eac077a713c57b4f4397629a4145982c661f48044dd3f96427d40b147d9742f",
        # negative xy
        "3eb858e78f5a7254d8c9731174a94f76755fd3941c0ac93735c07ba14579630e",
        "a45fdc55c76448c049a1ab33f17023edfb2be3581e9c7aade8a6125215e04220",
        # s = -1 -> y = 0
        "ecffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
    ]
    for h in bad:
        assert not O.point_valid(bytes.fromhex(h)), h


def test_reference_negative_encodings():
    assert not O.point_valid(b64("tNDkeYUVQWgh34d-RqaElOk7yFB8d2qCh5f4Vi2euT0"))      # serde.rs:402-404
    assert not O.scalar_is_canonical(b64("nN3xf7lSOX0_zs6QPBwWHYi0Dkx2Ln_z1MPwnbzaM_8"))  # serde.rs:427-429
    assert O.scalar_is_canonical(sc(L - 1)) and not O.scalar_is_canonical(L.to_bytes(32, "little"))


def test_scalar_arithmetic_vs_python():
    rnd = random.Random(1)
    for _ in range(200):
        wide = rnd.getrandbits(512).to_bytes(64, "little")
        assert int.from_bytes(O.scalar_reduce_wide(wide), "little") == int.from_bytes(wide, "little") % L
        a, b, c = (rnd.randrange(L) for _ in range(3))
        assert int.from_bytes(O.scalar_muladd(sc(a), sc(b), sc(c)), "little") == (a * b + c) % L
    for a in (1, 2, L - 1, rnd.randrange(L)):
        assert int.from_bytes(O.scalar_invert(sc(a)), "little") == pow(a, -1, L)
    assert O.scalar_reduce_wide(b"\xff" * 64) == sc(2**512 - 1)


def test_field_arithmetic_vs_python():
    rnd = random.Random(2)
    edge = [0, 1, 2, 19, P - 1, P - 2, 2**255 - 20, 2**254, (1 << 51) - 1]
    vals = edge + [rnd.randrange(P) for _ in range(100)]
    for a in vals:
        for b in vals[:12]:
            got = int.from_bytes(O.fe_mul(a.to_bytes(32, "little"), b.to_bytes(32, "little")), "little")
            assert got == a * b % P
    for a in vals[1:]:
        assert int.from_bytes(O.fe_invert(a.to_bytes(32, "little")), "little") == pow(a, -1, P)


def test_group_laws():
    rnd = random.Random(3)
    for _ in range(10):
        a, b = rnd.randrange(L), rnd.randrange(L)
        A, B = O.point_mul_generator(sc(a)), O.point_mul_generator(sc(b))
        assert O.point_add(A, B) == O.point_mul_generator(sc(a + b))
        assert O.point_sub(A, B) == O.point_mul_generator(sc(a - b))
        assert O.point_mul(sc(b), A) == O.point_mul_generator(sc(a * b))


def test_libsodium_cross_check():
    # products computed by libsodium, an independent implementation (SURVEY.md A.5), stored by
    # tests/golden/make_libsodium_vectors.py
    gold = json.loads((pathlib.Path(__file__).parent / "golden" / "libsodium_ristretto255.json").read_text())
    rnd = random.Random(4)
    for v in gold["vectors"]:
        k, k2 = sc(rnd.randrange(1, L)), sc(rnd.randrange(1, L))
        assert (k.hex(), k2.hex()) == (v["k"], v["k2"])
        assert O.point_mul_generator(k) == bytes.fromhex(v["k_base"])
        assert O.point_mul(k2, bytes.fromhex(v["k_base"])) == bytes.fromhex(v["k2_k_base"])
    assert len(gold["vectors"]) == 5


# ---------------------------------------------------------------- RangeDecomposition KATs

@pytest.mark.parametrize("ub,expected", [
    (5, "0..5"), (16, "4 * 0..4 + 0..4"), (60, "12 * 0..5 + 3 * 0..4 + 0..3"),
    (1000, "125 * 0..8 + 25 * 0..5 + 5 * 0..5 + 0..5"),
    (17, "4 * 0..4 + 0..5"), (101, "20 * 0..5 + 4 * 0..5 + 0..5"),
    (12345, "2880 * 0..4 + 720 * 0..5 + 90 * 0..9 + 15 * 0..7 + 3 * 0..5 + 0..3"),
    (777777, "125440 * 0..6 + 25088 * 0..6 + 3136 * 0..8 + 784 * 0..4 + 196 * 0..4 + 49 * 0..5 + 7 * 0..7 + 0..7"),
    (12345678, "3072000 * 0..4 + 768000 * 0..4 + 192000 * 0..4 + 48000 * 0..5 + 9600 * 0..6 + 1200 * 0..8 + "
               "300 * 0..4 + 75 * 0..5 + 15 * 0..5 + 3 * 0..6 + 0..3"),
    (42, "6 * 0..7 + 0..6"), (100, "20 * 0..5 + 4 * 0..5 + 0..4"),                 # range.rs:95-101
    (65536, "16384 * 0..4 + 4096 * 0..4 + 1024 * 0..4 + 256 * 0..4 + 64 * 0..4 + 16 * 0..4 + 4 * 0..4 + 0..4"),
    (21, "3 * 0..7 + 0..3"),                                                       # SURVEY.md 3.3
])
def test_range_decomposition_kats(ub, expected):
    r = O.range_optimal(ub)
    assert O.range_display(r) == expected
    assert O.lib().eo_range_upper_bound(O.C.byref(r)) == ub


def test_range_doc_table_proof_sizes():          # range.rs:56-65
    for ub, size in [(5, 6), (10, 10), (20, 12), (50, 17), (64, 17), (100, 19), (256, 23), (1000, 30)]:
        r = O.range_optimal(ub)
        assert r.rings_size + 2 * r.n_rings - 1 == size, ub


def test_isqrt():                                # quadratic_voting.rs:398-417
    rnd = random.Random(5)
    samples = list(range(1, 1000)) + [rnd.getrandbits(rnd.randrange(1, 64)) | 1 for _ in range(1000)] + [2**64 - 1]
    for x in samples:
        r = O.lib().eo_isqrt(x)
        assert r * r <= x < (r + 1) * (r + 1)


def test_lagrange_kats():                        # sharing/mod.rs:334-369
    inv = lambda x: pow(x, -1, L)
    c, s = O.lagrange_coefficients([0, 1])
    assert c == [sc(1), sc(-inv(2))] and s == sc(2)
    c, s = O.lagrange_coefficients([0, 2])
    assert c == [sc(inv(2)), sc(-inv(6))] and s == sc(3)
    c, s = O.lagrange_coefficients([0, 3, 4])
    assert c == [sc(inv(12)), sc(-inv(12)), sc(inv(20))] and s == sc(20)


# ---------------------------------------------------------------- protocol behaviours

@pytest.fixture(scope="module")
def keys():
    rng = O.rng_from_seed(bytes([5] * 32))
    sk, pk = O.keypair(rng)
    return rng, sk, pk


def flip(b, i, bit=1):
    b = bytearray(b)
    b[i] ^= bit
    return bytes(b)


def test_zero_proof_behaviour(keys):             # basic.rs:35-75
    rng, sk, pk = keys
    ct, proof = O.encrypt_zero(pk, rng)
    assert O.verify_zero(pk, ct, proof) == O.OK
    assert O.decrypt_to_element(sk, ct) == bytes(32)
    # blinded + G -> mismatch
    bad = ct[:32] + O.point_add(ct[32:], G_ENC)
    assert O.verify_zero(pk, bad, proof) == O.CHALLENGE_MISMATCH
    ct2, proof2 = O.encrypt_zero(pk, rng)
    assert O.verify_zero(pk, ct, proof2) == O.CHALLENGE_MISMATCH
    # proof for another key
    _, pk2 = O.keypair(rng)
    assert O.verify_zero(pk2, ct, proof) == O.CHALLENGE_MISMATCH
    # non-canonical scalar / invalid point are MALFORMED
    assert O.verify_zero(pk, ct, proof[:32] + b"\xff" * 32) == O.MALFORMED
    assert O.verify_zero(pk, b"\x01" + bytes(31) + ct[32:], proof) == O.MALFORMED


def test_bool_proof_behaviour(keys):             # basic.rs:116-141
    rng, sk, pk = keys
    for value in (False, True):
        ct, proof = O.encrypt_bool(pk, value, rng)
        assert O.verify_bool(pk, ct, proof) == O.OK
        assert O.decrypt_to_element(sk, ct) == (G_ENC if value else bytes(32))
        other, other_proof = O.encrypt_bool(pk, value, rng)
        assert O.verify_bool(pk, other, proof) == O.CHALLENGE_MISMATCH
        bad = ct[:32] + O.point_add(ct[32:], G_ENC)
        assert O.verify_bool(pk, bad, proof) == O.CHALLENGE_MISMATCH
        # swapped responses
        swapped = proof[:32] + proof[64:96] + proof[32:64]
        assert O.verify_bool(pk, ct, swapped) == O.CHALLENGE_MISMATCH
    # encryption of 2 cannot be proven: proof for `true` does not fit ct + G
    ct, proof = O.encrypt_bool(pk, True, rng)
    assert O.verify_bool(pk, ct[:32] + O.point_add(ct[32:], G_ENC), proof) == O.CHALLENGE_MISMATCH


@pytest.mark.parametrize("n", [2, 3, 5, 10, 15])   # basic.rs:164
def test_choice_behaviour(keys, n):
    rng, sk, pk = keys
    table = O.DlogTable(0, 2)
    for choice in {0, n // 2, n - 1}:
        cts, ring, sm = O.choice_new(pk, [i == choice for i in range(n)], True, rng)
        assert O.choice_verify(pk, n, True, cts, ring, sm) == O.OK
        dec = [table.get(O.decrypt_to_element(sk, cts[64 * i:64 * i + 64])) for i in range(n)]
        assert dec == [int(i == choice) for i in range(n)]
        # choice.rs:457-474: swapping two ciphertexts breaks the ring proof but not the sum proof
        if n > 1:
            j = (choice + 1) % n
            lo, hi = min(choice, j), max(choice, j)
            parts = [cts[64 * i:64 * i + 64] for i in range(n)]
            parts[lo], parts[hi] = parts[hi], parts[lo]
            assert O.choice_verify(pk, n, True, b"".join(parts), ring, sm) == O.CHOICE_RANGE
        # adding G to one blinded element breaks the sum proof first
        bad = bytearray(cts)
        bad[32:64] = O.point_add(cts[32:64], G_ENC)
        assert O.choice_verify(pk, n, True, bytes(bad), ring, sm) == O.CHOICE_SUM
    # multi-choice: no sum proof
    flags = [bool(i % 2) for i in range(n)]
    cts, ring, sm = O.choice_new(pk, flags, False, rng)
    assert sm is None and O.choice_verify(pk, n, False, cts, ring, None) == O.OK
    # a multi-choice with 2 selections does not pass single-choice verification with a bogus sum proof
    if n >= 4:
        assert O.choice_verify(pk, n, True, cts, ring, sc(1) + sc(2)) == O.CHOICE_SUM


@pytest.mark.parametrize("ub", [2, 5, 16, 100, 256, 1000])
def test_range_behaviour(keys, ub):              # range.rs:732-794
    rng, sk, pk = keys
    spec = O.range_optimal(ub)
    rnd = random.Random(ub)
    for value in {0, ub - 1, rnd.randrange(ub)}:
        ct, partial, ring, _ = O.range_prove(pk, spec, "ciphertext_range", value, rng)
        assert O.range_verify(pk, spec, "ciphertext_range", ct, partial, ring) == O.OK
        assert O.range_verify(pk, spec, "another_label", ct, partial, ring) == O.CHALLENGE_MISMATCH
        bad = ct[:32] + O.point_add(ct[32:], G_ENC)
        assert O.range_verify(pk, spec, "ciphertext_range", bad, partial, ring) == O.CHALLENGE_MISMATCH
        if spec.n_rings > 1:
            badp = bytearray(partial)
            badp[32:64] = O.point_add(partial[32:64], G_ENC)
            assert O.range_verify(pk, spec, "ciphertext_range", ct, bytes(badp), ring) == O.CHALLENGE_MISMATCH
        mal = ring[:-1] + b"\xff"
        assert O.range_verify(pk, spec, "ciphertext_range", ct, partial, mal) == O.MALFORMED


def test_qv_behaviour(keys):                     # quadratic_voting.rs:419-464
    rng, sk, pk = keys
    params = O.qv_params(5, 20)
    assert O.range_display(params.vote_range) == "0..5"
    assert O.range_display(params.credit_range) == "3 * 0..7 + 0..3"
    assert O.qv_ballot_size(params) == 2144
    ballot = O.qv_new(pk, params, [4, 0, 0, 1, 1], rng)       # quadratic_voting.rs:188
    assert O.qv_verify(pk, params, ballot) == O.OK
    vsz = 64 + 32 * 6
    # tamper vote 2's blinded element -> Variant{2}
    bad = bytearray(ballot)
    bad[vsz * 2 + 32:vsz * 2 + 64] = O.point_add(ballot[vsz * 2 + 32:vsz * 2 + 64], G_ENC)
    assert O.qv_verify(pk, params, bytes(bad)) == O.QV_VARIANT_BASE + 2
    # swap the credit ciphertext for one from another ballot -> CreditRange
    other = O.qv_new(pk, params, [1, 3, 0, 3, 1], rng)
    bad = bytearray(ballot)
    bad[vsz * 5:vsz * 5 + 64] = other[vsz * 5:vsz * 5 + 64]
    assert O.qv_verify(pk, params, bytes(bad)) == O.QV_CREDIT_RANGE
    # take the sum-of-squares proof from another ballot -> CreditEquivalence
    bad = ballot[:-384] + other[-384:]
    assert O.qv_verify(pk, params, bad) == O.QV_CREDIT_EQUIV
    # swapping two whole vote items keeps range proofs valid but breaks credit equivalence only if votes differ
    parts = [ballot[vsz * i:vsz * (i + 1)] for i in range(5)]
    parts[0], parts[1] = parts[1], parts[0]
    assert O.qv_verify(pk, params, b"".join(parts) + ballot[vsz * 5:]) == O.QV_CREDIT_EQUIV
    assert O.qv_verify(pk, params, ballot[:-1] + b"\xff") == O.MALFORMED


def test_sharing_round_trip():                   # sharing.rs:108-173 (3-of-5)
    rng = O.rng_from_seed(bytes([9] * 32))
    ks, secrets = O.dealer_new(5, 3, rng)
    shared = bytes(ks.shared_key)
    table = O.DlogTable(0, 1 << 10)
    for value in (0, 1, 777):
        ct = O.encrypt(shared, value, rng)
        shares = {}
        for i in (0, 2, 4):
            share, proof = O.decrypt_share(ks, i, secrets[i], ct, rng)
            assert O.verify_share(ks, i, ct, share, proof) == O.OK
            assert O.verify_share(ks, (i + 1) % 5, ct, share, proof) == O.CHALLENGE_MISMATCH
            other_ct = O.encrypt(shared, value, rng)
            assert O.verify_share(ks, i, other_ct, share, proof) == O.CHALLENGE_MISMATCH
            shares[i] = share
        rc, elem = O.combine_decrypt([0, 2, 4], [shares[0], shares[2], shares[4]], ct)
        assert rc == 0 and table.get(elem) == value
        # wrong index attribution gives garbage
        rc, elem = O.combine_decrypt([0, 1, 4], [shares[0], shares[2], shares[4]], ct)
        assert table.get(elem) is None


def test_dlog_table_semantics():                 # encryption.rs:260-298
    t = O.DlogTable(5, 10)
    assert t.get(bytes(32)) == 0                 # identity is always Some(0)
    assert t.get(O.point_mul_generator(sc(7))) == 7
    assert t.get(O.point_mul_generator(sc(4))) is None
    assert t.get(O.point_mul_generator(sc(10))) is None


def test_batch_generation_is_deterministic_and_threads_agree(keys):
    _, _, pk = keys
    seed = bytes([5] * 32)
    a = O.gen_choice_batch(pk, 5, seed, 16, threads=1)
    b = O.gen_choice_batch(pk, 5, seed, 16, threads=4)
    assert all((x == y).all() for x, y in zip(a, b))
    tail = O.gen_choice_batch(pk, 5, seed, 8, first=8, threads=2)
    assert (tail[0] == a[0][8:]).all()
    v1, t1 = O.verify_choice_batch(pk, 5, True, *a, threads=1)
    v4, t4 = O.verify_choice_batch(pk, 5, True, *a, threads=3)
    assert (v1 == 0).all() and (v1 == v4).all() and (t1 == t4).all()
