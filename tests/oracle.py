"""ctypes bindings for the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
`--impl reference` legs.  The product package (elastic_elgamal_b200) never imports this module.
"""
import ctypes as C
import os
import pathlib
import subprocess

ROOT = pathlib.Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
LIB_PATH = ORACLE_DIR / "liboracle.so"

EO_MAX_RINGS = 64

OK, MALFORMED, CHALLENGE_MISMATCH, CHOICE_SUM, CHOICE_RANGE, QV_CREDIT_RANGE, QV_CREDIT_EQUIV, MALFORMED_PARTICIPANT_KEYS = range(8)
QV_VARIANT_BASE = 16


def build(force=False):
    stale = LIB_PATH.exists() and any(p.stat().st_mtime > LIB_PATH.stat().st_mtime
                                      for p in list(ORACLE_DIR.glob("*.[ch]")) + [ORACLE_DIR / "Makefile"])
    if force or stale or not LIB_PATH.exists():
        subprocess.run(["make", "-C", str(ORACLE_DIR), "-B" if force else "-s", "liboracle.so"], check=True,
                       stdout=subprocess.DEVNULL)
    return LIB_PATH


class RngOverrun(AssertionError):
    """A replaying oracle rng was asked for more blocks than it was given."""


class Rng(C.Structure):
    """eo_rng (oracle/eg_oracle.h): a replaying rng keeps its state in the key bytes, so the layout is the same for both
    forms; its size is checked against eo_rng_size() when the library is loaded."""
    _fields_ = [("key", C.c_uint8 * 32), ("block", C.c_uint64)]


class Range(C.Structure):
    _fields_ = [("n_rings", C.c_uint32), ("size", C.c_uint64 * EO_MAX_RINGS), ("step", C.c_uint64 * EO_MAX_RINGS)]

    @property
    def rings(self):
        return [(self.size[i], self.step[i]) for i in range(self.n_rings)]

    @property
    def rings_size(self):
        return sum(self.size[i] for i in range(self.n_rings))


class QvParams(C.Structure):
    _fields_ = [("options", C.c_uint32), ("credits", C.c_uint64), ("vote_range", Range), ("credit_range", Range)]


class KeySet(C.Structure):
    _fields_ = [("shares", C.c_uint32), ("threshold", C.c_uint32), ("shared_key", C.c_uint8 * 32),
                ("participant_keys", (C.c_uint8 * 32) * 64)]


class Transcript(C.Structure):
    _fields_ = [("state", C.c_uint8 * 200), ("pos", C.c_uint8), ("pos_begin", C.c_uint8), ("cur_flags", C.c_uint8)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        try:
            _lib = C.CDLL(str(LIB_PATH))
        except OSError:
            build(force=True)
            _lib = C.CDLL(str(LIB_PATH))
        _lib.eo_range_upper_bound.restype = C.c_uint64
        _lib.eo_range_rings_size.restype = C.c_uint64
        _lib.eo_range_display.restype = C.c_size_t
        _lib.eo_qv_ballot_size.restype = C.c_size_t
        _lib.eo_isqrt.restype = C.c_uint64
        _lib.eo_isqrt.argtypes = [C.c_uint64]
        _lib.eo_dlog_table_new.restype = C.c_void_p
        _lib.eo_dlog_table_new.argtypes = [C.c_uint64, C.c_uint64]
        _lib.eo_dlog_table_free.argtypes = [C.c_void_p]
        _lib.eo_dlog_table_get.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_uint64)]
        _lib.eo_range_optimal.argtypes = [C.POINTER(Range), C.c_uint64]
        _lib.eo_rng_seed_from_u64.argtypes = [C.POINTER(Rng), C.c_uint64]
        _lib.eo_rng_from_seed.argtypes = [C.POINTER(Rng), C.c_char_p, C.c_uint64]
        _lib.eo_rng_from_blocks.argtypes = [C.POINTER(Rng), C.c_void_p, C.c_uint64]
        _lib.eo_rng_size.restype = C.c_size_t
        _lib.eo_rng_overrun.argtypes = [C.POINTER(Rng)]
        _lib.eo_rng_blocks_left.argtypes = [C.POINTER(Rng)]
        _lib.eo_rng_blocks_left.restype = C.c_uint64
        # a mirror that disagrees with the C struct would corrupt memory far from the cause
        assert _lib.eo_rng_size() == C.sizeof(Rng), (_lib.eo_rng_size(), C.sizeof(Rng))
    return _lib


def buf(n):
    return (C.c_uint8 * n)()


def raw(b):
    return bytes(b)


# ---------------------------------------------------------------- rng / primitives

def rng_from_u64(seed):
    r = Rng()
    lib().eo_rng_seed_from_u64(C.byref(r), seed)
    return r


def rng_from_seed(seed32, first_block=0):
    r = Rng()
    lib().eo_rng_from_seed(C.byref(r), bytes(seed32), first_block)
    return r


def rng_from_blocks(blocks):
    """An rng that replays `blocks` (a multiple of 64 bytes) in order, as the library's `wide_rand` form takes them; every
    wrapper below raises RngOverrun once a prover has drawn past the end."""
    blocks = bytes(blocks)
    assert len(blocks) % 64 == 0
    r = Rng()
    r._blocks = C.create_string_buffer(blocks, len(blocks))       # kept alive with the rng
    lib().eo_rng_from_blocks(C.byref(r), C.addressof(r._blocks), len(blocks) // 64)
    return r


def rng_blocks_left(rng):
    """Blocks a replaying rng has not handed out yet."""
    return lib().eo_rng_blocks_left(C.byref(rng))


def _drawn(rng):
    if lib().eo_rng_overrun(C.byref(rng)):
        raise RngOverrun(f"a prover drew more than the {rng.block - 1} blocks of its replay")


def rng_block(rng):
    out = buf(64)
    lib().eo_rng_block(C.byref(rng), out)
    _drawn(rng)
    return raw(out)


def keypair(rng):
    sk, pk = buf(32), buf(32)
    lib().eo_keypair_generate(C.byref(rng), sk, pk)
    _drawn(rng)
    return raw(sk), raw(pk)


def scalar_reduce_wide(b64):
    out = buf(32)
    lib().eo_scalar_reduce_wide_bytes(out, bytes(b64))
    return raw(out)


def scalar_is_canonical(b):
    return bool(lib().eo_scalar_is_canonical(bytes(b)))


def scalar_muladd(a, b, c):
    out = buf(32)
    lib().eo_scalar_muladd_bytes(out, bytes(a), bytes(b), bytes(c))
    return raw(out)


def scalar_invert(a):
    out = buf(32)
    lib().eo_scalar_invert_bytes(out, bytes(a))
    return raw(out)


def point_valid(b):
    return bool(lib().eo_point_decode_check(bytes(b)))


def point_mul(scalar, point):
    out = buf(32)
    if not lib().eo_point_mul_bytes(out, bytes(scalar), bytes(point)):
        return None
    return raw(out)


def point_mul_generator(scalar):
    out = buf(32)
    lib().eo_point_mul_generator_bytes(out, bytes(scalar))
    return raw(out)


def point_add(a, b):
    out = buf(32)
    if not lib().eo_point_add_bytes(out, bytes(a), bytes(b)):
        return None
    return raw(out)


def point_sub(a, b):
    out = buf(32)
    if not lib().eo_point_sub_bytes(out, bytes(a), bytes(b)):
        return None
    return raw(out)


def fe_mul(a, b):
    out = buf(32)
    lib().eo_fe_mul_bytes(out, bytes(a), bytes(b))
    return raw(out)


def fe_invert(a):
    out = buf(32)
    lib().eo_fe_invert_bytes(out, bytes(a))
    return raw(out)


def keccak_f1600(state200):
    s = (C.c_uint8 * 200).from_buffer_copy(bytes(state200))
    lib().eo_keccak_f1600(s)
    return raw(s)


class MerlinTranscript:
    def __init__(self, label):
        self.t = Transcript()
        lib().eo_transcript_new(C.byref(self.t), label.encode())

    def append_message(self, label, msg):
        lib().eo_transcript_append_message(C.byref(self.t), label.encode(), bytes(msg), C.c_size_t(len(msg)))

    def append_u64(self, label, x):
        lib().eo_transcript_append_u64(C.byref(self.t), label.encode(), C.c_uint64(x))

    def challenge_bytes(self, label, n):
        out = buf(n)
        lib().eo_transcript_challenge_bytes(C.byref(self.t), label.encode(), out, C.c_size_t(n))
        return raw(out)

    def state(self):
        return raw(self.t.state), self.t.pos, self.t.pos_begin


# ---------------------------------------------------------------- protocol objects

def encrypt(pk, value, rng):
    ct = buf(64)
    assert lib().eo_encrypt(pk, C.c_uint64(value), C.byref(rng), ct) == 0
    _drawn(rng)
    return raw(ct)


def decrypt_to_element(sk, ct):
    out = buf(32)
    assert lib().eo_decrypt_to_element(sk, ct, out) == 0
    return raw(out)


def encrypt_zero(pk, rng):
    ct, proof = buf(64), buf(64)
    assert lib().eo_encrypt_zero(pk, C.byref(rng), ct, proof) == 0
    _drawn(rng)
    return raw(ct), raw(proof)


def verify_zero(pk, ct, proof):
    return lib().eo_verify_zero(pk, bytes(ct), bytes(proof))


def encrypt_bool(pk, value, rng):
    ct, proof = buf(64), buf(96)
    assert lib().eo_encrypt_bool(pk, int(value), C.byref(rng), ct, proof) == 0
    _drawn(rng)
    return raw(ct), raw(proof)


def verify_bool(pk, ct, proof):
    return lib().eo_verify_bool(pk, bytes(ct), bytes(proof))


def choice_new(pk, choices, single, rng):
    n = len(choices)
    cts, ring, sm = buf(64 * n), buf(32 * (1 + 2 * n)), buf(64)
    flags = bytes(1 if c else 0 for c in choices)
    assert lib().eo_choice_new(pk, n, flags, int(single), C.byref(rng), cts, ring, sm) == 0
    _drawn(rng)
    return raw(cts), raw(ring), (raw(sm) if single else None)


def choice_verify(pk, n, single, cts, ring, sm):
    return lib().eo_choice_verify(pk, n, int(single), bytes(cts), bytes(ring), bytes(sm) if sm is not None else None)


def range_optimal(upper_bound):
    r = Range()
    assert lib().eo_range_optimal(C.byref(r), upper_bound) == 0
    return r


def range_display(r):
    b = C.create_string_buffer(4096)
    n = lib().eo_range_display(C.byref(r), b, C.c_size_t(4096))
    return b.raw[:n].decode()


def range_prove(pk, rng_spec, label, value, rng):
    total = rng_spec.rings_size
    ct, r_out = buf(64), buf(32)
    partial, ring = buf(max(1, 64 * (rng_spec.n_rings - 1))), buf(32 * (1 + total))
    assert lib().eo_range_prove(pk, C.byref(rng_spec), label.encode(), C.c_uint64(value), C.byref(rng), ct, r_out,
                                partial, ring) == 0
    _drawn(rng)
    return raw(ct), raw(partial)[:64 * (rng_spec.n_rings - 1)], raw(ring), raw(r_out)


def range_verify(pk, rng_spec, label, ct, partial, ring):
    return lib().eo_range_verify(pk, C.byref(rng_spec), label.encode(), bytes(ct), bytes(partial), bytes(ring))


def sumsq_prove(pk, cts, values, randomness, sum_ct, sum_randomness, label, rng):
    n = len(values)
    proof = buf(32 * (2 * n + 2))
    assert lib().eo_sumsq_prove(pk, n, b"".join(cts), b"".join(values), b"".join(randomness), sum_ct, sum_randomness,
                                label.encode(), C.byref(rng), proof) == 0
    _drawn(rng)
    return raw(proof)


def sumsq_verify(pk, cts, sum_ct, label, proof):
    return lib().eo_sumsq_verify(pk, len(cts), b"".join(cts), bytes(sum_ct), label.encode(), bytes(proof))


def qv_params(options, credits):
    p = QvParams()
    assert lib().eo_qv_params_new(C.byref(p), options, C.c_uint64(credits)) == 0
    return p


def qv_ballot_size(p):
    return lib().eo_qv_ballot_size(C.byref(p))


def qv_new(pk, p, votes, rng):
    ballot = buf(qv_ballot_size(p))
    v = (C.c_uint64 * len(votes))(*votes)
    assert lib().eo_qv_new(pk, C.byref(p), v, C.byref(rng), ballot) == 0
    _drawn(rng)
    return raw(ballot)


def qv_verify(pk, p, ballot):
    return lib().eo_qv_verify(pk, C.byref(p), bytes(ballot))


def dealer_new(shares, threshold, rng):
    ks = KeySet()
    secrets = buf(32 * shares)
    assert lib().eo_dealer_new(shares, threshold, C.byref(rng), C.byref(ks), secrets) == 0
    s = raw(secrets)
    _drawn(rng)
    return ks, [s[32 * i:32 * i + 32] for i in range(shares)]


def decrypt_share(ks, index, secret, ct, rng):
    share, proof = buf(32), buf(64)
    assert lib().eo_decrypt_share(C.byref(ks), index, secret, ct, C.byref(rng), share, proof) == 0
    _drawn(rng)
    return raw(share), raw(proof)


def verify_share(ks, index, ct, share, proof):
    return lib().eo_verify_share(C.byref(ks), index, bytes(ct), bytes(share), bytes(proof))


def decryption_prove(secret, label, ct, rng):
    dh, proof = buf(32), buf(64)
    assert lib().eo_decryption_prove(bytes(secret), label.encode(), bytes(ct), C.byref(rng), dh, proof) == 0
    _drawn(rng)
    return raw(dh), raw(proof)


def decryption_verify(key, label, ct, dh, proof):
    return lib().eo_decryption_verify(bytes(key), label.encode(), bytes(ct), bytes(dh), bytes(proof))


def lagrange_coefficients(indexes):
    t = len(indexes)
    idx = (C.c_uint32 * t)(*indexes)
    coeffs, scale = buf(32 * t), buf(32)
    lib().eo_lagrange_coefficients(idx, t, coeffs, scale)
    c = raw(coeffs)
    return [c[32 * i:32 * i + 32] for i in range(t)], raw(scale)


def combine_decrypt(indexes, shares, ct):
    t = len(indexes)
    idx = (C.c_uint32 * t)(*indexes)
    out = buf(32)
    rc = lib().eo_combine_decrypt(t, idx, b"".join(shares), bytes(ct), out)
    return rc, raw(out)


class DlogTable:
    def __init__(self, lo, hi):
        self.h = lib().eo_dlog_table_new(lo, hi)

    def get(self, element):
        v = C.c_uint64(0)
        rc = lib().eo_dlog_table_get(self.h, bytes(element), C.byref(v))
        return v.value if rc == 1 else None

    def __del__(self):
        if getattr(self, "h", None):
            lib().eo_dlog_table_free(self.h)
            self.h = None


# ---------------------------------------------------------------- batches (numpy in / out)

def _np():
    import numpy as np
    return np


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def gen_bool_batch(pk, seed, n, first=0, threads=0):
    np = _np()
    cts, proofs = np.empty((n, 64), np.uint8), np.empty((n, 96), np.uint8)
    assert lib().eo_gen_bool_batch(pk, bytes(seed), C.c_size_t(first), C.c_size_t(n), _ptr(cts), _ptr(proofs), threads) == 0
    return cts, proofs


def verify_bool_batch(pk, cts, proofs, threads=0):
    np = _np()
    n = cts.shape[0]
    verdicts = np.empty(n, np.uint8)
    cts, proofs = np.ascontiguousarray(cts), np.ascontiguousarray(proofs)
    assert lib().eo_verify_bool_batch(pk, C.c_size_t(n), _ptr(cts), _ptr(proofs), _ptr(verdicts), threads) == 0
    return verdicts


def gen_choice_batch(pk, options, seed, n, first=0, threads=0):
    np = _np()
    cts = np.empty((n, options, 64), np.uint8)
    rings = np.empty((n, 1 + 2 * options, 32), np.uint8)
    sums = np.empty((n, 64), np.uint8)
    assert lib().eo_gen_choice_batch(pk, options, bytes(seed), C.c_size_t(first), C.c_size_t(n), _ptr(cts), _ptr(rings),
                                     _ptr(sums), threads) == 0
    return cts, rings, sums


def verify_choice_batch(pk, options, single, cts, rings, sums, threads=0):
    np = _np()
    n = cts.shape[0]
    verdicts = np.empty(n, np.uint8)
    tally = np.empty((options, 64), np.uint8)
    cts, rings = np.ascontiguousarray(cts), np.ascontiguousarray(rings)
    sums_p = _ptr(np.ascontiguousarray(sums)) if sums is not None else None
    assert lib().eo_verify_choice_batch(pk, options, int(single), C.c_size_t(n), _ptr(cts), _ptr(rings), sums_p,
                                        _ptr(verdicts), _ptr(tally), threads) == 0
    return verdicts, tally


def gen_range_batch(pk, rng_spec, label, seed, values, first=0, threads=0):
    np = _np()
    values = np.ascontiguousarray(values, dtype=np.uint64)
    n = values.shape[0]
    total, nparts = rng_spec.rings_size, rng_spec.n_rings - 1
    cts = np.empty((n, 64), np.uint8)
    partials = np.empty((n, nparts, 64), np.uint8)
    rings = np.empty((n, 1 + total, 32), np.uint8)
    assert lib().eo_gen_range_batch(pk, C.byref(rng_spec), label.encode(), bytes(seed), C.c_size_t(first), C.c_size_t(n),
                                    _ptr(values), _ptr(cts), _ptr(partials), _ptr(rings), threads) == 0
    return cts, partials, rings


def verify_range_batch(pk, rng_spec, label, cts, partials, rings, threads=0):
    np = _np()
    n = cts.shape[0]
    verdicts = np.empty(n, np.uint8)
    cts, partials, rings = np.ascontiguousarray(cts), np.ascontiguousarray(partials), np.ascontiguousarray(rings)
    assert lib().eo_verify_range_batch(pk, C.byref(rng_spec), label.encode(), C.c_size_t(n), _ptr(cts), _ptr(partials),
                                       _ptr(rings), _ptr(verdicts), threads) == 0
    return verdicts


def gen_qv_batch(pk, p, seed, votes, first=0, threads=0):
    np = _np()
    votes = np.ascontiguousarray(votes, dtype=np.uint64)
    n = votes.shape[0]
    ballots = np.empty((n, qv_ballot_size(p)), np.uint8)
    assert lib().eo_gen_qv_batch(pk, C.byref(p), bytes(seed), C.c_size_t(first), C.c_size_t(n), _ptr(votes),
                                 _ptr(ballots), threads) == 0
    return ballots


def verify_qv_batch(pk, p, ballots, threads=0):
    np = _np()
    n = ballots.shape[0]
    verdicts = np.empty(n, np.uint8)
    tally = np.empty((p.options, 64), np.uint8)
    ballots = np.ascontiguousarray(ballots)
    assert lib().eo_verify_qv_batch(pk, C.byref(p), C.c_size_t(n), _ptr(ballots), _ptr(verdicts), _ptr(tally), threads) == 0
    return verdicts, tally


# ---------------------------------------------------------------- CommitmentEquivalenceProof / ProofOfPossession

def commitment_equiv_prove(pk, value, blinding_base, label, rng):
    ct, commitment, proof, blinding = buf(64), buf(32), buf(128), buf(32)
    assert lib().eo_commitment_equiv_prove(pk, C.c_uint64(value), bytes(blinding_base), label.encode(), C.byref(rng), ct,
                                           commitment, proof, blinding) == 0
    _drawn(rng)
    return raw(ct), raw(commitment), raw(proof), raw(blinding)


def commitment_equiv_verify(pk, blinding_base, label, ct, commitment, proof):
    return lib().eo_commitment_equiv_verify(pk, bytes(blinding_base), label.encode(), bytes(ct), bytes(commitment), bytes(proof))


def gen_ceq_batch(pk, blinding_base, label, seed, values, first=0, threads=0):
    np = _np()
    values = np.ascontiguousarray(values, dtype=np.uint64)
    n = values.shape[0]
    cts, commitments, proofs = np.empty((n, 64), np.uint8), np.empty((n, 32), np.uint8), np.empty((n, 128), np.uint8)
    assert lib().eo_gen_ceq_batch(pk, bytes(blinding_base), label.encode(), bytes(seed), C.c_size_t(first), C.c_size_t(n),
                                  _ptr(values), _ptr(cts), _ptr(commitments), _ptr(proofs), threads) == 0
    return cts, commitments, proofs


def verify_ceq_batch(pk, blinding_base, label, cts, commitments, proofs, threads=0):
    np = _np()
    n = cts.shape[0]
    verdicts = np.empty(n, np.uint8)
    cts, commitments, proofs = np.ascontiguousarray(cts), np.ascontiguousarray(commitments), np.ascontiguousarray(proofs)
    assert lib().eo_verify_ceq_batch(pk, bytes(blinding_base), label.encode(), C.c_size_t(n), _ptr(cts), _ptr(commitments),
                                     _ptr(proofs), _ptr(verdicts), threads) == 0
    return verdicts


def pop_prove(secrets, keys, label, rng):
    k = len(keys)
    proof = buf(32 * (1 + k))
    assert lib().eo_pop_prove(k, b"".join(secrets), b"".join(keys), label.encode(), C.byref(rng), proof) == 0
    _drawn(rng)
    return raw(proof)


def pop_verify(keys, label, proof):
    return lib().eo_pop_verify(len(keys), b"".join(keys), label.encode(), bytes(proof))


def gen_pop_batch(k, label, seed, n, first=0, threads=0):
    np = _np()
    keys, proofs = np.empty((n, k, 32), np.uint8), np.empty((n, 1 + k, 32), np.uint8)
    assert lib().eo_gen_pop_batch(k, label.encode(), bytes(seed), C.c_size_t(first), C.c_size_t(n), _ptr(keys), _ptr(proofs), threads) == 0
    return keys, proofs


def verify_pop_batch(label, keys, proofs, threads=0):
    np = _np()
    n, k = keys.shape[0], keys.shape[1]
    verdicts = np.empty(n, np.uint8)
    keys, proofs = np.ascontiguousarray(keys), np.ascontiguousarray(proofs)
    assert lib().eo_verify_pop_batch(k, label.encode(), C.c_size_t(n), _ptr(keys), _ptr(proofs), _ptr(verdicts), threads) == 0
    return verdicts


def keyset_from_participants(shares, threshold, keys):
    """-> (verdict, shared_key or None)"""
    out = buf(32)
    rc = lib().eo_keyset_from_participants(shares, threshold, b"".join(bytes(k) for k in keys), out)
    return rc, (raw(out) if rc == 0 else None)


def hw_threads():
    return lib().eo_hw_threads()
