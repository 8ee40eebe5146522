"""Edge values of the decryption side, shared by the CPU harness tests (test_hostsim_edges.py) and the `-m gpu` tests
(test_gpu_edges.py).  Random inputs almost never reach the values where integer code goes wrong, so these are chosen by hand:
discrete-log tables whose ranges do not start at 0 or end next to 2^64, u64 plaintexts at the ends of their range, and secret
keys and nonces whose recodings sit on the digit limits of the decryption kernels (sc_recode4, sc_wide_digit, sc_half).
Outputs are compared with the oracle, or -- for proofs on chosen nonces, which the oracle's ChaCha20-driven prover cannot
take -- checked by algebra with the oracle's point operations."""
import ctypes as C
import functools
import random

import numpy as np

import decrypt_common as D
import oracle as O
import parity_common as PC
import workloads as W

L = W.L
U64 = 1 << 64
USED = (0, 2, 4)                 # participants of the 3-of-5 key set whose shares are combined


def sc(x):
    return PC.sc(x)


def rows(blobs, width):
    return np.frombuffer(b"".join(blobs), np.uint8).reshape(len(blobs), width).copy()


def both_modes(e, fn):
    """fn() in the default and in the constant-time prover mode; the context is left in the default mode."""
    out = []
    for ct in (False, True):
        e.set_prover_mode(ct)
        try:
            out.append(fn())
        finally:
            e.set_prover_mode(False)
    return out


# ---------------------------------------------------------------- DiscreteLogTable ranges

TABLE_RANGES = [
    (5, 5),                                                          # empty
    (0, 1), (0, 31), (0, 32), (0, 33),                               # around the 32 values one build thread inserts
    (1, 8), (1000, 1015), (2**40, 2**40 + 1023),                     # n = 7, 15, 1023: 2n + 2 is the capacity (fullest)
    (37, 1037),
    (2**32 - 40, 2**32 + 40), (2**63 - 50, 2**63 + 50),
    (U64 - 2, U64 - 1), (U64 - 33, U64 - 1), (U64 - 100, U64 - 1),   # top slice of 32 ends past 2^64 / at 2^64 - 1
]


def table_values(lo, hi):
    """Every value of lo..hi, the outside neighbours that fit in u64, and 0 (the identity: found with value 0 whatever the
    range, encryption.rs:287-297)."""
    return list(range(lo, hi)) + ([lo - 1] if lo > 0 else []) + ([hi] if hi < U64 else []) + [0]


def expected_lookup(lo, hi, v):
    return (1, v) if lo <= v < hi else (1, 0) if v == 0 else (0, 0)


class TableCorpus:
    """The values of every range in one batch (`spans[k]` slices range k), encrypted by the oracle under the receiver key
    (cts_pk) and under the key set's shared key (cts_ks), with the oracle's decryption of cts_pk and the oracle's
    DiscreteLogTable::get on it."""

    def __init__(self, ranges):
        sk, pk = W.receiver()
        ks, _, _ = D.keyset()
        rng = O.rng_from_seed(bytes([0x5e] * 32))
        self.ranges, self.spans, self.values = list(ranges), [], []
        for lo, hi in self.ranges:
            vs = table_values(lo, hi)
            self.spans.append(slice(len(self.values), len(self.values) + len(vs)))
            self.values += vs
        self.cts_pk = rows([O.encrypt(pk, v, rng) for v in self.values], 64)
        self.cts_ks = rows([O.encrypt(bytes(ks.shared_key), v, rng) for v in self.values], 64)
        self.elements = [O.decrypt_to_element(sk, bytes(c)) for c in self.cts_pk]
        self.lookups = []
        for (lo, hi), sp in zip(self.ranges, self.spans):
            otable = O.DlogTable(lo, hi)
            for v, el in zip(self.values[sp], self.elements[sp]):
                ov = otable.get(el)
                got = (0, 0) if ov is None else (1, ov)
                assert got == expected_lookup(lo, hi, v), (hex(lo), hex(hi), hex(v), got)   # the oracle pins the semantics
                self.lookups.append(got)


@functools.lru_cache(maxsize=None)
def table_corpus():
    return TableCorpus(TABLE_RANGES)


def library_shares(e, corpus):
    """The key set's shares of cts_ks made by the library (decrypt_share, USED participants); the oracle combines them to
    the element the receiver key decrypts cts_pk to, which is [v]G for both."""
    ks, eks, secrets = D.keyset()
    n = len(corpus.values)
    shares = np.zeros((n, len(USED), 32), np.uint8)
    for j, idx in enumerate(USED):
        sh, _, ok = e.decrypt_share(eks, idx, secrets[idx], corpus.cts_ks, seed=D.SEED)
        assert ok.all()
        shares[:, j] = sh
    for i in range(n):
        rc, el = O.combine_decrypt(list(USED), [bytes(shares[i, j]) for j in range(len(USED))], bytes(corpus.cts_ks[i]))
        assert rc == 0 and el == corpus.elements[i], i
    return shares


def _mismatches(corpus, k, found, vals):
    """found / values of range k against the oracle, item for item, with the values read as exact u64: [] or a description."""
    lo, hi = corpus.ranges[k]
    sp = corpus.spans[k]
    assert vals.dtype == np.uint64
    got = list(zip(found.tolist(), [int(v) for v in vals]))
    want = corpus.lookups[sp]
    bad = [(hex(v), g, w) for v, g, w in zip(corpus.values[sp], got, want) if g != w]
    return [f"[{lo:#x}, {hi:#x}): {len(bad)} of {len(want)} lookups differ from the oracle, e.g. {bad[:3]}"] if bad else []


def _with_table(e, lo, hi, fn):
    table = e.dlog_table(lo, hi)
    try:
        return fn(table)
    finally:
        table.close()


def check_tables_decrypt(e, corpus):
    """eg_decrypt_batch with each table: elements as the oracle decrypts them, found / values as the oracle's table."""
    sk, _ = W.receiver()
    bad = []
    for k, (lo, hi) in enumerate(corpus.ranges):
        sp = corpus.spans[k]
        el, vals, found = _with_table(e, lo, hi, lambda t: e.decrypt(sk, corpus.cts_pk[sp], t))
        assert [bytes(x) for x in el] == corpus.elements[sp]
        bad += _mismatches(corpus, k, found, vals)
    assert not bad, "\n".join(bad)


def check_tables_combine(e, corpus, shares):
    """eg_combine_decrypt_batch (host pointers) with each table."""
    bad = []
    for k, (lo, hi) in enumerate(corpus.ranges):
        sp = corpus.spans[k]
        vals, found = _with_table(e, lo, hi, lambda t: e.combine_decrypt(list(USED), corpus.cts_ks[sp], shares[sp], t))
        bad += _mismatches(corpus, k, found, vals)
    assert not bad, "\n".join(bad)


def combine_decrypt_dev(e, dev, cts, shares, table):
    """eg_combine_decrypt_batch_dev through `dev` (up / empty / ptr / down: buffers in the context's device memory); the
    values come back as int64 and are read as uint64."""
    n = cts.shape[0]
    idx = (C.c_uint32 * len(USED))(*USED)
    d_c, d_s = dev.up(cts), dev.up(shares)
    d_vals, d_found = dev.empty(n, "int64"), dev.empty(n, "uint8")
    e._check(e.lib.eg_combine_decrypt_batch_dev(e.h, len(USED), idx, n, shares.shape[1], dev.ptr(d_c), dev.ptr(d_s), table.h,
                                                dev.ptr(d_vals), dev.ptr(d_found)))
    return dev.down(d_vals).view(np.uint64), dev.down(d_found)


def check_tables_combine_dev(e, corpus, shares, dev):
    bad = []
    for k, (lo, hi) in enumerate(corpus.ranges):
        sp = corpus.spans[k]
        vals, found = _with_table(e, lo, hi, lambda t: combine_decrypt_dev(e, dev, corpus.cts_ks[sp], shares[sp], t))
        bad += _mismatches(corpus, k, found, vals)
    assert not bad, "\n".join(bad)


def check_table_argument_errors(e, corpus):
    """hi < lo and hi - lo = 2^28 + 1 are EG_ERR_INVALID_ARG; the next call on the same context is unaffected."""
    from elastic_elgamal_b200 import EngineError, _ffi
    sk, _ = W.receiver()
    k = corpus.ranges.index((U64 - 100, U64 - 1))
    sp = corpus.spans[k]
    for lo, hi in ((10, 9), (U64 - 1, 0), (0, 2**28 + 1), (U64 - 2**28 - 2, U64 - 1)):
        try:
            e.dlog_table(lo, hi).close()
            raise AssertionError(f"table [{lo:#x}, {hi:#x}) accepted")
        except EngineError as err:
            assert err.status == _ffi.ERR_INVALID_ARG
        _, vals, found = _with_table(e, U64 - 100, U64 - 1, lambda t: e.decrypt(sk, corpus.cts_pk[sp], t))
        assert not _mismatches(corpus, k, found, vals)


def check_top_table_2_20(e, dev, samples=4096):
    """A 2^20-value table ending at 2^64 - 1 (32 768 build threads, the top slices next to the wrap), checked on the known
    plaintexts of `samples` values drawn from it, its lowest value and its top 64, its outside neighbours and 0; through
    eg_decrypt_batch and both forms of eg_combine_decrypt_batch."""
    lo, hi = U64 - (1 << 20) - 1, U64 - 1
    values = sorted(random.Random(20).sample(range(lo, hi - 64), samples)) + [lo] + list(range(hi - 64, hi)) + [lo - 1, hi, 0]
    want = [expected_lookup(lo, hi, v) for v in values]
    sk, pk = W.receiver()
    ks, eks, secrets = D.keyset()
    rng = O.rng_from_seed(bytes([0x20] * 32))
    cts_pk = rows([O.encrypt(pk, v, rng) for v in values], 64)
    cts_ks = rows([O.encrypt(bytes(ks.shared_key), v, rng) for v in values], 64)
    shares = np.zeros((len(values), len(USED), 32), np.uint8)
    for j, idx in enumerate(USED):
        shares[:, j] = e.decrypt_share(eks, idx, secrets[idx], cts_ks, seed=D.SEED)[0]
    table = e.dlog_table(lo, hi)
    try:
        _, vals, found = e.decrypt(sk, cts_pk, table)
        outs = [(vals, found), e.combine_decrypt(list(USED), cts_ks, shares, table), combine_decrypt_dev(e, dev, cts_ks, shares, table)]
    finally:
        table.close()
    for vals, found in outs:
        assert vals.dtype == np.uint64
        got = list(zip(found.tolist(), [int(v) for v in vals]))
        bad = [(hex(v), g, w) for v, g, w in zip(values, got, want) if g != w]
        assert not bad, f"{len(bad)} of {len(values)} lookups wrong, e.g. {bad[:4]}"


# ---------------------------------------------------------------- u64 plaintexts

U64_PLAINTEXTS = [0, 1, 2**32 - 1, 2**32, 2**63 - 1, 2**63, U64 - 2, U64 - 1]
FIRST_ITEM = 11                  # item i draws from per-item stream FIRST_ITEM + i


def check_u64_plaintexts(e):
    """encrypt with caller blocks and with seed= equals the oracle on the same per-item streams; every ciphertext decrypts to
    [v]G and round-trips through each table of TABLE_RANGES (2^64 - 1 lies above every u64 range)."""
    inside = {v for v in U64_PLAINTEXTS for lo, hi in TABLE_RANGES if lo <= v < hi}
    assert inside == set(U64_PLAINTEXTS) - {U64 - 1}
    sk, pk = W.receiver()
    e.set_receiver(pk)
    n = len(U64_PLAINTEXTS)
    values = np.array(U64_PLAINTEXTS, np.uint64)
    expected = [O.encrypt(pk, v, D.item_rng(FIRST_ITEM + i)) for i, v in enumerate(U64_PLAINTEXTS)]
    cts = e.encrypt(values, D.wide(FIRST_ITEM, n))
    assert [bytes(c) for c in cts] == expected
    assert [bytes(c) for c in e.encrypt(values, seed=D.SEED, counter_base=FIRST_ITEM << 20)] == expected
    mults = [O.point_mul_generator(sc(v)) for v in U64_PLAINTEXTS]
    assert [O.decrypt_to_element(sk, c) for c in expected] == mults
    for lo, hi in TABLE_RANGES:
        el, vals, found = _with_table(e, lo, hi, lambda t: e.decrypt(sk, cts, t))
        assert [bytes(x) for x in el] == mults and vals.dtype == np.uint64
        assert list(zip(found.tolist(), [int(v) for v in vals])) == [expected_lookup(lo, hi, v) for v in U64_PLAINTEXTS], (lo, hi)


# ---------------------------------------------------------------- secret keys and nonces

NIBBLES_8 = int("8" * 64, 16)


def recode4(a):
    """ge.cuh sc_recode4 + sc_digit4: 64 signed 4-bit digits, low to high, digit i = nibble i of (a + 0x88..8) - 8."""
    r = (a + NIBBLES_8) % (1 << 256)
    return [((r >> (4 * i)) & 15) - 8 for i in range(64)]


def wide_digits(a, bits):
    """ge.cuh sc_wide_digit_b<bits>: signed `bits`-bit digits in [-2^(bits-1), 2^(bits-1)) with a running carry."""
    out, carry = [], 0
    for i in range((254 + bits - 1) // bits):
        v = ((a >> (bits * i)) & ((1 << bits) - 1)) + carry
        carry = 1 if v >= 1 << (bits - 1) else 0
        out.append(v - (carry << bits))
    return out


def sc_half(x):
    """ge.cuh sc_half: x / 2 mod l as (x + (l if x is odd)) / 2."""
    return (x + (L if x & 1 else 0)) >> 1


RECODE4_PATTERNS = {             # all 64 digits, low to high; the top digit keeps the scalar in [0, l)
    "all -8": [-8] * 63 + [1],
    "all 7": [7] * 63 + [0],
    "-8 / 7 alternating": [-8, 7] * 31 + [-8, 1],
    "7 / -8 alternating": [7, -8] * 31 + [7, 0],
    "zero below the top digit": [0] * 63 + [1],
}


def pattern_scalars():
    return [sum(d << (4 * i) for i, d in enumerate(digits)) for digits in RECODE4_PATTERNS.values()]


# 1, 2, l - 1, l - 2; the odd / even boundary of sc_half; the top bit of a canonical scalar
EDGE_SCALARS = [1, 2, L - 1, L - 2, (L - 1) // 2, (L + 1) // 2, 2**252 - 1, 2**252]
WIDE_BITS = (16, 24)             # EG_WIDE_BITS of the CPU harness and of the device build


def _unique(xs):
    return list(dict.fromkeys(xs))


def edge_keys():
    """The edge scalars, the recode4 patterns p (eg_decrypt_batch recodes the key s itself) and 2p mod l (the proofs recode
    s / 2)."""
    pats = pattern_scalars()
    return _unique(EDGE_SCALARS + pats + [2 * p % L for p in pats])


def nonce_blocks():
    """64-byte blocks reduced to the nonce x: a target in the low 32 bytes and zeros above (x = target), the same targets as
    the keys and x = 0 ([x]G and [x]R are the identity in ge_double_compress_n<3>), l + target, and all-0xff."""
    blocks = [t.to_bytes(64, "little") for t in _unique([0] + edge_keys())]
    return blocks + [(L + t).to_bytes(64, "little") for t in (0, 1, L - 1)] + [b"\xff" * 64]


def wide_nonce_blocks():
    """Nonces x = 2w mod l, so that the kernels' [x/2]G walks the wide fixed-base digits of every w of
    parity_common.wide_window_edge_scalars() (16-, 20- and 24-bit window boundaries)."""
    return [(2 * int.from_bytes(w, "little") % L).to_bytes(64, "little") for w in PC.wide_window_edge_scalars()]


def nonce(block):
    x = int.from_bytes(block, "little") % L
    assert O.scalar_reduce_wide(block) == sc(x)
    return x


def check_recodings_hit_their_edges():
    """The key and nonce lists above really produce the digit patterns they are meant to: each recode4 pattern for the key
    itself (plain decryption) and for its half (the proofs' [s/2]R, [x/2]R and constant-time [x/2]G), and the extreme wide
    digits, with a carry into the top window, for the [x/2]G walk at the device's and the CPU harness's window width."""
    for digits, p in zip(RECODE4_PATTERNS.values(), pattern_scalars()):
        assert 0 < p < L and recode4(p) == digits and sum(d << (4 * i) for i, d in enumerate(recode4(p))) == p
    for x in (1, L - 1, 12345, 2**252):
        assert sc_half(x) == x * pow(2, -1, L) % L
    keys = edge_keys()
    nonces = [nonce(b) for b in nonce_blocks()]
    for name, digits in RECODE4_PATTERNS.items():
        assert any(recode4(s) == digits for s in keys), name
        assert any(recode4(sc_half(s)) == digits for s in keys), name
        assert any(recode4(sc_half(x)) == digits for x in nonces), name
    assert 0 in nonces and {L - 1, (L - 1) // 2, (L + 1) // 2} <= set(keys)
    halves = [sc_half(nonce(b)) for b in wide_nonce_blocks()]
    for bits in WIDE_BITS:
        top = 1 << (bits - 1)
        digits = [wide_digits(h, bits) for h in halves]
        for h, ds in zip(halves, digits):
            assert sum(d << (bits * i) for i, d in enumerate(ds)) == h and all(-top <= d < top for d in ds)
        below_top = {d for ds in digits for d in ds[:-1]}
        assert {-top, top - 1, -1, 0, 1} <= below_top, bits
        assert any(ds[-1] != h >> (bits * (len(ds) - 1)) for h, ds in zip(halves, digits)), bits   # a carry reaches the top


def edge_points():
    """Ciphertext R values: G, -G, [2]G, the identity and random points."""
    rnd = random.Random(31)
    return ([W.G_ENC, O.point_mul_generator(sc(L - 1)), O.point_mul_generator(sc(2)), bytes(32)]
            + [O.point_mul_generator(sc(rnd.randrange(L))) for _ in range(4)])


def plain_ciphertexts(s, n=40):
    """n >= 33 ciphertexts R | B over edge_points(); B = [s]R (the element is the identity) and B = identity once each."""
    rnd = random.Random(s % 1000003)
    Rs = edge_points()
    out = []
    for i in range(n):
        R = Rs[i % len(Rs)]
        B = O.point_mul(sc(s), R) if i == 4 else bytes(32) if i == 5 else O.point_mul_generator(sc(rnd.randrange(L)))
        out.append(R + B)
    return rows(out, 64)


def check_edge_keys_decrypt(e):
    """eg_decrypt_batch with every edge key and key 0 equals the oracle's decrypt_to_element, byte for byte, in both modes."""
    for s in [0] + edge_keys():
        cts = plain_ciphertexts(s)
        expected = [O.decrypt_to_element(sc(s), bytes(c)) for c in cts]
        for el, vals, found in both_modes(e, lambda: e.decrypt(sc(s), cts)):
            assert found.tolist() == [1] * len(cts)
            bad = [i for i in range(len(cts)) if bytes(el[i]) != expected[i]]
            assert not bad, f"key {s:#x}: items {bad} differ from the oracle"
        assert expected[4] == bytes(32)


def proof_items(blocks, n=40):
    """(nonce block, R) per item: x = 0 against every R, then `blocks` over the R values, then random nonces up to n."""
    Rs = edge_points()
    items = [(bytes(64), R) for R in Rs] + [(b, Rs[i % len(Rs)]) for i, b in enumerate(blocks)]
    rnd = random.Random(len(blocks))
    while len(items) < n:
        items.append((rnd.randbytes(64), Rs[len(items) % len(Rs)]))
    return items


def check_proofs(e, s, items):
    """eg_prove_decryption_batch with key s and the items' chosen nonces, in both modes (identical bytes).  The oracle cannot
    take a chosen nonce, so the proof is checked by algebra: dh = [s]R, the oracle's verifier accepts it, and
    [resp]G - [c][s]G = [x]G -- with c a function of the transcript, these fix c and resp exactly."""
    cts = rows([R + W.G_ENC for _, R in items], 64)
    wide = rows([b for b, _ in items], 64)
    (dh, pr, ok), (dh_ct, pr_ct, ok_ct) = both_modes(e, lambda: e.prove_decryption(D.LABEL, sc(s), cts, wide))
    assert ok.all() and ok_ct.all() and (dh_ct == dh).all() and (pr_ct == pr).all(), f"key {s:#x}: the modes differ"
    pk = O.point_mul_generator(sc(s))
    for i, (block, R) in enumerate(items):
        d, p = bytes(dh[i]), bytes(pr[i])
        assert d == O.point_mul(sc(s), R), (hex(s), i)
        assert O.decryption_verify(pk, D.LABEL, bytes(cts[i]), d, p) == O.OK, (hex(s), i)
        rG_minus_csG = O.point_sub(O.point_mul_generator(p[32:]), O.point_mul(p[:32], pk))
        assert rG_minus_csG == O.point_mul_generator(sc(nonce(block))), (hex(s), i)


def check_edge_keys_and_nonces_prove(e):
    items = proof_items(nonce_blocks())
    assert len(items) >= 33
    for s in edge_keys():
        check_proofs(e, s, items)


def check_wide_window_nonces_prove(e):
    items = proof_items(wide_nonce_blocks())
    for s in (1, pattern_scalars()[0], 2 * pattern_scalars()[0] % L, random.Random(7).randrange(1, L)):
        check_proofs(e, s, items)
