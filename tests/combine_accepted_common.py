"""eg_combine_decrypt_accepted_batch(_dev) (threshold decryption from the shares a tallier accepted), shared by the CPU
harness tests (test_hostsim_combine_accepted.py) and the `-m gpu` tests (test_gpu_combine_accepted.py).

The expected result of a tally is the reference tallier's: the first t columns whose verdict is EG_V_OK (0), in column order,
go to the oracle's combine_decrypt, whose element the oracle's DiscreteLogTable looks up; fewer than t accepted columns
give found 3 (combine_shares returns None).

Most batches are synthetic threshold tallies, which admit any participant indexes (also 2^31 and past): with a polynomial
f of degree t - 1 and the x coordinate index + 1 of sharing/mod.rs, the ciphertext of v is ([r]G, [v + r f(0)]G) and the
share of participant x is [r f(x + 1)]G.  The end-to-end check uses the dealer, decrypt_share and verify_shares instead."""
import ctypes as C
import functools
import random
import time

import numpy as np

import decrypt_common as D
import edge_common as EC
import oracle as O
import workloads as W

L = W.L
BAD = b"\xff" * 32                      # does not decode (non-canonical)
REJECT = (1, 2, 7)                      # verdict bytes other than EG_V_OK
TABLE = (0, 1024)


def element(k):
    return O.point_mul_generator(EC.sc(k % L))


class Batch:
    """n synthetic tallies of `threshold`-of-many sharing with one column per index: cts (n, 64), shares (n, S, 32) and
    the plaintexts (n,)."""

    def __init__(self, threshold, indexes, values, seed):
        rnd = random.Random(seed)
        self.t, self.indexes, self.values = threshold, list(indexes), list(values)
        n, S = len(values), len(indexes)
        self.cts = np.zeros((n, 64), np.uint8)
        self.shares = np.zeros((n, S, 32), np.uint8)
        for i, v in enumerate(values):
            f = [rnd.randrange(1, L) for _ in range(threshold)]
            r = rnd.randrange(1, L)
            self.cts[i] = np.frombuffer(element(r) + element(v + r * f[0]), np.uint8)
            for j, x in enumerate(indexes):
                fx = sum(c * pow(x + 1, d, L) for d, c in enumerate(f)) % L
                self.shares[i, j] = np.frombuffer(element(r * fx), np.uint8)


@functools.lru_cache(maxsize=None)
def batch(threshold, indexes, n, seed=1, values=None):
    rnd = random.Random(seed * 7919 + n)
    if values is None:
        values = tuple(rnd.choice([0, 1, 17, 1023, 1024, 5000, rnd.randrange(1024)]) for _ in range(n))
    return Batch(threshold, indexes, values, seed)


def oracle_lookup(lo, hi):
    table = O.DlogTable(lo, hi)
    return table.get


def known_lookup(lo, hi, values):
    """DiscreteLogTable::get on elements of known plaintexts (for tables too large for the oracle to build)."""
    known = {element(v): v for v in values}
    return lambda el: 0 if el == bytes(32) else (known[el] if el in known and lo <= known[el] < hi else None)


def expected(t, indexes, cts, shares, verdicts, lookup):
    """(found, values) of the reference tallier: combine the first t accepted columns, decrypt, look up."""
    n, S = shares.shape[0], shares.shape[1]
    found, vals = np.zeros(n, np.uint8), np.zeros(n, np.uint64)
    for i in range(n):
        cols = [j for j in range(S) if verdicts[i, j] == 0][:t]
        if len(cols) < t:
            found[i] = 3
            continue
        rc, el = O.combine_decrypt([indexes[j] for j in cols], [bytes(shares[i, j]) for j in cols], bytes(cts[i]))
        if rc != 0:
            found[i] = 2
            continue
        v = lookup(el)
        if v is not None:
            found[i], vals[i] = 1, v
    return found, vals


def random_verdicts(n, S, rnd, p_reject):
    return np.array([[rnd.choice(REJECT) if rnd.random() < p_reject else 0 for _ in range(S)] for _ in range(n)], np.uint8)


def with_table(e, lo, hi, fn, m=None):
    t = e.dlog_table(lo, hi, m)
    try:
        return fn(t)
    finally:
        t.close()


def check(e, b, verdicts, lookup=None, table=TABLE, m=None, what=""):
    lookup = lookup or oracle_lookup(*table)
    vals, found = with_table(e, table[0], table[1], lambda tb: e.combine_decrypt_accepted(b.t, b.indexes, b.cts, b.shares, verdicts, tb), m)
    want_f, want_v = expected(b.t, b.indexes, b.cts, b.shares, verdicts, lookup)
    bad = [i for i in range(len(found)) if (found[i], vals[i]) != (want_f[i], want_v[i])]
    assert not bad, f"{what}: {len(bad)} tallies differ, e.g. " + str([(i, found[i], int(vals[i]), want_f[i], int(want_v[i])) for i in bad[:4]])
    return vals, found


# ---------------------------------------------------------------- 1. every verdict pattern of 3-of-5

def check_patterns(e, copies=3):
    indexes = (0, 1, 2, 3, 4)
    b = batch(3, indexes, 32 * copies, seed=2)
    rnd = random.Random(5)
    verdicts = np.array([[0 if (p >> j) & 1 else rnd.choice(REJECT) for j in range(5)] for p in range(32) for _ in range(copies)],
                        np.uint8)
    vals, found = check(e, b, verdicts, what="3-of-5 patterns")
    few = np.array([bin(p).count("1") < 3 for p in range(32) for _ in range(copies)])
    assert (found[few] == 3).all() and not vals[few].any() and (found[~few] != 3).all()


# ---------------------------------------------------------------- 2. equal to the fixed subset when every share is accepted

def check_equivalence(e, t=3, indexes=(0, 1, 2, 3, 4), n=40):
    b = batch(t, tuple(indexes), n, seed=3)
    v = np.zeros((n, len(indexes)), np.uint8)

    def run(tb):
        return e.combine_decrypt_accepted(t, b.indexes, b.cts, b.shares, v, tb), e.combine_decrypt(b.indexes[:t], b.cts, b.shares, tb)
    (va, fa), (vb, fb) = with_table(e, *TABLE, run)
    assert (fa == fb).all() and (va == vb).all(), "all accepted differs from eg_combine_decrypt_batch(indexes[:t], share_stride = n_shares)"
    assert (fa == 1).any()


# ---------------------------------------------------------------- 3. shapes

def index_sets(S, rnd):
    perm = list(range(64))
    rnd.shuffle(perm)
    big = [2**31, 2**32 - 1, 2**31 + 1, 2**32 - 2, 0, 2**20, 12345] + [2**31 + 7 * k for k in range(2, 64)]
    return {"ascending": tuple(range(S)), "reversed": tuple(range(S))[::-1], "permuted": tuple(perm[:S]),
            "large": tuple(big[:S])}


def check_shape(e, t, S, n=12, p_reject=0.3):
    rnd = random.Random(t * 100 + S)
    for name, idx in index_sets(S, rnd).items():
        b = batch(t, idx, n, seed=t * 1000 + S)
        v = random_verdicts(n, S, rnd, p_reject if S > t else 0.1)
        v[0] = 0                                            # one tally of each: the first t columns
        check(e, b, v, what=f"t={t} n_shares={S} {name}")


def check_random_masks_64(e, n=24):
    rnd = random.Random(64)
    idx = tuple(index_sets(64, rnd)["permuted"])
    b = batch(16, idx, n, seed=64)
    for p in (0.1, 0.5, 0.75):
        check(e, b, random_verdicts(n, 64, rnd, p), what=f"16-of-64, reject probability {p}")


# ---------------------------------------------------------------- 4. fast path and other selections in one warp

def check_mixed_warps(e, runs=4):
    indexes = (4, 0, 3, 1, 2)
    n = 32 * runs
    b = batch(3, indexes, n, seed=6)
    rnd = random.Random(7)
    v = np.zeros((n, 5), np.uint8)
    for i in range(n):
        r, k = divmod(i, 32)
        if (r == 0 and k % 2) or (r == 1 and k % 3 == 0) or r == 3:    # run 2 stays all default
            v[i, rnd.randrange(3)] = rnd.choice(REJECT)
            if r == 3 and k % 4 == 0:
                v[i, 3] = 1
    check(e, b, v, what="mixed selections within warps")


# ---------------------------------------------------------------- 5. inputs that must not be read, and found 2 / 3

def check_garbage(e, n=40):
    indexes = (0, 1, 2, 3, 4)
    b = batch(3, indexes, n, seed=8)
    rnd = random.Random(9)
    v = random_verdicts(n, 5, rnd, 0.3)
    v[:4] = 0
    want_v, want_f = check(e, b, v, what="before garbage")
    g = Batch.__new__(Batch)
    g.t, g.indexes, g.values, g.cts, g.shares = b.t, b.indexes, b.values, b.cts.copy(), b.shares.copy()
    for i in range(n):
        acc = [j for j in range(5) if v[i, j] == 0]
        for j in range(5):
            if v[i, j] != 0 or j in acc[3:]:
                g.shares[i, j] = np.frombuffer(BAD, np.uint8)
    vals, found = with_table(e, *TABLE, lambda tb: e.combine_decrypt_accepted(3, indexes, g.cts, g.shares, v, tb))
    assert (found == want_f).all() and (vals == want_v).all(), "undecodable shares that are not selected changed the result"
    # a selected undecodable share, an undecodable ciphertext: 2; fewer than t accepted wins over both
    g.shares[0, 1] = np.frombuffer(BAD, np.uint8)
    g.cts[1, 32:] = np.frombuffer(BAD, np.uint8)
    g.cts[2, :32] = np.frombuffer(BAD, np.uint8)
    v2 = v.copy()
    v2[2, :3] = 1
    v2[2, 3:] = 0
    g.cts[3] = np.frombuffer(BAD + BAD, np.uint8)
    v2[3] = 7
    vals, found = check(e, g, v2, what="found 2 / 3")
    assert found[:4].tolist() == [2, 2, 3, 3] and not vals[:4].any()


# ---------------------------------------------------------------- 6. tables

def check_bsgs(e, lo, hi, m, values):
    """A baby-step giant-step table of m baby steps over [lo, hi) on known plaintexts (some outside the range)."""
    b = batch(3, (0, 1, 2, 3, 4), len(values), seed=10, values=tuple(values))
    v = random_verdicts(len(values), 5, random.Random(11), 0.25)
    check(e, b, v, lookup=known_lookup(lo, hi, values), table=(lo, hi), m=m, what=f"BSGS [{lo:#x}, {hi:#x}) m={m}")


def check_no_walk(e, m, n):
    """Every tally has fewer than t accepted shares and a B that a table of m baby steps and 2^32 giant steps does not hold
    at giant step 0: a walk would take hours, found 3 must come back at once."""
    hi = m * 2**32
    rnd = random.Random(12)
    b = batch(3, (0, 1, 2, 3, 4), n, seed=12, values=tuple(rnd.randrange(m, hi) for _ in range(n)))
    v = random_verdicts(n, 5, rnd, 0.5)
    for i in range(n):
        v[i, [j for j in range(5) if v[i, j] == 0][2:]] = 2
    t0 = time.perf_counter()
    vals, found = with_table(e, 0, hi, lambda tb: e.combine_decrypt_accepted(3, b.indexes, b.cts, b.shares, v, tb), m)
    took = time.perf_counter() - t0
    assert (found == 3).all() and not vals.any()
    return took


# ---------------------------------------------------------------- 7. chunks, device pointers, multi-device contexts

def mixed_batch(n=40, seed=13):
    b = batch(3, (2, 0, 4, 1, 3), n, seed=seed)
    v = random_verdicts(n, 5, random.Random(seed), 0.3)
    return b, v


def check_chunks(e, n=40):
    b, v = mixed_batch(n)
    want = expected(b.t, b.indexes, b.cts, b.shares, v, oracle_lookup(*TABLE))
    try:
        for chunk in (7, 0, 16):
            e.set_chunk_items(chunk)
            vals, found = with_table(e, *TABLE, lambda tb: e.combine_decrypt_accepted(3, b.indexes, b.cts, b.shares, v, tb))
            assert (found == want[0]).all() and (vals == want[1]).all(), f"chunk size {chunk}"
    finally:
        e.set_chunk_items(0)


def run_dev(e, dev, b, v, tb):
    n = b.cts.shape[0]
    d_c, d_s, d_v = dev.up(b.cts), dev.up(b.shares), dev.up(v)
    d_vals, d_found = dev.empty(n, "int64"), dev.empty(n, "uint8")
    e.combine_decrypt_accepted_dev(b.t, b.indexes, n, dev.ptr(d_c), dev.ptr(d_s), dev.ptr(d_v), tb, dev.ptr(d_vals), dev.ptr(d_found))
    return dev.down(d_vals).view(np.uint64), dev.down(d_found)


def check_dev(e, dev, n=40, chunk=0):
    b, v = mixed_batch(n)
    e.set_chunk_items(chunk)
    try:
        def run(tb):
            return e.combine_decrypt_accepted(3, b.indexes, b.cts, b.shares, v, tb), run_dev(e, dev, b, v, tb)
        (hv, hf), (dv, df) = with_table(e, *TABLE, run)
    finally:
        e.set_chunk_items(0)
    want = expected(b.t, b.indexes, b.cts, b.shares, v, oracle_lookup(*TABLE))
    assert (hf == want[0]).all() and (hv == want[1]).all()
    assert (df == hf).all() and (dv == hv).all(), "host and _dev forms differ"


def check_multi(m, e, n=40):
    b, v = mixed_batch(n, seed=14)
    a = with_table(m, *TABLE, lambda tb: m.combine_decrypt_accepted(3, b.indexes, b.cts, b.shares, v, tb))
    s = with_table(e, *TABLE, lambda tb: e.combine_decrypt_accepted(3, b.indexes, b.cts, b.shares, v, tb))
    want = expected(b.t, b.indexes, b.cts, b.shares, v, oracle_lookup(*TABLE))
    assert (a[1] == want[0]).all() and (a[0] == want[1]).all() and (a[1] == s[1]).all() and (a[0] == s[0]).all()


# ---------------------------------------------------------------- 8. end to end

def check_end_to_end(e, dev, n=60):
    """Encrypt, decrypt_share for all 5 participants of a 3-of-5 key set, tamper some proofs and some shares, verify_shares
    (host and _dev), then combine the accepted shares: every tally with at least 3 valid shares decrypts to its plaintext."""
    ks, eks, secrets = D.keyset()
    rnd = random.Random(15)
    values = np.array([rnd.randrange(1000) for _ in range(n)], np.uint64)
    e.set_receiver(bytes(ks.shared_key))
    cts = e.encrypt(values, seed=bytes([0x3c] * 32))
    indexes = [0, 1, 2, 3, 4]
    shares, proofs = np.zeros((n, 5, 32), np.uint8), np.zeros((n, 5, 64), np.uint8)
    for j in indexes:
        sh, pr, ok = e.decrypt_share(eks, j, secrets[j], cts, seed=D.SEED)
        assert ok.all()
        shares[:, j], proofs[:, j] = sh, pr
    bad = np.zeros((n, 5), bool)
    for i in range(n):
        for j in rnd.sample(range(5), rnd.choice([0, 0, 1, 2, 3])):
            bad[i, j] = True
            if rnd.random() < 0.5:
                proofs[i, j, 40] ^= 1                       # a wrong response: the share itself is right
            else:
                shares[i, j] = np.frombuffer(element(rnd.randrange(1, L)), np.uint8)     # a wrong share, a decodable one
    v = e.verify_shares(eks, indexes, cts, shares, proofs)
    assert ((v != 0) == bad).all()
    d_c, d_s, d_p, d_v = dev.up(cts), dev.up(shares), dev.up(proofs), dev.empty(n * 5, "uint8")
    idx = (C.c_uint32 * 5)(*indexes)
    e._check(e.lib.eg_verify_shares_batch_dev(e.h, C.byref(eks), n, 5, idx, dev.ptr(d_c), dev.ptr(d_s), dev.ptr(d_p), dev.ptr(d_v)))
    assert (dev.down(d_v).reshape(n, 5) == v).all()

    def run(tb):
        host = e.combine_decrypt_accepted(3, indexes, cts, shares, v, tb)
        d_vals, d_found = dev.empty(n, "int64"), dev.empty(n, "uint8")
        e.combine_decrypt_accepted_dev(3, indexes, n, dev.ptr(d_c), dev.ptr(d_s), dev.ptr(d_v), tb, dev.ptr(d_vals), dev.ptr(d_found))
        return host, (dev.down(d_vals).view(np.uint64), dev.down(d_found))
    (vals, found), (dvals, dfound) = with_table(e, *TABLE, run)
    enough = (~bad).sum(axis=1) >= 3
    assert (found[enough] == 1).all() and (vals[enough] == values[enough]).all()
    assert (found[~enough] == 3).all() and not vals[~enough].any()
    assert (dfound == found).all() and (dvals == vals).all()
    assert enough.any() and (~enough).any()


# ---------------------------------------------------------------- 9. at size

def check_at_size(e, n, unique=1000):
    b = batch(3, (0, 1, 2, 3, 4), unique, seed=16)
    rnd = random.Random(17)
    v = np.zeros((unique, 5), np.uint8)
    for i in rnd.sample(range(unique), unique // 100):
        v[i, rnd.randrange(5)] = rnd.choice(REJECT)
    want_f, want_v = expected(3, b.indexes, b.cts, b.shares, v, oracle_lookup(*TABLE))
    reps = (n + unique - 1) // unique
    tile = lambda a: np.concatenate([a] * reps)[:n]
    vals, found = with_table(e, *TABLE, lambda tb: e.combine_decrypt_accepted(3, b.indexes, tile(b.cts), tile(b.shares), tile(v), tb))
    assert (found == tile(want_f)).all() and (vals == tile(want_v)).all()


# ---------------------------------------------------------------- 10. argument errors

def check_argument_errors(e, other, multi=None):
    """Refused calls leave the context usable; n = 0 succeeds."""
    from elastic_elgamal_b200 import _ffi
    b, v = mixed_batch(8, seed=18)
    want = expected(3, b.indexes, b.cts, b.shares, v, oracle_lookup(*TABLE))
    vals, found = np.zeros(8, np.uint64), np.zeros(8, np.uint8)
    a = lambda x: None if x is None else x.ctypes.data
    u32 = lambda xs: (C.c_uint32 * len(xs))(*xs)
    big = np.zeros((8, 65, 32), np.uint8)
    bigv = np.zeros((8, 65), np.uint8)
    tb, foreign = e.dlog_table(*TABLE), other.dlog_table(*TABLE)
    try:
        calls = [
            (0, 5, u32(b.indexes), b.cts, b.shares, v, tb), (17, 20, u32(range(20)), b.cts, np.zeros((8, 20, 32), np.uint8),
                                                            np.zeros((8, 20), np.uint8), tb),
            (3, 2, u32(b.indexes[:2]), b.cts, b.shares, v, tb), (3, 65, u32(range(65)), b.cts, big, bigv, tb),
            (3, 5, u32([0, 1, 2, 3, 1]), b.cts, b.shares, v, tb), (3, 5, u32([4, 4, 0, 1, 2]), b.cts, b.shares, v, tb),
            (3, 5, None, b.cts, b.shares, v, tb),
            (3, 5, u32(b.indexes), None, b.shares, v, tb), (3, 5, u32(b.indexes), b.cts, None, v, tb),
            (3, 5, u32(b.indexes), b.cts, b.shares, None, tb), (3, 5, u32(b.indexes), b.cts, b.shares, v, foreign),
            (3, 5, u32(b.indexes), b.cts, b.shares, v, None),
        ]
        for t, S, idx, c, s, vv, table in calls:
            st = e.lib.eg_combine_decrypt_accepted_batch(e.h, t, S, idx, 8, a(c), a(s), a(vv), table.h if table else None, a(vals), a(found))
            assert st == _ffi.ERR_INVALID_ARG, (t, S)
            got = e.combine_decrypt_accepted(3, b.indexes, b.cts, b.shares, v, tb)
            assert (got[1] == want[0]).all() and (got[0] == want[1]).all(), "the context changed after a refused call"
        for out in ((None, found), (vals, None)):
            st = e.lib.eg_combine_decrypt_accepted_batch(e.h, 3, 5, u32(b.indexes), 8, a(b.cts), a(b.shares), a(v), tb.h, a(out[0]), a(out[1]))
            assert st == _ffi.ERR_INVALID_ARG
        st = e.lib.eg_combine_decrypt_accepted_batch(e.h, 3, 5, u32(b.indexes), 0, None, None, None, tb.h, None, None)
        assert st == _ffi.SUCCESS
        if multi is None:
            st = e.lib.eg_combine_decrypt_accepted_batch_dev(e.h, 3, 5, u32(b.indexes), 0, None, None, None, tb.h, None, None)
            assert st == _ffi.SUCCESS
    finally:
        tb.close()
        foreign.close()
    if multi is not None:
        mt = multi.dlog_table(*TABLE)
        try:
            st = multi.lib.eg_combine_decrypt_accepted_batch_dev(multi.h, 3, 5, u32(b.indexes), 8, a(b.cts), a(b.shares), a(v), mt.h,
                                                                 a(vals), a(found))
            assert st == _ffi.ERR_INVALID_ARG
            got = multi.combine_decrypt_accepted(3, b.indexes, b.cts, b.shares, v, mt)
            assert (got[1] == want[0]).all() and (got[0] == want[1]).all()
        finally:
            mt.close()
