"""eg_ciphertexts_weighted_sum (the weighted tally fold sum_i [k_i] cts[i]), shared by the CPU harness tests
(test_hostsim_weighted_sum.py) and the `-m gpu` tests (test_gpu_weighted_sum.py).  Every check compares bytes.

Elements are [x]G with known x, so a weighted sum is also [sum k_i x_i]G: small batches are checked against a fold of the
oracle's point_mul / point_add, larger ones against that one fixed-base product."""
import functools
import random

import numpy as np

import edge_common as EC
import oracle as O
import workloads as W

L = W.L
IDENTITY = bytes(32)
SPECIAL = [0, 1, 2, L - 1, L - 2, 2**64 - 1, 2**64, 2**252]


def sc(k):
    return (k % L).to_bytes(32, "little")


def scalar_rows(ks):
    return EC.rows([sc(k) for k in ks], 32)


@functools.lru_cache(maxsize=None)
def corpus(n, n_cts, seed=1):
    """(cts (n, n_cts, 64), logs (n, 2 n_cts)): ciphertext j of item i is ([x_{i,2j}]G, [x_{i,2j+1}]G)."""
    rnd = random.Random(seed * 1000003 + n * 131 + n_cts)
    logs = [[rnd.randrange(1, L) for _ in range(2 * n_cts)] for _ in range(n)]
    cts = np.frombuffer(b"".join(O.point_mul_generator(sc(x)) for row in logs for x in row), np.uint8).reshape(n, n_cts, 64)
    return cts, logs


def expected(cts, logs, ks, mask=None, fold=None):
    """The n_cts ciphertexts sum_i [k_i] cts[i] over the included items: by the oracle's point_mul / point_add (fold=True,
    the default for small batches) or as [sum k_i x_i]G."""
    n, n_cts = cts.shape[0], cts.shape[1]
    inc = [i for i in range(n) if mask is None or mask[i] == 0]
    if fold is None:
        fold = len(inc) * n_cts <= 600
    out = []
    for col in range(2 * n_cts):
        if fold:
            acc = IDENTITY
            for i in inc:
                acc = O.point_add(acc, O.point_mul(sc(ks[i]), bytes(cts[i, col // 2, 32 * (col % 2):32 * (col % 2) + 32])))
        else:
            acc = O.point_mul_generator(sc(sum(ks[i] * logs[i][col] for i in inc)))
        out.append(acc)
    return np.frombuffer(b"".join(out), np.uint8).reshape(n_cts, 64)


def check(e, cts, logs, ks, mask=None, what=""):
    out, ok = e.weighted_sum(cts, scalar_rows(ks), mask)
    assert ok, what
    want = expected(cts, logs, ks, mask)
    assert (out == want).all(), f"{what}: weighted sum differs from the oracle"
    return out


def random_scalars(n, rnd, kind):
    if kind == "u64":
        return [rnd.randrange(2**64) for _ in range(n)]
    if kind == "full":
        return [rnd.randrange(L) for _ in range(n)]
    base = SPECIAL + [rnd.randrange(L) for _ in range(4)] + [rnd.randrange(2**64) for _ in range(4)]
    return [base[i % len(base)] if i < 2 * len(base) else rnd.randrange(L) for i in range(n)]


# ---------------------------------------------------------------- 1. oracle parity

def check_parity(e, n, n_cts, kind, seed=3):
    cts, logs = corpus(n, n_cts)
    ks = random_scalars(n, random.Random(seed + n), kind)
    check(e, cts, logs, ks, what=f"n={n} n_cts={n_cts} {kind}")


def carry_scalars(c):
    """For window width c: digits at +2^(c-1) in every window (no carry), and 2^b - 1 for every b up to 253 bits, whose
    signed digits are -1 with a carry through every window but the top."""
    half = sum(2 ** (c - 1) << (c * w) for w in range(253 // c))
    ks = [half % L, (half >> c) % L]
    ks += [2**b - 1 for b in range(c - 1, 253, max(1, c - 1))]
    ks += [2 ** (c * w) * (2 ** (c - 1) + 1) for w in range(253 // c)]            # one digit just past the top: a carry
    return [k % L for k in ks]


def check_width(e, n, c, n_cts=2):
    cts, logs = corpus(n, n_cts)
    special = carry_scalars(c)
    ks = [special[i % len(special)] for i in range(n)]
    check(e, cts, logs, ks, what=f"width {c}, n={n}")
    # one scalar at a time among zeros: the windows follow the largest scalar, so each pattern sets the window count
    for k in special[:: max(1, len(special) // 6)]:
        ks = [0] * n
        ks[n // 2] = k
        check(e, cts, logs, ks, what=f"width {c}, single scalar {k:#x}")


# ---------------------------------------------------------------- 2. skew and cancellation

def check_skew(e, n, n_cts):
    cts, logs = corpus(n, n_cts)
    rnd = random.Random(17)
    out = check(e, cts, logs, [1] * n, what="all weights 1")
    plain = cts[0].copy()
    for i in range(1, n):
        for j in range(n_cts):
            for h in (0, 32):
                plain[j, h:h + 32] = np.frombuffer(O.point_add(bytes(plain[j, h:h + 32]), bytes(cts[i, j, h:h + 32])), np.uint8)
    assert (out == plain).all(), "weight 1 differs from the unweighted fold"
    k = rnd.randrange(L)
    check(e, cts, logs, [k] * n, what="all scalars equal")
    a, b = rnd.randrange(2**20), rnd.randrange(L)
    check(e, cts, logs, [a if rnd.random() < 0.5 else b for _ in range(n)], what="two scalars")
    ks = [0] * n
    ks[rnd.randrange(n)] = rnd.randrange(L)
    check(e, cts, logs, ks, what="all zero but one")
    check(e, cts, logs, [max(1, int(2**20 / (1 + rnd.paretovariate(1.2)))) for _ in range(n)], what="Zipf-like weights")
    # pairs that cancel: item 2t + 1 repeats item 2t's ciphertext with l - k
    m = n - n % 2
    if m:
        pc = cts[:m].copy()
        pc[1::2] = pc[0::2]
        pl = [logs[2 * (i // 2)] for i in range(m)]
        ks = []
        for _ in range(m // 2):
            k = rnd.randrange(1, L)
            ks += [k, L - k]
        out, ok = e.weighted_sum(pc, scalar_rows(ks))
        assert ok and not out.any(), "cancelling pairs do not give the identity"
        assert (out == expected(pc, pl, ks)).all()


# ---------------------------------------------------------------- 3. masks and validation

def check_choice_mask(e, n=64, m=5):
    sk, pk = W.receiver()
    e.set_receiver(pk)
    cts, rings, sums = O.gen_choice_batch(pk, m, W.SEED_CHOICE, n)
    cts, rings, sums = cts.copy(), rings.copy(), sums.copy()
    W.tamper_choice(cts, rings, sums, random.Random(5), frac=0.2)
    v, t = e.verify_choice(m, cts, rings, sums)
    assert (v != 0).any() and (v == 0).any()
    out, ok = e.weighted_sum(cts, np.arange(n) * 0 + 1, v)
    assert ok and (out == t).all(), "weights 1 under the verdicts differ from eg_verify_choice_batch's tally"


def qv_record(p):
    r = p.vote_range
    return 64 + 64 * (r.n_rings - 1) + 32 * (1 + r.rings_size)


def check_qv_mask(e, n=24, options=3, credits=10):
    sk, pk = W.receiver()
    e.set_receiver(pk)
    p = e.qv_params(options, credits)
    rnd = random.Random(9)
    votes = np.array([[rnd.randrange(2) for _ in range(options)] for _ in range(n)], np.uint64)
    ballots = O.gen_qv_batch(pk, O.qv_params(options, credits), W.SEED_QV, votes).copy()
    for i in range(0, n, 5):                         # flip a byte of a response in some ballots
        ballots[i, -40] ^= 1
    v, t = e.verify_qv(p, ballots)
    assert (v != 0).any() and (v == 0).any()
    out, ok = e.weighted_sum(ballots, [1] * n, v, ct_stride=qv_record(p), n_cts=options)
    assert ok and (out == t).all(), "weights 1 under the verdicts differ from eg_verify_qv_batch's tally"


def check_validation(e, n=40, n_cts=2):
    cts, logs = corpus(n, n_cts)
    rnd = random.Random(23)
    ks = [rnd.randrange(L) for _ in range(n)]
    bad_el, bad_sc = cts.copy(), scalar_rows(ks)
    bad_el[3, 1, 32:] = np.frombuffer(W.BAD_POINT, np.uint8)
    bad_sc[7] = np.frombuffer(W.BAD_SCALAR, np.uint8)
    mask = np.zeros(n, np.uint8)
    mask[[3, 7]] = 3
    want = expected(cts, logs, ks, mask)
    for c, s in ((bad_el, scalar_rows(ks)), (cts, bad_sc), (bad_el, bad_sc)):
        out, ok = e.weighted_sum(c, s, mask)
        assert ok and (out == want).all(), "a bad excluded item changed the result"
        out, ok = e.weighted_sum(c, s)
        assert not ok and not out.any(), "a bad included item must give ok = 0 and identity ciphertexts"
    out, ok = e.weighted_sum(cts, scalar_rows(ks), np.full(n, 1, np.uint8))
    assert ok and not out.any(), "no included item: identity"
    out, ok = e.weighted_sum(cts[:0], np.zeros((0, 32), np.uint8))
    assert ok and out.shape == (n_cts, 64) and not out.any(), "n = 0: identity"
    out, ok = e.weighted_sum(cts, [0] * n)
    assert ok and not out.any(), "all weights 0: identity"


# ---------------------------------------------------------------- 4. invariance

def check_chunks(e, n, n_cts, kind="mixed"):
    cts, logs = corpus(n, n_cts)
    ks = random_scalars(n, random.Random(41), kind)
    mask = np.array([0 if i % 7 else 1 for i in range(n)], np.uint8)
    want = expected(cts, logs, ks, mask)
    s = scalar_rows(ks)
    try:
        for chunk in (7, 0, 100):
            e.set_chunk_items(chunk)
            out, ok = e.weighted_sum(cts, s, mask)
            assert ok and (out == want).all(), f"chunk size {chunk}"
    finally:
        e.set_chunk_items(0)


def check_thresholds(e, sizes, n_cts=1):
    for n in sizes:
        cts, logs = corpus(n, n_cts)
        ks = random_scalars(n, random.Random(n), "mixed")
        check(e, cts, logs, ks, what=f"threshold batch n={n}")


def check_multi(m, e, n=100, n_cts=3):
    cts, logs = corpus(n, n_cts)
    ks = random_scalars(n, random.Random(43), "mixed")
    mask = np.array([i % 3 == 1 for i in range(n)], np.uint8)
    a, ok_a = m.weighted_sum(cts, scalar_rows(ks), mask)
    b, ok_b = e.weighted_sum(cts, scalar_rows(ks), mask)
    assert ok_a and ok_b and (a == b).all() and (a == expected(cts, logs, ks, mask)).all()
    bad = scalar_rows(ks)
    bad[n - 1] = np.frombuffer(W.BAD_SCALAR, np.uint8)
    a, ok_a = m.weighted_sum(cts, bad)
    assert not ok_a and not a.any()
    a, ok_a = m.weighted_sum(cts[:0], bad[:0])
    assert ok_a and not a.any()


def check_dev(e, dev, n=300, n_cts=2, chunk=0):
    cts, logs = corpus(n, n_cts)
    ks = random_scalars(n, random.Random(47), "mixed")
    mask = np.array([i % 5 == 2 for i in range(n)], np.uint8)
    host, ok = e.weighted_sum(cts, scalar_rows(ks), mask)
    assert ok and (host == expected(cts, logs, ks, mask)).all()
    e.set_chunk_items(chunk)
    try:
        d_cts, d_s, d_v = dev.up(cts.reshape(n, -1)), dev.up(scalar_rows(ks)), dev.up(mask)
        d_out, d_ok = dev.empty(n_cts * 64, "uint8"), dev.empty(1, "uint8")
        e.weighted_sum_dev(n, n_cts, 64 * n_cts, 64, dev.ptr(d_cts), dev.ptr(d_s), dev.ptr(d_v), dev.ptr(d_out), dev.ptr(d_ok))
        assert dev.down(d_ok)[0] == 1 and (dev.down(d_out).reshape(n_cts, 64) == host).all(), "host and _dev forms differ"
        e.weighted_sum_dev(n, n_cts, 64 * n_cts, 64, dev.ptr(d_cts), dev.ptr(d_s), 0, dev.ptr(d_out), dev.ptr(d_ok))
        assert (dev.down(d_out).reshape(n_cts, 64) == expected(cts, logs, ks)).all()
    finally:
        e.set_chunk_items(0)


# ---------------------------------------------------------------- 5. argument errors

def check_argument_errors(e, multi=None):
    from elastic_elgamal_b200 import _ffi
    cts, logs = corpus(8, 2)
    ks = [3, 5, 7, 11, 13, 17, 19, 23]
    s = scalar_rows(ks)
    want = expected(cts, logs, ks)
    out, ok = np.zeros(64 * 65, np.uint8), np.zeros(1, np.uint8)
    a = lambda x: None if x is None else x.ctypes.data
    calls = [
        (8, 0, 128, 64, cts, s, out, ok), (8, 65, 65 * 64, 64, cts, s, out, ok),
        (8, 2, 128, 32, cts, s, out, ok), (8, 2, 127, 64, cts, s, out, ok), (8, 1, 63, 64, cts, s, out, ok),
        (8, 2, 128, 64, None, s, out, ok), (8, 2, 128, 64, cts, None, out, ok), (8, 2, 128, 64, cts, s, None, ok),
        (8, 2, 128, 64, cts, s, out, None), (0, 2, 128, 64, None, None, None, ok),
    ]
    for n, k, istr, cstr, c, sc_, o, okb in calls:
        st = e.lib.eg_ciphertexts_weighted_sum(e.h, n, k, istr, cstr, a(c), a(sc_), None, a(o), a(okb))
        assert st == _ffi.ERR_INVALID_ARG, (n, k, istr, cstr)
        got, good = e.weighted_sum(cts, s)
        assert good and (got == want).all(), "the context changed after a refused call"
    if multi is not None:
        st = multi.lib.eg_ciphertexts_weighted_sum_dev(multi.h, 8, 2, 128, 64, a(cts), a(s), None, a(out), a(ok))
        assert st == _ffi.ERR_INVALID_ARG
        got, good = multi.weighted_sum(cts, s)
        assert good and (got == want).all()
