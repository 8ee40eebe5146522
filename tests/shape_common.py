"""Shapes at the limits of the verifiers and provers, shared by the CPU harness tests (test_hostsim_shapes.py) and the
`-m gpu` tests (test_gpu_shapes.py).  Every kernel has compile-time and run-time limits -- fixed local arrays (EG_MAX_RINGS,
EG_MSM_MAXV, EG_TERM_MAX), slot groups of EG_MAX_SLOTS per launch, the 4096-entry admissible-value cache -- and an
off-by-one or an overflowing array there shows as a wrong verdict rather than a crash.  So these checks run the shapes on
both sides of each limit and at the limit itself, compare the engine with the oracle bit for bit (verdict bytes, 64-byte
tallies, prover output bytes), and tamper with some items so that every rejection is shown, not assumed."""
import random

import numpy as np

import oracle as O
import parity_common as PC
import workloads as W

U64 = 1 << 64
RING_MODES = (1, 2, 3, 0)        # per-equation pipeline, one thread per ring, pair engine, the library's choice


def expect_invalid(fn):
    """fn() must raise EngineError with EG_ERR_INVALID_ARG."""
    from elastic_elgamal_b200 import EngineError, _ffi
    try:
        fn()
    except EngineError as exc:
        assert exc.status == _ffi.ERR_INVALID_ARG, exc.status
    else:
        raise AssertionError("accepted")


def in_ring_modes(e, fn, modes=RING_MODES):
    """[fn() for each ring mode]; the context is left in mode 0."""
    out = []
    for mode in modes:
        e.set_ring_mode(mode)
        try:
            out.append(fn())
        finally:
            e.set_ring_mode(0)
    return out


def with_chunk(e, items, fn):
    e.set_chunk_items(items)
    try:
        return fn()
    finally:
        e.set_chunk_items(0)


# ---------------------------------------------------------------- EncryptedChoice across the slot groups

# Around the commit groups (38 ring slots + the sum proof's 2 in the first launch of the per-equation pipeline, 40 after),
# the 40-slot decode and ring-hash groups, and EG_MAX_RINGS = 64 (2 * 64 + 2 = 130 = EG_TERM_MAX deferred terminal points)
CHOICE_OPTIONS = (1, 2, 19, 20, 21, 38, 39, 40, 41, 63, 64)
CHOICE_SEED = bytes([0x33] * 32)
FIRST = 3                        # item i draws from per-item stream FIRST + i


def choice_values(m, n, single):
    if single:
        v = np.zeros((n, m), np.uint8)
        for i in range(n):
            v[i, (FIRST + i) % m] = 1
        return v
    rnd = random.Random(m * 1000 + n)
    v = np.array([[rnd.randrange(2) for _ in range(m)] for _ in range(n)], np.uint8).reshape(n, m)
    v[0] = 0
    if n > 1:
        v[1] = 1
    return v


def oracle_choices(pk, m, values, single):
    """EncryptedChoice::new on the oracle for each row, item i from stream FIRST + i (block counter (FIRST + i) << 20)."""
    n = values.shape[0]
    if single:
        cts, rings, sums = O.gen_choice_batch(pk, m, CHOICE_SEED, n, first=FIRST)
        assert all(values[i].tolist() == [int(k == (FIRST + i) % m) for k in range(m)] for i in range(n))
        return cts, rings, sums
    out = [O.choice_new(pk, [bool(x) for x in values[i]], False, O.rng_from_seed(CHOICE_SEED, first_block=(FIRST + i) << 20))
           for i in range(n)]
    return (np.frombuffer(b"".join(o[0] for o in out), np.uint8).reshape(n, m, 64).copy(),
            np.frombuffer(b"".join(o[1] for o in out), np.uint8).reshape(n, 1 + 2 * m, 32).copy(), None)


def tamper_choice_at(cts, rings, sums, items, m):
    """One change per item, each on an option next to a group boundary (the last option, 0, 19, 38, 39, 40): G added to a
    blinded element, a flipped ring response bit, a non-canonical response, an undecodable element, a sum proof of another
    ballot (MultiChoice: a flipped common challenge bit)."""
    spots = [m - 1, 0, 19 % m, 38 % m, 39 % m, 40 % m]
    for k, i in enumerate(items):
        o = spots[k % len(spots)]
        kind = k % 5
        if kind == 0:
            cts[i, o, 32:] = np.frombuffer(O.point_add(bytes(cts[i, o, 32:]), W.G_ENC), np.uint8)
        elif kind == 1:
            rings[i, 1 + 2 * o, 0] ^= 1
        elif kind == 2:
            rings[i, 2 + 2 * o] = np.frombuffer(W.BAD_SCALAR, np.uint8)
        elif kind == 3:
            cts[i, o, :32] = np.frombuffer(W.BAD_POINT2, np.uint8)
        elif sums is not None:
            sums[i] = sums[(i + 1) % len(sums)]
        else:
            rings[i, 0, 0] ^= 1


def check_choice_shape(e, pk, sk, m, single, n=8, modes=RING_MODES, prove=True):
    """Prover (caller-supplied blocks and _seeded) -> oracle bytes; verify + tally in every ring mode -> oracle verdicts and
    tallies, with half of the items tampered; the tally decrypts to the per-option counts of the accepted ballots."""
    values = choice_values(m, n, single)
    cts, rings, sums = oracle_choices(pk, m, values, single)
    if prove:
        draws = 3 * m + (1 if single else 0)
        wide = np.frombuffer(b"".join(PC.item_blocks(CHOICE_SEED, FIRST + i, draws) for i in range(n)), np.uint8).reshape(n, draws, 64)
        for out in (e.encrypt_choice(m, values, wide, single=single),
                    e.encrypt_choice(m, values, single=single, seed=CHOICE_SEED, counter_base=FIRST << 20)):
            assert (out[0] == cts).all() and (out[1] == rings).all(), (m, single)
            assert (out[2] is None) if not single else (out[2] == sums).all(), (m, single)
    cts, rings = cts.copy(), rings.copy()
    sums = sums.copy() if sums is not None else None
    bad = list(range(1, n, 2))
    tamper_choice_at(cts, rings, sums, bad, m)
    expected, exp_tally = O.verify_choice_batch(pk, m, single, cts, rings, sums)
    assert (expected[bad] != 0).all() and (np.delete(expected, bad) == 0).all(), expected
    for mode, (got, tally) in zip(modes, in_ring_modes(e, lambda: e.verify_choice(m, cts, rings, sums, single=single, tally=True), modes)):
        assert got.tolist() == expected.tolist(), (m, single, mode, got, expected)
        assert (tally == exp_tally).all(), (m, single, mode)
    counts = values[expected == 0].sum(axis=0, dtype=np.int64)
    table = e.dlog_table(0, n + 1)
    try:
        el, vals, found = e.decrypt(sk, exp_tally, table)
    finally:
        table.close()
    assert found.tolist() == [1] * m and vals.tolist() == counts.tolist(), (m, single)


def check_choice_options_refused(e, pk):
    """0 and 65 options are EG_ERR_INVALID_ARG for the verifier and both prover forms; the context stays usable."""
    buf = np.zeros(65 * 200, np.uint8)
    p = buf.ctypes.data
    for m in (0, 65):
        for single in (0, 1):
            expect_invalid(lambda: e._check(e.lib.eg_verify_choice_batch(e.h, 1, m, single, p, p, p, p, p)))
            expect_invalid(lambda: e._check(e.lib.eg_encrypt_choice_batch(e.h, 1, m, single, p, p, p, p, p)))
            expect_invalid(lambda: e._check(e.lib.eg_encrypt_choice_batch_seeded(e.h, 1, m, single, p, p, 0, p, p, p)))
    cts, rings, sums = O.gen_choice_batch(pk, 3, W.SEED_CHOICE, 4)
    v, t = e.verify_choice(3, cts, rings, sums)
    ov, ot = O.verify_choice_batch(pk, 3, True, cts, rings, sums)
    assert v.tolist() == ov.tolist() == [0] * 4 and (t == ot).all()


# ---------------------------------------------------------------- RangeProof at its limits

def custom_range(rings):
    """(size, step) list, most significant ring first -> (oracle Range, engine Range)."""
    from elastic_elgamal_b200 import _ffi
    o, g = O.Range(), _ffi.Range()
    for r in (o, g):
        r.n_rings = len(rings)
        for i, (size, step) in enumerate(rings[:64]):
            r.size[i], r.step[i] = size, step
    return o, g


def upper_bound(rings):
    return 1 + sum((size - 1) * step for size, step in rings)


RANGE_SHAPES = {
    "32 rings of 4 (2^64)": [(4, 4**k) for k in reversed(range(32))],
    "64 rings of 2 (2^64)": [(2, 2**k) for k in reversed(range(64))],
    "64 rings, above 2^64": [(3, 2**63)] + [(2, 2**k) for k in reversed(range(63))],
    "63 rings": [(3, 2**62)] + [(2, 2**k) for k in reversed(range(62))],
    "one ring of 3500": [(3500, 1)],
}

# EG_ERR_INVALID_ARG: 65 rings, a ring of 4097, 3501 values in all, a zero step, and decompositions with gaps (a value
# below the upper bound that the greedy decomposition cannot reach)
REFUSED_RANGES = {
    "65 rings": [(2, 2**k) for k in reversed(range(64))] + [(2, 1)],
    "size 4097": [(4097, 1)],
    "total 3501": [(3000, 501), (501, 1)],
    "zero step": [(2, 0), (3, 1)],
    "gap above the last ring": [(2, 6), (5, 1)],
    "last step above 1": [(4, 2)],
    "gap in the middle": [(2, 100), (3, 20), (10, 1)],
}


def range_values(ub, between=3):
    """0, ub - 2, ub - 1 (ub capped at 2^64) and `between` values between."""
    top = min(ub, U64)
    rnd = random.Random(top)
    return [0, top - 2, top - 1] + [rnd.randrange(top) for _ in range(between)]


def check_range_shape(e, pk, rings, label="ciphertext_range", modes=RING_MODES, chunk=0, between=3, seed=b"\x44" * 32):
    """encrypt_range with caller blocks and _seeded equal the oracle's RangeProof::new byte for byte; values >= ub (when ub
    fits in u64) are refused; verify_range in every ring mode gives the oracle's verdicts for the proofs and for tampered
    copies of them."""
    ospec, espec = custom_range(rings)
    ub = upper_bound(rings)
    assert O.range_display(ospec) == e.range_display(espec)
    values = np.array(range_values(ub, between), np.uint64)
    n = len(values)
    cts, partials, rproofs = O.gen_range_batch(pk, ospec, label, seed, values)
    draws = e.lib.eg_range_prover_draws(O.C.byref(espec))
    assert draws == len(rings) + ospec.rings_size
    wide = np.frombuffer(b"".join(PC.item_blocks(seed, i, draws) for i in range(n)), np.uint8).reshape(n, draws, 64)

    def prove():
        return (e.encrypt_range(espec, label, values, wide), e.encrypt_range(espec, label, values, seed=seed))
    for c, p, r in with_chunk(e, chunk, prove):
        assert (c == cts).all() and (p == partials).all() and (r == rproofs).all()
    if ub < U64:
        expect_invalid(lambda: e.encrypt_range(espec, label, np.array([ub], np.uint64), wide[:1]))
    cts, partials, rproofs = (np.concatenate([a, a]) for a in (cts, partials, rproofs))
    bad = list(range(n, 2 * n))[:4]
    for k, i in enumerate(bad):               # the main ciphertext, the first ring, the last response, the common challenge
        if k == 0:
            cts[i, 32:] = np.frombuffer(O.point_add(bytes(cts[i, 32:]), W.G_ENC), np.uint8)
        elif k == 1 and len(rings) > 1:
            partials[i, 0, :32] = np.frombuffer(O.point_add(bytes(partials[i, 0, :32]), W.G_ENC), np.uint8)
        elif k == 1:
            rproofs[i, 1, 0] ^= 1
        elif k == 2:
            rproofs[i, -1] = np.frombuffer(W.BAD_SCALAR, np.uint8)
        else:
            rproofs[i, 0, 0] ^= 1
    expected = O.verify_range_batch(pk, ospec, label, cts, partials, rproofs)
    assert (expected[bad] != 0).all() and (np.delete(expected, bad) == 0).all(), expected
    for mode, got in zip(modes, in_ring_modes(e, lambda: e.verify_range(espec, label, cts, partials, rproofs), modes)):
        assert got.tolist() == expected.tolist(), (mode, got, expected)


def check_range_2_32(e, pk):
    """RangeDecomposition::optimal(2^32) on both sides: 16 rings and a `Display` string longer than the 166-byte STROBE rate
    of the transcript; values 0, 2^32 - 2 and 2^32 - 1 prove and verify, 2^32 is refused."""
    spec = O.range_optimal(1 << 32)
    espec = e.range_optimal(1 << 32)
    assert espec.rings == spec.rings and len(spec.rings) == 16 and len(O.range_display(spec)) > 166
    check_range_shape(e, pk, spec.rings)


def check_ranges_refused(e, pk):
    """Every decomposition of REFUSED_RANGES is EG_ERR_INVALID_ARG for the verifier and the provers; the context stays
    usable."""
    z = np.zeros(64 * 65 * 4097, np.uint8)
    p = z.ctypes.data
    values = np.zeros(1, np.uint64)
    for name, rings in REFUSED_RANGES.items():
        _, g = custom_range(rings)             # 65 rings: the struct holds the first 64, n_rings says 65
        for call in (lambda: e.lib.eg_verify_range_batch(e.h, O.C.byref(g), b"ciphertext_range", 1, p, p, p, p),
                     lambda: e.lib.eg_encrypt_range_batch(e.h, O.C.byref(g), b"ciphertext_range", 1, values.ctypes.data, p, p, p, p),
                     lambda: e.lib.eg_encrypt_range_batch_seeded(e.h, O.C.byref(g), b"ciphertext_range", 1, values.ctypes.data, p, 0,
                                                                 p, p, p)):
            expect_invalid(lambda: e._check(call()))
    PC.check_verify_range(e, pk, 21, n=6, frac=0.5)


def check_range_cache_eviction(e, pk, calls=2):
    """Two single-ring ranges of 3500 and 700 admissible values (4200 > the 4096-entry cache) alternated across calls, and a
    QV ballot whose vote range (2000 values) and credit range (2100) evict each other inside every call: the verdicts and
    tallies never change."""
    a, b = [(3500, 1)], [(700, 1)]
    runs = []
    for rings in (a, b):
        ospec, espec = custom_range(rings)
        values = np.array([0, 699, 350], np.uint64)
        c, p, r = O.gen_range_batch(pk, ospec, "ciphertext_range", b"\x55" * 32, values)
        c = c.copy()
        c[1, 32:] = np.frombuffer(O.point_add(bytes(c[1, 32:]), W.G_ENC), np.uint8)
        expected = O.verify_range_batch(pk, ospec, "ciphertext_range", c, p, r)
        assert expected.tolist() == [0, 2, 0]
        runs.append((espec, c, p, r, expected))
    for _ in range(calls):
        for espec, c, p, r, expected in runs:
            assert e.verify_range(espec, "ciphertext_range", c, p, r).tolist() == expected.tolist()
    op = O.QvParams()
    op.options, op.credits = 2, 2099
    op.vote_range, op.credit_range = custom_range([(2000, 1)])[0], custom_range([(2100, 1)])[0]
    ep = PC.as_engine_qv(op)
    votes = np.array([[0, 0], [45, 7], [3, 44]], np.uint64)
    ballots = O.gen_qv_batch(pk, op, W.SEED_QV, votes).copy()
    ballots[2, 40] ^= 1
    expected, exp_tally = O.verify_qv_batch(pk, op, ballots)
    assert expected[[0, 1]].tolist() == [0, 0] and expected[2] != 0
    for _ in range(calls):
        got, tally = e.verify_qv(ep, ballots)
        assert got.tolist() == expected.tolist() and (tally == exp_tally).all()
        espec, c, p, r, exp_range = runs[0]
        assert e.verify_range(espec, "ciphertext_range", c, p, r).tolist() == exp_range.tolist()


# ---------------------------------------------------------------- multi-scalar kernels at EG_MSM_MAXV = 16

def check_sumsq_15(e, pk, n=9):
    """SumOfSquaresProof::verify with 15 ciphertexts (k_msm: 16 variable-base terms) against the oracle with the reference's
    tamper patterns; 16 ciphertexts are refused."""
    PC.check_verify_sumsq(e, pk, n=n, count=15)
    expect_invalid(lambda: e.verify_sumsq("test", np.zeros((1, 16, 64), np.uint8), np.zeros((1, 64), np.uint8),
                                          np.zeros((1, 34, 32), np.uint8)))
    PC.check_verify_sumsq(e, pk, n=2, count=2)


QV15_CREDITS = 40                # vote range optimal(isqrt(40) + 1 = 7), credit range optimal(41)
QV15_VOTES = [[0] * 15, [1] * 15, [6] + [0] * 14, [2] * 10 + [0] * 5, [0] * 14 + [6], [3] * 4 + [1] * 4 + [0] * 7,
              [1, 2, 3, 4] + [0] * 11, [5, 3, 1] + [0] * 12]          # credits 0..40; rows 3 and 5 spend exactly 40


def check_qv_15(e, pk, sk, modes=RING_MODES, verify=True, chunk=0):
    """QV ballots with 15 options (the sum-of-squares proof's k_msm slots: 16 variable-base terms): the prover's bytes in both
    randomness forms; verify + tally in every ring mode against the oracle, with the reference's tamper patterns, and the
    tally decrypts to the vote sums of the accepted ballots; a vote above the vote range, a credit above the credit range
    and 16 options are refused."""
    m = 15
    p, ep = O.qv_params(m, QV15_CREDITS), e.qv_params(m, QV15_CREDITS)
    assert ep.vote_range.rings == p.vote_range.rings and ep.credit_range.rings == p.credit_range.rings
    votes = np.array(QV15_VOTES, np.uint64)
    n = len(votes)
    assert max(int((v * v).sum()) for v in votes) == QV15_CREDITS
    ballots = O.gen_qv_batch(pk, p, W.SEED_QV, votes)
    draws = e.lib.eg_qv_prover_draws(O.C.byref(ep))
    wide = np.frombuffer(b"".join(PC.item_blocks(W.SEED_QV, i, draws) for i in range(n)), np.uint8).reshape(n, draws, 64)
    got = with_chunk(e, chunk, lambda: (e.encrypt_qv(ep, votes, wide), e.encrypt_qv(ep, votes, seed=W.SEED_QV)))
    for g in got:
        bad = np.nonzero((g != ballots).any(axis=1))[0]
        assert bad.size == 0, bad
    expect_invalid(lambda: e.encrypt_qv(ep, np.array([[7] + [0] * 14], np.uint64), seed=W.SEED_QV))
    expect_invalid(lambda: e.encrypt_qv(ep, np.array([[6, 3] + [0] * 13], np.uint64), seed=W.SEED_QV))
    e16 = e.qv_params(16, QV15_CREDITS)
    expect_invalid(lambda: e.verify_qv(e16, np.zeros((1, e.qv_ballot_size(e16)), np.uint8)))
    expect_invalid(lambda: e.encrypt_qv(e16, np.zeros((1, 16), np.uint64), seed=W.SEED_QV))
    if not verify:
        return
    ballots = ballots.copy()
    vsz = 64 + 64 * (p.vote_range.n_rings - 1) + 32 * (1 + p.vote_range.rings_size)
    o = m - 1                                  # quadratic_voting.rs:433-464 on the last option
    ballots[1, vsz * o + 32:vsz * o + 64] = np.frombuffer(O.point_add(bytes(ballots[1, vsz * o + 32:vsz * o + 64]), W.G_ENC), np.uint8)
    ballots[2, vsz * m:vsz * m + 64] = ballots[3, vsz * m:vsz * m + 64]
    ballots[4, -32 * (2 * m + 2):] = ballots[5, -32 * (2 * m + 2):]
    ballots[6, -1] = 0xff
    ballots[7, 0:32] = np.frombuffer(W.BAD_POINT, np.uint8)
    expected, exp_tally = O.verify_qv_batch(pk, p, ballots)
    assert expected[1] == O.QV_VARIANT_BASE + o and expected[2] == O.QV_CREDIT_RANGE and expected[4] != 0
    assert expected[6] == O.MALFORMED and expected[7] == O.MALFORMED and expected[[0, 3, 5]].tolist() == [0, 0, 0]
    for mode, (v, t) in zip(modes, in_ring_modes(e, lambda: e.verify_qv(ep, ballots), modes)):
        assert v.tolist() == expected.tolist(), (mode, v, expected)
        assert (t == exp_tally).all(), mode
    table = e.dlog_table(0, 6 * n + 1)
    try:
        _, vals, found = e.decrypt(sk, exp_tally, table)
    finally:
        table.close()
    assert found.all() and vals.tolist() == votes[expected == 0].sum(axis=0).tolist()


def check_multi_mul_16(e, n=6):
    """eg_multi_mul_batch up to 16 terms against the oracle's point arithmetic; 17 terms are refused."""
    PC.check_multi_mul(e, n=n)
    expect_invalid(lambda: e.multi_mul(np.zeros((1, 17, 32), np.uint8), np.zeros((1, 17, 32), np.uint8)))


def check_combine_16(e, n=8):
    """Combine-and-decrypt with 16 shares of a 16-of-64 key set (participant indexes spread over 0..63) against the oracle's
    combination and table lookup, one item with a share of another participant; 17 shares are refused."""
    rng = O.rng_from_seed(bytes([0x16] * 32))
    ks, secrets = O.dealer_new(64, 16, rng)
    used = [0, 1, 5, 9, 17, 20, 31, 32, 33, 40, 47, 50, 55, 61, 62, 63]
    shared = bytes(ks.shared_key)
    values = [0, 63, 64, 1, 2, 33, 62, 7][:n]
    cts = [O.encrypt(shared, v, rng) for v in values]
    sh = np.array([[np.frombuffer(O.decrypt_share(ks, i, secrets[i], ct, rng)[0], np.uint8) for i in used] for ct in cts], np.uint8)
    sh[3, 7] = sh[3, 8]
    table = e.dlog_table(0, 64)
    otable = O.DlogTable(0, 64)
    try:
        vals, found = e.combine_decrypt(used, np.frombuffer(b"".join(cts), np.uint8).reshape(n, 64), sh, table)
        idx17 = used + [2]
        sh17 = np.concatenate([sh, sh[:, :1]], axis=1)
        expect_invalid(lambda: e.combine_decrypt(idx17, np.frombuffer(b"".join(cts), np.uint8).reshape(n, 64), sh17, table))
    finally:
        table.close()
    for i in range(n):
        rc, el = O.combine_decrypt(used, [bytes(s) for s in sh[i]], cts[i])
        assert rc == 0
        ov = otable.get(el)
        assert (found[i], int(vals[i])) == ((1, ov) if ov is not None else (0, 0)), i
    assert found.tolist() == [1, 1, 0, 0, 1, 1, 1, 1] and vals[1] == 63 and vals[6] == 62


def check_keysets_64_16(e):
    """PublicKeySet::from_participants with 64 keys and threshold 16 (k_msm: 16 Lagrange terms) against the oracle, with the
    tamper patterns of parity_common; threshold 17 and 65 keys are refused."""
    PC.check_keysets_validate(e, n_sets=6, shares=64, threshold=16)
    expect_invalid(lambda: e.keysets_validate(64, 17, np.zeros((1, 64, 32), np.uint8)))
    expect_invalid(lambda: e.keysets_validate(65, 3, np.zeros((1, 65, 32), np.uint8)))


# ---------------------------------------------------------------- chunking at the limits

def check_chunked_limits(e, pk, sk):
    """Several chunks with a remainder: 64-option ballots (verify + tally in chunks of 3, prover in chunks of 3), 15-option
    QV ballots (prover in chunks of 3) and the 2^64 range (prover in chunks of 4)."""
    with_chunk(e, 3, lambda: check_choice_shape(e, pk, sk, 64, True, n=8, modes=(0, 1)))
    check_qv_15(e, pk, sk, verify=False, chunk=3)
    check_range_shape(e, pk, RANGE_SHAPES["32 rings of 4 (2^64)"], modes=(0,), chunk=4)
