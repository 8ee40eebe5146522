"""Baby-step giant-step discrete-log tables (eg_dlog_table_create_bsgs) and the batch lookup eg_dlog_lookup_batch, shared by
the CPU harness tests (test_hostsim_dlog_bsgs.py, small baby-step counts) and the `-m gpu` tests (test_gpu_dlog_bsgs.py).

A BSGS table of m baby steps over [lo, hi) must answer every lookup exactly as eg_dlog_table_create(lo, hi) -- and the
oracle's DiscreteLogTable -- would.  The ranges below sit on the giant-step boundaries (hi - lo = m, m + 1, 2m - 1, ...), next
to 2^32 and 2^63, and at the top of u64, where lo + J m passes 2^64.  Ranges that no table can hold are checked on known
plaintexts: every value is encrypted by the oracle, so the expected lookup is known without a table."""
import random

import numpy as np

import decrypt_common as D
import edge_common as EC
import oracle as O
import workloads as W

L = W.L
U64 = EC.U64
USED = EC.USED
UNDECODABLE = [b"\xff" * 32, bytes([1]) + bytes(31)]        # non-canonical; "negative" (odd) s


def boundary_ranges(m):
    """Ranges on the giant-step boundaries of m baby steps, around 2^32 and 2^63, at the top of u64, and the empty range."""
    return [
        (0, m), (0, m + 1), (0, 2 * m - 1), (0, 2 * m), (0, 2 * m + 1), (3, 3 + 5 * m + 1), (37, 37 + 37 * m),
        (2**32 - 2 * m - 7, 2**32 + 2 * m + 9), (2**63 - m - 3, 2**63 + 2 * m + 1),
        (U64 - 4 * m - 3, U64 - 1),
        (5, 5),
    ]


def element(v):
    return O.point_mul_generator(EC.sc(v))


def elements(values):
    return EC.rows([element(v) for v in values], 32)


def as_pairs(found, vals):
    assert vals.dtype == np.uint64
    return list(zip(found.tolist(), [int(v) for v in vals]))


def diff(values, got, want, what):
    bad = [(hex(v), g, w) for v, g, w in zip(values, got, want) if g != w]
    return [f"{what}: {len(bad)} of {len(want)} lookups wrong, e.g. {bad[:3]}"] if bad else []


def with_table(e, lo, hi, m, fn):
    t = e.dlog_table(lo, hi, m)
    try:
        return fn(t)
    finally:
        t.close()


# ---------------------------------------------------------------- 1. equal to the range table

def check_equal_to_range_table(e, corpus, m, shares, dev):
    """Every range of `corpus` (an edge_common.TableCorpus) through eg_decrypt_batch, both forms of eg_combine_decrypt_batch
    and eg_dlog_lookup_batch with a BSGS table of m baby steps: item for item what eg_dlog_table_create(lo, hi) gives and what
    the oracle's DlogTable gives (corpus.lookups).  dev=None skips the device-pointer form (multi-device contexts)."""
    sk, _ = W.receiver()
    bad = []
    for k, (lo, hi) in enumerate(corpus.ranges):
        sp = corpus.spans[k]
        values, want = corpus.values[sp], corpus.lookups[sp]
        els = EC.rows(corpus.elements[sp], 32)
        ref = EC._with_table(e, lo, hi, lambda t: e.decrypt(sk, corpus.cts_pk[sp], t))
        bad += diff(values, as_pairs(ref[2], ref[1]), want, f"range table [{lo:#x}, {hi:#x})")

        def run(t):
            el, vals, found = e.decrypt(sk, corpus.cts_pk[sp], t)
            assert [bytes(x) for x in el] == corpus.elements[sp]
            outs = {"decrypt": (found, vals)}
            vals, found = e.combine_decrypt(list(USED), corpus.cts_ks[sp], shares[sp], t)
            outs["combine"] = (found, vals)
            if dev is not None:
                vals, found = EC.combine_decrypt_dev(e, dev, corpus.cts_ks[sp], shares[sp], t)
                outs["combine_dev"] = (found, vals)
            vals, found = e.dlog_lookup(t, els)
            outs["lookup"] = (found, vals)
            return outs

        for what, (found, vals) in with_table(e, lo, hi, m, run).items():
            bad += diff(values, as_pairs(found, vals), want, f"{what}, BSGS m={m} [{lo:#x}, {hi:#x})")
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------- 2. ranges no table can hold

def giants(lo, hi, m):
    return -(-(hi - lo) // m)


def known_values(lo, hi, m, samples, seed):
    """lo + j m + {-1, 0, 1} for j in {1, 2, J - 1, J}, hi - 2, hi - 1, hi and lo - 1 (absent when in u64), 0 and random
    samples of the range."""
    J = giants(lo, hi, m)
    vs = [lo + j * m + d for j in (1, 2, J - 1, J) for d in (-1, 0, 1)] + [hi - 2, hi - 1, hi, lo - 1, 0]
    rnd = random.Random(seed)
    vs += [rnd.randrange(lo, hi) for _ in range(samples)]
    return list(dict.fromkeys(v for v in vs if 0 <= v < U64))


def check_large_range(e, lo, hi, m, samples=8, misses=2, decrypt=True):
    """Known plaintexts of [lo, hi) with m baby steps through eg_dlog_lookup_batch (and eg_decrypt_batch on the values inside
    the range): the expected lookups follow from the values.  `misses` random group elements must come back absent, and
    undecodable encodings as found 2.  Each miss walks all J giant steps."""
    values = known_values(lo, hi, m, samples, seed=lo ^ hi ^ m)
    want = [EC.expected_lookup(lo, hi, v) for v in values]
    rnd = random.Random(m)
    rand_els = [element(rnd.randrange(1, L)) for _ in range(misses)]
    els = EC.rows([element(v) for v in values] + rand_els + UNDECODABLE, 32)
    sk, pk = W.receiver()
    inside = [v for v in values if lo <= v < hi or v == 0]
    rng = O.rng_from_seed(bytes([0x48] * 32))
    cts = EC.rows([O.encrypt(pk, v, rng) for v in inside], 64)

    def run(t):
        out = [e.dlog_lookup(t, els)]
        if decrypt:
            out.append(e.decrypt(sk, cts, t)[1:])
        return out

    outs = with_table(e, lo, hi, m, run)
    vals, found = outs[0]
    got = as_pairs(found, vals)
    bad = diff(values, got[:len(values)], want, f"lookup [{lo:#x}, {hi:#x}) m={m}")
    assert got[len(values):] == [(0, 0)] * misses + [(2, 0)] * len(UNDECODABLE), got[len(values):]
    if decrypt:
        vals, found = outs[1]
        bad += diff(inside, as_pairs(found, vals), [EC.expected_lookup(lo, hi, v) for v in inside], "decrypt")
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------- 3. the case that motivates this

def check_large_tally(e, values, lo, hi, m):
    """Tallies of `values` encrypted under the 3-of-5 key set's shared key, shares made by eg_decrypt_share_batch, combined by
    eg_combine_decrypt_batch with a BSGS table: the exact values.  eg_dlog_table_create(lo, hi) itself refuses the range
    when it is longer than 2^28."""
    from elastic_elgamal_b200 import EngineError, _ffi
    ks, eks, secrets = D.keyset()
    rng = O.rng_from_seed(bytes([0x7a] * 32))
    cts = EC.rows([O.encrypt(bytes(ks.shared_key), v, rng) for v in values], 64)
    shares = np.zeros((len(values), len(USED), 32), np.uint8)
    for j, idx in enumerate(USED):
        sh, _, ok = e.decrypt_share(eks, idx, secrets[idx], cts, seed=D.SEED)
        assert ok.all()
        shares[:, j] = sh
    vals, found = with_table(e, lo, hi, m, lambda t: e.combine_decrypt(list(USED), cts, shares, t))
    assert as_pairs(found, vals) == [(1, v) for v in values]
    if hi - lo > 2**28:
        try:
            e.dlog_table(lo, hi).close()
            raise AssertionError("eg_dlog_table_create accepted a range of more than 2^28 values")
        except EngineError as err:
            assert err.status == _ffi.ERR_INVALID_ARG


# ---------------------------------------------------------------- 4. shapes

def mixed_values(n, lo, hi, m, seed, walks, misses):
    """n values: `walks` of them at random giant steps >= 1, then `misses` outside the range (lo - 1 or hi), the rest found
    by giant step 0; positions shuffled."""
    rnd = random.Random(seed)
    idx = list(range(n))
    rnd.shuffle(idx)
    kinds = ["hit"] * n
    for i in idx[:walks]:
        kinds[i] = "walk"
    for i in idx[walks:walks + misses]:
        kinds[i] = "miss"
    outside = [v for v in (lo - 1, hi) if 0 < v < U64]
    return [rnd.choice(outside) if k == "miss" else rnd.randrange(lo + m, hi) if k == "walk" else rnd.randrange(lo, lo + m)
            for k in kinds]


def check_shapes(e, lo, hi, m, ns, walks, misses, chunk=None, ct_mode=False, decrypt=True):
    """Batches of each size in `ns` mixing giant-step-0 hits, long walks and misses, through eg_dlog_lookup_batch and
    eg_decrypt_batch (unless decrypt=False); optional chunk size (eg_ctx_set_chunk_items) and constant-time prover mode."""
    sk, pk = W.receiver()
    t = e.dlog_table(lo, hi, m)
    try:
        for n in ns:
            values = mixed_values(n, lo, hi, m, seed=n, walks=walks, misses=misses)
            want = [EC.expected_lookup(lo, hi, v) for v in values]
            assert n < 4 or {w[0] for w in want} == {0, 1}
            if chunk:
                e.set_chunk_items(chunk)
            try:
                vals, found = e.dlog_lookup(t, elements(values))
                assert not diff(values, as_pairs(found, vals), want, f"lookup n={n}")
                if not decrypt:
                    continue
                rng = O.rng_from_seed(bytes([n % 251] * 32))
                cts = EC.rows([O.encrypt(pk, v, rng) for v in values], 64)
                for ct in ([False, True] if ct_mode else [False]):
                    e.set_prover_mode(ct)
                    try:
                        _, vals, found = e.decrypt(sk, cts, t)
                    finally:
                        e.set_prover_mode(False)
                    assert not diff(values, as_pairs(found, vals), want, f"decrypt n={n} constant-time={ct}")
            finally:
                if chunk:
                    e.set_chunk_items(0)
    finally:
        t.close()


# ---------------------------------------------------------------- 5. multi-device

def check_multi(m_engine, corpus, m, shares):
    """The same checks as check_equal_to_range_table on a multi-device context (host-pointer forms)."""
    check_equal_to_range_table(m_engine, corpus, m, shares, None)


# ---------------------------------------------------------------- 6. argument errors

def check_argument_errors(e, other, m):
    """Refused shapes are EG_ERR_INVALID_ARG, a table of another context is refused by every lookup, and the next call on the
    context still works."""
    from elastic_elgamal_b200 import EngineError, _ffi
    sk, pk = W.receiver()
    good = [0, 1, m, m + 7, 3 * m + 1]
    cts = EC.rows([O.encrypt(pk, v, O.rng_from_seed(bytes([3] * 32))) for v in good], 64)
    want = [(1, v) for v in good]

    def still_works():
        _, vals, found = with_table(e, 0, 4 * m, m, lambda t: e.decrypt(sk, cts, t))
        assert as_pairs(found, vals) == want

    def refused(fn):
        try:
            fn()
            raise AssertionError("accepted")
        except EngineError as err:
            assert err.status == _ffi.ERR_INVALID_ARG, err
        still_works()

    for lo, hi, bs in ((0, 2**20, 255), (0, 2**40, 2**28 + 1), (10, 9, 256), (0, 2**32 * 256 + 1, 256),  # J = 2^32 + 1
                       (U64 - 2 - 2**40, U64 - 1, 256)):                                                   # J = 2^32 + 1
        refused(lambda: e.dlog_table(lo, hi, bs).close())
    for lo, hi, bs in ((0, 2**32 * 256, 256), (U64 - 1 - 2**40, U64 - 1, 256)):       # J = 2^32 exactly: accepted
        assert giants(lo, hi, bs) == 2**32
        e.dlog_table(lo, hi, bs).close()                                                 # (nothing walks its top here)
    assert e.lib.eg_dlog_table_create_bsgs(e.h, 0, 4 * m, m, None) == _ffi.ERR_INVALID_ARG
    still_works()
    foreign = other.dlog_table(0, 4 * m, m)
    try:
        els = elements(good)
        shares = np.zeros((len(good), len(USED), 32), np.uint8)
        refused(lambda: e.dlog_lookup(foreign, els))
        refused(lambda: e.decrypt(sk, cts, foreign))
        refused(lambda: e.combine_decrypt(list(USED), cts, shares, foreign))
    finally:
        foreign.close()
