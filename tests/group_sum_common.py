"""eg_ciphertexts_group_sum (the tally fold per group id), shared by the CPU harness tests (test_hostsim_group_sum.py) and the
`-m gpu` tests (test_gpu_group_sum.py).  Every check compares bytes.

Elements are [x]G with known x (weighted_sum_common.corpus), so each group's total is also [sum x]G: small groups are
checked against a fold of the oracle's point_add, larger ones against that one fixed-base product.  Empty groups and groups
with a bad included element are the identity."""
import random

import numpy as np
import pytest

import oracle as O
import weighted_sum_common as WS
import workloads as W

L = W.L
IDENTITY = WS.IDENTITY
MAX_CELLS = 1 << 22
DISTRIBUTIONS = ["one", "own", "uniform", "zipf", "last"]


def group_ids(n, n_groups, kind, seed=0):
    """n group ids below n_groups: all in one group, each item in its own group (n_groups >= n), uniform, Zipf-like (group
    k drawn with weight 1 / (k + 1), over a shuffled order of the groups) or only the last id."""
    rnd = random.Random(seed * 7919 + n * 31 + n_groups)
    if kind == "one":
        g = [rnd.randrange(n_groups)] * n
    elif kind == "own":
        assert n_groups >= n
        g = rnd.sample(range(n_groups), n)
    elif kind == "uniform":
        g = [rnd.randrange(n_groups) for _ in range(n)]
    elif kind == "zipf":
        order = list(range(n_groups))
        rnd.shuffle(order)
        w = np.cumsum(1.0 / np.arange(1, n_groups + 1))
        g = [order[int(k)] for k in np.searchsorted(w, np.array([rnd.random() for _ in range(n)]) * w[-1], side="right").clip(0, n_groups - 1)]
    elif kind == "last":
        g = [n_groups - 1] * n
    else:
        raise ValueError(kind)
    return np.array(g, np.uint32)


def expected(cts, logs, groups, n_groups, mask=None, fold=None):
    """(out (n_groups, n_cts, 64), ok) of the included items by group: the oracle's point_add fold (small groups) or
    [sum x]G; logs=None: always the fold."""
    n, n_cts = cts.shape[0], cts.shape[1]
    members = {}
    for i in range(n):
        if mask is None or mask[i] == 0:
            members.setdefault(int(groups[i]), []).append(i)
    out = np.zeros((n_groups, n_cts, 64), np.uint8)
    for g, inc in members.items():
        f = fold if fold is not None else (logs is None or len(inc) <= 8)
        for col in range(2 * n_cts):
            h = 32 * (col % 2)
            if f:
                acc = IDENTITY
                for i in inc:
                    acc = O.point_add(acc, bytes(cts[i, col // 2, h:h + 32]))
            else:
                acc = O.point_mul_generator(WS.sc(sum(logs[i][col] for i in inc)))
            out[g, col // 2, h:h + 32] = np.frombuffer(acc, np.uint8)
    return out, np.ones(n_groups, bool)


def check(e, cts, logs, groups, n_groups, mask=None, what=""):
    out, ok = e.group_sum(cts, groups, n_groups, mask)
    want, want_ok = expected(cts, logs, groups, n_groups, mask)
    assert out.shape == (n_groups, cts.shape[1], 64) and ok.shape == (n_groups,), what
    assert ok.all(), what
    bad = [g for g in range(n_groups) if not (out[g] == want[g]).all()]
    assert not bad, f"{what}: groups {bad[:8]} differ from the oracle"
    return out


# ---------------------------------------------------------------- 1. oracle parity and group-size distributions

def check_parity(e, n, n_cts, n_groups, kind="uniform"):
    cts, logs = WS.corpus(n, n_cts)
    check(e, cts, logs, group_ids(n, n_groups, kind), n_groups, what=f"n={n} n_cts={n_cts} n_groups={n_groups} {kind}")


def check_distribution(e, n, n_cts, kind):
    n_groups = {"one": 3, "own": n + 5, "uniform": 37, "zipf": 200, "last": 50}[kind]
    cts, logs = WS.corpus(n, n_cts)
    groups = group_ids(n, n_groups, kind, seed=1)
    mask = np.array([i % 9 == 4 for i in range(n)], np.uint8)
    check(e, cts, logs, groups, n_groups, what=f"{kind} n={n}")
    check(e, cts, logs, groups, n_groups, mask, what=f"{kind} n={n} masked")


# ---------------------------------------------------------------- 2. consistency with the other folds

def check_single_group_is_weighted_sum(e, n, n_cts):
    cts, logs = WS.corpus(n, n_cts)
    mask = np.array([i % 4 == 1 for i in range(n)], np.uint8)
    for m in (None, mask):
        out, ok = e.group_sum(cts, np.zeros(n, np.uint32), 1, m)
        ws, ws_ok = e.weighted_sum(cts, np.ones(n, np.uint64), m)
        assert ok.all() and ws_ok and (out[0] == ws).all(), "n_groups = 1 differs from the unit-weight weighted sum"


def _sum_groups(e, out):
    total, ok = e.ciphertexts_sum(out)
    assert ok
    return total


def check_choice_mask(e, n=64, m=5, n_groups=7):
    sk, pk = W.receiver()
    e.set_receiver(pk)
    cts, rings, sums = O.gen_choice_batch(pk, m, W.SEED_CHOICE, n)
    cts, rings, sums = cts.copy(), rings.copy(), sums.copy()
    W.tamper_choice(cts, rings, sums, random.Random(5), frac=0.2)
    v, t = e.verify_choice(m, cts, rings, sums)
    assert (v != 0).any() and (v == 0).any()
    groups = group_ids(n, n_groups, "zipf", seed=2)
    out, ok = e.group_sum(cts, groups, n_groups, v)
    assert ok.all()
    want, _ = expected(cts, None, groups, n_groups, v)
    assert (out == want).all()
    assert (_sum_groups(e, out) == t).all(), "the group totals do not add up to eg_verify_choice_batch's tally"


def check_qv_mask(e, n=24, options=3, credits=10, n_groups=5):
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
    groups = group_ids(n, n_groups, "uniform", seed=3)
    out, ok = e.group_sum(ballots, groups, n_groups, v, ct_stride=WS.qv_record(p), n_cts=options)
    assert ok.all() and out.shape == (n_groups, options, 64)
    assert (_sum_groups(e, out) == t).all(), "the group totals do not add up to eg_verify_qv_batch's tally"
    for g in range(n_groups):                        # each group equals the unit-weight weighted sum of its members
        sel = groups == g
        ws, ws_ok = e.weighted_sum(ballots[sel], np.ones(int(sel.sum()), np.uint64), v[sel], ct_stride=WS.qv_record(p), n_cts=options)
        assert ws_ok and (out[g] == ws).all(), f"group {g}"


# ---------------------------------------------------------------- 3. bad input

def check_bad_items(e, n=60, n_cts=2, n_groups=6):
    from elastic_elgamal_b200.engine import EngineError
    cts, logs = WS.corpus(n, n_cts)
    groups = group_ids(n, n_groups, "uniform", seed=4)
    want, _ = expected(cts, logs, groups, n_groups)
    bad = cts.copy()
    bad[3, 1, 32:] = np.frombuffer(W.BAD_POINT, np.uint8)
    g3 = int(groups[3])
    out, ok = e.group_sum(bad, groups, n_groups)
    assert not ok[g3] and not out[g3].any(), "a bad included element must give its group ok = 0 and the identity"
    others = [g for g in range(n_groups) if g != g3]
    assert ok[others].all() and (out[others] == want[others]).all(), "a bad element changed another group"
    mask = np.zeros(n, np.uint8)
    mask[3] = 1
    out, ok = e.group_sum(bad, groups, n_groups, mask)
    want_m, _ = expected(cts, logs, groups, n_groups, mask)
    assert ok.all() and (out == want_m).all(), "a bad excluded element changed the result"
    # an out-of-range group id: refused when the item is included, ignored when it is excluded
    for gid in (n_groups, n_groups + 1000, 2**32 - 1):
        g = groups.copy()
        g[5] = gid
        with pytest.raises(EngineError) as ex:
            e.group_sum(cts, g, n_groups)
        assert ex.value.status == 1
        mask = np.zeros(n, np.uint8)
        mask[5] = 2
        out, ok = e.group_sum(cts, g, n_groups, mask)
        want_m, _ = expected(cts, logs, g, n_groups, mask)
        assert ok.all() and (out == want_m).all(), "an excluded item's group id is not checked"
    out, ok = e.group_sum(cts, groups, n_groups)
    assert ok.all() and (out == want).all(), "the context changed after a refused call"
    out, ok = e.group_sum(cts, groups, n_groups, np.full(n, 1, np.uint8))
    assert ok.all() and not out.any(), "no included item: identity everywhere"
    out, ok = e.group_sum(cts[:0], groups[:0], n_groups)
    assert ok.all() and out.shape == (n_groups, n_cts, 64) and not out.any(), "n = 0: identity everywhere"


# ---------------------------------------------------------------- 4. call shapes

def check_chunks(e, n, n_cts, n_groups, chunks=(7, 0, 100)):
    cts, logs = WS.corpus(n, n_cts)
    groups = group_ids(n, n_groups, "zipf", seed=5)
    mask = np.array([0 if i % 7 else 1 for i in range(n)], np.uint8)
    want, _ = expected(cts, logs, groups, n_groups, mask)
    try:
        for chunk in chunks:
            e.set_chunk_items(chunk)
            out, ok = e.group_sum(cts, groups, n_groups, mask)
            assert ok.all() and (out == want).all(), f"chunk size {chunk}"
    finally:
        e.set_chunk_items(0)


def check_dev(e, dev, n=300, n_cts=2, n_groups=17, chunk=0):
    cts, logs = WS.corpus(n, n_cts)
    groups = group_ids(n, n_groups, "zipf", seed=6)
    mask = np.array([i % 5 == 2 for i in range(n)], np.uint8)
    bad = cts.copy()
    bad[8, 0, :32] = np.frombuffer(W.BAD_POINT, np.uint8)
    host, ok = e.group_sum(bad, groups, n_groups, mask)
    e.set_chunk_items(chunk)
    try:
        d_cts, d_g, d_v = dev.up(bad.reshape(n, -1)), dev.up(groups.view(np.uint8)), dev.up(mask)
        d_out, d_ok = dev.empty(n_groups * n_cts * 64, "uint8"), dev.empty(n_groups, "uint8")
        e.group_sum_dev(n, n_cts, 64 * n_cts, 64, dev.ptr(d_cts), dev.ptr(d_g), n_groups, dev.ptr(d_v), dev.ptr(d_out), dev.ptr(d_ok))
        assert (dev.down(d_ok) == ok).all() and (dev.down(d_out).reshape(n_groups, n_cts, 64) == host).all(), "host and _dev forms differ"
        assert not ok[groups[8]] if mask[8] == 0 else ok.all()
        d_cts = dev.up(cts.reshape(n, -1))
        e.group_sum_dev(n, n_cts, 64 * n_cts, 64, dev.ptr(d_cts), dev.ptr(d_g), n_groups, 0, dev.ptr(d_out), dev.ptr(d_ok))
        want, _ = expected(cts, logs, groups, n_groups)
        assert dev.down(d_ok).all() and (dev.down(d_out).reshape(n_groups, n_cts, 64) == want).all()
    finally:
        e.set_chunk_items(0)


def check_multi(m, e, n=100, n_cts=3, n_groups=9):
    cts, logs = WS.corpus(n, n_cts)
    groups = group_ids(n, n_groups, "zipf", seed=7)
    mask = np.array([i % 3 == 1 for i in range(n)], np.uint8)
    a, ok_a = m.group_sum(cts, groups, n_groups, mask)
    b, ok_b = e.group_sum(cts, groups, n_groups, mask)
    want, _ = expected(cts, logs, groups, n_groups, mask)
    assert ok_a.all() and ok_b.all() and (a == b).all() and (a == want).all()
    bad = cts.copy()
    bad[n - 1, 0, :32] = np.frombuffer(W.BAD_POINT, np.uint8)        # in the last device's shard
    a, ok_a = m.group_sum(bad, groups, n_groups)
    b, ok_b = e.group_sum(bad, groups, n_groups)
    gl = int(groups[n - 1])
    assert not ok_a[gl] and not a[gl].any() and (ok_a == ok_b).all() and (a == b).all()
    a, ok_a = m.group_sum(cts[:0], groups[:0], n_groups)
    assert ok_a.all() and not a.any()


# ---------------------------------------------------------------- 5. argument errors

def check_argument_errors(e, multi=None):
    from elastic_elgamal_b200 import _ffi
    cts, logs = WS.corpus(8, 2)
    groups = np.array([0, 1, 2, 0, 1, 2, 0, 1], np.uint32)
    want, _ = expected(cts, logs, groups, 3)
    out, ok = np.zeros(64 * 65 * 8, np.uint8), np.zeros(MAX_CELLS + 1, np.uint8)
    a = lambda x: None if x is None else x.ctypes.data
    calls = [
        (8, 2, 128, 64, cts, groups, 0, out, ok), (8, 1, 64, 64, cts, groups, MAX_CELLS + 1, out, ok),
        (8, 2, 128, 64, cts, groups, MAX_CELLS // 2 + 1, out, ok), (8, 64, 64 * 64, 64, cts, groups, MAX_CELLS // 64 + 1, out, ok),
        (8, 0, 128, 64, cts, groups, 3, out, ok), (8, 65, 65 * 64, 64, cts, groups, 3, out, ok),
        (8, 2, 128, 32, cts, groups, 3, out, ok), (8, 2, 127, 64, cts, groups, 3, out, ok), (8, 1, 63, 64, cts, groups, 3, out, ok),
        (8, 2, 128, 64, None, groups, 3, out, ok), (8, 2, 128, 64, cts, None, 3, out, ok), (8, 2, 128, 64, cts, groups, 3, None, ok),
        (8, 2, 128, 64, cts, groups, 3, out, None), (0, 2, 128, 64, None, None, 3, None, ok), (0, 2, 128, 64, None, None, 0, out, ok),
    ]
    for n, k, istr, cstr, c, g, ng, o, okb in calls:
        st = e.lib.eg_ciphertexts_group_sum(e.h, n, k, istr, cstr, a(c), a(g), ng, None, a(o), a(okb))
        assert st == _ffi.ERR_INVALID_ARG, (n, k, istr, cstr, ng)
        got, good = e.group_sum(cts, groups, 3)
        assert good.all() and (got == want).all(), "the context changed after a refused call"
    if multi is not None:
        st = multi.lib.eg_ciphertexts_group_sum_dev(multi.h, 8, 2, 128, 64, a(cts), a(groups), 3, None, a(out), a(ok))
        assert st == _ffi.ERR_INVALID_ARG
        got, good = multi.group_sum(cts, groups, 3)
        assert good.all() and (got == want).all()
