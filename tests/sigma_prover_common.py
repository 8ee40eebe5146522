"""Checks of the stand-alone sigma provers (eg_prove_commitment_equiv_batch*, eg_prove_sumsq_batch*,
eg_prove_possession_batch*) shared by the CPU harness tests (test_hostsim_sigma_provers.py) and the `-m gpu` tests
(test_gpu_sigma_provers.py): the reference snapshots regenerated, byte parity with the oracle's provers on the same ChaCha20
streams in both randomness forms, acceptance and rejection by the library's and the oracle's verifiers, the edges of the
value ranges and the argument errors."""
import json
import pathlib

import numpy as np

import oracle as O
import parity_common as PC
import workloads as W

SEED = bytes([0x2a] * 32)
SEED_R = bytes([0x17] * 32)          # ciphertext randomness of the sum-of-squares instances
LABEL = "test"
BB = PC.BLINDING_BASE
U64_MAX = (1 << 64) - 1
L = W.L


def gold(name):
    return json.loads((pathlib.Path(__file__).parent / "golden" / "ristretto_snapshots.json").read_text())[name]


def blocks(seed, first, count):
    rng = O.rng_from_seed(seed, first_block=first)
    return b"".join(O.rng_block(rng) for _ in range(count))


def item_wide(seed, counter_base, n, draws):
    """The caller-supplied form of the seeded draws: item i's blocks counter_base + (i << 20) + k."""
    return np.frombuffer(b"".join(blocks(seed, counter_base + (i << 20), draws) for i in range(n)), np.uint8).reshape(n, draws, 64).copy()


def reduced(seed, counter):
    return O.scalar_reduce_wide(blocks(seed, counter, 1))


def sc(v):
    return (v % L).to_bytes(32, "little")


def enc_with(pk, value_scalar, r):
    """([r]G, [v]G + [r]K) for a scalar value v (CiphertextWithValue arithmetic)."""
    return O.point_mul_generator(r) + O.point_add(O.point_mul_generator(value_scalar), O.point_mul(r, pk))


def as_np(rows, *shape):
    return np.frombuffer(b"".join(rows), np.uint8).reshape(*shape).copy()


def status(fn):
    from elastic_elgamal_b200 import EngineError, _ffi
    try:
        fn()
    except EngineError as err:
        return err.status
    return _ffi.SUCCESS


# ---------------------------------------------------------------- reference snapshots

def check_commitment_equiv_snapshot(e):
    """tests/snapshots.rs:163-189: key of seed_from_u64(12345) (block 0), value 123, r = block 1, then b, e_r, e_v, e_c."""
    g = gold("commitment-equiv-proof")
    rng = O.rng_from_u64(12345)
    key = bytes(rng.key)
    sk, pk = O.keypair(rng)
    e.set_receiver(pk)
    e.set_blinding_base(BB)
    r = reduced(key, 1)
    cts, coms, proofs, blind = e.prove_commitment_equiv(LABEL, [123], as_np([r], 1, 32), seed=key, counter_base=2)
    ct = bytes.fromhex(g["ciphertext"]["random_element"]) + bytes.fromhex(g["ciphertext"]["blinded_element"])
    proof = b"".join(bytes.fromhex(g["proof"][k]) for k in ("challenge", "randomness_response", "value_response", "commitment_response"))
    assert bytes(cts[0]) == ct and bytes(coms[0]) == bytes.fromhex(g["commitment"]) and bytes(proofs[0]) == proof
    _, _, _, oblind = O.commitment_equiv_prove(pk, 123, BB, LABEL, rng)
    assert bytes(blind[0]) == oblind
    got = e.prove_commitment_equiv(LABEL, [123], as_np([r], 1, 32), np.frombuffer(blocks(key, 2, 4), np.uint8))
    assert all((a == b).all() for a, b in zip(got, (cts, coms, proofs, blind)))


def check_sumsq_snapshot(e):
    """tests/snapshots.rs:132-151: values [1, 3, 3, 7, 5]; the sum ciphertext's r = block 1, the ciphertexts' r = blocks 2-6,
    the proof's draws from block 7."""
    g = gold("sum-sq-proof")
    rng = O.rng_from_u64(12345)
    key = bytes(rng.key)
    sk, pk = O.keypair(rng)
    e.set_receiver(pk)
    values = [1, 3, 3, 7, 5]
    sum_r = reduced(key, 1)
    rs = [reduced(key, 2 + j) for j in range(5)]
    cts = [enc_with(pk, sc(v), r) for v, r in zip(values, rs)]
    sum_ct = enc_with(pk, sc(sum(v * v for v in values)), sum_r)
    assert cts[0] == O.encrypt(pk, 1, O.rng_from_seed(key, first_block=2))
    args = (LABEL, as_np(cts, 1, 5, 64), [values], as_np(rs, 1, 5, 32), as_np([sum_ct], 1, 64), as_np([sum_r], 1, 32))
    proofs = e.prove_sumsq(*args, seed=key, counter_base=7)
    hx = bytes.fromhex
    assert bytes(proofs[0]) == hx(g["challenge"]) + b"".join(hx(x) for x in g["ciphertext_responses"]) + hx(g["sum_response"])
    assert (e.prove_sumsq(*args, np.frombuffer(blocks(key, 7, 11), np.uint8)) == proofs).all()


# ---------------------------------------------------------------- oracle parity

def ceq_values(n):
    vals = [(977 * i + 5) % 100000 for i in range(n)]
    vals[0], vals[-1] = 0, U64_MAX
    if n > 3:
        vals[2] = U64_MAX - 1
    return np.array(vals, np.uint64)


def ceq_inputs(n):
    values = ceq_values(n)
    ct_r = as_np([reduced(SEED, i << 20) for i in range(n)], n, 32)
    return values, ct_r


def check_ceq_parity(e, pk, n=9, label="ceq"):
    """Seeded (counter_base = 1, ct randomness = block i << 20) and blocks forms equal eo_gen_ceq_batch byte for byte,
    blindings included; the commitment opens to [v]G + [b]H; both verifiers accept; tampering is rejected."""
    e.set_receiver(pk)
    e.set_blinding_base(BB)
    values, ct_r = ceq_inputs(n)
    ocs, ocoms, oproofs = O.gen_ceq_batch(pk, BB, label, SEED, values)
    oblind = [O.commitment_equiv_prove(pk, int(values[i]), BB, label, O.rng_from_seed(SEED, first_block=i << 20))[3] for i in range(n)]
    cts, coms, proofs, blind = e.prove_commitment_equiv(label, values, ct_r, seed=SEED, counter_base=1)
    assert (cts == ocs).all() and (coms == ocoms).all() and (proofs == oproofs).all()
    assert [bytes(b) for b in blind] == oblind
    got = e.prove_commitment_equiv(label, values, ct_r, item_wide(SEED, 1, n, 4))
    assert all((a == b).all() for a, b in zip(got, (cts, coms, proofs, blind)))
    none, coms2, proofs2, _ = e.prove_commitment_equiv(label, values, ct_r, seed=SEED, counter_base=1, want_cts=False)
    assert none is None and (coms2 == coms).all() and (proofs2 == proofs).all()
    for i in range(n):        # C = [v]G + [b]H
        assert bytes(coms[i]) == O.point_add(O.point_mul_generator(sc(int(values[i]))), O.point_mul(bytes(blind[i]), BB))
    assert (e.verify_commitment_equiv(label, cts, coms, proofs) == O.OK).all()
    assert (O.verify_ceq_batch(pk, BB, label, cts, coms, proofs) == O.OK).all()
    bad_p, bad_c = proofs.copy(), coms.copy()
    bad_p[1, 32:64], bad_p[1, 64:96] = proofs[1, 64:96], proofs[1, 32:64]        # swapped responses
    bad_c[3] = np.frombuffer(O.point_add(bytes(coms[3]), W.G_ENC), np.uint8)      # C + G
    for lbl, c_, p_ in ((label, coms, bad_p), (label, bad_c, proofs)):
        want = O.verify_ceq_batch(pk, BB, lbl, cts, c_, p_)
        assert e.verify_commitment_equiv(lbl, cts, c_, p_).tolist() == want.tolist()
        assert (want != O.OK).sum() == 1
    assert not (e.verify_commitment_equiv(label + "x", cts, coms, proofs) == O.OK).any()
    assert not (O.verify_ceq_batch(pk, BB, label + "x", cts, coms, proofs) == O.OK).any()


def pop_secrets(n, k, seed=SEED):
    return as_np([reduced(seed, (i << 20) + j) for i in range(n) for j in range(k)], n, k, 32)


def check_pop_parity(e, k, n=5, label="pop"):
    """Secrets = blocks (i << 20) + j, nonces from counter_base = k: the keys and proofs of eo_gen_pop_batch, in both forms."""
    okeys, oproofs = O.gen_pop_batch(k, label, SEED, n)
    secrets = pop_secrets(n, k)
    keys, proofs = e.prove_possession(label, secrets, seed=SEED, counter_base=k)
    assert (keys == okeys).all() and (proofs == oproofs).all()
    keys2, proofs2 = e.prove_possession(label, secrets, item_wide(SEED, k, n, k))
    assert (keys2 == keys).all() and (proofs2 == proofs).all()
    assert (e.verify_possession(label, keys, proofs) == O.OK).all()
    assert (O.verify_pop_batch(label, keys, proofs) == O.OK).all()
    bad = proofs.copy()
    if k > 1:
        bad[0, 1], bad[0, 2] = proofs[0, 2], proofs[0, 1]          # swapped responses
    else:
        bad[0, 1] = proofs[1, 1]
    want = O.verify_pop_batch(label, keys, bad)
    assert want[0] == O.CHALLENGE_MISMATCH and e.verify_possession(label, keys, bad).tolist() == want.tolist()
    assert not (e.verify_possession(label + "x", keys, proofs) == O.OK).any()
    assert not (O.verify_pop_batch(label + "x", keys, proofs) == O.OK).any()


def sumsq_instances(pk, n, m, big=False, first=0):
    """n items of m ciphertexts; the sum ciphertext is built by scalar arithmetic (squares may exceed u64)."""
    rnd = np.random.default_rng(1000 * m + n + first)
    if big:
        values = rnd.integers(0, 1 << 63, size=(n, m), dtype=np.uint64) * 2 + 1
        values[0, 0] = U64_MAX
        values[-1, -1] = 0
    else:
        values = rnd.integers(0, 50, size=(n, m), dtype=np.uint64)
    rs = [[reduced(SEED_R, ((first + i) << 20) + j) for j in range(m)] for i in range(n)]
    sum_r = [reduced(SEED_R, ((first + i) << 20) + m) for i in range(n)]
    cts = [[enc_with(pk, sc(int(values[i, j])), rs[i][j]) for j in range(m)] for i in range(n)]
    sums = [sc(sum(int(v) ** 2 for v in values[i])) for i in range(n)]
    sum_cts = [enc_with(pk, sums[i], sum_r[i]) for i in range(n)]
    return (as_np([c for row in cts for c in row], n, m, 64), values, as_np([r for row in rs for r in row], n, m, 32),
            as_np(sum_cts, n, 64), as_np(sum_r, n, 32))


def oracle_sumsq(pk, inst, label, counter_base, first=0):
    cts, values, rs, sum_cts, sum_r = inst
    n, m = values.shape
    rows = [O.sumsq_prove(pk, [bytes(c) for c in cts[i]], [sc(int(v)) for v in values[i]], [bytes(r) for r in rs[i]],
                          bytes(sum_cts[i]), bytes(sum_r[i]), label, O.rng_from_seed(SEED, first_block=((first + i) << 20) + counter_base))
            for i in range(n)]
    return as_np(rows, n, 2 * m + 2, 32)


def check_sumsq_parity(e, pk, m, n=4, big=False, label="sumsq"):
    e.set_receiver(pk)
    inst = sumsq_instances(pk, n, m, big)
    cts, values, rs, sum_cts, sum_r = inst
    proofs = e.prove_sumsq(label, cts, values, rs, sum_cts, sum_r, seed=SEED, counter_base=3)
    assert (proofs == oracle_sumsq(pk, inst, label, 3)).all()
    assert (e.prove_sumsq(label, cts, values, rs, sum_cts, sum_r, item_wide(SEED, 3, n, 1 + 2 * m)) == proofs).all()
    assert (e.verify_sumsq(label, cts, sum_cts, proofs) == O.OK).all()
    assert all(O.sumsq_verify(pk, [bytes(c) for c in cts[i]], bytes(sum_cts[i]), label, bytes(proofs[i])) == O.OK for i in range(n))
    bad = proofs.copy()
    bad[0, 1], bad[0, 2] = proofs[0, 2], proofs[0, 1]
    assert e.verify_sumsq(label, cts, sum_cts, bad)[0] == O.CHALLENGE_MISMATCH
    assert O.sumsq_verify(pk, [bytes(c) for c in cts[0]], bytes(sum_cts[0]), label, bytes(bad[0])) == O.CHALLENGE_MISMATCH
    assert not (e.verify_sumsq(label + "x", cts, sum_cts, proofs) == O.OK).any()


def check_sumsq_inconsistent(e, pk, m=3, n=4, label="sumsq"):
    """The prover does not check its inputs (as mul.rs:107-181): an item whose sum ciphertext does not encrypt the sum of
    squares -- or whose ciphertext does not match its value -- gets a proof that both verifiers reject; the others verify."""
    e.set_receiver(pk)
    cts, values, rs, sum_cts, sum_r = sumsq_instances(pk, n, m)
    s1 = sum(int(v) ** 2 for v in values[1]) + 1
    sum_cts[1] = np.frombuffer(enc_with(pk, sc(s1), bytes(sum_r[1])), np.uint8)
    values2 = values.copy()
    values2[2, 0] += 1                                            # ciphertext 0 of item 2 does not encrypt this value
    proofs = e.prove_sumsq(label, cts, values2, rs, sum_cts, sum_r, seed=SEED)
    got = e.verify_sumsq(label, cts, sum_cts, proofs)
    want = [O.sumsq_verify(pk, [bytes(c) for c in cts[i]], bytes(sum_cts[i]), label, bytes(proofs[i])) for i in range(n)]
    assert got.tolist() == want and want[0] == O.OK and want[3] == O.OK
    assert want[1] == O.CHALLENGE_MISMATCH and want[2] == O.CHALLENGE_MISMATCH


def check_zero_possession_secret(e, label="pop"):
    """A zero secret: the identity as its key (the oracle's keypair of 0) and a proof the verifiers refuse as malformed."""
    k, n = 3, 2
    secrets = pop_secrets(n, k)
    secrets[1, 1] = 0
    keys, proofs = e.prove_possession(label, secrets, seed=SEED, counter_base=k)
    assert (keys[1, 1] == 0).all()
    for i in range(n):
        okeys = [O.point_mul_generator(bytes(s)) for s in secrets[i]]
        assert [bytes(x) for x in keys[i]] == okeys
        oproof = O.pop_prove([bytes(s) for s in secrets[i]], okeys, label, O.rng_from_seed(SEED, first_block=(i << 20) + k))
        assert bytes(proofs[i]) == oproof
    want = O.verify_pop_batch(label, keys, proofs)
    assert want.tolist() == [O.OK, O.MALFORMED] and e.verify_possession(label, keys, proofs).tolist() == want.tolist()


# ---------------------------------------------------------------- errors

def check_errors_leave_context_usable(e, new_engine, pk):
    """Refused shapes, non-canonical scalars, a missing blinding base or receiver, bad labels, null pointers: each reported as
    the header says, and the next call on the same context gives the same bytes as before.  n = 0 is a no-op."""
    from elastic_elgamal_b200 import _ffi
    e.set_receiver(pk)
    e.set_blinding_base(BB)
    values, ct_r = ceq_inputs(3)
    inst = sumsq_instances(pk, 2, 2)
    secrets = pop_secrets(2, 2)
    ref = (e.prove_commitment_equiv("x", values, ct_r, seed=SEED), e.prove_sumsq("x", *inst, seed=SEED),
           e.prove_possession("x", secrets, seed=SEED))

    def again():
        got = (e.prove_commitment_equiv("x", values, ct_r, seed=SEED), e.prove_sumsq("x", *inst, seed=SEED),
               e.prove_possession("x", secrets, seed=SEED))
        assert all((a == b).all() for a, b in zip(ref[0], got[0])) and (got[1] == ref[1]).all()
        assert all((a == b).all() for a, b in zip(ref[2], got[2]))

    cts, vals, rs, sum_cts, sum_r = inst
    bad_r = ct_r.copy()
    bad_r[1] = np.frombuffer(W.BAD_SCALAR, np.uint8)
    bad_rs, bad_sr = rs.copy(), sum_r.copy()
    bad_rs[1, 1] = np.frombuffer(W.BAD_SCALAR2, np.uint8)
    bad_sr[0] = np.frombuffer(W.BAD_SCALAR, np.uint8)
    bad_sec = secrets.copy()
    bad_sec[1, 0] = np.frombuffer(W.BAD_SCALAR2, np.uint8)
    cts16 = np.zeros((1, 16, 64), np.uint8)
    z16 = np.zeros((1, 16, 32), np.uint8)
    cases = [
        (lambda: e.prove_commitment_equiv("x", values, bad_r, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_sumsq("x", cts, vals, bad_rs, sum_cts, sum_r, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_sumsq("x", cts, vals, rs, sum_cts, bad_sr, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_possession("x", bad_sec, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_sumsq("x", cts16, np.zeros((1, 16)), z16, cts16[:, 0], z16[:, 0], seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_sumsq("x", cts16[:, :0], np.zeros((1, 0)), z16[:, :0], cts16[:, 0], z16[:, 0], seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_possession("x", np.zeros((1, 65, 32), np.uint8), seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_possession("x", np.zeros((1, 0, 32), np.uint8), seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_commitment_equiv("", values, ct_r, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_sumsq("y" * 256, *inst, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e.prove_possession("", secrets, seed=SEED), _ffi.ERR_INVALID_ARG),
        (lambda: e._check(e.lib.eg_prove_commitment_equiv_batch(e.h, b"x", 3, values.ctypes.data, ct_r.ctypes.data, None, None, None,
                                                                None, None)), _ffi.ERR_INVALID_ARG),
        (lambda: e._check(e.lib.eg_prove_commitment_equiv_batch_seeded(e.h, b"x", 3, values.ctypes.data, ct_r.ctypes.data, None, 0,
                                                                       None, None, None, None)), _ffi.ERR_INVALID_ARG),
        (lambda: e._check(e.lib.eg_prove_sumsq_batch_seeded(e.h, b"x", 2, 2, cts.ctypes.data, None, rs.ctypes.data, sum_cts.ctypes.data,
                                                            sum_r.ctypes.data, SEED, 0, None)), _ffi.ERR_INVALID_ARG),
        (lambda: e._check(e.lib.eg_prove_possession_batch(e.h, b"x", 2, 2, secrets.ctypes.data, None, None, None)), _ffi.ERR_INVALID_ARG),
    ]
    for fn, want in cases:
        assert status(fn) == want
        again()
    # n = 0 with null buffers: a successful no-op
    assert e.lib.eg_prove_commitment_equiv_batch(e.h, b"x", 0, None, None, None, None, None, None, None) == 0
    assert e.lib.eg_prove_commitment_equiv_batch_seeded(e.h, b"x", 0, None, None, SEED, 0, None, None, None, None) == 0
    assert e.lib.eg_prove_sumsq_batch(e.h, b"x", 3, 0, None, None, None, None, None, None, None) == 0
    assert e.lib.eg_prove_sumsq_batch_seeded(e.h, b"x", 3, 0, None, None, None, None, None, SEED, 0, None) == 0
    assert e.lib.eg_prove_possession_batch(e.h, b"x", 3, 0, None, None, None, None) == 0
    assert e.lib.eg_prove_possession_batch_seeded(e.h, b"x", 3, 0, None, SEED, 0, None, None) == 0
    again()
    # a context without a receiver key / without a blinding base
    f = new_engine()
    try:
        assert status(lambda: f.prove_commitment_equiv("x", values, ct_r, seed=SEED)) == _ffi.ERR_NO_RECEIVER
        assert status(lambda: f.prove_sumsq("x", *inst, seed=SEED)) == _ffi.ERR_NO_RECEIVER
        got = f.prove_possession("x", secrets, seed=SEED)                   # needs no receiver
        assert all((a == b).all() for a, b in zip(ref[2], got))
        f.set_receiver(pk)
        assert status(lambda: f.prove_commitment_equiv("x", values, ct_r, seed=SEED)) == _ffi.ERR_NO_RECEIVER
        assert "blinding" in f.lib.eg_last_error(f.h).decode()
        assert (f.prove_sumsq("x", *inst, seed=SEED) == ref[1]).all()
        f.set_blinding_base(BB)
        got = f.prove_commitment_equiv("x", values, ct_r, seed=SEED)
        assert all((a == b).all() for a, b in zip(ref[0], got))
    finally:
        f.close()


# ---------------------------------------------------------------- invariance

def all_outputs(e, pk):
    """Every output of the three provers on one seeded workload (for comparisons across contexts, chunkings and modes)."""
    e.set_receiver(pk)
    e.set_blinding_base(BB)
    n = 8
    values, ct_r = ceq_inputs(n)
    out = list(e.prove_commitment_equiv("inv", values, ct_r, seed=SEED, counter_base=1))
    out += list(e.prove_commitment_equiv("inv", values, ct_r, item_wide(SEED, 5, n, 4)))
    inst = sumsq_instances(pk, 7, 3, big=True)
    out.append(e.prove_sumsq("inv", *inst, seed=SEED, counter_base=2))
    out.append(e.prove_sumsq("inv", *inst, item_wide(SEED, 9, 7, 7)))
    secrets = pop_secrets(7, 4)
    out += list(e.prove_possession("inv", secrets, seed=SEED, counter_base=3))
    out += list(e.prove_possession("inv", secrets, item_wide(SEED, 3, 7, 4)))
    return out
