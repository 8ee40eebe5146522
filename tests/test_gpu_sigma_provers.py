"""`-m gpu`: the stand-alone sigma provers on the CUDA library -- the reference snapshots regenerated, oracle parity in both
randomness forms and both prover modes, the edges and argument errors, chunking invariance, 262 144 + 77 items of each kind
verified on the GPU (the first 64 byte-identical to the oracle), and multi-GPU sharding giving the bytes of one GPU."""
import numpy as np
import pytest

import oracle as O
import sigma_prover_common as S
import workloads as W

pytestmark = pytest.mark.gpu
N = (1 << 18) + 77


def gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
    yield eng
    eng.close()


@pytest.fixture(params=[False, True], ids=["default", "constant_time"])
def mode(request, e):
    e.set_prover_mode(request.param)
    yield request.param
    e.set_prover_mode(False)


def canonical(rnd, shape):
    """Uniform scalars below 2^252 (< l): canonical."""
    s = rnd.integers(0, 256, size=shape + (32,), dtype=np.uint8)
    s[..., 31] &= 0x0F
    return s


def test_snapshots_regenerated(e, mode):
    S.check_commitment_equiv_snapshot(e)
    S.check_sumsq_snapshot(e)


def test_parity_with_oracle(e, mode):
    pk = W.receiver()[1]
    S.check_ceq_parity(e, pk)
    for k in (1, 5, 64):
        S.check_pop_parity(e, k, n=3)
    for count in (1, 5, 15):
        S.check_sumsq_parity(e, pk, count, n=3)
    S.check_sumsq_parity(e, pk, 4, n=3, big=True)
    S.check_zero_possession_secret(e)


def test_edges_and_errors(e):
    from elastic_elgamal_b200 import Engine
    pk = W.receiver()[1]
    S.check_sumsq_inconsistent(e, pk)
    S.check_errors_leave_context_usable(e, lambda: Engine(device=0), pk)


def test_chunking_and_modes_give_the_same_bytes(e):
    pk = W.receiver()[1]
    ref = S.all_outputs(e, pk)
    e.set_chunk_items(3)
    try:
        chunked = S.all_outputs(e, pk)
    finally:
        e.set_chunk_items(0)
    e.set_prover_mode(True)
    try:
        ct = S.all_outputs(e, pk)
    finally:
        e.set_prover_mode(False)
    assert all((a == b).all() and (a == c).all() for a, b, c in zip(ref, chunked, ct))


def test_commitment_equiv_at_size(e):
    pk = W.receiver()[1]
    e.set_receiver(pk)
    e.set_blinding_base(S.BB)
    rnd = np.random.default_rng(11)
    values = rnd.integers(0, 1 << 63, size=N, dtype=np.uint64) * 2
    values[:9] = S.ceq_values(9)
    ct_r = canonical(rnd, (N,))
    ct_r[:64] = S.ceq_inputs(64)[1]
    cts, coms, proofs, blind = e.prove_commitment_equiv("size", values, ct_r, seed=S.SEED, counter_base=1)
    assert (e.verify_commitment_equiv("size", cts, coms, proofs) == O.OK).all()
    ocs, ocoms, oproofs = O.gen_ceq_batch(pk, S.BB, "size", S.SEED, values[:64])
    assert (cts[:64] == ocs).all() and (coms[:64] == ocoms).all() and (proofs[:64] == oproofs).all()
    for i in range(0, N, 4099):      # the re-encryption is ([r]G, [v]G + [r]K); C opens to [v]G + [b]H
        assert bytes(cts[i]) == S.enc_with(pk, S.sc(int(values[i])), bytes(ct_r[i]))
        assert bytes(coms[i]) == O.point_add(O.point_mul_generator(S.sc(int(values[i]))), O.point_mul(bytes(blind[i]), S.BB))


def test_possession_at_size(e):
    k = 5
    rnd = np.random.default_rng(12)
    secrets = canonical(rnd, (N, k))
    secrets[:64] = S.pop_secrets(64, k)
    keys, proofs = e.prove_possession("size", secrets, seed=S.SEED, counter_base=k)
    assert (e.verify_possession("size", keys, proofs) == O.OK).all()
    okeys, oproofs = O.gen_pop_batch(k, "size", S.SEED, 64)
    assert (keys[:64] == okeys).all() and (proofs[:64] == oproofs).all()


def test_sumsq_at_size(e):
    pk = W.receiver()[1]
    e.set_receiver(pk)
    m = 5
    rnd = np.random.default_rng(13)
    values = rnd.integers(0, 1 << 16, size=(N, m), dtype=np.uint64)
    r = canonical(rnd, (N, m))
    sum_r = canonical(rnd, (N,))
    pad = lambda s: np.concatenate([s.reshape(-1, 32), np.zeros_like(s.reshape(-1, 32))], axis=1)   # block = r || 0 reduces to r
    cts = e.encrypt(values.reshape(-1), pad(r)).reshape(N, m, 64)
    sum_cts = e.encrypt((values * values).sum(axis=1), pad(sum_r))
    proofs = e.prove_sumsq("size", cts, values, r, sum_cts, sum_r, seed=S.SEED, counter_base=3)
    assert (e.verify_sumsq("size", cts, sum_cts, proofs) == O.OK).all()
    inst = (cts[:64], values[:64], r[:64], sum_cts[:64], sum_r[:64])
    assert (proofs[:64] == S.oracle_sumsq(pk, inst, "size", 3)).all()


def test_two_gpus_match_one_gpu(e):
    if gpu_count() < 2:
        pytest.skip(f"needs 2 GPUs, {gpu_count()} visible")
    from elastic_elgamal_b200 import Engine
    pk = W.receiver()[1]
    ref = S.all_outputs(e, pk)
    m = Engine(devices=[0, 1])
    try:
        got = S.all_outputs(m, pk)
    finally:
        m.close()
    assert all((a == b).all() for a, b in zip(ref, got))
