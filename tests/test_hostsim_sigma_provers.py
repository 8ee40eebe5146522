"""The stand-alone sigma provers (eg_prove_commitment_equiv_batch*, eg_prove_sumsq_batch*, eg_prove_possession_batch*) on the
CPU-compiled library (TEST HARNESS ONLY, tests/hostsim): the reference snapshots regenerated, byte parity with the oracle in
both randomness forms and both prover modes, acceptance and rejection by both verifiers, the edges, the argument errors, and
chunking and multi-device sharding giving the same bytes."""
import pytest

import sigma_prover_common as S
import workloads as W
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build


@pytest.fixture(scope="module")
def e():
    eng = Engine(lib_path=build())
    yield eng
    eng.close()


@pytest.fixture(params=[False, True], ids=["default", "constant_time"])
def mode(request, e):
    e.set_prover_mode(request.param)
    yield request.param
    e.set_prover_mode(False)


def test_commitment_equiv_snapshot_regenerated(e, mode):
    S.check_commitment_equiv_snapshot(e)


def test_sumsq_snapshot_regenerated(e, mode):
    S.check_sumsq_snapshot(e)


def test_commitment_equiv_matches_oracle_and_verifies(e, mode):
    S.check_ceq_parity(e, W.receiver()[1])


@pytest.mark.parametrize("k", [1, 5, 64])
def test_possession_matches_oracle_and_verifies(e, mode, k):
    S.check_pop_parity(e, k, n=3 if k == 64 else 5)


@pytest.mark.parametrize("count", [1, 5, 15])
def test_sumsq_matches_oracle_and_verifies(e, mode, count):
    S.check_sumsq_parity(e, W.receiver()[1], count, n=3)


def test_sumsq_values_whose_squares_exceed_u64(e, mode):
    S.check_sumsq_parity(e, W.receiver()[1], 4, n=3, big=True)


def test_sumsq_inconsistent_items_are_rejected(e):
    S.check_sumsq_inconsistent(e, W.receiver()[1])


def test_zero_possession_secret(e, mode):
    S.check_zero_possession_secret(e)


def test_errors_leave_context_usable(e):
    S.check_errors_leave_context_usable(e, lambda: Engine(lib_path=build()), W.receiver()[1])


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


@pytest.mark.parametrize("children", [1, 3])
def test_multi_context_shards_to_the_same_bytes(e, children):
    pk = W.receiver()[1]
    ref = S.all_outputs(e, pk)
    m = Engine(lib_path=build(), devices=[0] * children)
    try:
        got = S.all_outputs(m, pk)
        S.check_errors_leave_context_usable(m, lambda: Engine(lib_path=build(), devices=[0] * children), pk)
    finally:
        m.close()
    assert all((a == b).all() for a, b in zip(ref, got))
