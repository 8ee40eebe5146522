"""The decryption side (eg_decrypt_batch, eg_decrypt_share_batch*, eg_prove_decryption_batch*) on the CPU-compiled library
(TEST HARNESS ONLY, tests/hostsim): byte parity with the oracle in both randomness forms and both prover modes, acceptance by
the library's verifiers, identity and undecodable ciphertexts, the argument errors, and sharding over multi-device contexts
with 1 and 3 children giving the bytes of a single context.  No receiver key is ever set: none of these operations needs one."""
import pytest

import decrypt_common as D
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


def test_decrypt_share_matches_oracle_and_verifies(e, mode):
    D.check_share_parity(e)


def test_prove_decryption_matches_oracle_and_verifies(e, mode):
    D.check_prove_decryption_parity(e)


def test_decrypt_matches_oracle_and_table(e, mode):
    D.check_plain_decrypt(e)


def test_undecodable_ciphertexts(e):
    D.check_undecodable_items(e)


def test_errors_leave_context_usable(e):
    D.check_errors_leave_context_usable(e)


def test_chunking_and_modes_give_the_same_bytes(e):
    ref = D.all_outputs(e)
    e.set_chunk_items(3)
    try:
        chunked = D.all_outputs(e)
    finally:
        e.set_chunk_items(0)
    e.set_prover_mode(True)
    try:
        ct = D.all_outputs(e)
    finally:
        e.set_prover_mode(False)
    assert all((a == b).all() and (a == c).all() for a, b, c in zip(ref, chunked, ct))


@pytest.mark.parametrize("children", [1, 3])
def test_multi_context_shards_to_the_same_bytes(e, children):
    ref = D.all_outputs(e)
    m = Engine(lib_path=build(), devices=[0] * children)
    try:
        got = D.all_outputs(m)
        D.check_errors_leave_context_usable(m)
    finally:
        m.close()
    assert all((a == b).all() for a, b in zip(ref, got))
