"""`-m gpu`: edge randomness on the encryption side on the CUDA library -- encrypt, encrypt_zero, encrypt_bool,
EncryptedChoice::new (single and multi), RangeProof::new / from_ciphertext and QuadraticVotingBallot::new on caller blocks that
put every scalar edge of encrypt_edge_common.py into each role, byte for byte against the oracle replaying the same blocks, in
both prover modes and in a chunked run with a remainder, verified in every ring mode (batches of many warps, so that
k_ring_pair pairs and k_terminal run in full warps next to ordinary items)."""
import pytest

import encrypt_edge_common as EE

pytestmark = pytest.mark.gpu

PROVERS = EE.provers(qv=(5, 20), range_bounds=(21, 100)) + [EE.Choice(5, True), EE.Choice(4, False), EE.QV(3, 9)]


@pytest.fixture(scope="module")
def env():
    import workloads as W
    from elastic_elgamal_b200 import Engine
    e = Engine(device=0)
    sk, pk = W.receiver()
    e.set_receiver(pk)
    yield e, sk, pk
    e.close()


def test_edge_lists_hit_their_patterns():
    EE.check_edge_lists_hit_their_patterns()


@pytest.mark.parametrize("P", PROVERS, ids=[P.name for P in PROVERS])
def test_draw_maps(env, P):
    EE.check_draw_maps(P, env[2])


@pytest.mark.parametrize("P", PROVERS, ids=[P.name for P in PROVERS])
def test_prover_edges(env, P):
    e, sk, pk = env
    items, wide = EE.all_cases(P, pk)
    assert len(items) > 64
    EE.check_prover_edges(e, sk, pk, P, items, wide, chunk=97)
