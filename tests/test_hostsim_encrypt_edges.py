"""Edge randomness on the encryption side on the CPU-compiled library (TEST HARNESS ONLY, tests/hostsim): encrypt,
encrypt_zero, encrypt_bool, EncryptedChoice::new, RangeProof::new / from_ciphertext and QuadraticVotingBallot::new on
caller blocks that put the scalar edges into each role (encrypt_edge_common.py), byte for byte against the oracle replaying
the same blocks, in both prover modes, verified in every ring mode."""
import ctypes as C

import pytest

import encrypt_edge_common as EE
import oracle as O
import parity_common as PC
import workloads as W
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build

PROVERS = EE.provers(qv=(2, 5), range_bounds=(21,))


@pytest.fixture(scope="module")
def env():
    e = Engine(lib_path=build())
    sk, pk = W.receiver()
    e.set_receiver(pk)
    yield e, sk, pk
    e.close()


def test_edge_lists_hit_their_patterns():
    EE.check_edge_lists_hit_their_patterns()


def test_replay_rng():
    """eo_rng keeps the 40 bytes (key + block counter) that callers allocating it themselves rely on, and the ctypes mirror
    matches; a replay hands out the caller's blocks in order and raises, rather than wrapping around or returning zeros, on a
    draw past the end -- also from inside a prover."""
    assert O.lib().eo_rng_size() == C.sizeof(O.Rng) == 40
    blocks = bytes(range(64)) + bytes(64) + b"\xff" * 64
    rng = O.rng_from_blocks(blocks)
    assert [O.rng_block(rng) for _ in range(3)] == [blocks[:64], blocks[64:128], blocks[128:]]
    assert O.rng_blocks_left(rng) == 0
    with pytest.raises(O.RngOverrun):
        O.rng_block(rng)
    _, pk = W.receiver()
    with pytest.raises(O.RngOverrun):
        O.encrypt_bool(pk, 1, O.rng_from_blocks(PC.item_blocks(W.SEED_CHOICE, 0, 2)))
    seeded = O.encrypt_bool(pk, 1, O.rng_from_seed(W.SEED_CHOICE, 0))
    assert O.encrypt_bool(pk, 1, O.rng_from_blocks(PC.item_blocks(W.SEED_CHOICE, 0, 3))) == seeded


@pytest.mark.parametrize("P", PROVERS, ids=[P.name for P in PROVERS])
def test_draw_maps(env, P):
    EE.check_draw_maps(P, env[2])


@pytest.mark.parametrize("P", PROVERS, ids=[P.name for P in PROVERS])
def test_prover_edges(env, P):
    e, sk, pk = env
    items, wide = EE.all_cases(P, pk, wide_stride=8)
    EE.check_prover_edges(e, sk, pk, P, items, wide, ring_modes=(1, 3), chunk=29)
