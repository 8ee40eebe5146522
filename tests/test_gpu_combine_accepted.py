"""`-m gpu`: eg_combine_decrypt_accepted_batch(_dev) on the CUDA library -- the CPU harness checks (combine_accepted_common.py)
at device chunk sizes, a [0, 2^32) baby-step giant-step table, found 3 against a table of 2^32 giant steps, 262 144 tallies
with 1 % rejected shares, and multi-GPU contexts where the machine has them."""
import pytest

import combine_accepted_common as CA
from tests.test_gpu_decrypt import counts
from tests.test_gpu_edges import TorchBuffers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
    yield eng
    eng.close()


def test_patterns(e):
    CA.check_patterns(e, copies=8)


@pytest.mark.parametrize("t,indexes", [(3, (0, 1, 2, 3, 4)), (16, tuple(range(63, -1, -1))), (1, (2**31, 5))])
def test_equivalence(e, t, indexes):
    CA.check_equivalence(e, t, indexes, n=200)


@pytest.mark.parametrize("t", [1, 2, 3, 16])
@pytest.mark.parametrize("extra", ["t", "t+1", "64"])
def test_shapes(e, t, extra):
    CA.check_shape(e, t, {"t": t, "t+1": t + 1, "64": 64}[extra], n=12)


def test_random_masks_64(e):
    CA.check_random_masks_64(e, n=48)


def test_mixed_warps(e):
    CA.check_mixed_warps(e, runs=8)


def test_garbage(e):
    CA.check_garbage(e, n=200)


def test_bsgs(e):
    CA.check_bsgs(e, 0, 2**32, 2**24 - 1, [2**28, 2**28 + 1, 2**30 + 12345, 10**9, 2**32 - 1, 2**24 - 2, 2**24 - 1, 0, 5, 2**32,
                                            2**33 + 1])


def test_found3_does_not_walk(e):
    took = CA.check_no_walk(e, 2**24 - 1, 1000)
    assert took < 60, f"{took:.1f} s: tallies that were not combined walked the giant steps"


def test_chunks(e):
    CA.check_chunks(e)


@pytest.mark.parametrize("chunk", [0, 7])
def test_dev(e, chunk):
    CA.check_dev(e, TorchBuffers(), n=200, chunk=chunk)


@pytest.mark.parametrize("n_dev", counts())
def test_multi_gpu(e, n_dev):
    from elastic_elgamal_b200 import Engine
    m = Engine(devices=list(range(n_dev)))
    try:
        CA.check_multi(m, e, n=200)
        CA.check_argument_errors(m, e, multi=m)
    finally:
        m.close()


def test_end_to_end(e):
    CA.check_end_to_end(e, TorchBuffers(), n=300)


def test_at_size(e):
    CA.check_at_size(e, 262144)


def test_argument_errors(e):
    from elastic_elgamal_b200 import Engine
    other = Engine(device=0)
    try:
        CA.check_argument_errors(e, other)
    finally:
        other.close()
