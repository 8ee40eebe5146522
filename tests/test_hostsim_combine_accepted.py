"""eg_combine_decrypt_accepted_batch(_dev) on the CPU-compiled library (TEST HARNESS ONLY, tests/hostsim): every verdict
pattern of 3-of-5, thresholds 1 .. 16 with up to 64 candidate shares and any participant indexes, selections that differ
inside a warp, unread garbage, range and baby-step giant-step tables, chunk sizes, device pointers, multi-device contexts,
an end-to-end tally and argument errors (combine_accepted_common.py)."""
import pytest

import combine_accepted_common as CA
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build
from test_hostsim_edges import HostBuffers


@pytest.fixture(scope="module")
def e():
    eng = Engine(lib_path=build())
    yield eng
    eng.close()


def test_patterns(e):
    CA.check_patterns(e)


@pytest.mark.parametrize("t,indexes", [(3, (0, 1, 2, 3, 4)), (16, tuple(range(63, -1, -1))), (1, (2**31, 5))])
def test_equivalence(e, t, indexes):
    CA.check_equivalence(e, t, indexes, n=20)


@pytest.mark.parametrize("t", [1, 2, 3, 16])
@pytest.mark.parametrize("extra", ["t", "t+1", "64"])
def test_shapes(e, t, extra):
    CA.check_shape(e, t, {"t": t, "t+1": t + 1, "64": 64}[extra], n=6)


def test_random_masks_64(e):
    CA.check_random_masks_64(e, n=12)


def test_mixed_warps(e):
    CA.check_mixed_warps(e)


def test_garbage(e):
    CA.check_garbage(e)


def test_bsgs(e):
    lo = 2**28 - 3000
    CA.check_bsgs(e, lo, 2**28 + 3000, 256, [lo, lo + 255, lo + 256, 2**28 - 1, 2**28, 2**28 + 2999, 2**28 + 3000, 0, 7, lo - 1])


def test_found3_does_not_walk(e):
    CA.check_no_walk(e, 256, 20)


def test_chunks(e):
    CA.check_chunks(e)


@pytest.mark.parametrize("chunk", [0, 7])
def test_dev(e, chunk):
    CA.check_dev(e, HostBuffers(), chunk=chunk)


@pytest.mark.parametrize("children", [1, 3])
def test_multi_context(e, children):
    m = Engine(lib_path=build(), devices=[0] * children)
    try:
        CA.check_multi(m, e)
        CA.check_argument_errors(m, e, multi=m)
    finally:
        m.close()


def test_end_to_end(e):
    CA.check_end_to_end(e, HostBuffers(), n=40)


def test_argument_errors(e):
    other = Engine(lib_path=build())
    try:
        CA.check_argument_errors(e, other)
    finally:
        other.close()
