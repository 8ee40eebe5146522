"""eg_ciphertexts_group_sum on the CPU-compiled library (TEST HARNESS ONLY, tests/hostsim): small batches against the
oracle over several group counts and group-size distributions (with the harness's 4-entry runs, a group holding every
item is reduced through several run levels), consistency with the weighted sum and the verifiers' tallies, bad elements
and group ids, chunk sizes, host vs _dev, multi-device contexts and argument errors (group_sum_common.py)."""
import pytest

import group_sum_common as GS
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build
from test_hostsim_edges import HostBuffers


@pytest.fixture(scope="module")
def e():
    eng = Engine(lib_path=build())
    yield eng
    eng.close()


@pytest.mark.parametrize("n,n_cts", [(0, 1), (1, 1), (2, 2), (31, 5), (257, 1), (257, 2), (2000, 1), (2, 64), (31, 64)])
@pytest.mark.parametrize("groups", ["1", "2", "7", "1000", "n+5"])
def test_parity(e, n, n_cts, groups):
    GS.check_parity(e, n, n_cts, n + 5 if groups == "n+5" else int(groups))


@pytest.mark.parametrize("kind", GS.DISTRIBUTIONS)
@pytest.mark.parametrize("n,n_cts", [(1, 1), (257, 2), (2000, 1)])
def test_distributions(e, n, n_cts, kind):
    GS.check_distribution(e, n, n_cts, kind)


@pytest.mark.parametrize("n,n_cts", [(1, 1), (300, 5)])
def test_single_group_is_weighted_sum(e, n, n_cts):
    GS.check_single_group_is_weighted_sum(e, n, n_cts)


def test_choice_mask(e):
    GS.check_choice_mask(e)


def test_qv_mask(e):
    GS.check_qv_mask(e)


def test_bad_items(e):
    GS.check_bad_items(e)


@pytest.mark.parametrize("n,n_cts,n_groups", [(50, 1, 1), (300, 5, 40), (300, 2, 1000)])
def test_chunks(e, n, n_cts, n_groups):
    GS.check_chunks(e, n, n_cts, n_groups)


@pytest.mark.parametrize("chunk", [0, 7])
def test_dev(e, chunk):
    GS.check_dev(e, HostBuffers(), chunk=chunk)


@pytest.mark.parametrize("children", [1, 3])
def test_multi_context(e, children):
    m = Engine(lib_path=build(), devices=[0] * children)
    try:
        GS.check_multi(m, e)
        GS.check_argument_errors(m, multi=m)
    finally:
        m.close()


def test_argument_errors(e):
    GS.check_argument_errors(e)
