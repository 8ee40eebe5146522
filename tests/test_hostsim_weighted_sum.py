"""eg_ciphertexts_weighted_sum on the CPU-compiled library (TEST HARNESS ONLY, tests/hostsim): small batches against the
oracle, every window width of the harness's window policy (2..5 bits, chosen at 32 / 64 / 128 / 256 items), skewed and
cancelling weights, verdict masks, chunk sizes, multi-device contexts and argument errors (weighted_sum_common.py)."""
import pytest

import weighted_sum_common as WS
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build
from test_hostsim_edges import HostBuffers


@pytest.fixture(scope="module")
def e():
    eng = Engine(lib_path=build())
    yield eng
    eng.close()


@pytest.mark.parametrize("n,n_cts", [(1, 1), (2, 2), (31, 5), (257, 1), (257, 2), (2000, 1), (2, 64), (31, 64)])
@pytest.mark.parametrize("kind", ["mixed", "u64", "full"])
def test_parity(e, n, n_cts, kind):
    WS.check_parity(e, n, n_cts, kind)


@pytest.mark.parametrize("n,c", [(20, 2), (40, 2), (64, 3), (100, 3), (128, 4), (200, 4), (256, 5), (300, 5)])
def test_widths(e, n, c):
    WS.check_width(e, n, c)


def test_thresholds(e):
    WS.check_thresholds(e, [31, 32, 63, 64, 127, 128, 255, 256])


@pytest.mark.parametrize("n,n_cts", [(1, 1), (33, 2), (300, 5)])
def test_skew(e, n, n_cts):
    WS.check_skew(e, n, n_cts)


def test_choice_mask(e):
    WS.check_choice_mask(e)


def test_qv_mask(e):
    WS.check_qv_mask(e)


def test_validation(e):
    WS.check_validation(e)


@pytest.mark.parametrize("n,n_cts", [(50, 1), (300, 5)])
def test_chunks(e, n, n_cts):
    WS.check_chunks(e, n, n_cts)


@pytest.mark.parametrize("chunk", [0, 7])
def test_dev(e, chunk):
    WS.check_dev(e, HostBuffers(), chunk=chunk)


@pytest.mark.parametrize("children", [1, 3])
def test_multi_context(e, children):
    m = Engine(lib_path=build(), devices=[0] * children)
    try:
        WS.check_multi(m, e)
        WS.check_argument_errors(m, multi=m)
    finally:
        m.close()


def test_argument_errors(e):
    WS.check_argument_errors(e)
