"""Shapes at the limits of the verifiers and provers on the CPU-compiled library (TEST HARNESS ONLY, tests/hostsim):
choice ballots of 1..64 options across the slot groups and EG_TERM_MAX, range proofs up to 64 rings, 3500 values and an
upper bound of 2^64 and beyond, the admissible-value cache evicting, the multi-scalar kernels at EG_MSM_MAXV, and chunking
at those shapes (shape_common.py)."""
import pytest

import shape_common as SC
import workloads as W
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build


@pytest.fixture(scope="module")
def env():
    e = Engine(lib_path=build())
    sk, pk = W.receiver()
    e.set_receiver(pk)
    yield e, sk, pk
    e.close()


@pytest.mark.parametrize("single", [True, False], ids=["single", "multi"])
@pytest.mark.parametrize("options", SC.CHOICE_OPTIONS)
def test_choice_shapes(env, options, single):
    e, sk, pk = env
    SC.check_choice_shape(e, pk, sk, options, single)


def test_choice_64_options_above_one_warp(env):
    e, sk, pk = env
    SC.check_choice_shape(e, pk, sk, 64, True, n=40, modes=(2, 3), prove=False)


def test_choice_options_refused(env):
    SC.check_choice_options_refused(env[0], env[2])


@pytest.mark.parametrize("shape", ["32 rings of 4 (2^64)", "64 rings of 2 (2^64)"])
def test_range_upper_bound_2_64(env, shape):
    """Upper bound exactly 2^64: 1 + sum (size - 1) * step wraps to 0 in u64, and a prover that compared with the wrapped
    bound refused every value."""
    SC.check_range_shape(env[0], env[2], SC.RANGE_SHAPES[shape])


@pytest.mark.parametrize("shape", ["64 rings, above 2^64", "63 rings", "one ring of 3500"])
def test_range_shapes(env, shape):
    SC.check_range_shape(env[0], env[2], SC.RANGE_SHAPES[shape], between=0 if shape == "one ring of 3500" else 3)


def test_range_2_32(env):
    SC.check_range_2_32(env[0], env[2])


def test_ranges_refused(env):
    SC.check_ranges_refused(env[0], env[2])


def test_range_cache_eviction(env):
    SC.check_range_cache_eviction(env[0], env[2])


def test_sumsq_15(env):
    SC.check_sumsq_15(env[0], env[2])


def test_qv_15_options(env):
    e, sk, pk = env
    SC.check_qv_15(e, pk, sk)


def test_multi_mul_16(env):
    SC.check_multi_mul_16(env[0])


def test_combine_threshold_16(env):
    SC.check_combine_16(env[0])


def test_keysets_64_threshold_16(env):
    SC.check_keysets_64_16(env[0])


def test_chunked_limits(env):
    e, sk, pk = env
    SC.check_chunked_limits(e, pk, sk)
