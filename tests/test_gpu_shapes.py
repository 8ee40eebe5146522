"""`-m gpu`: shapes at the limits of the verifiers and provers on the CUDA library -- choice ballots of 1..64 options across
the slot groups and EG_TERM_MAX (k_terminal with 130 deferred points, in full warps), range proofs up to 64 rings, 3500
values and an upper bound of 2^64 and beyond, the admissible-value cache evicting, k_msm at EG_MSM_MAXV, and chunking at
those shapes (shape_common.py)."""
import pytest

import shape_common as SC
import workloads as W

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    from elastic_elgamal_b200 import Engine
    e = Engine(device=0)
    sk, pk = W.receiver()
    e.set_receiver(pk)
    yield e, sk, pk
    e.close()


@pytest.mark.parametrize("single", [True, False], ids=["single", "multi"])
@pytest.mark.parametrize("options", SC.CHOICE_OPTIONS)
def test_choice_shapes(env, options, single):
    e, sk, pk = env
    SC.check_choice_shape(e, pk, sk, options, single)


@pytest.mark.parametrize("n", [40, 300])
def test_choice_64_options_full_warps(env, n):
    e, sk, pk = env
    SC.check_choice_shape(e, pk, sk, 64, True, n=n, prove=n == 40)


def test_choice_options_refused(env):
    SC.check_choice_options_refused(env[0], env[2])


@pytest.mark.parametrize("shape", ["32 rings of 4 (2^64)", "64 rings of 2 (2^64)"])
def test_range_upper_bound_2_64(env, shape):
    SC.check_range_shape(env[0], env[2], SC.RANGE_SHAPES[shape])


@pytest.mark.parametrize("shape", ["64 rings, above 2^64", "63 rings", "one ring of 3500"])
def test_range_shapes(env, shape):
    SC.check_range_shape(env[0], env[2], SC.RANGE_SHAPES[shape])


def test_range_2_32(env):
    SC.check_range_2_32(env[0], env[2])


def test_ranges_refused(env):
    SC.check_ranges_refused(env[0], env[2])


def test_range_cache_eviction(env):
    SC.check_range_cache_eviction(env[0], env[2], calls=3)


def test_sumsq_15(env):
    SC.check_sumsq_15(env[0], env[2], n=40)


def test_qv_15_options(env):
    e, sk, pk = env
    SC.check_qv_15(e, pk, sk)


def test_multi_mul_16(env):
    SC.check_multi_mul_16(env[0], n=40)


def test_combine_threshold_16(env):
    SC.check_combine_16(env[0])


def test_keysets_64_threshold_16(env):
    SC.check_keysets_64_16(env[0])


def test_chunked_limits(env):
    e, sk, pk = env
    SC.check_chunked_limits(e, pk, sk)
