"""`-m gpu`: the device transcript at every STROBE block offset on the CUDA library -- every labelled entry point (k_ring,
the pair engine and the per-equation pipeline with k_ring_final, k_rprove, k_sumsq_final, k_sumsq_prove, k_share_final,
k_decrypt<proof>, k_sigma_final, k_ceq_prove, k_pop_prove) gives the oracle's bytes and verdicts for every label length
1..255 and for non-ASCII labels; labels of 0 and 256 bytes are refused by every one of them, on one GPU and on a
multi-device context (transcript_common.py)."""
import pytest

import transcript_common as T
from tests.test_gpu_edges import TorchBuffers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def e():
    from elastic_elgamal_b200 import Engine
    eng = Engine(device=0)
    T.prepare(eng)
    yield eng
    eng.close()


@pytest.mark.parametrize("obj", T.OBJECTS)
def test_label_sweep_lengths_1_to_255(e, obj):
    T.check_sweep(e, obj, T.SWEEP, TorchBuffers())


@pytest.mark.parametrize("label", T.NON_ASCII_LABELS.values(), ids=T.NON_ASCII_LABELS.keys())
@pytest.mark.parametrize("obj", T.OBJECTS)
def test_non_ascii_labels(e, obj, label):
    T.check_label(e, obj, label, TorchBuffers())


@pytest.mark.parametrize("name", T.ENTRY_POINTS)
def test_label_arguments(e, name):
    T.check_label_arguments(e, name, TorchBuffers())


@pytest.fixture(scope="module")
def multi():
    from elastic_elgamal_b200 import Engine
    eng = Engine(devices=[0])
    T.prepare(eng)
    yield eng
    eng.close()


@pytest.mark.parametrize("name", T.HOST_ENTRY_POINTS)
def test_label_arguments_multi_context(multi, name):
    T.check_label_arguments(multi, name, None)
