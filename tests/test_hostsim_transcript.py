"""The device transcript at every STROBE block offset on the CPU-compiled library (TEST HARNESS ONLY, tests/hostsim): the
oracle's and pyref's transcripts agree for every label length 0..255; every labelled entry point -- range, sum-of-squares,
decryption, commitment-equivalence and possession verifiers and provers, the range verifier in ring modes 1, 2 and 3 --
gives the oracle's bytes and verdicts for every label length 1..255 (the full sweep, every phase) and for non-ASCII labels;
labels of 0 and 256 bytes are refused by every one of them (transcript_common.py)."""
import pytest

import transcript_common as T
from elastic_elgamal_b200 import Engine
from hostsim.build_hostsim import build
from tests.test_hostsim_edges import HostBuffers


@pytest.fixture(scope="module")
def e():
    eng = Engine(lib_path=build())
    T.prepare(eng)
    yield eng
    eng.close()


def test_references_agree_at_every_phase():
    T.check_references_agree()


def test_every_labelled_entry_point_is_covered():
    assert T.labelled_in_header() == set(T.ENTRY_POINTS)


@pytest.mark.parametrize("obj", T.OBJECTS)
def test_label_sweep_lengths_1_to_255(e, obj):
    T.check_sweep(e, obj, T.SWEEP, HostBuffers())


@pytest.mark.parametrize("label", T.NON_ASCII_LABELS.values(), ids=T.NON_ASCII_LABELS.keys())
@pytest.mark.parametrize("obj", T.OBJECTS)
def test_non_ascii_labels(e, obj, label):
    T.check_label(e, obj, label, HostBuffers())


@pytest.mark.parametrize("name", T.ENTRY_POINTS)
def test_label_arguments(e, name):
    T.check_label_arguments(e, name, HostBuffers())


@pytest.fixture(scope="module")
def multi():
    eng = Engine(lib_path=build(), devices=[0] * 3)
    T.prepare(eng)
    yield eng
    eng.close()


@pytest.mark.parametrize("name", T.HOST_ENTRY_POINTS)
def test_label_arguments_multi_context(multi, name):
    T.check_label_arguments(multi, name, None)
