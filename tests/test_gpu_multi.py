"""`-m gpu` tests of the multi-GPU paths that live inside the library (include/eg_b200.h "multi-GPU"):
eg_ctx_create_multi (one process, several devices) and eg_ctx_attach_comm (one process per GPU).  Verdicts and the
64-byte tally ciphertexts must be byte-identical to the single-GPU result and to the oracle for every device count the
box offers (N = 1 always; 2, 4, 8 when that many GPUs are visible)."""
import os
import pathlib
import random
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import oracle as O
import parity_common as PC
import workloads as W

pytestmark = pytest.mark.gpu
HERE = pathlib.Path(__file__).resolve().parent


def gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def counts():
    """Device counts 1, 2, 4 and 8; a count above what the machine has skips."""
    n = gpu_count()
    return [c if c <= max(n, 1) else pytest.param(c, marks=pytest.mark.skip(reason=f"needs {c} GPUs, {n} visible"))
            for c in (1, 2, 4, 8)]


@pytest.fixture(scope="module")
def batch():
    sk, pk = W.receiver()
    n, m = 3001, 5
    cts, rings, sums = O.gen_choice_batch(pk, m, W.SEED_CHOICE, n)
    cts, rings, sums = cts.copy(), rings.copy(), sums.copy()
    W.tamper_choice(cts, rings, sums, random.Random(5), frac=0.1)
    ov, ot = O.verify_choice_batch(pk, m, True, cts, rings, sums)
    return sk, pk, m, cts, rings, sums, ov, ot


@pytest.mark.parametrize("n_dev", counts())
def test_create_multi_matches_oracle_and_single_gpu(batch, n_dev):
    from elastic_elgamal_b200 import Engine
    sk, pk, m, cts, rings, sums, ov, ot = batch
    e = Engine(devices=list(range(n_dev)))
    try:
        assert e.comm_info()["devices"] == n_dev
        e.set_receiver(pk)
        e.set_ring_mode(2)
        v, t = e.verify_choice(m, cts, rings, sums)
        assert (v == ov).all() and (t == ot).all()
        # every other sharded entry point, on shapes that do not divide evenly
        PC.check_verify_bool(e, pk, n=301)
        PC.check_verify_range(e, pk, 100, n=45, frac=0.3)
        PC.check_verify_qv(e, pk, sk, n=13, options=3, credits=9)
        PC.check_shares_and_decrypt(e, n=37, shares=5, threshold=3, used=(0, 2, 4), table_hi=64)
        PC.check_empty_and_tiny(e, pk)
    finally:
        e.close()


def _run_ranks(world, n, options):
    with tempfile.TemporaryDirectory() as d:
        id_file = os.path.join(d, "nccl_id")
        outs = [os.path.join(d, f"out{r}.npz") for r in range(world)]
        procs = [subprocess.Popen([sys.executable, str(HERE / "comm_worker.py"), str(r), str(world), id_file, outs[r], str(n), str(options)])
                 for r in range(world)]
        for p in procs:
            assert p.wait(timeout=600) == 0
        return [dict(np.load(o)) for o in outs]


@pytest.mark.parametrize("world", counts())
def test_attach_comm_matches_oracle(world):
    """One process per GPU: the library creates the communicator from an id the ranks exchange through a file; the tally
    every rank returns is the global one."""
    sk, pk = W.receiver()
    n, m = 2003, 5
    cts, rings, sums = O.gen_choice_batch(pk, m, W.SEED_CHOICE, n)
    cts, rings, sums = cts.copy(), rings.copy(), sums.copy()
    W.tamper_choice(cts, rings, sums, random.Random(5), frac=0.1)
    ov, ot = O.verify_choice_batch(pk, m, True, cts, rings, sums)
    res = _run_ranks(world, n, m)
    for r in res:
        assert (r["verdicts"] == ov[int(r["lo"]):int(r["hi"])]).all()
        assert (r["tally"] == ot).all()
    # second call: the last rank had an empty slice
    if world > 1:
        hi = int(res[-1]["lo"])
        _, ot2 = O.verify_choice_batch(pk, m, True, cts[:hi], rings[:hi], sums[:hi])
        for r in res:
            assert (r["tally2"] == ot2).all()
