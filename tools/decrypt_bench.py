#!/usr/bin/env python3
"""tools/decrypt_bench.py -- the talliers' side at the config-5 shape: key set 3-of-5, N unique ciphertexts (default 2^20) of
values in [0, 2^20) under the shared key, made on the GPU with eg_encrypt_batch_seeded.  Prints one JSON line with

  * decryption shares per second for one participant (eg_decrypt_share_batch*): device-resident (_dev, seeded), host pinned
    and host pageable buffers, each in both prover modes;
  * eg_prove_decryption_batch_seeded and eg_decrypt_batch (with the 2^20 table) per second, pageable buffers;
  * eg_verify_shares_batch_dev per share on the same inputs (three shares per tally), the yardstick;
  * the oracle's eo_decrypt_share on one host thread and on all of them (ctypes releases the GIL during the call);
  * the GPU's name, power limit and SM clock, read in the same process.

Every timed output is checked: the first 64 items equal the oracle byte for byte, all shares and proofs are accepted by the
GPU verifier, and the decrypted values are the encrypted ones.

    python tools/decrypt_bench.py [--items 1048576] [--out FILE]
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import os
import pathlib
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
import numpy as np  # noqa: E402

import decrypt_common as D  # noqa: E402
import oracle as O  # noqa: E402
import workloads as W  # noqa: E402
from elastic_elgamal_b200 import Engine  # noqa: E402

USED = (0, 2, 4)
REPS = 3


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), (x.strip() for x in out.strip().split(","))))


def rate(n, fn, sync):
    fn()
    sync()
    t0 = time.perf_counter()
    for _ in range(REPS):
        fn()
    sync()
    return n * REPS / (time.perf_counter() - t0)


def oracle_rate(ks, secret, cts, items, threads):
    lib = O.lib()

    def work(lo, hi):
        share, proof = O.buf(32), O.buf(64)
        for i in range(lo, hi):
            rng = O.rng_from_seed(D.SEED, first_block=i << 20)
            assert lib.eo_decrypt_share(C.byref(ks), 2, secret, bytes(cts[i]), C.byref(rng), share, proof) == 0
    total = items * threads
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda t: work(t * items, (t + 1) * items), range(threads)))
    return total / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    n = args.items
    dev = torch.device("cuda", 0)
    sync = torch.cuda.synchronize
    info = gpu_info()
    e = Engine(device=0)
    ks, eks, secrets = D.keyset()
    values = np.random.default_rng(5).integers(0, 1 << 20, n, dtype=np.uint64)
    e.set_receiver(bytes(ks.shared_key))
    cts = e.encrypt(values, seed=bytes(range(32)))
    res = {"items": n, "gpu": info}

    def check_shares(j, sh, pr, ok, first=0):
        assert ok.all()
        osh, opr = D.oracle_shares(ks, j, secrets[j], cts[:64], first)
        assert (sh[:64] == osh).all() and (pr[:64] == opr).all()

    # ---- shares of participant 2: device-resident, pinned, pageable; both prover modes
    d_cts = torch.from_numpy(cts).to(dev)
    d_sh = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    d_pr = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    d_ok = torch.empty(n, dtype=torch.uint8, device=dev)
    p_cts = torch.from_numpy(cts).pin_memory()
    p_sh, p_pr, p_ok = (torch.empty(s, dtype=torch.uint8).pin_memory() for s in ((n, 32), (n, 64), (n,)))
    sec = np.frombuffer(secrets[2], np.uint8).copy()
    seed = np.frombuffer(D.SEED, np.uint8).copy()
    for ct_mode in (False, True):
        e.set_prover_mode(ct_mode)
        tag = "constant_time" if ct_mode else "default"
        res[f"shares_per_s_device_{tag}"] = rate(n, lambda: e.decrypt_share_dev(eks, 2, secrets[2], n, d_cts.data_ptr(), d_sh.data_ptr(),
                                                                                d_pr.data_ptr(), d_ok.data_ptr(), seed=D.SEED), sync)
        check_shares(2, d_sh.cpu().numpy(), d_pr.cpu().numpy(), d_ok.cpu().numpy())
        res[f"shares_per_s_pinned_{tag}"] = rate(n, lambda: e._check(e.lib.eg_decrypt_share_batch_seeded(
            e.h, C.byref(eks), 2, sec.ctypes.data, n, p_cts.data_ptr(), seed.ctypes.data, 0, p_sh.data_ptr(), p_pr.data_ptr(),
            p_ok.data_ptr())), sync)
        check_shares(2, p_sh.numpy(), p_pr.numpy(), p_ok.numpy())
        out = {}
        res[f"shares_per_s_pageable_{tag}"] = rate(n, lambda: out.update(r=e.decrypt_share(eks, 2, secrets[2], cts, seed=D.SEED)), sync)
        check_shares(2, *out["r"])
    e.set_prover_mode(False)

    # ---- the other two participants (device-resident), then the verifier on the same inputs
    shares = torch.empty((n, 3, 32), dtype=torch.uint8, device=dev)
    proofs = torch.empty((n, 3, 64), dtype=torch.uint8, device=dev)
    for j, idx in enumerate(USED):
        e.decrypt_share_dev(eks, idx, secrets[idx], n, d_cts.data_ptr(), d_sh.data_ptr(), d_pr.data_ptr(), d_ok.data_ptr(), seed=D.SEED)
        sync()
        assert (d_ok == 1).all()
        shares[:, j], proofs[:, j] = d_sh, d_pr
    idx = (C.c_uint32 * 3)(*USED)
    d_v = torch.empty((n, 3), dtype=torch.uint8, device=dev)
    res["verify_shares_dev_shares_per_s"] = 3 * rate(n, lambda: e._check(e.lib.eg_verify_shares_batch_dev(
        e.h, C.byref(eks), n, 3, idx, d_cts.data_ptr(), shares.data_ptr(), proofs.data_ptr(), d_v.data_ptr())), sync)
    res["verify_k_msm_ms_last_call"] = e.last_kernel_stats(2)["ms"]
    assert (d_v == 0).all()
    table = e.dlog_table(0, 1 << 20)
    vals, found = e.combine_decrypt(list(USED), cts, shares.cpu().numpy(), table)
    assert (found == 1).all() and (vals == values).all()

    # ---- VerifiableDecryption::new with a custom key, SecretKey::decrypt with the 2^20 table (pageable)
    sk, pk = W.receiver()
    e.set_receiver(pk)
    cts_pk = e.encrypt(values, seed=bytes([7] * 32))
    out = {}
    res["prove_decryption_per_s_pageable"] = rate(n, lambda: out.update(r=e.prove_decryption(D.LABEL, sk, cts_pk, seed=D.SEED)), sync)
    dh, pr, ok = out["r"]
    odh, opr = D.oracle_decryption_proofs(sk, cts_pk[:64], 0)
    assert ok.all() and (dh[:64] == odh).all() and (pr[:64] == opr).all()
    assert (e.verify_decryption(D.LABEL, pk, cts_pk, dh, pr) == 0).all()
    res["decrypt_per_s_pageable_table_2_20"] = rate(n, lambda: out.update(r=e.decrypt(sk, cts_pk, table)), sync)
    el, v, f = out["r"]
    assert (f == 1).all() and (v == values).all()
    assert all(bytes(el[i]) == O.decrypt_to_element(sk, bytes(cts_pk[i])) for i in range(64))
    table.close()

    # ---- the oracle port (one participant's shares)
    threads = os.cpu_count() or 1
    res["oracle_shares_per_s_1_thread"] = oracle_rate(ks, secrets[2], cts, 2000, 1)
    res["oracle_shares_per_s_all_threads"] = oracle_rate(ks, secrets[2], cts, max(1, 8000 // threads), threads)
    res["host_threads"] = threads
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        pathlib.Path(args.out).write_text(line + "\n")
    e.close()


if __name__ == "__main__":
    main()
