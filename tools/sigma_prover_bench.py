#!/usr/bin/env python3
"""tools/sigma_prover_bench.py -- the stand-alone sigma provers at N items (default 2^20).  Prints one JSON line with

  * eg_prove_commitment_equiv_batch*: caller-supplied blocks / seeded x default / constant-time prover mode, from pinned and
    from pageable host buffers;
  * eg_prove_sumsq_batch_seeded at count 5 (the quadratic-voting shape) and 15, pageable;
  * eg_prove_possession_batch_seeded at k = 1 and 8 keys per proof, pageable;
  * the oracle's provers on one host thread and on 16 (ctypes releases the GIL during each call);
  * the GPU's name, power limit and SM clock, read in the same process.

Every timed output is checked: the first 64 items equal the oracle byte for byte and every item is accepted by the GPU
verifier.

    python tools/sigma_prover_bench.py [--items 1048576] [--out FILE]
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import pathlib
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
import numpy as np  # noqa: E402

import oracle as O  # noqa: E402
import sigma_prover_common as S  # noqa: E402
import workloads as W  # noqa: E402
from elastic_elgamal_b200 import Engine  # noqa: E402

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


def canonical(rnd, shape):
    s = rnd.integers(0, 256, size=shape + (32,), dtype=np.uint8)
    s[..., 31] &= 0x0F
    return s


def oracle_rate(work, items, threads):
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda t: work(t * items, (t + 1) * items), range(threads)))
    return items * threads / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    n = args.items
    sync = torch.cuda.synchronize
    res = {"items": n, "gpu": gpu_info()}
    e = Engine(device=0)
    sk, pk = W.receiver()
    e.set_receiver(pk)
    e.set_blinding_base(S.BB)
    rnd = np.random.default_rng(21)
    seed = np.frombuffer(S.SEED, np.uint8).copy()

    # ---- CommitmentEquivalenceProof::new
    values = rnd.integers(0, 1 << 63, size=n, dtype=np.uint64)
    ct_r = canonical(rnd, (n,))
    ct_r[:64] = S.ceq_inputs(64)[1]
    wide = np.frombuffer(b"".join(S.blocks(S.SEED, 1 + (i << 20), 4) for i in range(64)), np.uint8).reshape(64, 4, 64)
    wide = np.concatenate([wide, rnd.integers(0, 256, size=(n - 64, 4, 64), dtype=np.uint8)])
    ocs, ocoms, oproofs = O.gen_ceq_batch(pk, S.BB, "bench", S.SEED, values[:64])
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    p_vals, p_r, p_wide = pin(values), pin(ct_r), pin(wide)
    p_out = [torch.empty(s, dtype=torch.uint8).pin_memory() for s in ((n, 64), (n, 32), (n, 128), (n, 32))]
    for ct_mode in (False, True):
        e.set_prover_mode(ct_mode)
        tag = "constant_time" if ct_mode else "default"
        for form in ("blocks", "seeded"):
            out = {}
            kw = dict(seed=S.SEED, counter_base=1) if form == "seeded" else dict(wide_rand=wide)
            res[f"ceq_per_s_pageable_{form}_{tag}"] = rate(n, lambda: out.update(r=e.prove_commitment_equiv("bench", values, ct_r, **kw)), sync)
            if form == "seeded":
                res[f"ceq_per_s_pinned_{form}_{tag}"] = rate(n, lambda: e._check(e.lib.eg_prove_commitment_equiv_batch_seeded(
                    e.h, b"bench", n, p_vals.data_ptr(), p_r.data_ptr(), seed.ctypes.data, 1, *(t.data_ptr() for t in p_out))), sync)
            else:
                res[f"ceq_per_s_pinned_{form}_{tag}"] = rate(n, lambda: e._check(e.lib.eg_prove_commitment_equiv_batch(
                    e.h, b"bench", n, p_vals.data_ptr(), p_r.data_ptr(), p_wide.data_ptr(), *(t.data_ptr() for t in p_out))), sync)
            cts, coms, proofs, _ = out["r"]
            for got in (out["r"], [t.numpy() for t in p_out]):
                assert (got[0][:64] == ocs).all() and (got[1][:64] == ocoms).all() and (got[2][:64] == oproofs).all()
                assert (got[0] == cts).all() and (got[2] == proofs).all()
            assert (e.verify_commitment_equiv("bench", cts, coms, proofs) == O.OK).all()
    e.set_prover_mode(False)
    res["ceq_h2d_d2h_bytes_per_item_blocks"] = [8 + 32 + 256, 64 + 32 + 128 + 32]
    del wide, p_wide

    # ---- SumOfSquaresProof::new at count 5 and 15
    for m in (5, 15):
        vals = rnd.integers(0, 1 << 16, size=(n, m), dtype=np.uint64)
        r, sum_r = canonical(rnd, (n, m)), canonical(rnd, (n,))
        pad = lambda s: np.concatenate([s.reshape(-1, 32), np.zeros_like(s.reshape(-1, 32))], axis=1)
        cts = e.encrypt(vals.reshape(-1), pad(r)).reshape(n, m, 64)
        sum_cts = e.encrypt((vals * vals).sum(axis=1), pad(sum_r))
        out = {}
        res[f"sumsq_{m}_per_s_pageable_seeded"] = rate(n, lambda: out.update(r=e.prove_sumsq("bench", cts, vals, r, sum_cts, sum_r,
                                                                                             seed=S.SEED, counter_base=3)), sync)
        proofs = out["r"]
        assert (e.verify_sumsq("bench", cts, sum_cts, proofs) == O.OK).all()
        assert (proofs[:64] == S.oracle_sumsq(pk, (cts[:64], vals[:64], r[:64], sum_cts[:64], sum_r[:64]), "bench", 3)).all()
        del cts, r, proofs

    # ---- Keypair::from + ProofOfPossession::from_keys at k = 1 and 8
    for k in (1, 8):
        secrets = canonical(rnd, (n, k))
        secrets[:64] = S.pop_secrets(64, k)
        out = {}
        res[f"pop_{k}_per_s_pageable_seeded"] = rate(n, lambda: out.update(r=e.prove_possession("bench", secrets, seed=S.SEED,
                                                                                                  counter_base=k)), sync)
        keys, proofs = out["r"]
        okeys, oproofs = O.gen_pop_batch(k, "bench", S.SEED, 64)
        assert (keys[:64] == okeys).all() and (proofs[:64] == oproofs).all()
        assert (e.verify_possession("bench", keys, proofs) == O.OK).all()

    # ---- the oracle port
    lib = O.lib()

    def ceq_work(lo, hi):
        ct, com, pr, bl = O.buf(64), O.buf(32), O.buf(128), O.buf(32)
        for i in range(lo, hi):
            rng = O.rng_from_seed(S.SEED, first_block=i << 20)
            assert lib.eo_commitment_equiv_prove(pk, C.c_uint64(i), S.BB, b"bench", C.byref(rng), ct, com, pr, bl) == 0

    inst = S.sumsq_instances(pk, 1, 5)
    scts, svals, srs, ssum, ssr = (b"".join(bytes(x) for x in inst[0][0]), b"".join(S.sc(int(v)) for v in inst[1][0]),
                                   b"".join(bytes(x) for x in inst[2][0]), bytes(inst[3][0]), bytes(inst[4][0]))

    def sumsq_work(lo, hi):
        pr = O.buf(32 * 12)
        for i in range(lo, hi):
            rng = O.rng_from_seed(S.SEED, first_block=i << 20)
            assert lib.eo_sumsq_prove(pk, 5, scts, svals, srs, ssum, ssr, b"bench", C.byref(rng), pr) == 0

    psec = S.pop_secrets(1, 1)[0].tobytes()
    pkey = O.point_mul_generator(psec)

    def pop_work(lo, hi):
        pr = O.buf(64)
        for i in range(lo, hi):
            rng = O.rng_from_seed(S.SEED, first_block=i << 20)
            assert lib.eo_pop_prove(1, psec, pkey, b"bench", C.byref(rng), pr) == 0

    for name, work, items in (("ceq", ceq_work, 2000), ("sumsq_5", sumsq_work, 500), ("pop_1", pop_work, 4000)):
        res[f"oracle_{name}_per_s_1_thread"] = oracle_rate(work, items, 1)
        res[f"oracle_{name}_per_s_16_threads"] = oracle_rate(work, max(1, items // 4), 16)
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        pathlib.Path(args.out).write_text(line + "\n")
    e.close()


if __name__ == "__main__":
    main()
