"""Baby-step giant-step discrete-log tables on one GPU: build time and device bytes, lookups/s through eg_dlog_lookup_batch and
eg_decrypt_batch at several batch sizes (values uniform in the range), the worst case (the top of the range) at n = 1, and
giant steps/s on a batch of misses, which walk every giant step.  Every output is checked against the known plaintexts.

    python tools/dlog_bsgs_bench.py [--out profiles/dlog_bsgs_bench_b200.json] [--max-steps 2**34]

Batches whose expected walk exceeds --max-steps giant steps are reported as skipped.  The card's name, power limit and SM
clock are read in the same run and stored with the numbers."""
import argparse
import json
import pathlib
import random
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

CONFIGS = [(2**32, 2**20 - 1), (2**32, 2**24 - 1), (2**40, 2**24 - 1), (2**48, 2**24 - 1), (2**40, 2**28 - 1)]
SIZES = [1, 5, 1024, 65536]
SEED = bytes([0x5b] * 32)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.splitlines()[0].split(",")])) if out.strip() else {}


def timed(fn, reps):
    fn()                                                   # warm-up (module load, scratch growth)
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    return (time.perf_counter() - t0) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "dlog_bsgs_bench_b200.json"))
    ap.add_argument("--max-steps", type=float, default=2.0**34)
    args = ap.parse_args()
    import workloads as W
    from elastic_elgamal_b200 import Engine
    sk, pk = W.receiver()
    e = Engine(device=0)
    e.set_receiver(pk)
    result = {"card": card(), "configs": []}
    for hi, m in CONFIGS:
        J = -(-hi // m)
        row = {"range": f"[0, 2^{hi.bit_length() - 1})", "baby_steps": m, "giant_steps": J}
        t0 = time.perf_counter()
        table = e.dlog_table(0, hi, m)
        row["build_s"] = time.perf_counter() - t0
        cap = 16
        while cap < 2 * m + 2:
            cap <<= 1
        row["device_bytes"] = cap * 40
        rnd = random.Random(hi ^ m)

        def inputs(values):
            v = np.array(values, np.uint64)
            cts = e.encrypt(v, seed=SEED)
            elements = e.decrypt(sk, cts)[0]
            return v, cts, elements

        for n in SIZES:
            if n * J / 2 > args.max_steps:
                row[f"n{n}"] = "skipped: expected walk above --max-steps"
                continue
            v, cts, els = inputs([rnd.randrange(hi) for _ in range(n)])
            reps = 5 if n * J < 2**28 else 1
            t_l, (vals, found) = timed(lambda: e.dlog_lookup(table, els), reps)
            t_d, (_, vals_d, found_d) = timed(lambda: e.decrypt(sk, cts, table), reps)
            assert found.all() and (vals == v).all() and found_d.all() and (vals_d == v).all(), (hi, m, n)
            row[f"n{n}"] = {"lookup_s": t_l, "lookups_per_s": n / t_l, "decrypt_s": t_d, "decrypts_per_s": n / t_d}
        v, cts, els = inputs([hi - 1])
        t_w, (vals, found) = timed(lambda: e.dlog_lookup(table, els), 3)
        assert found.all() and (vals == v).all()
        row["worst_n1_s"] = t_w
        n_miss = int(max(1, min(65536, 2**31 // J)))
        misses = e.decrypt(sk, e.encrypt(np.array([rnd.randrange(2**64 - 2**40, 2**64) for _ in range(n_miss)], np.uint64),
                                          seed=SEED))[0]
        t_m, (vals, found) = timed(lambda: e.dlog_lookup(table, misses), 1)
        assert not found.any()
        row["miss_batch"] = n_miss
        row["giant_steps_per_s"] = n_miss * (J - 1) / t_m
        table.close()
        result["configs"].append(row)
        print(json.dumps(row), flush=True)
    e.close()
    pathlib.Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
