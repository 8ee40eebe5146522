"""The weighted tally fold on one GPU: eg_ciphertexts_weighted_sum_dev and the host form at n in {10^4, 2^18, 10^6} items of
n_cts in {1, 5} ciphertexts, with u64 weights and with full 253-bit scalars; beside it, the lower bound of the per-item path
(eg_ciphertexts_lincomb_batch with one term per ciphertext, its n x n_cts products left unsummed) on the same inputs, and
eg_verify_choice_batch on the same 10^6 five-option ballots.  Each weighted sum is checked against the products of the
per-item path added up by eg_ciphertexts_sum.

    python tools/weighted_sum_bench.py [--out profiles/weighted_sum_bench_b200.json] [--reps 5]

Every shape is run once before it is timed.  Times are host clocks around calls that end in a device synchronisation
(every entry point here is synchronous), medians of --reps calls.  The card's name and power limit are read in the same run."""
import argparse
import json
import pathlib
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

SIZES = [10**4, 2**18, 10**6]
N_CTS = [1, 5]
SEED = bytes([0x3c] * 32)
L = 2**252 + 27742317777372353535851937790883648493


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.splitlines()[0].split(",")])) if out.strip() else {}


def timed(fn, reps):
    out = fn()                                             # warm-up of this shape
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def scalars(n, kind, rng):
    s = np.zeros((n, 32), np.uint8)
    if kind == "u64":
        s[:, :8] = rng.integers(0, 256, (n, 8), dtype=np.uint8)
    else:
        s[:] = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        s[:, 31] &= 0x0f                                   # < 2^252 < l: canonical
    return s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "weighted_sum_bench_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default=",".join(map(str, SIZES)))
    args = ap.parse_args()
    import torch
    import workloads as W
    from elastic_elgamal_b200 import Engine
    e = Engine(device=0)
    sk, pk = W.receiver()
    e.set_receiver(pk)
    rng = np.random.default_rng(7)
    res = {"card": card(), "reps": args.reps, "timer": "host clock around synchronous calls, median", "rows": []}
    sizes = [int(x) for x in args.sizes.split(",")]
    for n_cts in N_CTS:
        for n in sizes:
            cts = e.encrypt(rng.integers(0, 2, n * n_cts, dtype=np.uint64), seed=SEED).reshape(n, n_cts, 64)
            d_cts = torch.from_numpy(cts.reshape(n, -1)).cuda()
            d_out, d_ok = torch.zeros(64 * n_cts, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.uint8, device="cuda")
            for kind in ("u64", "full"):
                s = scalars(n, kind, rng)
                d_s = torch.from_numpy(s).cuda()
                torch.cuda.synchronize()

                def dev():
                    e.weighted_sum_dev(n, n_cts, 64 * n_cts, 64, d_cts.data_ptr(), d_s.data_ptr(), 0, d_out.data_ptr(), d_ok.data_ptr())
                    torch.cuda.synchronize()
                t_dev, _ = timed(dev, args.reps)
                t_host, (out, ok) = timed(lambda: e.weighted_sum(cts, s), args.reps)
                assert ok and int(d_ok.cpu()[0]) == 1 and (d_out.cpu().numpy().reshape(n_cts, 64) == out).all()
                # the per-item path: one product per ciphertext (the fold left out of the timing)
                ls = np.repeat(s, n_cts, axis=0).reshape(n * n_cts, 1, 32)
                lc = cts.reshape(n * n_cts, 1, 64)
                t_lin, (prods, pok) = timed(lambda: e.ciphertexts_lincomb(ls, lc), args.reps)
                total, sok = e.ciphertexts_sum(prods.reshape(n, n_cts, 64))
                assert pok.all() and sok and (total == out).all(), "the weighted sum differs from the per-item path"
                row = {"n": n, "n_cts": n_cts, "scalars": kind, "dev_ms": t_dev * 1e3, "host_ms": t_host * 1e3,
                       "lincomb_bound_ms": t_lin * 1e3, "dev_items_per_s": n / t_dev, "gain_over_lincomb_dev": t_lin / t_dev}
                res["rows"].append(row)
                print(json.dumps(row), flush=True)
            del d_cts
    if 10**6 in sizes:
        n, m = 10**6, 5
        values = np.zeros((n, m), np.uint8)
        values[np.arange(n), rng.integers(0, m, n)] = 1
        choices, rings, sums = e.encrypt_choice(m, values, seed=SEED)
        t_v, (v, t) = timed(lambda: e.verify_choice(m, choices, rings, sums), args.reps)
        assert (v == 0).all()
        t_w, (out, ok) = timed(lambda: e.weighted_sum(choices, np.ones(n, np.uint64), v), args.reps)
        assert ok and (out == t).all()
        w = rng.integers(1, 2**20, n, dtype=np.uint64)
        t_ww, _ = timed(lambda: e.weighted_sum(choices, w, v), args.reps)
        res["choice_1m_5"] = {"verify_choice_ms": t_v * 1e3, "weighted_sum_weights1_ms": t_w * 1e3,
                              "weighted_sum_u20_weights_ms": t_ww * 1e3, "weighted_over_verify": t_ww / t_v}
        print(json.dumps(res["choice_1m_5"]), flush=True)
    pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    e.close()


if __name__ == "__main__":
    main()
