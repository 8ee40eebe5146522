"""Threshold decryption from the accepted shares on one GPU: eg_combine_decrypt_accepted_batch(_dev) at 2^20 tallies of a 3-of-5
key set, all 5 shares per tally and a [0, 2^20) table, in three verdict cases, beside eg_combine_decrypt_batch(_dev) on the
all-accepted batch with the fixed columns 0, 1, 2 (share_stride 5):

  all_accepted      every share accepted: every tally takes k_combine_select's copy of the batch coefficients
  one_pct_rejected  1 % of the tallies have one rejected share among their first three columns: those invert
  half_p0_rejected  participant 0 is rejected on a random half of the tallies: half of every warp inverts

    python tools/combine_accepted_bench.py [--out profiles/combine_accepted_bench_b200.json] [--reps 7]

Every call is run once before it is timed, and the calls of a round alternate between the cases.  Device times are CUDA
events on the library's stream around the _dev calls; host times are host clocks around the synchronous host-pointer calls;
both are medians over --reps rounds.  Every output is checked against the plaintexts in the same run.  The card's name and
power limit are read in the same run."""
import argparse
import ctypes as C
import json
import pathlib
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

N = 2**20
SEED = bytes([0x3c] * 32)
INDEXES = [0, 1, 2, 3, 4]


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.splitlines()[0].split(",")])) if out.strip() else {}


def verdict_cases(n, rng):
    all_ok = np.zeros((n, 5), np.uint8)
    one = all_ok.copy()
    rows = rng.choice(n, n // 100, replace=False)
    one[rows, rng.integers(0, 3, rows.size)] = 2
    half = all_ok.copy()
    half[rng.random(n) < 0.5, 0] = 2
    return {"all_accepted": all_ok, "one_pct_rejected": one, "half_p0_rejected": half}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "combine_accepted_bench_b200.json"))
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--n", type=int, default=N)
    args = ap.parse_args()
    import torch
    import decrypt_common as D
    from elastic_elgamal_b200 import Engine
    n = args.n
    e = Engine(device=0)
    ks, eks, secrets = D.keyset()
    rng = np.random.default_rng(19)
    values = rng.integers(0, 2**20, n, dtype=np.uint64)
    e.set_receiver(bytes(ks.shared_key))
    cts = e.encrypt(values, seed=SEED)
    shares = np.zeros((n, 5, 32), np.uint8)
    for j in INDEXES:
        sh, _, ok = e.decrypt_share(eks, j, secrets[j], cts, seed=D.SEED)
        assert ok.all()
        shares[:, j] = sh
    cases = verdict_cases(n, rng)
    table = e.dlog_table(0, 2**20)
    stream = torch.cuda.ExternalStream(e.stream)
    d_cts, d_shares = torch.from_numpy(cts).cuda(), torch.from_numpy(shares).cuda()
    d_vals, d_found = torch.zeros(n, dtype=torch.int64, device="cuda"), torch.zeros(n, dtype=torch.uint8, device="cuda")
    d_verdicts = {k: torch.from_numpy(v).cuda() for k, v in cases.items()}
    torch.cuda.synchronize()
    idx3 = (C.c_uint32 * 3)(0, 1, 2)

    def check(vals, found, what):
        assert (np.asarray(found) == 1).all() and (np.asarray(vals).view(np.uint64) == values).all(), what

    def dev_call(name):
        if name == "fixed_subset":
            return lambda: e._check(e.lib.eg_combine_decrypt_batch_dev(e.h, 3, idx3, n, 5, d_cts.data_ptr(), d_shares.data_ptr(), table.h,
                                                                        d_vals.data_ptr(), d_found.data_ptr()))
        return lambda: e.combine_decrypt_accepted_dev(3, INDEXES, n, d_cts.data_ptr(), d_shares.data_ptr(), d_verdicts[name].data_ptr(),
                                                      table, d_vals.data_ptr(), d_found.data_ptr())

    def host_call(name):
        if name == "fixed_subset":
            return lambda: e.combine_decrypt([0, 1, 2], cts, shares, table)
        return lambda: e.combine_decrypt_accepted(3, INDEXES, cts, shares, cases[name], table)

    names = ["fixed_subset"] + list(cases)
    dev_ms = {k: [] for k in names}
    host_ms = {k: [] for k in names}
    stats = {}
    for rnd in range(args.reps + 1):                     # round 0 warms every call up
        for name in names:
            d_found.zero_()
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            dev_call(name)()
            ev1.record(stream)
            ev1.synchronize()
            stats[name] = e.last_kernel_stats(2)
            check(d_vals.cpu().numpy(), d_found.cpu().numpy(), f"{name} (_dev)")
            t0 = time.perf_counter()
            vals, found = host_call(name)()
            t = time.perf_counter() - t0
            check(vals, found, f"{name} (host)")
            if rnd:
                dev_ms[name].append(ev0.elapsed_time(ev1))
                host_ms[name].append(t * 1e3)
    table.close()
    base = float(np.median(dev_ms["fixed_subset"]))
    res = {"card": card(), "n": n, "threshold": 3, "n_shares": 5, "table": [0, 2**20], "reps": args.reps,
           "timer": "dev: CUDA events on the library stream around the _dev call; host: host clock around the host-pointer call; "
                    "medians over alternating rounds",
           "rows": []}
    for name in names:
        d, h = float(np.median(dev_ms[name])), float(np.median(host_ms[name]))
        row = {"case": name, "entry_point": "eg_combine_decrypt_batch" if name == "fixed_subset" else "eg_combine_decrypt_accepted_batch",
               "dev_ms": d, "dev_ms_min": float(min(dev_ms[name])), "dev_ms_max": float(max(dev_ms[name])), "host_ms": h,
               "dev_tallies_per_s": n / (d * 1e-3), "dev_over_fixed_subset": d / base, "k_msm_stats": stats[name]}
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
    pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    e.close()


if __name__ == "__main__":
    main()
