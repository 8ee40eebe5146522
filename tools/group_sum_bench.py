"""The grouped tally fold on one GPU: eg_ciphertexts_group_sum_dev and the host form over 10^6 five-option choice buffers
(1 % tampered) with eg_verify_choice_batch's verdicts as the mask, at n_groups in {1, 10^3, 2 * 10^5} with uniform, Zipf-like
and single-group distributions.  Beside it, on the same buffers: eg_ciphertexts_weighted_sum with unit weights (the same
fold with n_groups = 1), eg_verify_choice_batch itself, and the loop the grouped fold replaces -- one unit-weight weighted
sum per group over host-sorted items -- at 10^3 groups.  Every grouped result is checked: its groups add up (by
eg_ciphertexts_sum) to the verifier's tally, and the _dev form equals the host form.

    python tools/group_sum_bench.py [--out profiles/group_sum_bench_b200.json] [--reps 5]

Every shape is run once before it is timed.  Times are host clocks around calls that end in a device synchronisation
(every entry point here is synchronous), medians of --reps calls.  The card's name and power limit are read in the same run.
A last, separate pass records per-kernel device times of single _dev calls with torch.profiler (the single-thread scan
k_ws_hist_scan among them, up to 2^22 groups)."""
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

N, OPTIONS = 10**6, 5
GROUPS = [1, 10**3, 2 * 10**5]
SEED = bytes([0x3c] * 32)


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


def kernel_times(fn):
    """Device time per kernel name (ms, summed over launches) of one call of fn, by torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t and ("k_gs_" in ev.key or "k_ws_" in ev.key):
            out[ev.key] = out.get(ev.key, 0.0) + t / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "group_sum_bench_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n", type=int, default=N)
    args = ap.parse_args()
    import torch
    import group_sum_common as GS
    import workloads as W
    from elastic_elgamal_b200 import Engine
    n, m = args.n, OPTIONS
    e = Engine(device=0)
    sk, pk = W.receiver()
    e.set_receiver(pk)
    rng = np.random.default_rng(7)
    res = {"card": card(), "reps": args.reps, "n": n, "options": m, "timer": "host clock around synchronous calls, median", "rows": []}
    values = np.zeros((n, m), np.uint8)
    values[np.arange(n), rng.integers(0, m, n)] = 1
    choices, rings, sums = e.encrypt_choice(m, values, seed=SEED)
    choices, rings, sums = choices.copy(), rings.copy(), sums.copy()
    W.tamper_choice(choices, rings, sums, random.Random(5), frac=0.01)
    t_v, (v, tally) = timed(lambda: e.verify_choice(m, choices, rings, sums), args.reps)
    t_w, (ws, ws_ok) = timed(lambda: e.weighted_sum(choices, np.ones(n, np.uint64), v), args.reps)
    assert ws_ok and (ws == tally).all()
    d_cts, d_v = torch.from_numpy(choices.reshape(n, -1)).cuda(), torch.from_numpy(v).cuda()
    d_w = torch.from_numpy(np.ones(n, np.uint64).view(np.uint8).reshape(n, 8)).cuda()
    d_s = torch.zeros((n, 32), dtype=torch.uint8, device="cuda")
    d_s[:, :8] = d_w
    d_wout, d_wok = torch.zeros(64 * m, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def ws_dev():
        e.weighted_sum_dev(n, m, 64 * m, 64, d_cts.data_ptr(), d_s.data_ptr(), d_v.data_ptr(), d_wout.data_ptr(), d_wok.data_ptr())
        torch.cuda.synchronize()
    t_wd, _ = timed(ws_dev, args.reps)
    assert (d_wout.cpu().numpy().reshape(m, 64) == tally).all()
    res["yardsticks"] = {"verify_choice_ms": t_v * 1e3, "weighted_sum_weights1_host_ms": t_w * 1e3,
                         "weighted_sum_weights1_dev_ms": t_wd * 1e3, "rejected": int((v != 0).sum())}
    print(json.dumps(res["yardsticks"]), flush=True)
    shapes = [(1, "single")] + [(g, k) for g in GROUPS[1:] for k in ("uniform", "zipf", "single")]
    kinds = {"single": "one", "uniform": "uniform", "zipf": "zipf"}
    for ng, kind in shapes:
        groups = GS.group_ids(n, ng, kinds[kind], seed=3)
        d_g = torch.from_numpy(groups.view(np.int32)).cuda()
        d_out, d_ok = torch.zeros(ng * m * 64, dtype=torch.uint8, device="cuda"), torch.zeros(ng, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()

        def dev():
            e.group_sum_dev(n, m, 64 * m, 64, d_cts.data_ptr(), d_g.data_ptr(), ng, d_v.data_ptr(), d_out.data_ptr(), d_ok.data_ptr())
            torch.cuda.synchronize()
        t_dev, _ = timed(dev, args.reps)
        t_host, (out, ok) = timed(lambda: e.group_sum(choices, groups, ng, v), args.reps)
        assert ok.all() and d_ok.cpu().numpy().all() and (d_out.cpu().numpy().reshape(ng, m, 64) == out).all()
        total, sok = e.ciphertexts_sum(out)
        assert sok and (total == tally).all(), "the group totals do not add up to the verifier's tally"
        sizes = np.bincount(groups[v == 0], minlength=ng)
        row = {"n_groups": ng, "distribution": kind, "dev_ms": t_dev * 1e3, "host_ms": t_host * 1e3,
               "largest_group": int(sizes.max()), "empty_groups": int((sizes == 0).sum()),
               "dev_over_weighted_sum_dev": t_dev / t_wd, "dev_over_verify_choice": t_dev / t_v}
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
        del d_g, d_out, d_ok
    # the loop the grouped fold replaces: host-sorted items, one unit-weight weighted sum per group
    ng = 10**3
    groups = GS.group_ids(n, ng, "uniform", seed=3)
    out, _ = e.group_sum(choices, groups, ng, v)

    def loop():
        order = np.argsort(groups, kind="stable")
        bounds = np.searchsorted(groups[order], np.arange(ng + 1))
        c, vv = choices[order], v[order]
        ones = np.ones(n, np.uint64)
        res_ = np.empty((ng, m, 64), np.uint8)
        for g in range(ng):
            a, b = bounds[g], bounds[g + 1]
            res_[g], ok_ = e.weighted_sum(c[a:b], ones[a:b], vv[a:b])
            assert ok_
        return res_
    t_loop, lo = timed(loop, max(1, args.reps // 2))
    assert (lo == out).all()
    grouped = [r for r in res["rows"] if r["n_groups"] == ng and r["distribution"] == "uniform"][0]
    res["per_group_loop"] = {"n_groups": ng, "distribution": "uniform", "loop_ms": t_loop * 1e3,
                             "loop_over_group_sum_host": t_loop / (grouped["host_ms"] / 1e3)}
    print(json.dumps(res["per_group_loop"]), flush=True)
    if torch.cuda.device_count() > 1:
        k = torch.cuda.device_count()
        mc = Engine(devices=list(range(k)))
        mc.set_receiver(pk)
        res["multi"] = {"devices": k, "rows": []}
        for ng in (1, 2 * 10**5):
            groups = GS.group_ids(n, ng, "uniform", seed=3)
            t_m, (out, ok) = timed(lambda: mc.group_sum(choices, groups, ng, v), args.reps)
            assert ok.all() and (e.ciphertexts_sum(out)[0] == tally).all()
            res["multi"]["rows"].append({"n_groups": ng, "host_ms": t_m * 1e3})
        mc.close()
        print(json.dumps(res["multi"]), flush=True)
    # per-kernel device times, in a separate pass (profiling slows the host)
    prof = {}
    for ng, nn, mm in ((2 * 10**5, n, m), (GS.MAX_CELLS, 10**5, 1)):
        groups = GS.group_ids(nn, ng, "uniform", seed=4)
        d_g = torch.from_numpy(groups.view(np.int32)).cuda()
        d_out, d_ok = torch.zeros(ng * mm * 64, dtype=torch.uint8, device="cuda"), torch.zeros(ng, dtype=torch.uint8, device="cuda")
        d_c = d_cts if mm == m else torch.from_numpy(choices[:nn, 0].copy()).cuda()
        torch.cuda.synchronize()

        def one():
            e.group_sum_dev(nn, mm, 64 * mm, 64, d_c.data_ptr(), d_g.data_ptr(), ng, 0, d_out.data_ptr(), d_ok.data_ptr())
            torch.cuda.synchronize()
        t_one, _ = timed(one, args.reps)
        key = f"n={nn} n_cts={mm} n_groups={ng}"
        prof[key] = {"dev_ms": t_one * 1e3, "kernels_ms": kernel_times(one)}
        print(key, json.dumps(prof[key]), flush=True)
        del d_g, d_out, d_ok
    res["kernels"] = prof
    pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    e.close()


if __name__ == "__main__":
    main()
