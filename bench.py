#!/usr/bin/env python3
"""bench.py -- the five BASELINE.json configs through the C ABI of libeg_b200.so; config 2 is the headline and the default.

    python bench.py [--config C] --gpus N --steps K --warmup W [--dump-outputs DIR]     (N > 1: launched under torchrun)
    python bench.py [--config C] --impl reference --gpus N --steps K --warmup W     (the CPU restatement of the same path)

    C = 1  encrypt_bool + RingProof verify of 10 000 Boolean ciphertexts (benches/basics.rs:60-82 shape; latency-bound at
           that size, so the line also carries the saturated rate at 4 M ciphertexts)
        2  EncryptedChoice::single, 5 options: batch verify 1 M ballots + homomorphic tally      [default, BASELINE `metric`]
        3  QuadraticVotingBallot 5 options / 20 credits: batch verify 1 M ballots + tally
        4  RangeProof for [0, 2^16) (RangeDecomposition::optimal: 8 rings x 4), 1 M proofs
        5  3-of-5 verifiable decryption shares (LogEqualityProof) on 1 M tallies + combine + DiscreteLogTable lookup

One step = one pass of the hot path over one batch of `--items` units per GPU.  `value` is measured with the inputs
already resident in HBM (device-pointer entry points, CUDA events on the context's stream); `e2e` goes through the
host-pointer entry points with PINNED host buffers, H2D + D2H inside the timed region (`e2e.pageable` = the same with
ordinary pageable arrays, what a Rust Vec<u8> caller gets).  `roofline` = the dominant kernel against the INT32
multiply-add issue rate measured live by tools/microbench/int_pipe_bench; `cpu_baseline` = the oracle port on this
box's host cores.  Multi-GPU: one process per GPU; units shard across ranks; the partial tallies of configs 2 and 3 are
combined INSIDE the library (eg_ctx_attach_comm: ncclAllGather + point-add kernel) -- torch.distributed only carries
the 128-byte NCCL id and the barriers of the timing protocol.  `--scaling strong` keeps the total at the BASELINE size.

Synthetic data: `--unique` distinct items are produced by the oracle's prover from the seeded ChaCha streams of SURVEY.md
8(d) (1 % tampered with the reference's tamper patterns) and tiled to the batch size; cost does not depend on contents
(uniform control flow); every timed batch's verdicts / tallies / values are checked against the oracle's.  With the same
arguments the inputs are the same from run to run: `--dump-outputs DIR` writes what the last timed step returned as
DIR/<name>.npy, so that two builds of the library can be compared output for output.
"""
import argparse
import json
import os
import pathlib
import random
import subprocess
import sys
import tempfile
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
for p in (str(ROOT), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

# Reference-equivalent algorithmic work (SURVEY.md 8(d), A.6): one verification-equation side = half of a (double-base +
# 2-term) pair, 4956 / 2 field operations, plus one compression of 280; 144 IMAD-class instructions per field operation.
FIELD_OPS_PER_SIDE = 4956 / 2 + 280                      # 2758
FIELD_OPS_3TERM_SUM = 0.75 * 4956                        # a 3-term multi-scalar sum (Lagrange recombination)
IMAD_PER_FIELD_OP = 144
# executed work: one fixed-base term = one mixed addition (7 field operations) per window of the wide tables (24-bit windows:
# 11; elastic_elgamal_b200/csrc/ge.cuh EG_WIDE_BITS)
FIXED_TERM_OPS = 11 * 7
L2_BYTES = 126 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--items", "--ballots", type=int, default=0, help="units per GPU per step (0 = the BASELINE size)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: the BASELINE size is the total over all GPUs")
    ap.add_argument("--unique", type=int, default=0, help="distinct oracle-generated items that are tiled (0 = per config)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="items in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ring-mode", type=int, default=-1, choices=[-1, 0, 1, 2, 3], help="-1: per config (2 = k_ring for the large batches)")
    ap.add_argument("--chunk", type=int, default=0, help="items per internal chunk (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32 / float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 arm: the reference arm times the oracle on samples it does not keep")
    return args


# =============================================================================== workloads

def tile(a, n):
    import numpy as np
    reps = (n + a.shape[0] - 1) // a.shape[0]
    return np.ascontiguousarray(np.tile(a, (reps,) + (1,) * (a.ndim - 1))[:n])


class Workload:
    """One BASELINE config: unique oracle-made inputs, expected outputs, the device / host steps and the CPU leg."""
    cid = 0
    metric = unit = workload = ""
    default_items = 1 << 20
    default_unique = 2053                 # a prime: the tampered positions of the tiled batch do not line up with warps / CTAs
    bytes_per_item = 0
    ref_field_ops_per_item = 0.0
    ring_mode = 2
    kernel = "k_ring"
    kernel_kind = 1                       # eg_last_kernel_stats kind of the dominant kernel
    field_ops_per_task = FIELD_OPS_PER_SIDE
    executed_field_ops_per_task = None
    has_tally = False
    options = 0
    output_names = ("verdicts",)

    def make(self, unique, threads):      # -> None; fills self.inputs (list of unique arrays) and expectations
        raise NotImplementedError

    def setup(self, e):
        pass

    def outputs(self, n):                 # [(shape, numpy dtype)], in the order of output_names
        raise NotImplementedError

    def step_dev(self, e, n, d_in, d_out):
        raise NotImplementedError

    def step_host(self, e, n, h_in, h_out):
        raise NotImplementedError

    def check(self, n, out, world, unique):
        raise NotImplementedError

    def cpu(self, sample, threads):       # -> seconds for `sample` items
        raise NotImplementedError


class Bool(Workload):
    cid = 1
    metric = "verified Boolean ciphertexts/sec (encrypt_bool RingProof)"
    unit = "ciphertexts/s"
    workload = "PublicKey::verify_bool on 10k Boolean ciphertexts (BASELINE configs[0], benches/basics.rs:60-82)"
    default_items = 10000
    bytes_per_item = 160
    ref_field_ops_per_item = 12.1e3
    ring_mode = 0                         # the library picks the pair engine (k_ring_pair) for a batch this small
    executed_field_ops_per_task = 1949.5 - 1.25 * (112 - FIXED_TERM_OPS)      # as config 2's ring sides

    def make(self, unique, threads):
        import oracle as O
        import workloads as W
        self.sk, self.pk = W.receiver()
        cts, proofs = O.gen_bool_batch(self.pk, W.SEED_CHOICE, unique, threads=threads)
        cts, proofs = cts.copy(), proofs.copy()
        W.tamper_bool(cts, proofs, random.Random(1), frac=0.01)
        self.inputs = [cts, proofs]
        self.expected = O.verify_bool_batch(self.pk, cts, proofs, threads=threads)

    def setup(self, e):
        e.set_receiver(self.pk)

    def outputs(self, n):
        import numpy as np
        return [((n,), np.uint8)]

    def step_dev(self, e, n, d_in, d_out):
        e._check(e.lib.eg_verify_bool_batch_dev(e.h, n, d_in[0], d_in[1], d_out[0]))

    def step_host(self, e, n, h_in, h_out):
        e._check(e.lib.eg_verify_bool_batch(e.h, n, h_in[0], h_in[1], h_out[0]))

    def check(self, n, out, world, unique):
        assert (out[0] == tile(self.expected, n)).all(), "verdict mismatch against the oracle"

    def cpu(self, sample, threads):
        import oracle as O
        c, p = tile(self.inputs[0], sample), tile(self.inputs[1], sample)
        t0 = time.perf_counter()
        O.verify_bool_batch(self.pk, c, p, threads=threads)
        return time.perf_counter() - t0


class Choice(Workload):
    cid = 2
    metric = "verified ballots/sec (5-option choice)"
    unit = "ballots/s"
    workload = "EncryptedChoice::single 5 options: batch verify + homomorphic tally (BASELINE configs[1])"
    default_unique = 4099
    options = 5
    bytes_per_item = 5 * 64 + 11 * 32 + 64         # 736, SURVEY.md 8(a) a12
    ref_field_ops_per_item = 4956 * 11 + 280 * (34 + 10)      # 66 836
    has_tally = True
    output_names = ("verdicts", "tally")
    # what k_ring executes per equation side of a two-equation ring (DESIGN.md 5): 2 x 1603 table build + 4 sides x (435 + 497
    # + 112) + 112 for [e a]G + 304 for encoding the first equation's pair
    executed_field_ops_per_task = (2 * 1603 + 4 * (435 + 497 + FIXED_TERM_OPS) + FIXED_TERM_OPS + 304) / 4

    def make(self, unique, threads):
        import oracle as O
        import workloads as W
        self.sk, self.pk = W.receiver()
        cts, rings, sums = O.gen_choice_batch(self.pk, 5, W.SEED_CHOICE, unique, threads=threads)
        cts, rings, sums = cts.copy(), rings.copy(), sums.copy()
        W.tamper_choice(cts, rings, sums, random.Random(2), frac=0.01)
        self.inputs = [cts, rings, sums]
        self.expected, _ = O.verify_choice_batch(self.pk, 5, True, cts, rings, sums, threads=threads)

    def setup(self, e):
        e.set_receiver(self.pk)

    def outputs(self, n):
        import numpy as np
        return [((n,), np.uint8), ((5, 64), np.uint8)]

    def step_dev(self, e, n, d_in, d_out):
        e._check(e.lib.eg_verify_choice_batch_dev(e.h, n, 5, 1, d_in[0], d_in[1], d_in[2], d_out[0], d_out[1]))

    def step_host(self, e, n, h_in, h_out):
        e._check(e.lib.eg_verify_choice_batch(e.h, n, 5, 1, h_in[0], h_in[1], h_in[2], h_out[0], h_out[1]))

    def check(self, n, out, world, unique):
        import numpy as np
        import oracle as O
        ev = tile(self.expected, n)
        assert (out[0] == ev).all(), "verdict mismatch against the oracle"
        if world * n + 1 <= (1 << 22) + 1:
            # the tally of the timed batch (over ALL ranks: every rank runs the same tiled batch) decrypts to the number of
            # accepted ballots per option
            table = O.DlogTable(0, world * n + 1)
            idx = np.arange(n)
            for k in range(5):
                expect = world * int(np.count_nonzero((ev == 0) & ((idx % unique) % 5 == k)))
                got = table.get(O.decrypt_to_element(self.sk, bytes(out[1][k])))
                assert got == expect, (k, got, expect)

    def cpu(self, sample, threads):
        import oracle as O
        c, r, s = (tile(a, sample) for a in self.inputs)
        t0 = time.perf_counter()
        O.verify_choice_batch(self.pk, 5, True, c, r, s, threads=threads)
        return time.perf_counter() - t0


class Qv(Workload):
    cid = 3
    metric = "verified quadratic-voting ballots/sec (5 options, 20 credits)"
    unit = "ballots/s"
    workload = "QuadraticVotingBallot 5 options / 20 credits: batch verify + tally (BASELINE configs[2])"
    options = 5
    ref_field_ops_per_item = 256e3
    has_tally = True
    output_names = ("verdicts", "tally")

    def make(self, unique, threads):
        import numpy as np
        import oracle as O
        import parity_common as PC
        import workloads as W
        self.sk, self.pk = W.receiver()
        self.p = O.qv_params(5, 20)
        self.votes = np.array([PC.QV_VOTES[i % 4] for i in range(unique)], np.uint64)
        ballots = O.gen_qv_batch(self.pk, self.p, W.SEED_QV, self.votes, threads=threads).copy()
        self.bytes_per_item = int(ballots.shape[1])
        rnd = random.Random(3)
        for k, i in enumerate(sorted(rnd.sample(range(unique), max(1, unique // 100)))):
            if k % 3 == 0:
                ballots[i, 32:64] = np.frombuffer(O.point_add(bytes(ballots[i, 32:64]), W.G_ENC), np.uint8)
            elif k % 3 == 1:
                ballots[i, -32 * 12:] = ballots[(i + 1) % unique, -32 * 12:]
            else:
                ballots[i, -1] = 0xff
        self.inputs = [ballots]
        self.expected, _ = O.verify_qv_batch(self.pk, self.p, ballots, threads=threads)

    def setup(self, e):
        import ctypes as C
        e.set_receiver(self.pk)
        self.ep = e.qv_params(5, 20)
        self.ep_ref = C.byref(self.ep)

    def outputs(self, n):
        import numpy as np
        return [((n,), np.uint8), ((5, 64), np.uint8)]

    def step_dev(self, e, n, d_in, d_out):
        e._check(e.lib.eg_verify_qv_batch_dev(e.h, self.ep_ref, n, d_in[0], d_out[0], d_out[1]))

    def step_host(self, e, n, h_in, h_out):
        e._check(e.lib.eg_verify_qv_batch(e.h, self.ep_ref, n, h_in[0], h_out[0], h_out[1]))

    def check(self, n, out, world, unique):
        import oracle as O
        ev = tile(self.expected, n)
        assert (out[0] == ev).all(), "verdict mismatch against the oracle"
        if 4 * world * n + 1 <= (1 << 23):
            table = O.DlogTable(0, 4 * world * n + 1)
            vt = tile(self.votes, n)
            for k in range(5):
                got = table.get(O.decrypt_to_element(self.sk, bytes(out[1][k])))
                assert got == world * int(vt[ev == 0, k].sum()), (k, got)

    def cpu(self, sample, threads):
        import oracle as O
        b = tile(self.inputs[0], sample)
        t0 = time.perf_counter()
        O.verify_qv_batch(self.pk, self.p, b, threads=threads)
        return time.perf_counter() - t0


class Range(Workload):
    cid = 4
    metric = "verified range proofs/sec ([0, 2^16))"
    unit = "proofs/s"
    workload = "RangeProof verification for ciphertexts in [0, 2^16) via RangeDecomposition::optimal (BASELINE configs[3])"
    bytes_per_item = 64 + 7 * 64 + 33 * 32        # 1568
    ref_field_ops_per_item = 185.5e3
    # k_ring<256,2,8> per side of a four-equation ring: 2 x 2072 table build (224 doublings + 56 additions per point) + 8 sides
    # x (196 + 497 + 112) + 3 x 112 for [e a]G + 3 x 304 encodings, over 8 sides
    executed_field_ops_per_task = (2 * 2072 + 8 * (196 + 497 + FIXED_TERM_OPS) + 3 * FIXED_TERM_OPS + 3 * 304) / 8

    def make(self, unique, threads):
        import numpy as np
        import oracle as O
        import parity_common as PC
        import workloads as W
        self.sk, self.pk = W.receiver()
        self.spec = O.range_optimal(65536)
        values = (np.arange(unique, dtype=np.uint64) * 40503) % 65536
        cts, partials, rings = O.gen_range_batch(self.pk, self.spec, "ciphertext_range", W.SEED_CHOICE, values, threads=threads)
        cts, partials, rings = cts.copy(), partials.copy(), rings.copy()
        PC.tamper_range(cts, partials, rings, random.Random(4), 0.01)
        self.inputs = [cts, partials, rings]
        self.expected = O.verify_range_batch(self.pk, self.spec, "ciphertext_range", cts, partials, rings, threads=threads)

    def setup(self, e):
        import ctypes as C
        import parity_common as PC
        e.set_receiver(self.pk)
        self.espec = PC.to_engine_range(e, self.spec)
        self.espec_ref = C.byref(self.espec)

    def outputs(self, n):
        import numpy as np
        return [((n,), np.uint8)]

    def step_dev(self, e, n, d_in, d_out):
        e._check(e.lib.eg_verify_range_batch_dev(e.h, self.espec_ref, b"ciphertext_range", n, d_in[0], d_in[1], d_in[2], d_out[0]))

    def step_host(self, e, n, h_in, h_out):
        e._check(e.lib.eg_verify_range_batch(e.h, self.espec_ref, b"ciphertext_range", n, h_in[0], h_in[1], h_in[2], h_out[0]))

    def check(self, n, out, world, unique):
        assert (out[0] == tile(self.expected, n)).all(), "verdict mismatch against the oracle"

    def cpu(self, sample, threads):
        import oracle as O
        c, p, r = (tile(a, sample) for a in self.inputs)
        t0 = time.perf_counter()
        O.verify_range_batch(self.pk, self.spec, "ciphertext_range", c, p, r, threads=threads)
        return time.perf_counter() - t0


class Shares(Workload):
    cid = 5
    metric = "threshold-decrypted tallies/sec (3-of-5 shares verified + combined + dlog lookup)"
    unit = "tallies/s"
    workload = "3-of-5 verifiable decryption shares (LogEqualityProof) + combine_shares + DiscreteLogTable(0..2^20) (BASELINE configs[4])"
    default_unique = 1031                 # the oracle's share prover runs item by item through ctypes
    bytes_per_item = 64 + 3 * (32 + 64)   # 352
    ref_field_ops_per_item = 27e3
    kernel = "k_msm"
    kernel_kind = 2
    output_names = ("share_verdicts", "values", "found")
    # k_msm tasks per tally: 6 equation sides (3 shares x 2) + one 3-term recombination
    field_ops_per_task = (6 * FIELD_OPS_PER_SIDE + FIELD_OPS_3TERM_SUM) / 7
    USED = (0, 2, 4)
    TABLE_HI = 1 << 20

    def make(self, unique, threads):
        import numpy as np
        import oracle as O
        rng = O.rng_from_seed(bytes([9] * 32))
        self.ks, secrets = O.dealer_new(5, 3, rng)
        shared = bytes(self.ks.shared_key)
        rnd = random.Random(5)
        self.values = np.array([rnd.randrange(self.TABLE_HI) for _ in range(unique)], np.uint64)
        cts = [O.encrypt(shared, int(v), rng) for v in self.values]
        rows = [[O.decrypt_share(self.ks, i, secrets[i], ct, rng) for i in self.USED] for ct in cts]
        cts_a = np.frombuffer(b"".join(cts), np.uint8).reshape(unique, 64).copy()
        sh_a = np.frombuffer(b"".join(b"".join(r[0] for r in row) for row in rows), np.uint8).reshape(unique, 3, 32).copy()
        pr_a = np.frombuffer(b"".join(b"".join(r[1] for r in row) for row in rows), np.uint8).reshape(unique, 3, 64).copy()
        for k, i in enumerate(sorted(rnd.sample(range(unique), max(1, unique // 100)))):
            pr_a[i, k % 3] = pr_a[(i + 1) % unique, k % 3]        # proof of another tally: share rejected, decryption unaffected
        self.inputs = [cts_a, sh_a, pr_a]
        self.expected = np.array([[O.verify_share(self.ks, self.USED[j], bytes(cts_a[i]), bytes(sh_a[i, j]), bytes(pr_a[i, j]))
                                   for j in range(3)] for i in range(unique)], np.uint8)

    def setup(self, e):
        import ctypes as C
        import parity_common as PC
        self.eks = PC.as_engine_keyset(self.ks)
        self.eks_ref = C.byref(self.eks)
        self.idx = (C.c_uint32 * 3)(*self.USED)
        t0 = time.perf_counter()
        self.table = e.dlog_table(0, self.TABLE_HI)
        self.table_build_s = time.perf_counter() - t0

    def outputs(self, n):
        import numpy as np
        return [((n, 3), np.uint8), ((n,), np.uint64), ((n,), np.uint8)]

    def step_dev(self, e, n, d_in, d_out):
        e._check(e.lib.eg_verify_shares_batch_dev(e.h, self.eks_ref, n, 3, self.idx, d_in[0], d_in[1], d_in[2], d_out[0]))
        self.stats = e.last_kernel_stats(2)
        e._check(e.lib.eg_combine_decrypt_batch_dev(e.h, 3, self.idx, n, 3, d_in[0], d_in[1], self.table.h, d_out[1], d_out[2]))

    def step_host(self, e, n, h_in, h_out):
        e._check(e.lib.eg_verify_shares_batch(e.h, self.eks_ref, n, 3, self.idx, h_in[0], h_in[1], h_in[2], h_out[0]))
        e._check(e.lib.eg_combine_decrypt_batch(e.h, 3, self.idx, n, 3, h_in[0], h_in[1], self.table.h, h_out[1], h_out[2]))

    def check(self, n, out, world, unique):
        assert (out[0] == tile(self.expected, n)).all(), "share verdict mismatch against the oracle"
        assert (out[2] == 1).all() and (out[1] == tile(self.values, n)).all(), "decrypted value mismatch"

    def cpu(self, sample, threads):
        import oracle as O
        from concurrent.futures import ThreadPoolExecutor
        cts_a, sh_a, pr_a = self.inputs
        u = cts_a.shape[0]
        used = list(self.USED)

        def work(rng):                    # per-item ctypes calls into the C oracle; ctypes drops the GIL for their duration
            for q in range(*rng):
                i = q % u
                ct = bytes(cts_a[i])
                sh = [bytes(sh_a[i, j]) for j in range(3)]
                for j in range(3):
                    O.verify_share(self.ks, self.USED[j], ct, sh[j], bytes(pr_a[i, j]))
                O.combine_decrypt(used, sh, ct)

        t0 = time.perf_counter()
        if threads <= 1:
            work((0, sample))
        else:
            step = (sample + threads - 1) // threads
            with ThreadPoolExecutor(threads) as pool:
                list(pool.map(work, [(lo, min(sample, lo + step)) for lo in range(0, sample, step)]))
        return time.perf_counter() - t0



WORKLOADS = {1: Bool, 2: Choice, 3: Qv, 4: Range, 5: Shares}


# =============================================================================== instrumentation

class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def int32_peak():
    """Measured INT32 multiply-add issue rate (lane-ops / s) of this GPU: tools/microbench/int_pipe_bench."""
    exe = ROOT / "tools" / "microbench" / "int_pipe_bench"
    try:
        with tempfile.TemporaryDirectory() as tmp:
            if not exe.exists():  # built by __graft_entry__.build(); otherwise compiled here, outside the tree
                src, exe = str(exe) + ".cu", pathlib.Path(tmp) / exe.name
                subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-o", str(exe),
                                src], check=True, timeout=600)
            out = subprocess.run([str(exe), "8192"], check=True, stdout=subprocess.PIPE, text=True, timeout=120).stdout
        return json.loads(out.strip().splitlines()[-1])
    except Exception as exc:      # the bench line then carries peak = None
        return {"error": repr(exc), "tests": {}}


def hbm_peak():
    try:
        return float(json.loads((ROOT / "MEASURED_PEAKS.json").read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


_REAL_STDOUT = None


def emit(line):
    """The one JSON line of the contract goes to the process's original stdout."""
    data = (line + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line + "\n")
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def cpu_rates(wl, threads, target_s, sample_override=0):
    """(all-thread rate, single-thread rate, sample, seconds): the oracle on a bounded sample sized for ~target_s seconds."""
    probe = 64 if wl.cid in (3, 4) else 256
    single = probe / wl.cpu(probe, 1)
    if getattr(wl, "cpu_single_thread_only", False):
        sample = sample_override or max(probe, int(single * target_s))
        dt = wl.cpu(sample, 1)
        return sample / dt, sample / dt, sample, dt, 1
    sample = sample_override or max(probe, int(single * threads * target_s) // 64 * 64)
    dt = wl.cpu(sample, threads)
    return sample / dt, single, sample, dt, threads


DUMP_BYTES = 64_000_000


def dump_outputs(directory, names, arrays, n):
    """DIR/<name>.npy for every output of a step over `n` items: float32 for bytes and flags, float64 for wider integers
    (both exact).  When the files would exceed DUMP_BYTES in all, every per-item output keeps the same seeded sample of
    items, whose indices go to DIR/sample_index.npy."""
    import numpy as np
    outs = {name: a.astype(np.float32 if a.dtype.itemsize == 1 else np.float64) for name, a in zip(names, arrays)}
    per_item = [k for k, a in outs.items() if a.shape[0] == n]
    total, budget = sum(a.nbytes for a in outs.values()), DUMP_BYTES - 4096       # 4096: room for the .npy headers
    if total > budget:
        fixed = total - sum(outs[k].nbytes for k in per_item)
        row = sum(outs[k].nbytes for k in per_item) // n + 8                         # + its float64 sample index
        idx = np.sort(np.random.default_rng(0).choice(n, (budget - fixed) // row, replace=False))
        outs = {k: (a[idx] if k in per_item else a) for k, a in outs.items()}
        outs["sample_index"] = idx.astype(np.float64)
    directory.mkdir(parents=True, exist_ok=True)
    for k, a in outs.items():
        np.save(directory / f"{k}.npy", a)


# =============================================================================== reference arm

def run_reference(args):
    """`--impl reference`: the reference crate is Rust and cannot be built in this image (no cargo/rustc), so the arm times
    the oracle port of the same path on all host cores (cpu_baseline.kind = "port"), each step a bounded sample."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import oracle as O
    threads = O.hw_threads()
    wl = WORKLOADS[args.config]()
    wl.make(min(args.unique or wl.default_unique, 2048), threads)
    _, single, sample, _, used = cpu_rates(wl, threads, 2.0, args.cpu_sample)
    t = 1 if used == 1 else threads
    for _ in range(args.warmup):
        wl.cpu(max(32, sample // 8), t)
    t_tot = sum(wl.cpu(sample, t) for _ in range(args.steps))
    value = sample * args.steps / t_tot
    line = {
        "impl": "reference", "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "u64 limbs (GF(2^255-19), radix 2^51)", "data": "synthetic seeded items (oracle prover)",
        "config": {"workload": wl.workload, "config": wl.cid, "items_per_step": sample,
                   "note": "bounded sample of the BASELINE-size workload; units are independent"},
        "cpu_baseline": {"value": value, "unit": wl.unit, "cores": used, "kind": "port",
                         "sample": f"{sample} items/step x {args.steps} steps, {used} threads; single thread {single:.1f} {wl.unit}"},
        "e2e": {"value": value, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(line))


# =============================================================================== the B200 arm

def main():
    global _REAL_STDOUT
    args = parse_args()
    # Libraries print to stdout behind our back (NCCL's version banner when NCCL_DEBUG=VERSION, for one): route file
    # descriptor 1 to stderr for the whole run and keep the original stdout for the JSON line alone.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch

    import oracle as O
    from elastic_elgamal_b200 import Engine
    from elastic_elgamal_b200 import build as eg_build

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not eg_build.LIB.exists() and "EG_B200_LIB" not in os.environ:
        # __graft_entry__.build() leaves the CUDA library in the package.  Without it, compile it (nvcc, sm_100a) into the
        # temporary directory, never into the tree, which may be read-only.  Rank 0 of a node builds, the others wait for
        # an up-to-date file.  There is no other implementation to fall back to.
        lib = pathlib.Path(tempfile.gettempdir()) / f"eg_b200_bench_{os.getuid()}" / eg_build.LIB.name
        lib.parent.mkdir(exist_ok=True)
        if local_rank == 0:
            eg_build.build(lib=lib)
        else:
            for _ in range(1200):
                if not eg_build.needs_build(lib):
                    break
                time.sleep(0.5)
        os.environ["EG_B200_LIB"] = str(lib)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    wl = WORKLOADS[args.config]()
    threads = O.hw_threads()
    gen_threads = max(1, threads // max(1, min(world, 8)))
    unique = args.unique or wl.default_unique
    wl.make(unique, gen_threads)
    B = args.items or (wl.default_items // world if args.scaling == "strong" else wl.default_items)

    e = Engine(device=local_rank)
    if world > 1:
        # control plane only: rank 0's NCCL id reaches the other ranks through torch.distributed; the communicator, the
        # all-gather of the partial tallies and the point addition live inside libeg_b200.so (eg_ctx_attach_comm)
        uid = torch.from_numpy(e.comm_unique_id() if rank == 0 else np.zeros(128, np.uint8)).to(dev)
        dist.broadcast(uid, 0)
        e.attach_comm(uid.cpu().numpy(), rank, world)
    wl.setup(e)
    e.set_ring_mode(args.ring_mode if args.ring_mode >= 0 else wl.ring_mode)
    if args.chunk:
        e.set_chunk_items(args.chunk)

    h_in = [tile(a, B) for a in wl.inputs]
    in_bytes = sum(a.nbytes for a in h_in)
    d_in = [torch.from_numpy(a).to(dev) for a in h_in]
    out_specs = wl.outputs(B)
    tdt = {np.dtype(np.uint8): torch.uint8, np.dtype(np.uint64): torch.int64}
    d_out = [torch.empty(shape, dtype=tdt[np.dtype(dt)], device=dev) for shape, dt in out_specs]
    out_bytes = sum(t.numel() * t.element_size() for t in d_out)
    stream = torch.cuda.ExternalStream(e.stream, device=dev)
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev) if in_bytes < 2 * L2_BYTES else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_dev():
        wl.step_dev(e, B, [t.data_ptr() for t in d_in], [t.data_ptr() for t in d_out])

    # ---------------- device-resident throughput (`value`): CUDA events on the context's stream around every step
    for _ in range(args.warmup):
        run_dev()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = e.kernel_launches
    k_ms, k_tasks, k_launches = 0.0, 0, 0
    o_ms, o_tasks, o_launches = 0.0, 0, 0
    p_ms, p_tasks, p_launches = 0.0, 0, 0
    pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with torch.cuda.stream(stream):
        for ev0, ev1 in pairs:
            if flush is not None:
                flush.zero_()           # inputs smaller than the L2: evict them between timed iterations (outside the events)
            ev0.record(stream)
            run_dev()
            ev1.record(stream)
            st = getattr(wl, "stats", None) if wl.cid == 5 else None
            st2 = e.last_kernel_stats(wl.kernel_kind)
            for s in ([st, st2] if st else [st2]):
                k_ms += s["ms"]; k_tasks += s["tasks"]; k_launches += s["launches"]
            if wl.kernel_kind == 1:
                s = e.last_kernel_stats(0)
                o_ms += s["ms"]; o_tasks += s["tasks"]; o_launches += s["launches"]
                s = e.last_kernel_stats(3)
                p_ms += s["ms"]; p_tasks += s["tasks"]; p_launches += s["launches"]
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in pairs)
    launches = e.kernel_launches - launches0
    sampler.stop_flag = True
    sampler.join()
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    per_rank = None
    if world > 1:
        # every rank's own device time and median SM clock (reporting only): the step ends in the tally all-gather, so the
        # job runs at the pace of the slowest GPU
        mine = torch.tensor([dev_ms / args.steps, float(sampler.summary().get("sm_mhz") or 0)], dtype=torch.float64, device=dev)
        allr = torch.empty(2 * world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allr, mine)
        per_rank = allr.cpu().numpy().reshape(world, 2)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())

    # ---------------- correctness of what was timed
    def host_outs(tensors):
        return [x.cpu().numpy().view(np.dtype(dt)).reshape(shape) for x, (shape, dt) in zip(tensors, out_specs)]
    last = host_outs(d_out)
    wl.check(B, last, world, unique)
    if args.dump_outputs and rank == 0:
        dump_outputs(pathlib.Path(args.dump_outputs), wl.output_names, last, B)

    # ---------------- end-to-end through the host C ABI (`e2e`): host buffers, H2D + D2H inside, every step
    def e2e_run(h_arrays, h_outs, steps):
        ins, outs = [a.ctypes.data for a in h_arrays], [a.ctypes.data for a in h_outs]
        wl.step_host(e, B, ins, outs)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            wl.step_host(e, B, ins, outs)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    keep = []

    def pinned_like(a):
        tp = torch.empty(a.shape, dtype=tdt.get(a.dtype, torch.uint8), pin_memory=True)
        keep.append(tp)
        return tp.numpy().view(a.dtype)
    p_in = []
    for a in h_in:
        pa = pinned_like(a)
        pa[...] = a
        p_in.append(pa)
    p_out = [pinned_like(np.empty(shape, dt)) for shape, dt in out_specs]
    e2e_pinned_s = e2e_run(p_in, p_out, args.steps)
    wl.check(B, p_out, world, unique)
    g_out = [np.empty(shape, dt) for shape, dt in out_specs]
    page_steps = max(1, min(args.steps, 3))
    e2e_page_s = e2e_run(h_in, g_out, page_steps)
    wl.check(B, g_out, world, unique)

    # config 1 is latency-bound at its stated size: also report the saturated rate (4 M ciphertexts, device-resident)
    saturated = None
    if wl.cid == 1 and not args.items:
        n_sat = 1 << 22
        s_in = [torch.from_numpy(tile(a, n_sat)).to(dev) for a in wl.inputs]
        s_out = torch.empty(n_sat, dtype=torch.uint8, device=dev)
        e.set_ring_mode(2)
        sat = lambda: wl.step_dev(e, n_sat, [x.data_ptr() for x in s_in], [s_out.data_ptr()])
        sat()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            a.record(stream)
            sat(); sat()
            b.record(stream)
        torch.cuda.synchronize()
        st = e.last_kernel_stats(1)
        assert (s_out.cpu().numpy() == tile(wl.expected, n_sat)).all()
        saturated = {"items": n_sat, "value": 2 * n_sat / (a.elapsed_time(b) * 1e-3), "unit": wl.unit, "ring_mode": 2,
                     "k_ring_ms_per_launch": st["ms"] / max(1, st["launches"]), "k_ring_sides_per_launch": st["tasks"] / max(1, st["launches"])}
        e.set_ring_mode(args.ring_mode if args.ring_mode >= 0 else wl.ring_mode)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel + CPU baseline (rank 0)
    peak = int32_peak()
    imad = peak.get("tests", {}).get("imad", {})
    clk = sampler.summary()
    # peak = IMAD lane-ops/s measured with CUDA events by the microbenchmark, rescaled by (SM clock sampled during the
    # timed region) / (SM clock probed in the microbenchmark) when the two differ
    peak_ops = None
    if imad.get("per_s"):
        peak_ops = imad["per_s"]
        if clk.get("sm_mhz") and peak.get("sm_clock_mhz_probed"):
            peak_ops *= clk["sm_mhz"] / peak["sm_clock_mhz_probed"]
    dom_kernel, dom_kind = wl.kernel, wl.kernel_kind
    if wl.kernel_kind == 1 and k_ms == 0 and p_ms > 0:      # the library chose the pair engine (small batch of rings only)
        dom_kernel, k_ms, k_tasks, k_launches = "k_ring_pair (two lanes per ring, ring mode 3)", p_ms, p_tasks, p_launches
    elif wl.kernel_kind == 1 and k_ms == 0 and o_ms > 0:    # the library chose the per-equation pipeline (small batch)
        dom_kernel, k_ms, k_tasks, k_launches, o_ms = "k_commit (per-equation pipeline, ring mode 1)", o_ms, o_tasks, o_launches, 0.0
    achieved_ops = k_tasks * wl.field_ops_per_task * IMAD_PER_FIELD_OP / (k_ms * 1e-3) if k_ms > 0 else None
    traffic, traffic_src = None, None
    tfile = ROOT / "profiles" / "k_ring_traffic.json"
    if dom_kernel == "k_ring" and wl.cid == 2 and tfile.exists():
        try:        # dram bytes of one ncu-captured launch, rescaled to this run's equation sides per launch
            tj = json.loads(tfile.read_text())
            traffic = tj["dram_bytes_per_launch"] * (k_tasks / max(1, k_launches)) / tj["equation_sides_per_launch"]
            traffic_src = "from profiles/k_ring_traffic.json (one `ncu --set full` capture: dram__bytes_read.sum + dram__bytes_write.sum), rescaled by equation sides per launch; not measured in this run"
        except Exception:
            traffic = None
    hbm, hbm_src = hbm_peak()
    step_gbs = world * B * (wl.bytes_per_item + out_bytes / B) * args.steps / (dev_ms_max * 1e-3) / 1e9
    roofline = {
        "kernel": dom_kernel, "bound": "int32",
        "achieved": achieved_ops / 1e12 if achieved_ops else None, "peak": peak_ops / 1e12 if peak_ops else None,
        "unit": "T int32 multiply-add lane-ops/s",
        "frac": (achieved_ops / peak_ops) if achieved_ops and peak_ops else None,
        "peak_source": "measured live: tools/microbench/int_pipe_bench `imad` lane-ops/s (CUDA events; = 63 of the nominal 64 "
                       "lanes/clk/SM) at the SM clock sampled during the timed region (MEASURED_PEAKS.json has no integer peak)",
        "traffic": traffic, "traffic_source": traffic_src,
        "launches": k_launches, "avg_launch_ms": k_ms / max(1, k_launches),
        "share_of_step": k_ms / dev_ms if dev_ms else None,
        "algorithmic": {"field_ops_per_task": wl.field_ops_per_task, "imad_per_field_op": IMAD_PER_FIELD_OP,
                        "tasks_per_launch": k_tasks / max(1, k_launches),
                        "task": "multi-scalar sum (equation side or recombination)" if dom_kind == 2 else "verification-equation side"},
        # `achieved` counts the reference's algorithm (SURVEY 8(d)); the engine does less work per side (shared doublings,
        # chunked tables, inversion-only encoding), so the fraction of the pipe it really keeps busy is the lower one:
        "executed": ({"field_ops_per_task": wl.executed_field_ops_per_task,
                      "frac": achieved_ops * wl.executed_field_ops_per_task / wl.field_ops_per_task / peak_ops}
                     if achieved_ops and peak_ops and wl.executed_field_ops_per_task and dom_kernel == "k_ring" else None),
        "second_kernel": ({"kernel": "k_commit", "launches": o_launches, "equation_sides": o_tasks, "ms": o_ms,
                           "share_of_step": o_ms / dev_ms if dev_ms else None} if o_ms else None),
        "whole_step": {"ref_field_ops_per_item": wl.ref_field_ops_per_item,
                       "frac": (world * B * args.steps / (dev_ms_max * 1e-3) * wl.ref_field_ops_per_item * IMAD_PER_FIELD_OP / (world * peak_ops))
                       if peak_ops else None},
        "hbm": {"bound": "hbm", "achieved": step_gbs / world, "peak": hbm, "unit": "GB/s", "frac": step_gbs / world / hbm, "peak_source": hbm_src,
                "note": "input + output streaming of the whole step per GPU; the path is integer-pipe bound"},
        "microbench": {k: v.get("per_clk_per_sm") for k, v in peak.get("tests", {}).items()},
    }
    cpu = None
    if not args.no_cpu_baseline:
        rate, single, sample, dt, used = cpu_rates(wl, threads, 6.0, args.cpu_sample)
        cpu = {"value": rate, "unit": wl.unit, "cores": used, "kind": "port",
               "sample": f"{sample} items of the same workload on {used} thread(s) ({dt:.1f} s); single thread {single:.1f} {wl.unit}",
               "single_thread": single}

    value = world * B * args.steps / (dev_ms_max * 1e-3)
    line = {
        "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "u32 limbs (GF(2^255-19), integers mod l)",
        "data": f"synthetic: {unique} seeded oracle-proved items (1% tampered) tiled to {B}/GPU",
        "config": {"workload": wl.workload, "config": wl.cid, "items_per_gpu": B, "global_items": world * B,
                   "bytes_per_item": wl.bytes_per_item,
                   "l2": ("inputs and scratch exceed the 126 MB L2" if flush is None else "inputs fit the L2: a 252 MB buffer is rewritten between timed iterations"),
                   "parallelism": f"dp{world} over items; tally combine inside the library (ncclAllGather + point-add)" if world > 1 else "dp1",
                   "ring_mode": args.ring_mode if args.ring_mode >= 0 else wl.ring_mode},
        "e2e": {"value": world * B * args.steps / e2e_pinned_s, "unit": wl.unit, "h2d_bytes_per_step": in_bytes,
                "d2h_bytes_per_step": out_bytes, "steps": args.steps, "host_buffers": "pinned",
                "pageable": {"value": world * B * page_steps / e2e_page_s, "steps": page_steps}},
        "gpu_launches": launches,
        "clocks": clk,
        "roofline": roofline,
        "cpu_baseline": cpu,
    }
    if per_rank is not None:
        line["per_rank"] = {"ms_per_step": [round(float(x), 3) for x in per_rank[:, 0]], "sm_mhz": [int(x) for x in per_rank[:, 1]]}
    if saturated:
        line["saturated"] = saturated
    if wl.cid == 5:
        line["config"]["dlog_table"] = {"entries": wl.TABLE_HI, "build_s": wl.table_build_s}
    emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
