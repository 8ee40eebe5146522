"""The Merlin / STROBE-128 transcript at every block offset, shared by the CPU harness tests (test_hostsim_transcript.py) and
the `-m gpu` tests (test_gpu_transcript.py).

The host builds each call's transcript prefix (Transcript::new(label), the proof's dom-sep, the range `Display`, the key)
and the kernels continue it on the device.  STROBE absorbs into a 166-byte block, and meta-AD / AD never force a
permutation, so the offset in that block at which a kernel absorbs its elements, LE32 lengths and 2-byte op headers -- its
phase -- is (c + len(label)) mod 166, with c fixed by the entry point and shape, until the first challenge's PRF forces a
permutation.  Fixed labels check a handful of phases; these checks sweep the label length over 1..255, which reaches every
phase of every labelled entry point, and compare every output byte and verdict with the oracle.  Labels are built so that
their bytes vary with the length too, and a label of the same length (same phase) with another last byte must make every
proof fail, so the label's bytes -- not only its length -- are shown to reach the device prefix."""
import collections
import re

import numpy as np

import decrypt_common as D
import oracle as O
import pyref
import shape_common as SC
import sigma_prover_common as S
import workloads as W

RATE = 166
SWEEP = range(1, 256)
N = 3                                # items per call
SEED = bytes([0x6d] * 32)
RANGE_UB = 27                        # RangeDecomposition::optimal(27): three rings of 3
RING_MODES = (1, 2, 3)               # per-equation pipeline, k_ring, pair engine
MESSAGE_LENGTHS = (0, 1, 3, 4, 31, 32, 33, 165, 166, 167)
ALPHABET = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789_-"
NON_ASCII_LABELS = {"166 bytes": "é" * 83, "255 bytes": "€" * 85}


def label_of(length):
    """`length` ASCII bytes; the content depends on the length as well as on the position."""
    return "".join(ALPHABET[(5 * length + 7 * i) % len(ALPHABET)] for i in range(length))


def same_length_sibling(label):
    """The label with bit 0 of its last code point flipped: the same UTF-8 length (so the same phase), another last byte."""
    sib = label[:-1] + chr(ord(label[-1]) ^ 1)
    assert len(sib.encode()) == len(label.encode()) and sib.encode()[-1] != label.encode()[-1]
    return sib


# ---------------------------------------------------------------- the two references at every phase

def check_references_agree(lengths=range(256)):
    """The oracle's transcript (oracle/transcript.c) and pyref's independent STROBE / Merlin give the same state after
    Transcript::new(label) with every label length, after each message of MESSAGE_LENGTHS, and the same 64 challenge bytes."""
    for length in lengths:
        label = label_of(length)
        o, p = O.MerlinTranscript(label), pyref.Transcript(label.encode())
        steps = [("new", None)] + [("msg", m) for m in MESSAGE_LENGTHS]
        for k, (what, m) in enumerate(steps):
            if m is not None:
                msg = bytes((length + 31 * k + i) & 0xff for i in range(m))
                o.append_message("msg", msg)
                p.append_message(b"msg", msg)
            state, pos, pos_begin = o.state()
            assert (state, pos, pos_begin) == (bytes(p.strobe.state), p.strobe.pos, p.strobe.pos_begin), (length, what, m)
        assert o.challenge_bytes("challenge", 64) == p.challenge_bytes(b"challenge", 64), length


# ---------------------------------------------------------------- the labelled entry points

# run(label) -> the library's outputs; want -> the oracle's outputs for the label the entry was built with; reverify(label)
# -> the oracle's verdicts on the same inputs under another label (verifiers only)
Entry = collections.namedtuple("Entry", "run want reverify")


def prepare(e):
    """The receiver key and blinding base every entry point below uses."""
    e.set_receiver(W.receiver()[1])
    e.set_blinding_base(S.BB)


def tampered(verdicts, t):
    """The oracle gives CHALLENGE_MISMATCH for item t, whose challenge has a flipped bit, and Ok for the others."""
    want = [O.CHALLENGE_MISMATCH if i == t else O.OK for i in range(N)]
    assert verdicts.tolist() == want, (verdicts.tolist(), want)
    return verdicts


def range_entries(e, label, dev):
    pk = W.receiver()[1]
    spec, espec = O.range_optimal(RANGE_UB), e.range_optimal(RANGE_UB)
    assert espec.rings == spec.rings and spec.n_rings == 3
    values = np.array([0, RANGE_UB - 1, 13], np.uint64)
    cts, partials, rings = O.gen_range_batch(pk, spec, label, SEED, values)
    draws = e.lib.eg_range_prover_draws(O.C.byref(espec))
    wide = S.item_wide(SEED, 0, N, draws)
    ct_r = np.stack([np.frombuffer(O.scalar_reduce_wide(bytes(wide[i, 0])), np.uint8) for i in range(N)])
    t = len(label.encode()) % N
    bad = rings.copy()
    bad[t, 0, 0] ^= 1
    verdicts = tampered(O.verify_range_batch(pk, spec, label, cts, partials, bad), t)
    seed = np.frombuffer(SEED, np.uint8).copy()
    T = espec.rings_size

    def verify_dev(lbl):
        d_c, d_p, d_r, d_v = dev.up(cts), dev.up(partials), dev.up(bad), dev.empty(N, "uint8")
        e._check(e.lib.eg_verify_range_batch_dev(e.h, O.C.byref(espec), lbl.encode(), N, dev.ptr(d_c), dev.ptr(d_p), dev.ptr(d_r),
                                                 dev.ptr(d_v)))
        return (dev.down(d_v),)

    def encrypt_dev(lbl):
        d_v = dev.up(values.view(np.uint8))
        d_c, d_p, d_r = dev.empty(N * 64, "uint8"), dev.empty(N * 2 * 64, "uint8"), dev.empty(N * (1 + T) * 32, "uint8")
        e._check(e.lib.eg_encrypt_range_batch_dev(e.h, O.C.byref(espec), lbl.encode(), N, dev.ptr(d_v), None, seed.ctypes.data, 0,
                                                  dev.ptr(d_c), dev.ptr(d_p), dev.ptr(d_r)))
        return dev.down(d_c).reshape(N, 64), dev.down(d_p).reshape(N, 2, 64), dev.down(d_r).reshape(N, 1 + T, 32)

    again = lambda lbl: O.verify_range_batch(pk, spec, lbl, cts, partials, bad)
    return {
        "eg_verify_range_batch": Entry(lambda lbl: tuple(SC.in_ring_modes(e, lambda: e.verify_range(espec, lbl, cts, partials, bad),
                                                                          RING_MODES)),
                                       (verdicts,) * len(RING_MODES), again),
        "eg_verify_range_batch_dev": Entry(verify_dev, (verdicts,), again),
        "eg_encrypt_range_batch": Entry(lambda lbl: e.encrypt_range(espec, lbl, values, wide), (cts, partials, rings), None),
        "eg_encrypt_range_batch_seeded": Entry(lambda lbl: e.encrypt_range(espec, lbl, values, seed=SEED), (cts, partials, rings), None),
        "eg_encrypt_range_batch_dev": Entry(encrypt_dev, (cts, partials, rings), None),
        "eg_prove_range_batch": Entry(lambda lbl: e.prove_range(espec, lbl, values, ct_r, wide[:, 1:]), (cts, partials, rings), None),
        "eg_prove_range_batch_seeded": Entry(lambda lbl: e.prove_range(espec, lbl, values, ct_r, seed=SEED, counter_base=1),
                                             (cts, partials, rings), None),
    }


_sumsq_inputs = {}


def sumsq_entries(e, label, count):
    pk = W.receiver()[1]
    if count not in _sumsq_inputs:
        _sumsq_inputs[count] = S.sumsq_instances(pk, N, count)
    inst = _sumsq_inputs[count]
    cts, _, _, sum_cts, _ = inst
    proofs = S.oracle_sumsq(pk, inst, label, 2)
    t = len(label.encode()) % N
    bad = proofs.copy()
    bad[t, 0, 0] ^= 1

    def oracle_verify(lbl):
        return np.array([O.sumsq_verify(pk, [bytes(c) for c in cts[i]], bytes(sum_cts[i]), lbl, bytes(bad[i])) for i in range(N)],
                        np.uint8)
    return {
        "eg_verify_sumsq_batch": Entry(lambda lbl: (e.verify_sumsq(lbl, cts, sum_cts, bad),), (tampered(oracle_verify(label), t),),
                                       oracle_verify),
        "eg_prove_sumsq_batch": Entry(lambda lbl: (e.prove_sumsq(lbl, *inst, S.item_wide(S.SEED, 2, N, 1 + 2 * count)),), (proofs,),
                                      None),
        "eg_prove_sumsq_batch_seeded": Entry(lambda lbl: (e.prove_sumsq(lbl, *inst, seed=S.SEED, counter_base=2),), (proofs,), None),
    }


def decryption_entries(e, label):
    sk, pk = W.receiver()
    cts = D.ciphertexts(pk, [0, 1, 12345])
    rows = [O.decryption_prove(sk, label, bytes(cts[i]), D.item_rng(i)) for i in range(N)]
    dh = np.frombuffer(b"".join(r[0] for r in rows), np.uint8).reshape(N, 32)
    proofs = np.frombuffer(b"".join(r[1] for r in rows), np.uint8).reshape(N, 64)
    t = len(label.encode()) % N
    bad = proofs.copy()
    bad[t, 0] ^= 1

    def oracle_verify(lbl):
        return np.array([O.decryption_verify(pk, lbl, bytes(cts[i]), bytes(dh[i]), bytes(bad[i])) for i in range(N)], np.uint8)
    ok = np.ones(N, bool)
    return {
        "eg_verify_decryption_batch": Entry(lambda lbl: (e.verify_decryption(lbl, pk, cts, dh, bad),),
                                            (tampered(oracle_verify(label), t),), oracle_verify),
        "eg_prove_decryption_batch": Entry(lambda lbl: e.prove_decryption(lbl, sk, cts, D.wide(0, N)), (dh, proofs, ok), None),
        "eg_prove_decryption_batch_seeded": Entry(lambda lbl: e.prove_decryption(lbl, sk, cts, seed=D.SEED), (dh, proofs, ok), None),
    }


def commitment_equiv_entries(e, label):
    pk = W.receiver()[1]
    values, ct_r = S.ceq_inputs(N)
    cts, coms, proofs = O.gen_ceq_batch(pk, S.BB, label, S.SEED, values)
    blind = S.as_np([O.commitment_equiv_prove(pk, int(values[i]), S.BB, label, O.rng_from_seed(S.SEED, first_block=i << 20))[3]
                     for i in range(N)], N, 32)
    t = len(label.encode()) % N
    bad = proofs.copy()
    bad[t, 0] ^= 1
    again = lambda lbl: O.verify_ceq_batch(pk, S.BB, lbl, cts, coms, bad)
    want = (cts, coms, proofs, blind)
    return {
        "eg_verify_commitment_equiv_batch": Entry(lambda lbl: (e.verify_commitment_equiv(lbl, cts, coms, bad),),
                                                  (tampered(again(label), t),), again),
        "eg_prove_commitment_equiv_batch": Entry(lambda lbl: e.prove_commitment_equiv(lbl, values, ct_r, S.item_wide(S.SEED, 1, N, 4)),
                                                 want, None),
        "eg_prove_commitment_equiv_batch_seeded": Entry(lambda lbl: e.prove_commitment_equiv(lbl, values, ct_r, seed=S.SEED, counter_base=1),
                                                        want, None),
    }


def possession_entries(e, label, k):
    keys, proofs = O.gen_pop_batch(k, label, S.SEED, N)
    secrets = S.pop_secrets(N, k)
    t = len(label.encode()) % N
    bad = proofs.copy()
    bad[t, 0, 0] ^= 1
    again = lambda lbl: O.verify_pop_batch(lbl, keys, bad)
    return {
        "eg_verify_possession_batch": Entry(lambda lbl: (e.verify_possession(lbl, keys, bad),), (tampered(again(label), t),), again),
        "eg_prove_possession_batch": Entry(lambda lbl: e.prove_possession(lbl, secrets, S.item_wide(S.SEED, k, N, k)), (keys, proofs),
                                           None),
        "eg_prove_possession_batch_seeded": Entry(lambda lbl: e.prove_possession(lbl, secrets, seed=S.SEED, counter_base=k),
                                                  (keys, proofs), None),
    }


OBJECTS = {
    "range": lambda e, label, dev: range_entries(e, label, dev),
    "sumsq_1": lambda e, label, dev: sumsq_entries(e, label, 1),
    "sumsq_5": lambda e, label, dev: sumsq_entries(e, label, 5),
    "decryption": lambda e, label, dev: decryption_entries(e, label),
    "commitment_equiv": lambda e, label, dev: commitment_equiv_entries(e, label),
    "possession_1": lambda e, label, dev: possession_entries(e, label, 1),
    "possession_5": lambda e, label, dev: possession_entries(e, label, 5),
}

# every entry point that takes a transcript label -> the object whose inputs it is called with
ENTRY_POINTS = {
    **dict.fromkeys(("eg_verify_range_batch", "eg_verify_range_batch_dev", "eg_encrypt_range_batch", "eg_encrypt_range_batch_seeded",
                     "eg_encrypt_range_batch_dev", "eg_prove_range_batch", "eg_prove_range_batch_seeded"), "range"),
    **dict.fromkeys(("eg_verify_sumsq_batch", "eg_prove_sumsq_batch", "eg_prove_sumsq_batch_seeded"), "sumsq_5"),
    **dict.fromkeys(("eg_verify_decryption_batch", "eg_prove_decryption_batch", "eg_prove_decryption_batch_seeded"), "decryption"),
    **dict.fromkeys(("eg_verify_commitment_equiv_batch", "eg_prove_commitment_equiv_batch", "eg_prove_commitment_equiv_batch_seeded"),
                    "commitment_equiv"),
    **dict.fromkeys(("eg_verify_possession_batch", "eg_prove_possession_batch", "eg_prove_possession_batch_seeded"), "possession_5"),
}
HOST_ENTRY_POINTS = [name for name in ENTRY_POINTS if not name.endswith("_dev")]     # the forms a multi-device context serves


def labelled_in_header():
    """The entry points include/eg_b200.h declares with a `transcript_label` parameter."""
    text = (O.ROOT / "include" / "eg_b200.h").read_text()
    return set(re.findall(r"eg_status\s+(eg_\w+)\(eg_ctx \*ctx,[^;]*?const char \*transcript_label", text))


def same(got, want):
    return len(got) == len(want) and all(np.array_equal(np.asarray(a), np.asarray(b)) for a, b in zip(got, want))


def check_label(e, obj, label, dev):
    """Every entry point of `obj` under `label`: the oracle's bytes and verdicts (one item tampered); under a label of the same
    length with another last byte, every proof is rejected by the library and by the oracle."""
    sib = same_length_sibling(label)
    for name, en in OBJECTS[obj](e, label, dev).items():
        assert same(en.run(label), en.want), name
        if en.reverify is not None:
            assert all((v != O.OK).all() for v in en.run(sib)), (name, "accepted under", sib)
            assert (en.reverify(sib) != O.OK).all(), (name, "oracle accepted under", sib)


def check_sweep(e, obj, lengths, dev):
    """check_label for label_of(L), L in `lengths`; reports every length that fails."""
    failed = []
    for length in lengths:
        try:
            check_label(e, obj, label_of(length), dev)
        except AssertionError as exc:
            failed.append(f"L = {length}: {exc}")
    assert not failed, f"{len(failed)} of {len(lengths)} label lengths fail:\n" + "\n".join(failed)


# ---------------------------------------------------------------- label arguments

def check_label_arguments(e, name, dev):
    """A 255-byte label is accepted and gives the oracle's outputs; "" and a 256-byte label are EG_ERR_INVALID_ARG, after
    which the same call gives the same bytes as before."""
    from elastic_elgamal_b200 import _ffi
    label = label_of(255)
    en = OBJECTS[ENTRY_POINTS[name]](e, label, dev)[name]
    ref = en.run(label)
    assert same(ref, en.want), name
    for bad in ("", label_of(256)):
        assert S.status(lambda: en.run(bad)) == _ffi.ERR_INVALID_ARG, (name, len(bad))
        assert same(en.run(label), ref), (name, len(bad))
