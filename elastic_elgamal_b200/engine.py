"""Thin numpy-facing wrapper over the C ABI: one Engine = one eg_ctx = one GPU."""
import ctypes as C

import numpy as np

from . import _ffi


class EngineError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"{_ffi.STATUS_NAMES[status] if 0 <= status < len(_ffi.STATUS_NAMES) else status}: {message}")
        self.status = status


def _u8(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _addr(a):
    return None if a is None else a.ctypes.data


class Engine:
    """Owns an eg_ctx on `device`, or -- with `devices=[...]` -- a multi-device context (eg_ctx_create_multi) whose batch
    calls shard across those GPUs inside the library.  `lib_path` exists for the test harness; the default is the in-tree
    CUDA library."""

    def __init__(self, device=0, lib_path=None, devices=None):
        self.lib = _ffi.load(lib_path)
        h = C.c_void_p()
        if devices is not None:
            ids = (C.c_int * len(devices))(*devices)
            st = self.lib.eg_ctx_create_multi(ids, len(devices), C.byref(h))
            device = devices[0] if devices else 0
        else:
            st = self.lib.eg_ctx_create(device, C.byref(h))
        if st != _ffi.SUCCESS:
            raise EngineError(st, "eg_ctx_create failed (no CUDA device / NCCL? the engine has no CPU fallback)")
        self.h = h
        self.device = device

    # ---- multi-GPU: one process per GPU (torchrun style); the library owns the NCCL communicator
    def comm_unique_id(self):
        """128-byte NCCL unique id (rank 0 calls this; the host distributes it to the other ranks)."""
        buf = np.zeros(_ffi.COMM_ID_BYTES, np.uint8)
        st = self.lib.eg_comm_unique_id(_addr(buf))
        if st != _ffi.SUCCESS:
            raise EngineError(st, "eg_comm_unique_id failed (libnccl.so.2 not loadable?)")
        return buf

    def attach_comm(self, unique_id, rank, world):
        unique_id = _u8(unique_id, (_ffi.COMM_ID_BYTES,))
        self._check(self.lib.eg_ctx_attach_comm(self.h, _addr(unique_id), rank, world))

    def comm_info(self):
        r, w, d = C.c_int(0), C.c_int(0), C.c_int(0)
        self._check(self.lib.eg_ctx_comm_info(self.h, C.byref(r), C.byref(w), C.byref(d)))
        return {"rank": r.value, "world": w.value, "devices": d.value}

    def close(self):
        if getattr(self, "h", None):
            self.lib.eg_ctx_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, st):
        if st != _ffi.SUCCESS:
            raise EngineError(st, self.lib.eg_last_error(self.h).decode())

    @property
    def kernel_launches(self):
        return self.lib.eg_kernel_launch_count(self.h)

    @property
    def stream(self):
        return self.lib.eg_ctx_stream(self.h)

    def last_timings(self):
        t = (C.c_float * 5)()
        self._check(self.lib.eg_last_timings(self.h, C.byref(t)))
        return dict(zip(("decode_ms", "verify_ms", "commit_kernel_ms", "tally_ms", "total_ms"), t))

    def last_commit_stats(self):
        launches, tasks, ms = C.c_uint64(0), C.c_uint64(0), C.c_float(0)
        self._check(self.lib.eg_last_commit_stats(self.h, C.byref(launches), C.byref(tasks), C.byref(ms)))
        return {"launches": launches.value, "tasks": tasks.value, "ms": ms.value}

    def last_kernel_stats(self, kind):
        """kind 0: k_commit, 1: k_ring, 2: k_msm, 3: k_ring_pair -- launches, tasks (equation sides / sums) and summed device
        ms in the last batch call."""
        launches, tasks, ms = C.c_uint64(0), C.c_uint64(0), C.c_float(0)
        self._check(self.lib.eg_last_kernel_stats(self.h, kind, C.byref(launches), C.byref(tasks), C.byref(ms)))
        return {"launches": launches.value, "tasks": tasks.value, "ms": ms.value}

    def selftest_field(self, n=1 << 16, seed=1):
        m = C.c_uint64(0)
        self._check(self.lib.eg_selftest_field(self.h, n, seed, C.byref(m)))
        return m.value

    def set_chunk_items(self, items):
        self._check(self.lib.eg_ctx_set_chunk_items(self.h, items))

    def set_ring_mode(self, mode):
        self._check(self.lib.eg_ctx_set_ring_mode(self.h, mode))

    def set_key_table_min(self, min_tallies):
        """Tallies per call from which verify_shares / verify_decryption build fixed-base tables for the keys (0 = always)."""
        self._check(self.lib.eg_ctx_set_key_table_min(self.h, min_tallies))

    def set_prover_mode(self, constant_time):
        """True: constant-time fixed-base arithmetic for the provers' secret scalars (include/eg_b200.h)."""
        self._check(self.lib.eg_ctx_set_prover_mode(self.h, 1 if constant_time else 0))

    @staticmethod
    def _seed(seed):
        return _u8(np.frombuffer(bytes(seed), dtype=np.uint8), (32,))

    # ---- PublicKey::from_bytes
    def set_receiver(self, key):
        key = _u8(np.frombuffer(bytes(key), dtype=np.uint8), (32,))
        self._check(self.lib.eg_ctx_set_receiver(self.h, _addr(key)))

    # ---- Pedersen blinding base H (CommitmentEquivalenceProof)
    def set_blinding_base(self, base):
        base = _u8(np.frombuffer(bytes(base), dtype=np.uint8), (32,))
        self._check(self.lib.eg_ctx_set_blinding_base(self.h, _addr(base)))

    # ---- wire format: unpadded base64url of fixed-size fields (serde.rs:19-80)
    def base64url_decode(self, text, bytes_per_item):
        chars = self.lib.eg_base64url_chars(bytes_per_item)
        text = _u8(text, (-1, chars))
        n = text.shape[0]
        raw, ok = np.empty((n, bytes_per_item), np.uint8), np.empty(n, np.uint8)
        self._check(self.lib.eg_base64url_decode_batch(self.h, n, bytes_per_item, _addr(text), _addr(raw), _addr(ok)))
        return raw, ok.astype(bool)

    def base64url_encode(self, raw):
        raw = _u8(raw)
        n, b = raw.shape[0], int(np.prod(raw.shape[1:]))
        raw = raw.reshape(n, b)
        text = np.empty((n, self.lib.eg_base64url_chars(b)), np.uint8)
        self._check(self.lib.eg_base64url_encode_batch(self.h, n, b, _addr(raw), _addr(text)))
        return text

    # ---- struct-level wire format: objects of F base64url fields of 43 characters (serde.rs:179-355)
    def wire_fields(self, kind, count=0):
        return self.lib.eg_wire_fields(kind, count)

    def wire_decode(self, text, fields):
        if fields == 0:     # a vector below the reference's minimum length: the library reports EG_ERR_LEN_MISMATCH
            self._check(self.lib.eg_wire_decode_batch(self.h, 0, 1, None, None, None))
        text = _u8(text, (-1, fields * 43))
        n = text.shape[0]
        raw, ok = np.empty((n, fields * 32), np.uint8), np.empty(n, np.uint8)
        self._check(self.lib.eg_wire_decode_batch(self.h, fields, n, _addr(text), _addr(raw), _addr(ok)))
        return raw, ok.astype(bool)

    def wire_encode(self, raw, fields):
        raw = _u8(raw, (-1, fields * 32))
        n = raw.shape[0]
        text = np.empty((n, fields * 43), np.uint8)
        self._check(self.lib.eg_wire_encode_batch(self.h, fields, n, _addr(raw), _addr(text)))
        return text

    # ---- group helpers
    def elements_validate(self, enc):
        enc = _u8(enc, (-1, 32))
        ok = np.empty(enc.shape[0], np.uint8)
        self._check(self.lib.eg_elements_validate(self.h, enc.shape[0], _addr(enc), _addr(ok)))
        return ok.astype(bool)

    def scalars_validate(self, s):
        s = _u8(s, (-1, 32))
        ok = np.empty(s.shape[0], np.uint8)
        self._check(self.lib.eg_scalars_validate(self.h, s.shape[0], _addr(s), _addr(ok)))
        return ok.astype(bool)

    def scalars_from_wide(self, wide):
        wide = _u8(wide, (-1, 64))
        out = np.empty((wide.shape[0], 32), np.uint8)
        self._check(self.lib.eg_scalars_from_wide(self.h, wide.shape[0], _addr(wide), _addr(out)))
        return out

    def double_mul_generator(self, a, A, b):
        a, A, b = _u8(a, (-1, 32)), _u8(A, (-1, 32)), _u8(b, (-1, 32))
        n = a.shape[0]
        out, ok = np.empty((n, 32), np.uint8), np.empty(n, np.uint8)
        self._check(self.lib.eg_double_mul_generator_batch(self.h, n, _addr(a), _addr(A), _addr(b), _addr(out), _addr(ok)))
        return out, ok.astype(bool)

    def mul_generator(self, k):
        k = _u8(k, (-1, 32))
        n = k.shape[0]
        out, ok = np.empty((n, 32), np.uint8), np.empty(n, np.uint8)
        self._check(self.lib.eg_mul_generator_batch(self.h, n, _addr(k), _addr(out), _addr(ok)))
        return out, ok.astype(bool)

    def multi_mul(self, scalars, points):
        scalars = _u8(scalars)
        n, t = scalars.shape[0], scalars.shape[1]
        scalars, points = scalars.reshape(n, t, 32), _u8(points, (n, t, 32))
        out, ok = np.empty((n, 32), np.uint8), np.empty(n, np.uint8)
        self._check(self.lib.eg_multi_mul_batch(self.h, n, t, _addr(scalars), _addr(points), _addr(out), _addr(ok)))
        return out, ok.astype(bool)

    def ciphertexts_lincomb(self, scalars, cts):
        """Ciphertext Add / Sub / Neg / Mul<&Scalar> (encryption.rs:160-226) as out[i] = sum_j [scalars[i][j]] cts[i][j]."""
        scalars = _u8(scalars)
        n, t = scalars.shape[0], scalars.shape[1]
        scalars, cts = scalars.reshape(n, t, 32), _u8(cts, (n, t, 64))
        out, ok = np.empty((n, 64), np.uint8), np.empty(n, np.uint8)
        self._check(self.lib.eg_ciphertexts_lincomb_batch(self.h, n, t, _addr(scalars), _addr(cts), _addr(out), _addr(ok)))
        return out, ok.astype(bool)

    def ciphertexts_sum(self, parts):
        parts = _u8(parts)
        n_parts, n_cts = parts.shape[0], parts.shape[1]
        parts = parts.reshape(n_parts, n_cts, 64)
        out, ok = np.empty((n_cts, 64), np.uint8), np.zeros(1, np.uint8)
        self._check(self.lib.eg_ciphertexts_sum(self.h, n_parts, n_cts, _addr(parts), _addr(out), _addr(ok)))
        return out, bool(ok[0])

    # ---- proofs
    def verify_zero(self, cts, proofs):
        cts, proofs = _u8(cts, (-1, 64)), _u8(proofs, (-1, 64))
        n = cts.shape[0]
        assert proofs.shape[0] == n
        v = np.empty(n, np.uint8)
        self._check(self.lib.eg_verify_zero_batch(self.h, n, _addr(cts), _addr(proofs), _addr(v)))
        return v

    def verify_bool(self, cts, proofs):
        cts, proofs = _u8(cts, (-1, 64)), _u8(proofs, (-1, 96))
        n = cts.shape[0]
        assert proofs.shape[0] == n
        v = np.empty(n, np.uint8)
        self._check(self.lib.eg_verify_bool_batch(self.h, n, _addr(cts), _addr(proofs), _addr(v)))
        return v

    def verify_choice(self, options, choices, rings, sums=None, single=True, tally=True):
        choices = _u8(choices, (-1, options, 64))
        n = choices.shape[0]
        rings = _u8(rings, (n, 1 + 2 * options, 32))
        if single:
            sums = _u8(sums, (n, 64))
        v = np.empty(n, np.uint8)
        t = np.empty((options, 64), np.uint8) if tally else None
        self._check(self.lib.eg_verify_choice_batch(self.h, n, options, int(single), _addr(choices), _addr(rings),
                                                    _addr(sums) if single else None, _addr(v), _addr(t)))
        return v, t

    def verify_commitment_equiv(self, label, cts, commitments, proofs):
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        commitments, proofs = _u8(commitments, (n, 32)), _u8(proofs, (n, 128))
        v = np.empty(n, np.uint8)
        self._check(self.lib.eg_verify_commitment_equiv_batch(self.h, label.encode(), n, _addr(cts), _addr(commitments),
                                                              _addr(proofs), _addr(v)))
        return v

    def verify_possession(self, label, keys, proofs):
        keys = _u8(keys)
        n, k = keys.shape[0], keys.shape[1]
        keys, proofs = keys.reshape(n, k, 32), _u8(proofs, (n, 1 + k, 32))
        v = np.empty(n, np.uint8)
        self._check(self.lib.eg_verify_possession_batch(self.h, label.encode(), k, n, _addr(keys), _addr(proofs), _addr(v)))
        return v

    # ---- encryption side (randomness supplied by the caller as 64-byte blocks in the reference's draw order)
    # Every encrypt_* takes either `wide_rand` (the blocks themselves) or `seed=` (32 bytes) + `counter_base=`: the seeded
    # form generates the blocks in the kernel (eg_*_batch_seeded).
    def encrypt(self, values, wide_rand=None, seed=None, counter_base=0):
        values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1)
        n = values.shape[0]
        cts = np.empty((n, 64), np.uint8)
        if seed is not None:
            self._check(self.lib.eg_encrypt_batch_seeded(self.h, n, _addr(values), _addr(self._seed(seed)), counter_base, _addr(cts)))
            return cts
        wide_rand = _u8(wide_rand, (n, 64))
        self._check(self.lib.eg_encrypt_batch(self.h, n, _addr(values), _addr(wide_rand), _addr(cts)))
        return cts

    def encrypt_zero(self, wide_rand=None, seed=None, counter_base=0, n=None):
        if seed is not None:
            cts, proofs = np.empty((n, 64), np.uint8), np.empty((n, 64), np.uint8)
            self._check(self.lib.eg_encrypt_zero_batch_seeded(self.h, n, _addr(self._seed(seed)), counter_base, _addr(cts), _addr(proofs)))
            return cts, proofs
        wide_rand = _u8(wide_rand, (-1, 2, 64))
        n = wide_rand.shape[0]
        cts, proofs = np.empty((n, 64), np.uint8), np.empty((n, 64), np.uint8)
        self._check(self.lib.eg_encrypt_zero_batch(self.h, n, _addr(wide_rand), _addr(cts), _addr(proofs)))
        return cts, proofs

    def encrypt_bool(self, values, wide_rand=None, seed=None, counter_base=0):
        values = _u8(values, (-1,))
        n = values.shape[0]
        cts, proofs = np.empty((n, 64), np.uint8), np.empty((n, 96), np.uint8)
        if seed is not None:
            self._check(self.lib.eg_encrypt_bool_batch_seeded(self.h, n, _addr(values), _addr(self._seed(seed)), counter_base, _addr(cts),
                                                              _addr(proofs)))
            return cts, proofs
        wide_rand = _u8(wide_rand, (n, 3, 64))
        self._check(self.lib.eg_encrypt_bool_batch(self.h, n, _addr(values), _addr(wide_rand), _addr(cts), _addr(proofs)))
        return cts, proofs

    def encrypt_choice(self, options, values, wide_rand=None, single=True, seed=None, counter_base=0):
        values = _u8(values, (-1, options))
        n = values.shape[0]
        draws = 3 * options + (1 if single else 0)
        cts, rings = np.empty((n, options, 64), np.uint8), np.empty((n, 1 + 2 * options, 32), np.uint8)
        sums = np.empty((n, 64), np.uint8) if single else None
        if seed is not None:
            self._check(self.lib.eg_encrypt_choice_batch_seeded(self.h, n, options, int(single), _addr(values), _addr(self._seed(seed)),
                                                                counter_base, _addr(cts), _addr(rings), _addr(sums)))
            return cts, rings, sums
        wide_rand = _u8(wide_rand, (n, draws, 64))
        self._check(self.lib.eg_encrypt_choice_batch(self.h, n, options, int(single), _addr(values), _addr(wide_rand), _addr(cts),
                                                     _addr(rings), _addr(sums)))
        return cts, rings, sums

    # ---- RangeDecomposition / RangeProof
    def range_optimal(self, upper_bound):
        r = _ffi.Range()
        self._check(self.lib.eg_range_optimal(upper_bound, C.byref(r)))
        return r

    def range_display(self, r):
        b = C.create_string_buffer(4096)
        n = self.lib.eg_range_display(C.byref(r), b, 4096)
        return b.raw[:n].decode()

    def verify_range(self, rng, label, cts, partials, rings):
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        partials = _u8(partials, (n, max(0, rng.n_rings - 1), 64))
        rings = _u8(rings, (n, 1 + rng.rings_size, 32))
        v = np.empty(n, np.uint8)
        self._check(self.lib.eg_verify_range_batch(self.h, C.byref(rng), label.encode(), n, _addr(cts),
                                                   _addr(partials) if rng.n_rings > 1 else None, _addr(rings), _addr(v)))
        return v

    def encrypt_range(self, rng, label, values, wide_rand=None, seed=None, counter_base=0):
        values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1)
        n = values.shape[0]
        draws = self.lib.eg_range_prover_draws(C.byref(rng))
        cts = np.empty((n, 64), np.uint8)
        partials = np.empty((n, max(0, rng.n_rings - 1), 64), np.uint8)
        rings = np.empty((n, 1 + rng.rings_size, 32), np.uint8)
        if seed is not None:
            self._check(self.lib.eg_encrypt_range_batch_seeded(self.h, C.byref(rng), label.encode(), n, _addr(values), _addr(self._seed(seed)),
                                                               counter_base, _addr(cts), _addr(partials) if rng.n_rings > 1 else None,
                                                               _addr(rings)))
            return cts, partials, rings
        wide_rand = _u8(wide_rand, (n, draws, 64))
        self._check(self.lib.eg_encrypt_range_batch(self.h, C.byref(rng), label.encode(), n, _addr(values), _addr(wide_rand),
                                                    _addr(cts), _addr(partials) if rng.n_rings > 1 else None, _addr(rings)))
        return cts, partials, rings

    def prove_range(self, rng, label, values, ct_randomness, wide_rand=None, seed=None, counter_base=0, want_cts=True):
        """RangeProof::from_ciphertext: proofs for existing ciphertexts with known values and randomness."""
        values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1)
        n = values.shape[0]
        ct_randomness = _u8(ct_randomness, (n, 32))
        draws = self.lib.eg_range_prover_draws(C.byref(rng)) - 1
        cts = np.empty((n, 64), np.uint8) if want_cts else None
        partials = np.empty((n, max(0, rng.n_rings - 1), 64), np.uint8)
        rings = np.empty((n, 1 + rng.rings_size, 32), np.uint8)
        pp = _addr(partials) if rng.n_rings > 1 else None
        if seed is not None:
            self._check(self.lib.eg_prove_range_batch_seeded(self.h, C.byref(rng), label.encode(), n, _addr(values), _addr(ct_randomness),
                                                             _addr(self._seed(seed)), counter_base, _addr(cts), pp, _addr(rings)))
        else:
            wide_rand = _u8(wide_rand, (n, draws, 64))
            self._check(self.lib.eg_prove_range_batch(self.h, C.byref(rng), label.encode(), n, _addr(values), _addr(ct_randomness),
                                                      _addr(wide_rand), _addr(cts), pp, _addr(rings)))
        return cts, partials, rings

    # ---- QuadraticVotingBallot
    def qv_params(self, options, credits):
        p = _ffi.QvParams()
        self._check(self.lib.eg_qv_params_new(options, credits, C.byref(p)))
        return p

    def qv_ballot_size(self, p):
        return self.lib.eg_qv_ballot_size(C.byref(p))

    def verify_qv(self, p, ballots, tally=True):
        bsz = self.qv_ballot_size(p)
        ballots = _u8(ballots, (-1, bsz))
        n = ballots.shape[0]
        v = np.empty(n, np.uint8)
        t = np.empty((p.options, 64), np.uint8) if tally else None
        self._check(self.lib.eg_verify_qv_batch(self.h, C.byref(p), n, _addr(ballots), _addr(v), _addr(t)))
        return v, t

    def encrypt_qv(self, p, votes, wide_rand=None, seed=None, counter_base=0):
        votes = np.ascontiguousarray(votes, dtype=np.uint64).reshape(-1, p.options)
        n = votes.shape[0]
        draws = self.lib.eg_qv_prover_draws(C.byref(p))
        ballots = np.empty((n, self.qv_ballot_size(p)), np.uint8)
        if seed is not None:
            self._check(self.lib.eg_encrypt_qv_batch_seeded(self.h, C.byref(p), n, _addr(votes), _addr(self._seed(seed)), counter_base,
                                                            _addr(ballots)))
            return ballots
        wide_rand = _u8(wide_rand, (n, draws, 64))
        self._check(self.lib.eg_encrypt_qv_batch(self.h, C.byref(p), n, _addr(votes), _addr(wide_rand), _addr(ballots)))
        return ballots

    # ---- SumOfSquaresProof::verify / CandidateDecryption::verify as entry points of their own
    def verify_sumsq(self, label, cts, sum_cts, proofs):
        cts = _u8(cts)
        n, m = cts.shape[0], cts.shape[1]
        cts, sum_cts, proofs = cts.reshape(n, m, 64), _u8(sum_cts, (n, 64)), _u8(proofs, (n, 2 * m + 2, 32))
        v = np.empty(n, np.uint8)
        self._check(self.lib.eg_verify_sumsq_batch(self.h, label.encode(), m, n, _addr(cts), _addr(sum_cts), _addr(proofs), _addr(v)))
        return v

    def verify_decryption(self, label, key, cts, dh_elements, proofs):
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        dh_elements, proofs = _u8(dh_elements, (n, 32)), _u8(proofs, (n, 64))
        key = _u8(np.frombuffer(bytes(key), dtype=np.uint8), (32,))
        v = np.empty(n, np.uint8)
        self._check(self.lib.eg_verify_decryption_batch(self.h, label.encode(), _addr(key), n, _addr(cts), _addr(dh_elements),
                                                        _addr(proofs), _addr(v)))
        return v

    # ---- threshold decryption
    def verify_shares(self, keyset, indexes, cts, shares, proofs):
        s = len(indexes)
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        shares, proofs = _u8(shares, (n, s, 32)), _u8(proofs, (n, s, 64))
        idx = (C.c_uint32 * s)(*indexes)
        v = np.empty((n, s), np.uint8)
        self._check(self.lib.eg_verify_shares_batch(self.h, C.byref(keyset), n, s, idx, _addr(cts), _addr(shares), _addr(proofs), _addr(v)))
        return v

    def keysets_validate(self, shares, threshold, keys):
        keys = _u8(keys, (-1, shares, 32))
        n = keys.shape[0]
        shared, v = np.empty((n, 32), np.uint8), np.empty(n, np.uint8)
        self._check(self.lib.eg_keysets_validate_batch(self.h, shares, threshold, n, _addr(keys), _addr(shared), _addr(v)))
        return shared, v

    def dlog_table(self, lo, hi):
        return DlogTable(self, lo, hi)

    def combine_decrypt(self, indexes, cts, shares, table):
        t = len(indexes)
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        shares = _u8(shares, (n, -1, 32))
        idx = (C.c_uint32 * t)(*indexes)
        values, found = np.zeros(n, np.uint64), np.zeros(n, np.uint8)
        self._check(self.lib.eg_combine_decrypt_batch(self.h, t, idx, n, shares.shape[1], _addr(cts), _addr(shares), table.h,
                                                      _addr(values), _addr(found)))
        return values, found

    # ---- decryption side (the holder's secret key; randomness as for encrypt_*: `wide_rand` blocks or `seed=`)
    @staticmethod
    def _secret(secret):
        return _u8(np.frombuffer(bytes(secret), dtype=np.uint8), (32,))

    def decrypt(self, secret, cts, table=None):
        """SecretKey::decrypt_to_element / decrypt: (elements, values, found); values is None without a table, found as
        eg_decrypt_batch (1 found / decoded, 0 absent from the table, 2 the ciphertext does not decode)."""
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        elements, found = np.empty((n, 32), np.uint8), np.empty(n, np.uint8)
        values = np.zeros(n, np.uint64) if table is not None else None
        sec = self._secret(secret)
        self._check(self.lib.eg_decrypt_batch(self.h, _addr(sec), n, _addr(cts), table.h if table is not None else None,
                                              _addr(elements), _addr(values), _addr(found)))
        return elements, values, found

    def decrypt_share(self, keyset, index, secret, cts, wide_rand=None, seed=None, counter_base=0):
        """ActiveParticipant::decrypt_share: (shares, proofs, ok) in the layouts verify_shares reads (one share per tally)."""
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        shares, proofs, ok = np.empty((n, 32), np.uint8), np.empty((n, 64), np.uint8), np.empty(n, np.uint8)
        sec = self._secret(secret)
        if seed is not None:
            seed = self._seed(seed)
            self._check(self.lib.eg_decrypt_share_batch_seeded(self.h, C.byref(keyset), index, _addr(sec), n, _addr(cts),
                                                               _addr(seed), counter_base, _addr(shares), _addr(proofs),
                                                               _addr(ok)))
        else:
            wide_rand = _u8(wide_rand, (n, 64))
            self._check(self.lib.eg_decrypt_share_batch(self.h, C.byref(keyset), index, _addr(sec), n, _addr(cts),
                                                        _addr(wide_rand), _addr(shares), _addr(proofs), _addr(ok)))
        return shares, proofs, ok.astype(bool)

    def prove_decryption(self, label, secret, cts, wide_rand=None, seed=None, counter_base=0):
        """VerifiableDecryption::new with the key pair (secret, [secret]G): (dh_elements, proofs, ok)."""
        cts = _u8(cts, (-1, 64))
        n = cts.shape[0]
        dh, proofs, ok = np.empty((n, 32), np.uint8), np.empty((n, 64), np.uint8), np.empty(n, np.uint8)
        sec = self._secret(secret)
        if seed is not None:
            seed = self._seed(seed)
            self._check(self.lib.eg_prove_decryption_batch_seeded(self.h, label.encode(), _addr(sec), n, _addr(cts),
                                                                  _addr(seed), counter_base, _addr(dh), _addr(proofs), _addr(ok)))
        else:
            wide_rand = _u8(wide_rand, (n, 64))
            self._check(self.lib.eg_prove_decryption_batch(self.h, label.encode(), _addr(sec), n, _addr(cts),
                                                           _addr(wide_rand), _addr(dh), _addr(proofs), _addr(ok)))
        return dh, proofs, ok.astype(bool)

    # ---- device-pointer variants (ints are raw device addresses, e.g. torch.Tensor.data_ptr())
    def decrypt_share_dev(self, keyset, index, secret, n, d_cts, d_shares, d_proofs, d_ok, d_wide_rand=None, seed=None, counter_base=0):
        sec, seed = self._secret(secret), (self._seed(seed) if seed is not None else None)
        self._check(self.lib.eg_decrypt_share_batch_dev(self.h, C.byref(keyset), index, _addr(sec), n, d_cts, d_wide_rand, _addr(seed),
                                                        counter_base, d_shares, d_proofs, d_ok))

    def verify_bool_dev(self, n, d_cts, d_proofs, d_verdicts):
        self._check(self.lib.eg_verify_bool_batch_dev(self.h, n, d_cts, d_proofs, d_verdicts))

    def ciphertexts_sum_dev(self, n_parts, n_cts, d_parts, d_out, d_bad=None):
        self._check(self.lib.eg_ciphertexts_sum_dev(self.h, n_parts, n_cts, d_parts, d_out, d_bad))

    def verify_choice_dev(self, n, options, single, d_choices, d_rings, d_sums, d_verdicts, d_tally):
        self._check(self.lib.eg_verify_choice_batch_dev(self.h, n, options, int(single), d_choices, d_rings, d_sums,
                                                        d_verdicts, d_tally))


class DlogTable:
    """DiscreteLogTable::new(lo..hi) resident on the engine's GPU."""

    def __init__(self, engine, lo, hi):
        self.engine = engine
        h = C.c_void_p()
        engine._check(engine.lib.eg_dlog_table_create(engine.h, lo, hi, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and self.engine.h:
            self.engine.lib.eg_dlog_table_destroy(self.h)
        self.h = None

    __del__ = close
