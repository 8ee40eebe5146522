"""Edge randomness on the encryption side, shared by the CPU harness tests (test_hostsim_encrypt_edges.py) and the `-m gpu`
tests (test_gpu_encrypt_edges.py).  The provers take their randomness from the caller as 64-byte blocks in the reference's
draw order, so a block can put any scalar into any role: the ciphertext randomness r, the real nonce x of a ring, a forged
response s, the nonce of a sum proof.  The library computes every commitment as a fixed-base multiple of a *halved, derived*
scalar ([r/2], [x/2], [(s - e r)/2] with ge_fixed_adds, or ge_fixed_adds_ct in constant-time mode) and encodes the results
with ge_double_compress2, whose zero-product branch handles the identity -- none of which random blocks reach at its edges.

The oracle replays the same blocks (oracle.rng_from_blocks), so every output byte is compared with the reference's algorithm,
not checked by algebra.  The draw-position maps below are derived from the oracle's draw order (oracle/proofs.c: Ring::new
draws r, x and the forged responses after the real index; Ring::finalize the forged responses before it, once the common
challenge e0 is known) and are themselves tested against the oracle's outputs."""
import random

import numpy as np

import edge_common as EC
import oracle as O
import parity_common as PC
import shape_common as SC
import workloads as W

L = W.L


def blk(x):
    """The 64-byte block that Ristretto::generate_scalar reduces to x mod l (x < 2^512, not necessarily reduced)."""
    return int(x).to_bytes(64, "little")


def red(block):
    return int.from_bytes(block, "little") % L


def sc(x):
    return PC.sc(x)


# ---------------------------------------------------------------- scalar targets

BASIC = [0, 1, 2, L - 1, L - 2, (L - 1) // 2, (L + 1) // 2]          # (l -+ 1) / 2: sc_half's odd / even boundary
UNREDUCED = [L, L + 1, 2 * L - 1, 2**256 - 1, 2**512 - 1, L * 2**259 + 5, L * (2**259 - 1) + (L + 1) // 2]


def _unique(xs):
    return list(dict.fromkeys(xs))


def doubled_wide_edges():
    """2w mod l for every w of parity_common.wide_window_edge_scalars(): the halves the fixed-base walk sees sit on the window
    boundaries of every width the library is built with (16 in the CPU harness, 24 on the device, 20 as a build option)."""
    return [2 * int.from_bytes(w, "little") % L for w in PC.wide_window_edge_scalars()]


def doubled_patterns():
    """2p mod l for every recode4 pattern p of edge_common: the constant-time walk recodes the half, p."""
    return [2 * p % L for p in EC.pattern_scalars()]


def target_blocks(wide_stride=1):
    """One block per target: the basic scalars, the doubled patterns and window edges (zero-extended; every `wide_stride`-th
    of the latter), then blocks that are not reduced (>= l, 2^512 - 1, l k + t)."""
    wide = doubled_wide_edges()[::wide_stride]
    return [blk(t) for t in _unique(BASIC + doubled_patterns() + wide)] + [blk(x) for x in UNREDUCED]


def derived_offsets(wide_stride=1):
    """t of the derived targets s = e0 r + t: 0 (forged commitments [0]G = O and [e0 (a - v)]G) and twice each edge."""
    return _unique([0] + [red(b) for b in target_blocks(wide_stride)])


def check_edge_lists_hit_their_patterns():
    """Each list produces, after halving, the digit patterns it is meant to: every recode4 pattern (constant-time walk) and the
    extreme signed digits of 16- and 24-bit windows with a carry into the top window (ge_fixed_adds); both parities around
    (l - 1) / 2; blocks >= l that the oracle reduces as the Python model does."""
    scalars = [red(b) for b in target_blocks()]
    halves = [EC.sc_half(x) for x in scalars]
    for x, h in zip(scalars, halves):
        assert h == x * pow(2, -1, L) % L
    for name, digits in EC.RECODE4_PATTERNS.items():
        assert any(EC.recode4(h) == digits for h in halves), name
    wide_halves = [EC.sc_half(x) for x in doubled_wide_edges()]
    for bits in EC.WIDE_BITS:
        top = 1 << (bits - 1)
        digits = [EC.wide_digits(h, bits) for h in wide_halves]
        below_top = {d for ds in digits for d in ds[:-1]}
        assert {-top, top - 1, -1, 0, 1} <= below_top, bits
        assert any(ds[-1] != h >> (bits * (len(ds) - 1)) for h, ds in zip(wide_halves, digits)), bits
    assert set(BASIC) <= set(scalars)
    for x in UNREDUCED:
        assert x >= L and O.scalar_reduce_wide(blk(x)) == sc(x)
    assert set(derived_offsets()) == set(scalars) and 0 in derived_offsets()


# ---------------------------------------------------------------- draw-position maps
# A role is (part, kind, ring, eq): part numbers the proofs of one item (the options of a QV ballot, then its credit), kind is
# "r" (ciphertext randomness; ring None = the item's ciphertext), "x" (real nonce of a ring), "s" (forged response drawn before
# e0, eq > index), "f" (forged response drawn after e0, eq < index; eq 0 runs on e0 itself) or "n" (nonce of a sum proof).

def ring_map(rings, part=0):
    """rings: [(size, real index, draws r)] in the order RingProofBuilder adds them."""
    out = []
    for k, (size, idx, draws_r) in enumerate(rings):
        if draws_r:
            out.append((part, "r", k, None))
        out.append((part, "x", k, None))
        out += [(part, "s", k, eq) for eq in range(idx + 1, size)]
    for k, (size, idx, _) in enumerate(rings):
        out += [(part, "f", k, eq) for eq in range(idx)]
    return out


def decompose(spec, value):
    """RangeDecomposition::decompose (range.rs:199-210): the real index of each ring."""
    out = []
    for size, step in spec.rings:
        i = min(value // step, size - 1)
        out.append(i)
        value -= i * step
    return out


def range_map(spec, value, part=0):
    idx = decompose(spec, value)
    n = spec.n_rings
    return [(part, "r", None, None)] + ring_map([(size, idx[k], k < n - 1) for k, (size, _) in enumerate(spec.rings)], part)


def response_offsets(spec):
    """Offset of each ring's first response among a range proof's responses."""
    out, off = [], 0
    for size, _ in spec.rings:
        out.append(off)
        off += size
    return out


# ---------------------------------------------------------------- provers
# Each prover: items (plaintexts), draw_map(item), oracle(pk, item, rng) -> output bytes, engine(e, items, wide) -> output rows,
# verify(e, pk, rows) -> (engine verdicts, oracle verdicts, engine tally, oracle tally), plaintexts(item) -> [(ct offset, value)],
# and the layout accessors R(row, part, ring) / response(row, part, ring, eq) / e0(row, part) / ring_r(item, blocks, part, k).

def _rows(blobs):
    return np.frombuffer(b"".join(blobs), np.uint8).reshape(len(blobs), -1).copy()


def _cat(*arrs):
    n = arrs[0].shape[0]
    return np.concatenate([a.reshape(n, -1) for a in arrs if a is not None], axis=1)


class Encrypt:
    name = "encrypt"
    rings = False

    def items(self):
        return [0, 1, 2**63, 2**64 - 1]

    def draw_map(self, v):
        return [(0, "r", None, None)]

    def oracle(self, pk, v, rng):
        return O.encrypt(pk, v, rng)

    def engine(self, e, items, wide):
        return e.encrypt(np.array(items, np.uint64), wide[:, 0])

    def verify(self, e, pk, rows):
        return None

    def plaintexts(self, v):
        return [(0, v)]

    def R(self, row, part, ring):
        return bytes(row[:32])


class EncryptZero(Encrypt):
    name = "encrypt_zero"

    def items(self):
        return [0]

    def draw_map(self, v):
        return [(0, "r", None, None), (0, "n", None, None)]

    def oracle(self, pk, v, rng):
        c, p = O.encrypt_zero(pk, rng)
        return c + p

    def engine(self, e, items, wide):
        return _cat(*e.encrypt_zero(wide))

    def verify(self, e, pk, rows):
        got = e.verify_zero(rows[:, :64], rows[:, 64:])
        return got, [O.verify_zero(pk, bytes(r[:64]), bytes(r[64:])) for r in rows], None, None


class Choice:
    """EncryptedChoice::new over m options (bool encryption is the choice of one option with no sum proof: encrypt_bool
    draws and lays out exactly as a one-option MultiChoice)."""
    rings = True

    def __init__(self, m, single, as_bool=False):
        self.m, self.single, self.as_bool = m, single, as_bool
        self.name = "encrypt_bool" if as_bool else f"choice_{'single' if single else 'multi'}_{m}"

    def items(self):
        m = self.m
        if self.as_bool:
            return [(0,), (1,)]
        if self.single:
            return [tuple(int(k == c) for k in range(m)) for c in range(m)]
        return [tuple([0] * m), tuple([1] * m)] + [tuple((c >> k) & 1 for k in range(m)) for c in range(1, 2**m - 1)]

    def draw_map(self, item):
        return ring_map([(2, v, True) for v in item]) + ([(0, "n", None, None)] if self.single else [])

    def oracle(self, pk, item, rng):
        if self.as_bool:
            c, p = O.encrypt_bool(pk, item[0], rng)
            return c + p
        c, r, s = O.choice_new(pk, [bool(v) for v in item], self.single, rng)
        return c + r + (s if self.single else b"")

    def engine(self, e, items, wide):
        vals = np.array(items, np.uint8)
        if self.as_bool:
            return _cat(*e.encrypt_bool(vals[:, 0], wide))
        return _cat(*e.encrypt_choice(self.m, vals, wide, single=self.single))

    def split(self, rows):
        m = self.m
        return (rows[:, :64 * m].reshape(-1, m, 64), rows[:, 64 * m:64 * m + 32 * (1 + 2 * m)].reshape(-1, 1 + 2 * m, 32),
                rows[:, 64 * m + 32 * (1 + 2 * m):] if self.single else None)

    def verify(self, e, pk, rows):
        if self.as_bool:
            got = e.verify_bool(rows[:, :64], rows[:, 64:])
            return got, O.verify_bool_batch(pk, rows[:, :64], rows[:, 64:]), None, None
        cts, rings, sums = self.split(rows)
        got, tally = e.verify_choice(self.m, cts, rings, sums, single=self.single, tally=True)
        exp, exp_tally = O.verify_choice_batch(pk, self.m, self.single, cts, rings, sums)
        return got, exp, tally, exp_tally

    def plaintexts(self, item):
        return [(64 * k, v) for k, v in enumerate(item)]

    def R(self, row, part, ring):
        return bytes(row[64 * ring:64 * ring + 32])

    def e0(self, row, part):
        return bytes(row[64 * self.m:64 * self.m + 32])

    def response(self, row, part, ring, eq):
        o = 64 * self.m + 32 + 32 * (2 * ring + eq)
        return bytes(row[o:o + 32])

    def ring_r(self, item, blocks, roles, part, k):
        return red(blocks[roles.index((part, "r", k, None))])


class Range:
    """RangeProof::new (caller blocks for the ciphertext too) or RangeProof::from_ciphertext (ct_randomness given; the
    oracle replays it as the first block)."""
    rings = True

    def __init__(self, upper_bound, from_ct=False, label="ciphertext_range"):
        self.ub, self.from_ct, self.label = upper_bound, from_ct, label
        self.spec = O.range_optimal(upper_bound)
        self.name = f"{'prove' if from_ct else 'encrypt'}_range_{upper_bound}"

    def items(self):
        # every real index of every ring, both ends of the range
        return _unique([0, self.ub - 1] + [v for v in range(self.ub) if v % 7 in (0, 3)])

    def draw_map(self, v):
        return range_map(self.spec, v)

    def oracle(self, pk, v, rng):
        c, p, r, _ = O.range_prove(pk, self.spec, self.label, v, rng)
        return c + p + r

    def engine(self, e, items, wide):
        espec = PC.to_engine_range(e, self.spec)
        vals = np.array(items, np.uint64)
        if self.from_ct:
            ct_r = _rows([sc(red(bytes(w[0]))) for w in wide])
            return _cat(*e.prove_range(espec, self.label, vals, ct_r, np.ascontiguousarray(wide[:, 1:])))
        return _cat(*e.encrypt_range(espec, self.label, vals, wide))

    def split(self, rows):
        np_ = self.spec.n_rings - 1
        return (rows[:, :64], rows[:, 64:64 + 64 * np_].reshape(-1, np_, 64),
                rows[:, 64 + 64 * np_:].reshape(-1, 1 + self.spec.rings_size, 32))

    def verify(self, e, pk, rows):
        espec = PC.to_engine_range(e, self.spec)
        c, p, r = self.split(rows)
        return (e.verify_range(espec, self.label, c, p, r), O.verify_range_batch(pk, self.spec, self.label, c, p, r), None, None)

    def plaintexts(self, v):
        return [(0, v)]

    # layout of one range proof at byte offset `base`
    def _R(self, row, base, ring):
        o = base if ring is None else base + 64 + 64 * ring
        return bytes(row[o:o + 32])

    def _e0(self, row, base):
        o = base + 64 * self.spec.n_rings
        return bytes(row[o:o + 32])

    def _response(self, row, base, ring, eq):
        o = base + 64 * self.spec.n_rings + 32 + 32 * (response_offsets(self.spec)[ring] + eq)
        return bytes(row[o:o + 32])

    def _ring_r(self, blocks, roles, part, k, n_rings):
        if k < n_rings - 1:
            return red(blocks[roles.index((part, "r", k, None))])
        r = red(blocks[roles.index((part, "r", None, None))])
        return (r - sum(red(blocks[roles.index((part, "r", j, None))]) for j in range(n_rings - 1))) % L

    def R(self, row, part, ring):
        return self._R(row, 0, ring)

    def e0(self, row, part):
        return self._e0(row, 0)

    def response(self, row, part, ring, eq):
        return self._response(row, 0, ring, eq)

    def ring_r(self, item, blocks, roles, part, k):
        return self._ring_r(blocks, roles, part, k, self.spec.n_rings)


class QV(Range):
    """QuadraticVotingBallot::new: a range proof per option (parts 0 .. n-1), one for the credit (part n), then the
    sum-of-squares proof's nonces (kind "n")."""

    def __init__(self, options, credits):
        self.n, self.credits = options, credits
        self.p = O.qv_params(options, credits)
        self.vote = Range(int(O.lib().eo_isqrt(credits)) + 1, label="quadratic_voting_variant")
        self.credit = Range(credits + 1, label="quadratic_voting_credit_range")
        self.name = f"qv_{options}_{credits}"
        self.vsz = 64 * self.vote.spec.n_rings + 32 * (1 + self.vote.spec.rings_size)

    def items(self):
        mv = int(O.lib().eo_isqrt(self.credits))
        rnd = random.Random(self.n * 100 + self.credits)
        out = [tuple([0] * self.n), tuple([mv] + [0] * (self.n - 1))]
        while len(out) < 8:
            v = tuple(rnd.randrange(mv + 1) for _ in range(self.n))
            if sum(x * x for x in v) <= self.credits:
                out.append(v)
        return _unique(out)

    def _spec(self, part):
        return (self.vote if part < self.n else self.credit).spec

    def draw_map(self, votes):
        out = []
        for j, v in enumerate(votes):
            out += range_map(self.vote.spec, v, part=j)
        out += range_map(self.credit.spec, sum(v * v for v in votes), part=self.n)
        return out + [(self.n + 1, "n", None, k) for k in range(1 + 2 * self.n)]

    def oracle(self, pk, votes, rng):
        return O.qv_new(pk, self.p, list(votes), rng)

    def engine(self, e, items, wide):
        return e.encrypt_qv(e.qv_params(self.n, self.credits), np.array(items, np.uint64), wide)

    def verify(self, e, pk, rows):
        got, tally = e.verify_qv(e.qv_params(self.n, self.credits), rows)
        exp, exp_tally = O.verify_qv_batch(pk, self.p, rows)
        return got, exp, tally, exp_tally

    def plaintexts(self, votes):
        return [(self.vsz * j, v) for j, v in enumerate(votes)] + [(self.vsz * self.n, sum(v * v for v in votes))]

    def R(self, row, part, ring):
        return (self.vote if part < self.n else self.credit)._R(row, self.vsz * part, ring)

    def response(self, row, part, ring, eq):
        return (self.vote if part < self.n else self.credit)._response(row, self.vsz * part, ring, eq)

    def e0(self, row, part):
        return (self.vote if part < self.n else self.credit)._e0(row, self.vsz * part)

    def ring_r(self, item, blocks, roles, part, k):
        return self._ring_r(blocks, roles, part, k, self._spec(part).n_rings)


def provers(qv=(3, 9), range_bounds=(21, 100)):
    out = [Encrypt(), EncryptZero(), Choice(1, False, as_bool=True), Choice(3, True), Choice(3, False)]
    for ub in range_bounds:
        out += [Range(ub), Range(ub, from_ct=True)]
    return out + [QV(*qv)]


# ---------------------------------------------------------------- the maps against the oracle

def _oracle_rows(P, pk, items, wide):
    """The replaying oracle on each item's blocks; every block is drawn, none past the end."""
    out = []
    for item, blocks in zip(items, wide):
        rng = O.rng_from_blocks(bytes(blocks))
        out.append(P.oracle(pk, item, rng))
        assert O.rng_blocks_left(rng) == 0, (P.name, item, O.rng_blocks_left(rng))
    return _rows(out)


def _random_wide(P, items, rnd):
    d = len(P.draw_map(items[0]))
    assert all(len(P.draw_map(it)) == d for it in items)
    return np.frombuffer(rnd.randbytes(len(items) * d * 64), np.uint8).reshape(len(items), d, 64).copy()


def check_draw_maps(P, pk, seed=1):
    """On random blocks: each r position gives the R its ciphertext carries ([r]G), each forged-response position is the
    response the proof carries; changing one forged-response block changes that response to the new block's scalar and no
    other forged response.  Replaying the blocks of ChaCha20 streams gives the seeded oracle's bytes (gen_*_batch included)."""
    rnd = random.Random(seed)
    items = P.items()
    wide = _random_wide(P, items, rnd)
    rows = _oracle_rows(P, pk, items, wide)
    for i, item in enumerate(items):
        roles = P.draw_map(item)
        blocks = [bytes(b) for b in wide[i]]
        forged = [(p, r) for p, r in enumerate(roles) if r[1] in ("s", "f")]
        for pos, (part, kind, ring, eq) in enumerate(roles):
            if kind == "r":
                assert P.R(rows[i], part, ring) == O.point_mul_generator(sc(red(blocks[pos]))), (P.name, item, pos)
            if kind in ("s", "f"):
                assert P.response(rows[i], part, ring, eq) == sc(red(blocks[pos])), (P.name, item, pos)
            if kind == "x" and hasattr(P, "e0") and not any(r[:3] == (part, "f", ring) for r in roles):
                # real index 0: the response is e0 r + x
                e0 = int.from_bytes(P.e0(rows[i], part), "little")
                r = P.ring_r(item, blocks, roles, part, ring)
                assert P.response(rows[i], part, ring, 0) == sc(e0 * r + red(blocks[pos])), (P.name, item, pos)
            if kind == "n" and isinstance(P, (EncryptZero, Choice)):
                # the log-equality proof (c, s) of a zero encryption / a single choice's sum: s = c r + x, r the sum of the r
                c, s = int.from_bytes(bytes(rows[i, -64:-32]), "little"), bytes(rows[i, -32:])
                r = sum(red(blocks[p]) for p, ro in enumerate(roles) if ro[1] == "r")
                assert s == sc(c * r + red(blocks[pos])), (P.name, item, pos)
        if forged:
            pos, (part, _, ring, eq) = forged[i % len(forged)]
            changed = wide[i].copy()
            changed[pos] = np.frombuffer(rnd.randbytes(64), np.uint8)
            row2 = _oracle_rows(P, pk, [item], changed[None])[0]
            assert P.response(row2, part, ring, eq) == sc(red(bytes(changed[pos])))
            for p, (pa, _, ri, q) in forged:
                if p != pos:
                    assert P.response(row2, pa, ri, q) == P.response(rows[i], pa, ri, q), (P.name, item, pos, p)
    try:                                        # one block short: the replay refuses the last draw
        _oracle_rows(P, pk, items[:1], wide[:1, :-1])
    except O.RngOverrun:
        pass
    else:
        raise AssertionError(f"{P.name}: a replay one block short was accepted")
    check_replay_matches_seeded(P, pk, items)


def check_replay_matches_seeded(P, pk, items, seed=b"\x71" * 32, first=5):
    """Replaying item i's ChaCha20 stream (block counter (first + i) << 20) gives the seeded oracle call's bytes."""
    n = len(items)
    if isinstance(P, Choice) and P.as_bool:         # gen_bool_batch encrypts (first + i) mod 2
        items = [((first + i) & 1,) for i in range(n)]
    elif isinstance(P, Choice) and P.single:        # gen_choice_batch marks option (first + i) mod m
        items = [tuple(int(k == (first + i) % P.m) for k in range(P.m)) for i in range(n)]
    d = len(P.draw_map(items[0]))
    seeded = [P.oracle(pk, it, O.rng_from_seed(seed, (first + i) << 20)) for i, it in enumerate(items)]
    wide = np.frombuffer(b"".join(PC.item_blocks(seed, first + i, d) for i in range(len(items))), np.uint8).reshape(len(items), d, 64)
    assert _oracle_rows(P, pk, items, wide).tobytes() == b"".join(seeded), P.name
    if isinstance(P, Choice) and P.as_bool:
        c, p = O.gen_bool_batch(pk, seed, n, first=first)
        batch = _cat(c, p)
    elif isinstance(P, Choice) and P.single:
        batch = _cat(*O.gen_choice_batch(pk, P.m, seed, n, first=first))
    elif isinstance(P, QV):
        batch = O.gen_qv_batch(pk, P.p, seed, np.array(items, np.uint64), first=first)
    elif isinstance(P, Range) and not P.from_ct:
        batch = _cat(*O.gen_range_batch(pk, P.spec, P.label, seed, np.array(items, np.uint64), first=first))
    else:
        return
    assert batch.tobytes() == b"".join(seeded), P.name


# ---------------------------------------------------------------- cases

def role_cases(P, wide_stride=1, kinds=("r", "x", "s", "f", "n"), seed=2):
    """(items, wide): each target block in each role kind the prover has, over its items and positions in turn; the other
    blocks random."""
    rnd = random.Random(seed)
    base = P.items()
    targets = target_blocks(wide_stride)
    kinds = [k for k in kinds if any(r[1] == k for it in base for r in P.draw_map(it))]
    items, wide = [], []
    for t_i, t in enumerate(targets):
        for k_i, kind in enumerate(kinds):
            cands = [(it, p) for it in base for p, r in enumerate(P.draw_map(it)) if r[1] == kind]
            item, pos = cands[(7 * t_i + k_i) % len(cands)]
            d = len(P.draw_map(item))
            blocks = [rnd.randbytes(64) for _ in range(d)]
            blocks[pos] = t
            items.append(item)
            wide.append(b"".join(blocks))
    return items, np.frombuffer(b"".join(wide), np.uint8).reshape(len(items), -1, 64).copy()


def derived_cases(P, pk, wide_stride=1, seed=3):
    """Forged equations on e0 (kind "f", eq 0: the value-1 ring of bool / choice, range rings whose real index is not 0)
    with s = e0 r + t, so that s - e0 r = t: t = 0 makes the forged commitments O and [e0 (a - v)]G, t = 2 edge puts the edge
    into the halved scalar.  e0 is read from a first run; it does not depend on these draws, which is asserted."""
    rnd = random.Random(seed)
    base = [it for it in P.items() if any(r[1] == "f" and r[3] == 0 for r in P.draw_map(it))]
    offsets = derived_offsets(wide_stride)
    items = [base[k % len(base)] for k in range(len(offsets))]
    wide = _random_wide(P, items, rnd)
    first = _oracle_rows(P, pk, items, wide)
    def e0s(rows):
        return [{part: int.from_bytes(P.e0(rows[i], part), "little") for part in {r[0] for r in P.draw_map(it) if r[1] != "n"}}
                for i, it in enumerate(items)]
    before = e0s(first)
    for i, item in enumerate(items):
        roles = P.draw_map(item)
        blocks = [bytes(b) for b in wide[i]]
        for pos, (part, kind, ring, eq) in enumerate(roles):
            if kind == "f" and eq == 0:
                r = P.ring_r(item, blocks, roles, part, ring)
                wide[i, pos] = np.frombuffer(blk((before[i][part] * r + offsets[i]) % L), np.uint8)
    second = _oracle_rows(P, pk, items, wide)
    assert e0s(second) == before, P.name
    for i, item in enumerate(items):            # the forged responses are what was aimed at
        roles = P.draw_map(item)
        for part, kind, ring, eq in roles:
            if kind == "f" and eq == 0:
                r = P.ring_r(item, [bytes(b) for b in wide[i]], roles, part, ring)
                s = int.from_bytes(P.response(second[i], part, ring, 0), "little")
                assert (s - before[i][part] * r) % L == offsets[i], (P.name, item)
    return items, wide


def cancel_cases(P, seed=4):
    """Randomness that cancels: r = 0 with the value 0 (the ciphertext (O, O)) and, for choices, rings whose r sum to 0 mod l
    (sum ciphertext (O, [count]G); for a single choice the sum proof then runs on (O, O))."""
    rnd = random.Random(seed)
    items, wide = [], []
    for item in P.items():
        roles = P.draw_map(item)
        zero_value = item in (0, (0,)) or (isinstance(item, tuple) and not any(item))
        variants = []
        r_pos = [p for p, r in enumerate(roles) if r[1] == "r"]
        if zero_value or isinstance(P, (Range, QV)):
            variants.append({p: blk(0) for p in r_pos} if zero_value else {r_pos[0]: blk(0)})
        if isinstance(P, Choice) and not P.as_bool and len(r_pos) > 1:
            rs = [rnd.randrange(L) for _ in r_pos[:-1]]
            v = {p: blk(r) for p, r in zip(r_pos, rs)}
            v[r_pos[-1]] = blk((-sum(rs)) % L)
            variants.append(v)
            v = dict(v)
            v[r_pos[-1]] = blk((-sum(rs)) % L + L)             # the same sum, from a block that is not reduced
            variants.append(v)
        for v in variants:
            blocks = [rnd.randbytes(64) for _ in roles]
            for p, b in v.items():
                blocks[p] = b
            items.append(item)
            wide.append(b"".join(blocks))
    if not items:
        return [], None
    return items, np.frombuffer(b"".join(wide), np.uint8).reshape(len(items), -1, 64).copy()


def all_cases(P, pk, wide_stride=1):
    """Role targets, derived targets and cancelling randomness in one batch; wide_stride > 1 takes every wide_stride-th
    window edge only (the CPU harness, where every item costs a full host-side prover and verifier run)."""
    parts = [role_cases(P, wide_stride)]
    if P.rings and any(r[1] == "f" and r[3] == 0 for it in P.items() for r in P.draw_map(it)):
        parts.append(derived_cases(P, pk, wide_stride))
    c = cancel_cases(P)
    if c[0]:
        parts.append(c)
    items = [it for p in parts for it in p[0]]
    return items, np.concatenate([p[1] for p in parts])


# ---------------------------------------------------------------- the checks

def _tamper(rows):
    """One item per batch: a flipped low bit in the last scalar of the output (a response, or a sum proof's)."""
    bad = rows.copy()
    i = rows.shape[0] // 2
    bad[i, -32] ^= 1
    return bad, i


def check_prover_edges(e, sk, pk, P, items, wide, ring_modes=SC.RING_MODES, chunk=None):
    """The engine's output on the chosen blocks equals the replaying oracle's byte for byte in both prover modes (and, with
    `chunk`, in a chunked run with a remainder); the engine's verifiers in every ring mode give the oracle's verdicts and
    tallies for the outputs and for the outputs with one item tampered; the ciphertexts decrypt to their values."""
    n = len(items)
    expected = _oracle_rows(P, pk, items, wide)
    fast, slow = EC.both_modes(e, lambda: P.engine(e, items, wide))
    bad = np.nonzero((fast != expected).any(axis=1))[0]
    assert bad.size == 0, (P.name, "default mode", bad[:6].tolist(), [items[i] for i in bad[:3]])
    bad = np.nonzero((slow != expected).any(axis=1))[0]
    assert bad.size == 0, (P.name, "constant-time mode", bad[:6].tolist(), [items[i] for i in bad[:3]])
    if chunk:
        chunked = SC.with_chunk(e, chunk, lambda: P.engine(e, items, wide))
        assert (chunked == expected).all(), P.name
    tampered, ti = _tamper(expected)
    for rows, ok in ((expected, True), (tampered, False)):
        results = SC.in_ring_modes(e, lambda: P.verify(e, pk, rows), ring_modes)
        if chunk:
            results.append(SC.with_chunk(e, chunk, lambda: P.verify(e, pk, rows)))
        for res in results:
            if res is None:
                continue
            got, exp, tally, exp_tally = res
            exp = np.asarray(exp)
            assert got.tolist() == exp.tolist(), (P.name, ok, np.nonzero(got != exp)[0][:6].tolist())
            if ok:
                assert (exp == 0).all(), (P.name, np.nonzero(exp)[0][:6].tolist())
            else:
                assert exp[ti] != 0 and (np.delete(exp, ti) == 0).all(), P.name
            if exp_tally is not None:
                assert (tally == exp_tally).all(), (P.name, ok)
    cts, values = [], []
    for row, item in zip(expected, items):
        for off, v in P.plaintexts(item):
            cts.append(bytes(row[off:off + 64]))
            values.append(v)
    el, _, found = e.decrypt(sk, _rows(cts))
    assert (found == 1).all()
    want = {v: O.point_mul_generator(sc(v)) for v in set(values)}
    bad = [i for i, v in enumerate(values) if bytes(el[i]) != want[v]]
    assert not bad, (P.name, bad[:6])
    identity = [c for c, v in zip(cts, values) if v == 0 and c == bytes(64)]
    return n, len(identity)
