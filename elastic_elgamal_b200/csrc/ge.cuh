// ge.cuh -- ristretto255 group elements: extended twisted-Edwards arithmetic (a = -1), the RFC 9496
// encoding, and the multi-scalar chain used by every verification equation.
//
// Replaces curve25519-dalek's RistrettoPoint / CompressedRistretto / RISTRETTO_BASEPOINT_TABLE /
// VartimeMultiscalarMul as reached through src/group/ristretto.rs:72-146:
//   serialize_element :88 -> ge_encode, deserialize_element :93 -> ge_decode,
//   vartime_double_mul_generator :131 and vartime_multi_mul :139 -> ge_msm_chain (Straus with shared
//   doublings and fixed 4-bit signed windows for per-item bases; doubling-free walks over wide-window
//   affine tables for the batch-constant bases G, K, H).  Results are group elements, so the choice of
//   algorithm is invisible in the canonical encodings the verifier hashes.
#pragma once
#include "fe.cuh"
#include "sc.cuh"

namespace eg {

struct ge_ext { fe X, Y, Z, T; };             // x = X/Z, y = Y/Z, xy = T/Z
struct ge_cached { fe YpX, YmX, Z, T2d; };    // (Y+X, Y-X, Z, 2dT)
struct ge_niels { fe ypx, ymx, xy2d; };       // affine: (y+x, y-x, 2dxy)
struct ge_p1p1 { fe E, F, G, H; };            // completed: X = EF, Y = GH, Z = FG, T = EH

EG_HD ge_ext ge_identity() { ge_ext r; r.X = fe_zero(); r.Y = fe_one(); r.Z = fe_one(); r.T = fe_zero(); return r; }

EG_HD ge_ext ge_generator() {
    ge_ext r;
    r.X = fe_make(0x8f25d51au, 0xc9562d60u, 0x9525a7b2u, 0x692cc760u, 0xfdd6dc5cu, 0xc0a4e231u, 0xcd6e53feu, 0x216936d3u);
    r.Y = fe_make(0x66666658u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u);
    r.Z = fe_one();
    r.T = fe_make(0xa5b7dda3u, 0x6dde8ab3u, 0x775152f5u, 0x20f09f80u, 0x64abe37du, 0x66ea4e8eu, 0xd78b7665u, 0x67875f0fu);
    return r;
}

// Field multiply / square policies for the point formulas below.  `fe_ops_call` goes through the non-inlined
// fe_mul / fe_sq (compact code: setup, encodings, cold paths); `fe_ops_inline` expands the tuned PTX sequence in place and
// is used only inside the three hot point operations (ge_hot_*), which are themselves non-inlined: the hot code stays
// ~50 KB (instruction cache) and the by-value call ABI's register moves -- which ptxas issues as IMAD.MOV on the same
// pipe as the multiplier -- disappear from the inner loops.
struct fe_ops_call {
    static EG_HD void mul(fe &r, const fe &a, const fe &b) { fe_mul(r, a, b); }
    static EG_HD void sq(fe &r, const fe &a) { fe_sq(r, a); }
};
struct fe_ops_inline {
    static EG_HD void mul(fe &r, const fe &a, const fe &b) {
#if defined(__CUDA_ARCH__) && !defined(EG_PORTABLE_FE)
        fe_mul_ptx(r, a, b);
#else
        fe_mul_portable(r, a, b);
#endif
    }
    static EG_HD void sq(fe &r, const fe &a) {
#if defined(__CUDA_ARCH__) && !defined(EG_PORTABLE_FE)
        fe_sq_ptx(r, a);
#else
        fe_sq_portable(r, a);
#endif
    }
};

template <class O = fe_ops_call>
EG_HD void ge_p1p1_to_ext(ge_ext &r, const ge_p1p1 &p) {
    O::mul(r.X, p.E, p.F); O::mul(r.Y, p.G, p.H); O::mul(r.Z, p.F, p.G); O::mul(r.T, p.E, p.H);
}

// projective only (T left stale): enough when a doubling follows
template <class O = fe_ops_call>
EG_HD void ge_p1p1_to_proj(ge_ext &r, const ge_p1p1 &p) {
    O::mul(r.X, p.E, p.F); O::mul(r.Y, p.G, p.H); O::mul(r.Z, p.F, p.G);
}

// dbl-2008-hwcd; reads X, Y, Z only
template <class O = fe_ops_call>
EG_HD void ge_dbl_p1p1(ge_p1p1 &r, const ge_ext &p) {
    fe a, b, c, t;
    O::sq(a, p.X); O::sq(b, p.Y);
    O::sq(c, p.Z); fe_add(c, c, c);
    fe_add(t, p.X, p.Y); O::sq(t, t);
    fe_add(r.H, a, b);              // A + B
    fe_sub(r.E, t, r.H);            // E = (X+Y)^2 - A - B
    fe_sub(r.G, b, a);              // G = B - A
    fe_sub(r.F, r.G, c);            // F = G - C
    fe_neg(r.H, r.H);               // H = -(A + B)
}

EG_HD void ge_to_cached(ge_cached &c, const ge_ext &p) {
    fe_add(c.YpX, p.Y, p.X); fe_sub(c.YmX, p.Y, p.X); c.Z = p.Z; fe_mul(c.T2d, p.T, fe_const_2d());
}

// add-2008-hwcd-3 with a cached second operand; neg subtracts it
template <class O = fe_ops_call>
EG_HD void ge_add_cached_p1p1(ge_p1p1 &r, const ge_ext &p, const ge_cached &q, bool neg) {
    fe a, b, c, d, pm, pp;
    fe_sub(a, p.Y, p.X); fe_add(b, p.Y, p.X);
    fe_select(pm, q.YmX, q.YpX, neg); fe_select(pp, q.YpX, q.YmX, neg);
    O::mul(a, a, pm); O::mul(b, b, pp);
    O::mul(c, p.T, q.T2d);
    O::mul(d, p.Z, q.Z); fe_add(d, d, d);
    fe_sub(r.E, b, a); fe_add(r.H, b, a);
    fe nf, ng;
    fe_sub(nf, d, c); fe_add(ng, d, c);
    fe_select(r.F, nf, ng, neg); fe_select(r.G, ng, nf, neg);     // negating q flips the sign of C
}

// mixed addition with an affine Niels operand (Z2 = 1)
template <class O = fe_ops_call>
EG_HD void ge_add_niels_p1p1(ge_p1p1 &r, const ge_ext &p, const ge_niels &q, bool neg) {
    fe a, b, c, d, pm, pp;
    fe_sub(a, p.Y, p.X); fe_add(b, p.Y, p.X);
    fe_select(pm, q.ymx, q.ypx, neg); fe_select(pp, q.ypx, q.ymx, neg);
    O::mul(a, a, pm); O::mul(b, b, pp);
    O::mul(c, p.T, q.xy2d);
    fe_add(d, p.Z, p.Z);
    fe_sub(r.E, b, a); fe_add(r.H, b, a);
    fe nf, ng;
    fe_sub(nf, d, c); fe_add(ng, d, c);
    fe_select(r.F, nf, ng, neg); fe_select(r.G, ng, nf, neg);
}

EG_HD void ge_add(ge_ext &r, const ge_ext &p, const ge_ext &q) {
    ge_cached c; ge_p1p1 t;
    ge_to_cached(c, q);
    ge_add_cached_p1p1(t, p, c, false);
    ge_p1p1_to_ext(r, t);
}

EG_HD void ge_sub(ge_ext &r, const ge_ext &p, const ge_ext &q) {
    ge_cached c; ge_p1p1 t;
    ge_to_cached(c, q);
    ge_add_cached_p1p1(t, p, c, true);
    ge_p1p1_to_ext(r, t);
}

EG_HD void ge_dbl(ge_ext &r, const ge_ext &p) { ge_p1p1 t; ge_dbl_p1p1(t, p); ge_p1p1_to_ext(r, t); }

EG_HD void ge_neg(ge_ext &r, const ge_ext &p) { fe_neg(r.X, p.X); r.Y = p.Y; r.Z = p.Z; fe_neg(r.T, p.T); }

// ristretto equality with the identity class: X == 0 or Y == 0
EG_HD bool ge_is_identity(const ge_ext &p) { return fe_iszero(p.X) || fe_iszero(p.Y); }

// ------------------------------------------------------------------ RFC 9496 4.3.1 / 4.3.2

// s: canonical little-endian words of the 32-byte encoding.  Returns false (and the identity) when the
// encoding is rejected: non-canonical, negative, non-square, negative t, or y = 0.
EG_HD bool ge_decode(ge_ext &p, const uint32_t w[8]) {
    fe s, ss, u1, u2, u2s, v, t, inv, denx, deny, x, y;
    bool ok = fe_fromwords_canonical(s, w);
    ok = ok && ((w[0] & 1u) == 0);
    if (!ok) s = fe_zero();
    fe_sq(ss, s);
    fe_sub(u1, fe_one(), ss);
    fe_add(u2, fe_one(), ss);
    fe_sq(u2s, u2);
    fe_sq(t, u1); fe_mul(t, t, fe_const_d()); fe_neg(t, t);
    fe_sub(v, t, u2s);
    fe_mul(t, v, u2s);
    bool was_square = fe_invsqrt(inv, t);
    fe_mul(denx, inv, u2);
    fe_mul(deny, inv, denx); fe_mul(deny, deny, v);
    fe_add(t, s, s); fe_mul(x, t, denx);
    fe_abs(x, x);
    fe_mul(y, u1, deny);
    fe_mul(t, x, y);
    ok = ok && was_square && !fe_isneg(t) && !fe_iszero(y);
    if (!ok) { p = ge_identity(); return false; }
    p.X = x; p.Y = y; p.Z = fe_one(); p.T = t;
    return true;
}

EG_HD void ge_encode(uint32_t w[8], const ge_ext &p) {
    fe u1, u2, t, inv, den1, den2, zinv, ix, iy, ench, x, y, deninv, s;
    const fe sqrtm1 = fe_const_sqrtm1();
    fe_add(u1, p.Z, p.Y); fe_sub(t, p.Z, p.Y); fe_mul(u1, u1, t);
    fe_mul(u2, p.X, p.Y);
    fe_sq(t, u2); fe_mul(t, t, u1);
    fe_invsqrt(inv, t);
    fe_mul(den1, inv, u1);
    fe_mul(den2, inv, u2);
    fe_mul(zinv, den1, den2); fe_mul(zinv, zinv, p.T);
    fe_mul(ix, p.X, sqrtm1);
    fe_mul(iy, p.Y, sqrtm1);
    fe_mul(ench, den1, fe_const_invsqrt_a_minus_d());
    fe_mul(t, p.T, zinv);
    bool rotate = fe_isneg(t);
    fe_select(x, p.X, iy, rotate);
    fe_select(y, p.Y, ix, rotate);
    fe_select(deninv, den2, ench, rotate);
    fe_mul(t, x, zinv);
    fe_cneg(y, y, fe_isneg(t));
    fe_sub(t, p.Z, y);
    fe_mul(s, deninv, t);
    fe_abs(s, s);
    fe_towords(w, s);
}

// ------------------------------------------------------------------ fixed-base tables
//
// [b] F for the batch-constant bases (G, the receiver key K, the Pedersen base H) never doubles: the scalar is cut into
// EG_WIDE_WINDOWS signed windows of EG_WIDE_BITS bits, b = sum_i d_i 2^(W i) with d_i in [-2^(W-1), 2^(W-1)), and the table
// holds every |d| 2^(W i) F as an affine Niels point (96 B); [b] F costs one mixed addition (7 multiplications) per window.
// The width is a memory-for-arithmetic trade that HBM decides: every lookup is an independent 96-byte read (three 32-byte
// sectors) that is requested one window ahead, so the tables need not fit the L2.  Measured on B200, 5-option ballots/s:
//   W = 11 / 13 / 15 / 16 (24 .. 16 windows, <= 48 MiB per base): 1.860 / 1.895 / 1.922 / 1.934 M (profiles/r1_wide_tables_ab.txt;
//     8-bit windows over 4 chunks staged in shared memory: 1.865 M);
//   W = 16 / 20 / 24 (16 / 13 / 11 windows; 48 MiB / 0.61 GiB / 8.25 GiB per base): 2.072 / 2.100 / 2.128 M, range proofs
//     905 / 922 / 934 k/s (profiles/r2_ab_wide_bits.txt).
// W = 24 is the device default: 11 additions per fixed-base term, 2 x 8.25 GiB for G and K (+ 8.25 GiB with a Pedersen base)
// out of 180 GB of HBM, built on the device in tens of milliseconds.  W = 26 .. 31 would save one more addition (10 windows)
// for 4 x .. 128 x the memory.  A build with -DEG_WIDE_BITS=16 (or 20) keeps the small tables; the CPU test harness
// (tests/hostsim) uses 16.  W must be a multiple of 4 (ge_fixed_adds_ct).

#ifndef EG_WIDE_BITS
#ifdef EG_HOSTSIM
#define EG_WIDE_BITS 16
#else
#define EG_WIDE_BITS 24
#endif
#endif
static_assert(EG_WIDE_BITS % 4 == 0 && EG_WIDE_BITS >= 8 && EG_WIDE_BITS <= 28, "EG_WIDE_BITS: a multiple of 4 in 8..28");
#ifndef EG_WIDE_PREFETCH
#define EG_WIDE_PREFETCH 1
#endif
#define EG_WIDE_WINDOWS ((254 + EG_WIDE_BITS - 1) / EG_WIDE_BITS)     // W * windows >= 254: the top digit absorbs the last carry
#define EG_WIDE_ENTRIES (1 << (EG_WIDE_BITS - 1))                     // |d| = 1 .. 2^(W-1) per window
#define EG_WIDE_TABLE_WORDS ((size_t)EG_WIDE_WINDOWS * EG_WIDE_ENTRIES * 24)
#define EG_WIDE_BLOCK 32                                              // entries normalised together by the table builder
#define EG_WIDE_SCRATCH_WORDS (EG_WIDE_WINDOWS * 32)                  // window bases 2^(W i) F (extended), behind the table
// Narrow tables (16-bit windows, 48 MiB, ~1 ms to build) for bases that are constant for one call only -- the participant
// keys of a key set (PublicKeySet::verify_share): same layout and walk, built per call and cached by key bytes.
#define EG_NARROW_BITS 16
#define EG_BITS_WINDOWS(B) ((254 + (B) - 1) / (B))
#define EG_BITS_ENTRIES(B) (1 << ((B) - 1))
#define EG_BITS_TABLE_WORDS(B) ((size_t)EG_BITS_WINDOWS(B) * EG_BITS_ENTRIES(B) * 24)
#define EG_NARROW_ALLOC_WORDS (EG_BITS_TABLE_WORDS(EG_NARROW_BITS) + EG_BITS_WINDOWS(EG_NARROW_BITS) * 32)

EG_HD void ge_niels_load(ge_niels &n, const uint32_t *tbl, int idx) {
    const uint32_t *e = tbl + idx * 24;
    for (int i = 0; i < 8; i++) { n.ypx.v[i] = e[i]; n.ymx.v[i] = e[8 + i]; n.xy2d.v[i] = e[16 + i]; }
}

// one table entry: (k F) normalised to affine Niels form
EG_HD void ge_niels_from_ext(uint32_t out[24], const ge_ext &p) {
    fe zi, x, y, t;
    fe_invert(zi, p.Z);
    fe_mul(x, p.X, zi); fe_mul(y, p.Y, zi);
    fe_add(t, y, x); fe_towords(out, t);
    fe_sub(t, y, x); fe_towords(out + 8, t);
    fe_mul(t, x, y); fe_mul(t, t, fe_const_2d()); fe_towords(out + 16, t);
}

EG_HD void ge_niels_load4(ge_niels &n, const uint32_t *tbl, int idx) {
#if defined(__CUDA_ARCH__)
    const uint4 *q = reinterpret_cast<const uint4 *>(tbl + idx * 24);
    uint4 a;
    a = q[0]; n.ypx.v[0] = a.x; n.ypx.v[1] = a.y; n.ypx.v[2] = a.z; n.ypx.v[3] = a.w;
    a = q[1]; n.ypx.v[4] = a.x; n.ypx.v[5] = a.y; n.ypx.v[6] = a.z; n.ypx.v[7] = a.w;
    a = q[2]; n.ymx.v[0] = a.x; n.ymx.v[1] = a.y; n.ymx.v[2] = a.z; n.ymx.v[3] = a.w;
    a = q[3]; n.ymx.v[4] = a.x; n.ymx.v[5] = a.y; n.ymx.v[6] = a.z; n.ymx.v[7] = a.w;
    a = q[4]; n.xy2d.v[0] = a.x; n.xy2d.v[1] = a.y; n.xy2d.v[2] = a.z; n.xy2d.v[3] = a.w;
    a = q[5]; n.xy2d.v[4] = a.x; n.xy2d.v[5] = a.y; n.xy2d.v[6] = a.z; n.xy2d.v[7] = a.w;
#else
    ge_niels_load(n, tbl, idx);
#endif
}

EG_HD void ge_cached_store(uint32_t *e, const ge_cached &c) {
#if defined(__CUDA_ARCH__)
    uint4 *q = reinterpret_cast<uint4 *>(e);
    q[0] = make_uint4(c.YpX.v[0], c.YpX.v[1], c.YpX.v[2], c.YpX.v[3]); q[1] = make_uint4(c.YpX.v[4], c.YpX.v[5], c.YpX.v[6], c.YpX.v[7]);
    q[2] = make_uint4(c.YmX.v[0], c.YmX.v[1], c.YmX.v[2], c.YmX.v[3]); q[3] = make_uint4(c.YmX.v[4], c.YmX.v[5], c.YmX.v[6], c.YmX.v[7]);
    q[4] = make_uint4(c.Z.v[0], c.Z.v[1], c.Z.v[2], c.Z.v[3]);         q[5] = make_uint4(c.Z.v[4], c.Z.v[5], c.Z.v[6], c.Z.v[7]);
    q[6] = make_uint4(c.T2d.v[0], c.T2d.v[1], c.T2d.v[2], c.T2d.v[3]); q[7] = make_uint4(c.T2d.v[4], c.T2d.v[5], c.T2d.v[6], c.T2d.v[7]);
#else
    for (int k = 0; k < 8; k++) { e[k] = c.YpX.v[k]; e[8 + k] = c.YmX.v[k]; e[16 + k] = c.Z.v[k]; e[24 + k] = c.T2d.v[k]; }
#endif
}

EG_HD void ge_cached_load(ge_cached &c, const uint32_t *e) {
#if defined(__CUDA_ARCH__)
    const uint4 *q = reinterpret_cast<const uint4 *>(e);
    uint4 a;
    a = q[0]; c.YpX.v[0] = a.x; c.YpX.v[1] = a.y; c.YpX.v[2] = a.z; c.YpX.v[3] = a.w;
    a = q[1]; c.YpX.v[4] = a.x; c.YpX.v[5] = a.y; c.YpX.v[6] = a.z; c.YpX.v[7] = a.w;
    a = q[2]; c.YmX.v[0] = a.x; c.YmX.v[1] = a.y; c.YmX.v[2] = a.z; c.YmX.v[3] = a.w;
    a = q[3]; c.YmX.v[4] = a.x; c.YmX.v[5] = a.y; c.YmX.v[6] = a.z; c.YmX.v[7] = a.w;
    a = q[4]; c.Z.v[0] = a.x; c.Z.v[1] = a.y; c.Z.v[2] = a.z; c.Z.v[3] = a.w;
    a = q[5]; c.Z.v[4] = a.x; c.Z.v[5] = a.y; c.Z.v[6] = a.z; c.Z.v[7] = a.w;
    a = q[6]; c.T2d.v[0] = a.x; c.T2d.v[1] = a.y; c.T2d.v[2] = a.z; c.T2d.v[3] = a.w;
    a = q[7]; c.T2d.v[4] = a.x; c.T2d.v[5] = a.y; c.T2d.v[6] = a.z; c.T2d.v[7] = a.w;
#else
    for (int k = 0; k < 8; k++) { c.YpX.v[k] = e[k]; c.YmX.v[k] = e[8 + k]; c.Z.v[k] = e[16 + k]; c.T2d.v[k] = e[24 + k]; }
#endif
}

// ------------------------------------------------------------------ the three hot point operations
//
// Every inner loop of the multi-scalar kernels is a sequence of these three calls on an accumulator that lives in the
// caller's frame.  EG_HOT_OPS selects the field policy inside them: with fe_ops_inline the three bodies are ~58 KB of
// SASS and, because the warps of a persistent kernel sit in different functions at the same time, overflow the 32 KB
// L1.5 instruction cache (ncu: `no_instruction` becomes the top stall, profiles/r1_k_ring_hot_inline.txt); fe_ops_call
// keeps the resident hot set near 20 KB.
#ifndef EG_HOT_OPS
#define EG_HOT_OPS fe_ops_call
#endif
// The shared doubling callee (ge_hot_dbl: table builds, the single-use chains of k_commit / k_msm) expands its field
// operations in place: one 14 KB body next to the 4 KB of fe_mul / fe_sq still fits the instruction cache and drops the
// ~20 register moves per field operation of the call ABI from 56 % of the point operations.  Measured
// (profiles/r2_ab_inline_doubling.txt): k_msm -12 %, k_ring<256,2,8> -1.4 %, k_commit -8 %; expanding the additions or the
// evaluation loop as well loses 1.5-4 % (instruction cache).
#ifndef EG_HOT_DBL_OPS
#define EG_HOT_DBL_OPS fe_ops_inline
#endif
#ifndef EG_HOT_DBL_PROJ_OPS
#define EG_HOT_DBL_PROJ_OPS EG_HOT_DBL_OPS
#endif
#ifndef EG_EVAL_DBL_OPS
#define EG_EVAL_DBL_OPS fe_ops_call
#endif
#ifndef EG_EVAL_PROJ_OPS
#define EG_EVAL_PROJ_OPS fe_ops_call
#endif

// acc = 2^n acc (n >= 1); intermediate doublings stay projective, T is produced by the last one
static EG_HD_NOINLINE void ge_hot_dbl(ge_ext &acc, int n) {
    ge_ext a = acc;
    ge_p1p1 t;
#pragma unroll 1
    for (int k = 0; k < n; k++) {
        ge_dbl_p1p1<EG_HOT_DBL_OPS>(t, a);
        ge_p1p1_to_proj<EG_HOT_DBL_PROJ_OPS>(a, t);
        if (k == n - 1) EG_HOT_DBL_PROJ_OPS::mul(a.T, t.E, t.H);
    }
    acc = a;
}

// acc += (neg ? -Q : Q), Q a cached point at `entry` (32 words, 16-byte aligned)
// need_t = false leaves T stale: enough when a doubling follows
static EG_HD_NOINLINE void ge_hot_add_cached(ge_ext &acc, const uint32_t *entry, bool neg, bool need_t = true) {
    ge_cached q;
    ge_cached_load(q, entry);
    ge_p1p1 t;
    ge_add_cached_p1p1<EG_HOT_OPS>(t, acc, q, neg);
    ge_p1p1_to_proj<EG_HOT_OPS>(acc, t);
    if (need_t) EG_HOT_OPS::mul(acc.T, t.E, t.H);
}

// acc += (neg ? -Q : Q), Q = entry `idx` of an affine Niels table (24 words per entry, 16-byte aligned)
static EG_HD_NOINLINE void ge_hot_add_niels(ge_ext &acc, const uint32_t *table, int idx, bool neg) {
    ge_niels q;
    ge_niels_load4(q, table, idx);
    ge_p1p1 t;
    ge_add_niels_p1p1<EG_HOT_OPS>(t, acc, q, neg);
    ge_p1p1_to_ext<EG_HOT_OPS>(acc, t);
}

// ------------------------------------------------------------------ scalar recoding

// 4-bit signed windows: a + 0x888...8 so that digit_i = nibble_i - 8 in [-8, 7]  (a < 2^253)
EG_HD void sc_recode4(uint32_t out[8], const sc &a) {
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (uint64_t)a.v[i] + 0x88888888u; out[i] = (uint32_t)c; c >>= 32; }
}
EG_HD int sc_digit4(const uint32_t r[8], int i) { return (int)((r[i >> 3] >> ((i & 7) * 4)) & 15u) - 8; }

// EG_WIDE_BITS-bit signed windows, produced low to high with a running carry: digit i of `a` in [-2^(W-1), 2^(W-1)).
// a < 2^253 and W * EG_WIDE_WINDOWS >= 254, so the top window never carries out.
template <int BITS>
EG_HD int sc_wide_digit_b(const sc &a, int i, uint32_t &carry) {
    const int o = i * BITS, word = o >> 5, sh = o & 31;
    uint32_t v = word < 8 ? a.v[word] >> sh : 0u;
    if (sh + BITS > 32 && word + 1 < 8) v |= a.v[word + 1] << (32 - sh);
    v = (v & ((1u << BITS) - 1u)) + carry;
    carry = (v >> (BITS - 1)) != 0u;                 // v >= 2^(W-1) (v <= 2^W): borrow 2^W from the next window
    return (int)v - (int)(carry << BITS);
}
EG_HD int sc_wide_digit(const sc &a, int i, uint32_t &carry) { return sc_wide_digit_b<EG_WIDE_BITS>(a, i, carry); }

// the (at most two) 128-byte lines of a 96-byte table entry, requested ahead of its use
EG_HD void ge_wide_prefetch(const uint32_t *entry) {
#if defined(__CUDA_ARCH__) && EG_WIDE_PREFETCH == 2
    asm volatile("prefetch.global.L1 [%0];" :: "l"(entry));
    asm volatile("prefetch.global.L1 [%0];" :: "l"(entry + 23));
#elif defined(__CUDA_ARCH__) && EG_WIDE_PREFETCH == 1
    asm volatile("prefetch.global.L2 [%0];" :: "l"(entry));
    asm volatile("prefetch.global.L2 [%0];" :: "l"(entry + 23));
#else
    (void)entry;
#endif
}

// ------------------------------------------------------------------ the multi-scalar chain

// acc = sum_{v<NV} a_v P_v + sum_{f<NF} b_f F_f
//   P_v : per-item points (extended), windows of 4 bits over a per-thread table of [1..8]P_v
//   F_f : fixed bases, added afterwards from their wide-window tables (ge_fixed_accumulate: no doublings)
// One shared doubling chain of 252 doublings (Straus) for the per-item points.  NV, NF are compile-time.
#if defined(__CUDACC__)
#define EG_ALIGN16 __align__(16)
#else
#define EG_ALIGN16 alignas(16)
#endif

// table of [1..8] P as cached points (per-thread, local memory)
EG_HD void ge_window_table(ge_cached tbl[8], const ge_ext &P) {
    ge_ext cur = P;
    ge_to_cached(tbl[0], cur);
#pragma unroll 1
    for (int k = 1; k < 8; k++) {
        ge_hot_add_cached(cur, (const uint32_t *)&tbl[0], false);
        ge_to_cached(tbl[k], cur);
    }
}

// acc += [b] F from the wide table of F (EG_WIDE_WINDOWS mixed additions, no doublings)
template <int BITS>
static EG_HD_NOINLINE void ge_fixed_accumulate_b(ge_ext &acc, const uint32_t *wide, const sc &b) {
    uint32_t carry = 0;
#pragma unroll 1
    for (int i = 0; i < EG_BITS_WINDOWS(BITS); i++) {
        const int d = sc_wide_digit_b<BITS>(b, i, carry);
        if (d != 0) ge_hot_add_niels(acc, wide + (size_t)i * (EG_BITS_ENTRIES(BITS) * 24), (d < 0 ? -d : d) - 1, d < 0);
    }
}
// `narrow`: the table has EG_NARROW_BITS-bit windows (a per-call base) instead of the context's EG_WIDE_BITS
EG_HD void ge_fixed_accumulate(ge_ext &acc, const uint32_t *wide, const sc &b, bool narrow = false) {
    if (EG_NARROW_BITS != EG_WIDE_BITS && narrow) ge_fixed_accumulate_b<EG_NARROW_BITS>(acc, wide, b);
    else ge_fixed_accumulate_b<EG_WIDE_BITS>(acc, wide, b);
}

template <int NV, int NF>
EG_HD void ge_msm_chain(ge_ext &out, const ge_ext *P, const sc *a, const uint32_t *const *ftab, const sc *b) {
    EG_ALIGN16 ge_cached tbl[NV > 0 ? NV : 1][8];
    uint32_t ra[NV > 0 ? NV : 1][8];
#pragma unroll 1
    for (int v = 0; v < NV; v++) {
        ge_window_table(tbl[v], P[v]);
        sc_recode4(ra[v], a[v]);
    }
    ge_ext acc = ge_identity();
    if (NV > 0) {
#pragma unroll 1
        for (int i = 63; i >= 0; i--) {
            if (i != 63) ge_hot_dbl(acc, 4);
#pragma unroll 1
            for (int v = 0; v < NV; v++) {
                int d = sc_digit4(ra[v], i);
                if (d != 0) ge_hot_add_cached(acc, (const uint32_t *)&tbl[v][(d < 0 ? -d : d) - 1], d < 0, v != NV - 1 || i == 0);
            }
        }
    }
#pragma unroll 1
    for (int f = 0; f < NF; f++) ge_fixed_accumulate(acc, ftab[f], b[f]);
    out = acc;
}


// Same chain with run-time term counts (nv <= MAXV, nf <= 2), for the equations that are not of the [a]P + [b]F shape:
// share verification (two per-item bases), SumOfSquaresProof (G, K and one per-item base; (n+2)-term sums) and
// Lagrange recombination.  Replaces the general vartime_multi_mul (ristretto.rs:139-146).
template <int MAXV>
EG_HD void ge_msm_chain_rt(ge_ext &out, int nv, const ge_ext *P, const sc *a, int nf, const uint32_t *const *ftab, const sc *b,
                           const bool *narrow = nullptr) {
    EG_ALIGN16 ge_cached tbl[MAXV][8];
    uint32_t ra[MAXV][8];
#pragma unroll 1
    for (int v = 0; v < nv; v++) {
        ge_window_table(tbl[v], P[v]);
        sc_recode4(ra[v], a[v]);
    }
    ge_ext acc = ge_identity();
    if (nv > 0) {
#pragma unroll 1
        for (int i = 63; i >= 0; i--) {
            if (i != 63) ge_hot_dbl(acc, 4);
#pragma unroll 1
            for (int v = 0; v < nv; v++) {
                int d = sc_digit4(ra[v], i);
                if (d != 0) ge_hot_add_cached(acc, (const uint32_t *)&tbl[v][(d < 0 ? -d : d) - 1], d < 0, v != nv - 1 || i == 0);
            }
        }
    }
#pragma unroll 1
    for (int f = 0; f < nf; f++) ge_fixed_accumulate(acc, ftab[f], b[f], narrow && narrow[f]);
    out = acc;
}

// ------------------------------------------------------------------ chunked tables: 64 doublings per equation
//
// A ring proof evaluates several equations on the SAME ciphertext points (one per admissible value, ring.rs:333-361)
// with different challenges.  Splitting a 253-bit scalar into four 64-bit chunks, a = sum_c 2^(64c) a_c, turns
// [a]P into sum_c [a_c] P_c with P_c = [2^(64c)] P: the 192 doublings that produce P_1..P_3 (and the four window
// tables [1..8] P_c) are paid once per point, every equation then needs only 64 shared doublings.  The fixed-base
// terms are added afterwards from the wide tables.

// The chunk count is a compile-time parameter of the table builder and the evaluator: 4 chunks for rings of two
// equations (ballot choices), 8 chunks (32 doublings per equation, 224 for the tables) for the longer rings of range
// proofs -- measured on B200 (profiles/r1_wide_tables_ab.txt): 8 chunks -1.8 % on 5-option ballots, +3.7 % on
// RangeProof [0, 2^16).
#ifndef EG_EVAL_VIA_HOT_DBL
#define EG_EVAL_VIA_HOT_DBL 0
#endif
#ifndef EG_VTAB_PREFETCH
#define EG_VTAB_PREFETCH 1
#endif
#define EG_VCHUNKS_SHORT 4
#define EG_VCHUNKS_LONG 8
#define EG_VTAB_ENTRY_WORDS 32                                  // one cached point
#define EG_VTAB_WORDS (EG_VCHUNKS_LONG * 8 * EG_VTAB_ENTRY_WORDS)   // scratch reserved per point: 8 KB

// tab[(c * 8 + k) * 32 ..] = cached((k + 1) * 2^(256 c / C) * P), c < C, k < 8.  `tab` is 16-byte aligned scratch.
template <int C>
static EG_HD_NOINLINE void ge_vtab_build(uint32_t *tab, const ge_ext &P) {
    ge_ext base = P;
#pragma unroll 1
    for (int c = 0; c < C; c++) {
        uint32_t *t0 = tab + (c * 8) * EG_VTAB_ENTRY_WORDS;
        ge_cached ck;
        ge_to_cached(ck, base);
        ge_cached_store(t0, ck);
        ge_ext cur = base;
#pragma unroll 1
        for (int k = 1; k < 8; k++) {
            ge_hot_add_cached(cur, t0, false);
            ge_to_cached(ck, cur);
            ge_cached_store(t0 + k * EG_VTAB_ENTRY_WORDS, ck);
        }
        if (c + 1 < C) ge_hot_dbl(base, 256 / C);
    }
}

// acc += [b0] F0 (+ [b1] F1 when nf == 2) from the wide tables; `t` is the caller's scratch.  Inlined into its callers so
// that the accumulator stays in registers.
EG_HD void ge_fixed_adds(ge_ext &acc, ge_p1p1 &t, int nf, const uint32_t *ftab0, const sc &b0, const uint32_t *ftab1, const sc &b1) {
#pragma unroll 1
    for (int f = 0; f < nf; f++) {
        const uint32_t *ft = f ? ftab1 : ftab0;
        const sc &b = f ? b1 : b0;
        uint32_t carry = 0;
        int d = sc_wide_digit(b, 0, carry);
        const uint32_t *entry = ft + (size_t)((d < 0 ? -d : d) - (d != 0)) * 24;
#pragma unroll 1
        for (int i = 0; i < EG_WIDE_WINDOWS; i++) {
            const int dc = d;
            const uint32_t *ec = entry;
            if (i + 1 < EG_WIDE_WINDOWS) {          // digit and address of the next window; its lines are requested now
                d = sc_wide_digit(b, i + 1, carry);
                entry = ft + ((size_t)(i + 1) * EG_WIDE_ENTRIES + (size_t)((d < 0 ? -d : d) - (d != 0))) * 24;
                ge_wide_prefetch(entry);
            }
            if (dc != 0) {
                ge_niels n;
                ge_niels_load4(n, ec, 0);
                ge_add_niels_p1p1(t, acc, n, dc < 0);
                ge_p1p1_to_ext(acc, t);
            }
        }
    }
}

// out = [a] P + [b0] F0 (+ [b1] F1 when nf == 2): vtab from ge_vtab_build<C>(P) (or null: fixed-base terms only), ftab* = wide
// fixed-base tables.  256 / C - 4 doublings and 64 additions for the per-item point, EG_WIDE_WINDOWS mixed additions per
// fixed base.
template <int C>
static EG_HD_NOINLINE void ge_eval64(ge_ext &out, const uint32_t *vtab, const sc &a, int nf, const uint32_t *ftab0, const sc &b0,
                     const uint32_t *ftab1, const sc &b1) {
    constexpr int W = 64 / C;                  // 4-bit windows per chunk
    // the accumulator stays in registers for the whole function: the point formulas are expanded here once each (rolled
    // loops), with the field operations as calls (see EG_HOT_OPS above for why they are not expanded)
    ge_ext acc = ge_identity();
    ge_p1p1 t;
    if (vtab) {
        uint32_t ra[8];
        sc_recode4(ra, a);
#pragma unroll 1
        for (int i = W - 1; i >= 0; i--) {
#if defined(__CUDA_ARCH__) && EG_VTAB_PREFETCH
            // the C table entries of this window are needed after the four doublings below: request their lines now (the
            // per-thread tables miss L1 in ~11 % of the loads and then come from L2 / HBM, ncu long_scoreboard)
#pragma unroll 1
            for (int c = 0; c < C; c++) {
                const int d = sc_digit4(ra, W * c + i);
                if (d != 0) asm volatile("prefetch.global.L1 [%0];" :: "l"(vtab + (c * 8 + (d < 0 ? -d : d) - 1) * EG_VTAB_ENTRY_WORDS));
            }
#endif
            if (i != W - 1) {
#if EG_EVAL_VIA_HOT_DBL
                ge_hot_dbl(acc, 4);         // A/B: the shared doubling callee (with EG_HOT_DBL_OPS=fe_ops_inline: no per-field-op calls)
#else
#pragma unroll 1
                for (int k = 0; k < 4; k++) {
                    ge_dbl_p1p1<EG_EVAL_DBL_OPS>(t, acc);
                    ge_p1p1_to_proj<EG_EVAL_PROJ_OPS>(acc, t);
                    if (k == 3) fe_mul(acc.T, t.E, t.H);
                }
#endif
            }
#pragma unroll 1
            for (int c = 0; c < C; c++) {
                int d = sc_digit4(ra, W * c + i);
                if (d != 0) {
                    ge_cached q;
                    ge_cached_load(q, vtab + (c * 8 + (d < 0 ? -d : d) - 1) * EG_VTAB_ENTRY_WORDS);
                    ge_add_cached_p1p1(t, acc, q, d < 0);
                    ge_p1p1_to_proj(acc, t);
                    if (c != C - 1 || i == 0) fe_mul(acc.T, t.E, t.H);     // T is dead when doublings follow
                }
            }
        }
    }
    ge_fixed_adds(acc, t, nf, ftab0, b0, ftab1, b1);
    out = acc;
}

// Constant-time form of ge_fixed_adds for SECRET scalars (the provers' randomness r and nonces x; the reference uses the
// constant-time G::mul_generator / multi_mul there, src/proofs/ring.rs:99,115-116).  The scalar is cut into 64 signed
// 4-bit windows; window i needs |d| * 16^i F with |d| <= 8, which is entry |d| * 16^(i mod N) of wide window i / N
// (N = EG_WIDE_BITS / 4 nibbles per wide window), so no second table is needed.  Every window reads all eight candidates and
// keeps one with masks, conditionally negates with masks and always adds (d = 0 adds the identity in Niels form): no branch
// and no address depends on the scalar.  64 mixed additions and 512 entry reads per base instead of EG_WIDE_WINDOWS of each:
// four to six times the fixed-base work (eg_ctx_set_prover_mode).
EG_HD void ge_fixed_adds_ct(ge_ext &acc, ge_p1p1 &t, int nf, const uint32_t *ftab0, const sc &b0, const uint32_t *ftab1, const sc &b1) {
#pragma unroll 1
    for (int f = 0; f < nf; f++) {
        const uint32_t *ft = f ? ftab1 : ftab0;
        uint32_t ra[8];
        sc_recode4(ra, f ? b1 : b0);
#pragma unroll 1
        for (int i = 0; i < 64; i++) {
            const int d = sc_digit4(ra, i);                         // secret, in [-8, 7]
            const uint32_t sign = (uint32_t)(d >> 31);              // all ones when negative
            const uint32_t mag = ((uint32_t)d ^ sign) - sign;       // |d|
            constexpr int NIB = EG_WIDE_BITS / 4;                    // 4-bit windows per wide window
            const uint32_t *win = ft + (size_t)(i / NIB) * (EG_WIDE_ENTRIES * 24);
            const uint32_t stride = 1u << (4 * (i % NIB));
            uint32_t e[24];
            for (int w = 0; w < 24; w++) e[w] = 0;
            e[0] = 1; e[8] = 1;                                     // identity: (y + x, y - x, 2dxy) = (1, 1, 0)
#pragma unroll 1
            for (uint32_t k = 1; k <= 8; k++) {
                const uint32_t *q = win + (size_t)(k * stride - 1) * 24;
                const uint32_t m = (uint32_t)0 - (uint32_t)((((mag ^ k) - 1u) >> 31) & 1u);      // all ones iff mag == k
                for (int w = 0; w < 24; w++) e[w] = (e[w] & ~m) | (q[w] & m);
            }
            ge_niels n;
            for (int w = 0; w < 8; w++) {
                n.ypx.v[w] = (e[w] & ~sign) | (e[8 + w] & sign);    // negation swaps y + x and y - x ...
                n.ymx.v[w] = (e[8 + w] & ~sign) | (e[w] & sign);
                n.xy2d.v[w] = e[16 + w];
            }
            fe nx;
            fe_neg(nx, n.xy2d);                                     // ... and negates 2dxy
            for (int w = 0; w < 8; w++) n.xy2d.v[w] = (n.xy2d.v[w] & ~sign) | (nx.v[w] & sign);
            ge_add_niels_p1p1(t, acc, n, false);
            ge_p1p1_to_ext(acc, t);
        }
    }
}

// out = [a] P from the per-thread window table of P (ge_window_table), variable time: 252 doublings, an addition per non-zero
// 4-bit digit.  For scalars whose digits are the same in every lane (a decryption key), the branches do not diverge.
static EG_HD_NOINLINE void ge_var_mul(ge_ext &out, const ge_cached tbl[8], const sc &a) {
    uint32_t ra[8];
    sc_recode4(ra, a);
    ge_ext acc = ge_identity();
#pragma unroll 1
    for (int i = 63; i >= 0; i--) {
        if (i != 63) ge_hot_dbl(acc, 4);
        const int d = sc_digit4(ra, i);
        if (d != 0) ge_hot_add_cached(acc, (const uint32_t *)&tbl[(d < 0 ? -d : d) - 1], d < 0, i == 0);
    }
    out = acc;
}

// Constant-time variable-base multiplication for SECRET scalars (a decryption key, a proof nonce): 64 signed 4-bit windows
// over the table [1..8] P; every window reads all eight entries and keeps one with masks, negates it with masks (swap
// Y + X / Y - X, negate 2dT) and always adds (digit 0 adds the identity (1, 1, 1, 0)).  No branch and no address depends
// on the scalar; 252 doublings and 64 additions.
static EG_HD_NOINLINE void ge_var_mul_ct(ge_ext &out, const ge_cached tbl[8], const sc &a) {
    uint32_t ra[8];
    sc_recode4(ra, a);
    ge_ext acc = ge_identity();
    ge_p1p1 t;
#pragma unroll 1
    for (int i = 63; i >= 0; i--) {
        if (i != 63) ge_hot_dbl(acc, 4);
        const int d = sc_digit4(ra, i);                         // secret, in [-8, 7]
        const uint32_t sign = (uint32_t)(d >> 31);              // all ones when negative
        const uint32_t mag = ((uint32_t)d ^ sign) - sign;       // |d|
        ge_cached e;
        e.YpX = fe_one(); e.YmX = fe_one(); e.Z = fe_one(); e.T2d = fe_zero();
#pragma unroll 1
        for (uint32_t k = 1; k <= 8; k++) {
            const uint32_t m = (uint32_t)0 - (uint32_t)((((mag ^ k) - 1u) >> 31) & 1u);      // all ones iff mag == k
            const ge_cached &q = tbl[k - 1];
            for (int w = 0; w < 8; w++) {
                e.YpX.v[w] = (e.YpX.v[w] & ~m) | (q.YpX.v[w] & m);
                e.YmX.v[w] = (e.YmX.v[w] & ~m) | (q.YmX.v[w] & m);
                e.Z.v[w] = (e.Z.v[w] & ~m) | (q.Z.v[w] & m);
                e.T2d.v[w] = (e.T2d.v[w] & ~m) | (q.T2d.v[w] & m);
            }
        }
        fe nt;
        fe_neg(nt, e.T2d);
        for (int w = 0; w < 8; w++) {
            const uint32_t p = e.YpX.v[w], q = e.YmX.v[w];
            e.YpX.v[w] = (p & ~sign) | (q & sign);
            e.YmX.v[w] = (q & ~sign) | (p & sign);
            e.T2d.v[w] = (e.T2d.v[w] & ~sign) | (nt.v[w] & sign);
        }
        ge_add_cached_p1p1(t, acc, e, false);
        ge_p1p1_to_ext(acc, t);
    }
    out = acc;
}

// fixed-base-only form (the provers' [x] G, [x] K + [y] G); ct selects the constant-time table walk for secret scalars
static EG_HD_NOINLINE void ge_eval_fixed(ge_ext &out, int nf, const uint32_t *ftab0, const sc &b0, const uint32_t *ftab1, const sc &b1,
                                         bool ct = false) {
    ge_ext acc = ge_identity();
    ge_p1p1 t;
    if (ct) ge_fixed_adds_ct(acc, t, nf, ftab0, b0, ftab1, b1);
    else ge_fixed_adds(acc, t, nf, ftab0, b0, ftab1, b1);
    out = acc;
}

// x / 2 mod l
EG_HD void sc_half(sc &r, const sc &x) {
    uint32_t t[8];
    uint64_t c = 0;
    const uint32_t odd = (uint32_t)0 - (x.v[0] & 1u);       // mask: x may be secret (prover nonces), no branch on it
    for (int i = 0; i < 8; i++) { c += (uint64_t)x.v[i] + (sc_L(i) & odd); t[i] = (uint32_t)c; c >>= 32; }
    for (int i = 0; i < 7; i++) r.v[i] = (t[i] >> 1) | (t[i + 1] << 31);
    r.v[7] = t[7] >> 1;          // x + l < 2^254: no carry out of limb 7
}

// ------------------------------------------------------------------ double-and-compress
//
// encode(2Q) for several Q with ONE field inversion and no square root (the doubling makes the quantity under the
// RFC 9496 square root a known square).  A verifier that needs encode(C), C = sum [x_i] P_i, evaluates
// Q = sum [x_i / 2 mod l] P_i instead: 2Q = C + (a 4-torsion point), and all representatives of a ristretto255
// element encode identically.  Same bytes as serialize_element (ristretto.rs:88-90) on C.

struct ge_dc_state { fe e, f, g, h, eg, fh; };

EG_HD void ge_dc_prepare(ge_dc_state &s, fe &efgh, const ge_ext &P) {
    fe xx, yy, zz, dtt, t;
    fe_sq(xx, P.X); fe_sq(yy, P.Y); fe_sq(zz, P.Z);
    fe_sq(t, P.T); fe_mul(dtt, t, fe_const_d());
    fe_add(t, P.Y, P.Y); fe_mul(s.e, P.X, t);       // 2XY
    fe_add(s.f, zz, dtt);
    fe_add(s.g, yy, xx);
    fe_sub(s.h, zz, dtt);
    fe_mul(s.eg, s.e, s.g);
    fe_mul(s.fh, s.f, s.h);
    fe_mul(efgh, s.eg, s.fh);
}

// inv = 1 / (eg * fh), or 0 when that product is 0 (2Q in the identity coset: the encoding is all zeros)
EG_HD void ge_dc_finish(uint32_t w[8], const ge_dc_state &s, const fe &inv) {
    fe zinv, tinv, t, e, g, h, magic, s_out;
    fe_mul(zinv, s.eg, inv);
    fe_mul(tinv, s.fh, inv);
    fe_mul(t, s.eg, zinv);
    const bool rot = fe_isneg(t);
    fe ne, fi;
    fe_neg(ne, s.e);
    fe_mul(fi, s.f, fe_const_sqrtm1());
    fe_select(e, s.e, s.g, rot);
    fe_select(g, s.g, ne, rot);
    fe_select(h, s.h, fi, rot);
    fe_select(magic, fe_const_invsqrt_a_minus_d(), fe_const_sqrtm1(), rot);
    fe_mul(t, h, e); fe_mul(t, t, zinv);
    fe_cneg(g, g, fe_isneg(t));
    fe_mul(t, g, tinv); fe_mul(t, magic, t);
    fe hg;
    fe_sub(hg, h, g);
    fe_mul(s_out, hg, t);
    fe_abs(s_out, s_out);
    fe_towords(w, s_out);
}

// w0 = encode(2 Q0), w1 = encode(2 Q1)
static EG_HD_NOINLINE void ge_double_compress2(uint32_t w0[8], uint32_t w1[8], const ge_ext &Q0, const ge_ext &Q1) {
    ge_dc_state s0, s1;
    fe t0, t1, u0, u1, p, ip, i0, i1;
    ge_dc_prepare(s0, t0, Q0);
    ge_dc_prepare(s1, t1, Q1);
    const bool z0 = fe_iszero(t0), z1 = fe_iszero(t1);
    fe_select(u0, t0, fe_one(), z0);
    fe_select(u1, t1, fe_one(), z1);
    fe_mul(p, u0, u1);
    fe_invert(ip, p);
    fe_mul(i0, ip, u1);
    fe_mul(i1, ip, u0);
    fe_select(i0, i0, fe_zero(), z0);
    fe_select(i1, i1, fe_zero(), z1);
    ge_dc_finish(w0, s0, i0);
    ge_dc_finish(w1, s1, i1);
}

// w[k] = encode(2 Q[k]), k < N, with one inversion: Montgomery's trick over ge_dc_prepare's products, as k_terminal.  The
// per-point states live in local arrays walked by rolled loops (N x 48 words would not stay in registers anyway).
template <int N>
static EG_HD_NOINLINE void ge_double_compress_n(uint32_t w[N][8], const ge_ext Q[N]) {
    ge_dc_state st[N];
    fe prefix[N], u[N];
    bool z[N];
    fe run = fe_one();
#pragma unroll 1
    for (int k = 0; k < N; k++) {
        fe t;
        ge_dc_prepare(st[k], t, Q[k]);
        z[k] = fe_iszero(t);
        fe_select(u[k], t, fe_one(), z[k]);
        fe_mul(run, run, u[k]);
        prefix[k] = run;
    }
    fe inv;
    fe_invert(inv, run);
#pragma unroll 1
    for (int k = N - 1; k >= 0; k--) {
        fe ik;
        if (k) { fe_mul(ik, inv, prefix[k - 1]); fe_mul(inv, inv, u[k]); } else ik = inv;
        fe_select(ik, ik, fe_zero(), z[k]);
        ge_dc_finish(w[k], st[k], ik);
    }
}

EG_HD void ge_double_compress1(uint32_t w[8], const ge_ext &Q) {
    ge_dc_state s;
    fe t, u, i;
    ge_dc_prepare(s, t, Q);
    const bool z = fe_iszero(t);
    fe_select(u, t, fe_one(), z);
    fe_invert(i, u);
    fe_select(i, i, fe_zero(), z);
    ge_dc_finish(w, s, i);
}

}  // namespace eg
