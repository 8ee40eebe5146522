// kernels.cuh -- batch kernels of the verification hot path (sm_100a).
//
// Data layout in HBM (DESIGN.md "Layout"): per-batch scratch is *planar* -- word w of object q of item i
// lives at base[(q * W + w) * n + i] -- so that a warp of 32 consecutive items reads/writes 128 contiguous
// bytes per word.  Inputs stay in the reference's own array-of-structures byte layouts (to_bytes forms).
//
// The kernel bodies are __host__ __device__ functions of (item, slot) so that tests/hostsim can run the very
// same logic on the CPU (test harness only; the product library launches only the __global__ wrappers).
#pragma once
#include "chacha.cuh"
#include "fe.cuh"
#include "ge.cuh"
#include "merlin.cuh"
#include "sc.cuh"

namespace eg {

#define EG_MAX_SLOTS 40
#define EG_MAX_RINGS 64

// ------------------------------------------------------------------ planar accessors

EG_HD void planar_store_words(uint32_t *base, size_t n, size_t q, int W, size_t i, const uint32_t *w) {
    for (int k = 0; k < W; k++) base[(q * W + k) * n + i] = w[k];
}
EG_HD void planar_load_words(uint32_t *w, const uint32_t *base, size_t n, size_t q, int W, size_t i) {
    for (int k = 0; k < W; k++) w[k] = base[(q * W + k) * n + i];
}
EG_HD void planar_store_point(uint32_t *base, size_t n, size_t q, size_t i, const ge_ext &p) {
    for (int k = 0; k < 8; k++) {
        base[(q * 32 + k) * n + i] = p.X.v[k];
        base[(q * 32 + 8 + k) * n + i] = p.Y.v[k];
        base[(q * 32 + 16 + k) * n + i] = p.Z.v[k];
        base[(q * 32 + 24 + k) * n + i] = p.T.v[k];
    }
}
EG_HD void planar_load_point(ge_ext &p, const uint32_t *base, size_t n, size_t q, size_t i) {
    for (int k = 0; k < 8; k++) {
        p.X.v[k] = base[(q * 32 + k) * n + i];
        p.Y.v[k] = base[(q * 32 + 8 + k) * n + i];
        p.Z.v[k] = base[(q * 32 + 16 + k) * n + i];
        p.T.v[k] = base[(q * 32 + 24 + k) * n + i];
    }
}

// 32 bytes at an arbitrary (4-byte aligned or not) address -> little-endian words
EG_HD void load32_bytes(uint32_t w[8], const uint8_t *p) {
    if ((((uintptr_t)p) & 3u) == 0) {
        const uint32_t *q = (const uint32_t *)p;
        for (int k = 0; k < 8; k++) w[k] = q[k];
    } else {
        for (int k = 0; k < 8; k++)
            w[k] = (uint32_t)p[4 * k] | ((uint32_t)p[4 * k + 1] << 8) | ((uint32_t)p[4 * k + 2] << 16) | ((uint32_t)p[4 * k + 3] << 24);
    }
}
EG_HD void store32_bytes(uint8_t *p, const uint32_t w[8]) {
    if ((((uintptr_t)p) & 3u) == 0) {
        uint32_t *q = (uint32_t *)p;
        for (int k = 0; k < 8; k++) q[k] = w[k];
    } else {
        for (int k = 0; k < 8; k++) { p[4 * k] = (uint8_t)w[k]; p[4 * k + 1] = (uint8_t)(w[k] >> 8); p[4 * k + 2] = (uint8_t)(w[k] >> 16); p[4 * k + 3] = (uint8_t)(w[k] >> 24); }
    }
}

// ------------------------------------------------------------------ decode / validate

// Input buffers of a batch call (array-of-structures, reference byte layouts)
struct in_bufs {
    const uint8_t *buf[4];
    uint32_t stride[4];         // bytes per outer item in buf[k]
    uint32_t group[4];          // items per outer item (0 or 1: flat).  Lets "item = (ballot, option)" address proofs that
    uint32_t inner[4];          // are embedded in a larger record: addr = buf + (item / group) * stride + (item % group) * inner
};

EG_HD const uint8_t *in_ptr(const in_bufs &in, int k, size_t item) {
    if (in.group[k] > 1) return in.buf[k] + (item / in.group[k]) * in.stride[k] + (item % in.group[k]) * in.inner[k];
    return in.buf[k] + item * in.stride[k];
}

struct decode_slot {
    uint8_t buf;                // which input buffer
    uint8_t want_enc;           // also store the 8 encoding words (for transcript "enc" messages)
    uint8_t reject_identity;    // the element is a PublicKey: the identity is malformed too (keys/mod.rs:161-176)
    uint16_t enc_index;         // planar index in enc (8 words each)
    uint32_t offset;            // byte offset inside the item
    uint32_t p_index;           // planar point index
    uint32_t flag_offset;       // malformed flag goes to flags[item * flag_stride + flag_offset]
};

struct decode_params {
    in_bufs in;
    size_t n;
    int n_slots;
    decode_slot slots[EG_MAX_SLOTS];
    uint32_t *pts;              // planar points
    uint32_t *enc;              // planar encodings
    uint32_t *flags;            // bit 0 = malformed
    uint32_t flag_stride;       // 0 is treated as 1
};

EG_HD void decode_body(const decode_params &P, size_t item, int slot) {
    const decode_slot &s = P.slots[slot];
    uint32_t w[8];
    load32_bytes(w, in_ptr(P.in, s.buf, item) + s.offset);
    ge_ext p;
    bool ok = ge_decode(p, w);
    if (s.reject_identity && ge_is_identity(p)) ok = false;
    planar_store_point(P.pts, P.n, s.p_index, item, p);
    if (s.want_enc) planar_store_words(P.enc, P.n, s.enc_index, 8, item, w);
    if (!ok) {
        size_t fi = item * (P.flag_stride ? P.flag_stride : 1) + s.flag_offset;
#if defined(__CUDA_ARCH__)
        atomicOr(&P.flags[fi], 1u);
#else
        P.flags[fi] |= 1u;
#endif
    }
}

struct scalar_slot { uint8_t buf; uint32_t offset; uint32_t count; uint32_t flag_offset; };   // `count` consecutive scalars

struct scalars_params {
    in_bufs in;
    size_t n;
    int n_slots;
    scalar_slot slots[8];
    uint32_t *flags;
    uint32_t flag_stride;
};

EG_HD void scalars_body(const scalars_params &P, size_t item) {
    for (int s = 0; s < P.n_slots; s++) {
        bool ok = true;
        const uint8_t *base = in_ptr(P.in, P.slots[s].buf, item) + P.slots[s].offset;
        for (uint32_t k = 0; k < P.slots[s].count; k++) {
            uint32_t w[8];
            load32_bytes(w, base + 32 * k);
            ok = ok && sc_is_canonical_words(w);
        }
        if (!ok) {
            size_t fi = item * (P.flag_stride ? P.flag_stride : 1) + P.slots[s].flag_offset;
#if defined(__CUDA_ARCH__)
            atomicOr(&P.flags[fi], 1u);
#else
            P.flags[fi] |= 1u;
#endif
        }
    }
}

// ------------------------------------------------------------------ commitments (the hot kernel)

// One slot = one verification equation side:  C = [-e] (P - X) + [s] F
//   reference: ring.rs:342-350, log_equality.rs:160-164 (vartime_double_mul_generator / vartime_multi_mul)
struct commit_slot {
    uint32_t p_index;           // planar index of P
    int32_t adm_index;          // admissible value X (cached form) to subtract, -1 for none (x = identity)
    uint8_t base;               // 0: G, 1: K
    uint8_t e_planar;           // challenge from the planar `chal` buffer (1) or from an input buffer (0)
    uint8_t e_buf, s_buf;       // input buffers of the challenge / response scalars
    uint32_t e_offset;          // byte offset in item (e_planar = 0) or planar scalar index (e_planar = 1)
    uint32_t s_offset;          // byte offset of the response scalar in its item
    uint32_t out_index;         // planar index of the 8-word commitment encoding
};

struct commit_params {
    in_bufs in;
    size_t n;
    int n_slots;
    commit_slot slots[EG_MAX_SLOTS];
    const uint32_t *pts;
    const uint32_t *chal;       // planar scalars (8 words)
    uint32_t *commit;           // planar encodings (8 words)
    const uint32_t *adm;        // admissible values: cached points, 32 words each (YpX, YmX, Z, T2d)
    const uint32_t *table_g;    // wide fixed-base tables (ge.cuh)
    const uint32_t *table_k;
    uint32_t *term_pts;         // when set: slot k stores the half-scalar point Q (2Q = C) at planar index term_base + k
    uint32_t term_base;         //   of this buffer instead of encoding C; k_terminal encodes all of an item's points at once
};

EG_HD void commit_body(const commit_params &P, size_t item, int slot, const uint32_t *tab_g, const uint32_t *tab_k) {
    const commit_slot &s = P.slots[slot];
    ge_ext pt;
    planar_load_point(pt, P.pts, P.n, s.p_index, item);
    if (s.adm_index >= 0) {
        ge_cached x;
        const uint32_t *a = P.adm + (size_t)s.adm_index * 32;
        for (int k = 0; k < 8; k++) { x.YpX.v[k] = a[k]; x.YmX.v[k] = a[8 + k]; x.Z.v[k] = a[16 + k]; x.T2d.v[k] = a[24 + k]; }
        ge_p1p1 t;
        ge_add_cached_p1p1(t, pt, x, true);
        ge_p1p1_to_ext(pt, t);
    }
    uint32_t w[8];
    sc e, r, ne;
    if (s.e_planar) planar_load_words(w, P.chal, P.n, s.e_offset, 8, item);
    else load32_bytes(w, in_ptr(P.in, s.e_buf, item) + s.e_offset);
    bool ok = sc_from_words(e, w);
    load32_bytes(w, in_ptr(P.in, s.s_buf, item) + s.s_offset);
    ok = sc_from_words(r, w) && ok;
    if (!ok) { e = sc_zero(); r = sc_zero(); }      // malformed items are already flagged; keep the math defined
    sc_neg(ne, e);
    ge_ext acc;
    const uint32_t *ft[1] = {s.base ? tab_k : tab_g};
    if (P.term_pts) {
        sc hne, hr;
        sc_half(hne, ne);
        sc_half(hr, r);
        ge_msm_chain<1, 1>(acc, &pt, &hne, ft, &hr);
        planar_store_point(P.term_pts, P.n, P.term_base + slot, item, acc);
        return;
    }
    ge_msm_chain<1, 1>(acc, &pt, &ne, ft, &r);
    ge_encode(w, acc);
    planar_store_words(P.commit, P.n, s.out_index, 8, item, w);
}


EG_HD void point_to_words32(uint32_t *o, const ge_ext &p) {
    for (int k = 0; k < 8; k++) { o[k] = p.X.v[k]; o[8 + k] = p.Y.v[k]; o[16 + k] = p.Z.v[k]; o[24 + k] = p.T.v[k]; }
}
EG_HD void point_from_words32(ge_ext &p, const uint32_t *o) {
    for (int k = 0; k < 8; k++) { p.X.v[k] = o[k]; p.Y.v[k] = o[8 + k]; p.Z.v[k] = o[16 + k]; p.T.v[k] = o[24 + k]; }
}

// ------------------------------------------------------------------ general multi-scalar equations

#define EG_MSM_MAXV 16

// where a scalar comes from
struct scalar_src {
    uint8_t kind;               // 0: input buffer (AoS bytes), 1: planar `chal` buffer, 2: constant table
    uint8_t buf;                // input buffer (kind 0)
    uint8_t negate;             // use l - x
    uint8_t pad;
    uint32_t offset;            // byte offset in the item (kind 0), planar index (kind 1), table index (kind 2)
};

struct msm_slot {
    uint8_t nv, nf;             // per-item / constant bases ; fixed bases (G / K tables)
    uint8_t out_enc;            // 1: store the 8-word encoding at commit[out_index]; 2: deferred to k_terminal (see `term`)
    uint8_t out_point;          // store the extended point at pts[out_index]
    uint32_t out_index;
    uint32_t p_index[EG_MSM_MAXV];   // planar point index, or index into const_pts when bit 31 is set
    scalar_src vs[EG_MSM_MAXV];
    uint8_t fbase[2];           // 0: G, 1: K, 2: H (Pedersen blinding base, eg_ctx_set_blinding_base), 3 + j: per-call narrow table j
    uint8_t term;               // out_enc == 2: index of the half-scalar point in msm_params::term_pts (encoded by k_terminal)
    uint8_t pad2;
    scalar_src fs[2];
};

struct msm_params {
    in_bufs in;
    size_t n;
    int n_slots;
    const msm_slot *slots;      // device memory
    const uint32_t *pts;        // planar per-item points
    const uint32_t *const_pts;  // batch-constant points, 32 words each (X, Y, Z, T)
    const uint32_t *chal;       // planar scalars
    const uint32_t *const_scalars;   // batch-constant scalars, 8 words each
    uint32_t *commit;           // planar encodings out
    uint32_t *pts_out;          // planar points out
    const uint32_t *table_g, *table_k;
    const uint32_t *table_h;    // may be null when no slot uses base 2
    const uint32_t *table_x;    // per-call narrow tables (EG_NARROW_ALLOC_WORDS apart), null when no slot uses a base >= 3
    uint32_t *term_pts;         // planar points of the deferred encodings (slots with out_enc == 2)
};

EG_HD bool load_scalar(sc &out, const msm_params &P, const scalar_src &src, size_t item) {
    uint32_t w[8];
    if (src.kind == 0) load32_bytes(w, in_ptr(P.in, src.buf, item) + src.offset);
    else if (src.kind == 1) planar_load_words(w, P.chal, P.n, src.offset, 8, item);
    else for (int k = 0; k < 8; k++) w[k] = P.const_scalars[(size_t)src.offset * 8 + k];
    sc x;
    bool ok = sc_from_words(x, w);
    if (!ok) x = sc_zero();
    if (src.negate) sc_neg(out, x); else out = x;
    return ok;
}

EG_HD void msm_body(const msm_params &P, size_t item, int slot, const uint32_t *tab_g, const uint32_t *tab_k, const uint32_t *tab_h) {
    const msm_slot &s = P.slots[slot];
    ge_ext pts[EG_MSM_MAXV];
    sc a[EG_MSM_MAXV], b[2];
    const uint32_t *ft[2];
    bool narrow[2] = {false, false};
#pragma unroll 1
    for (int v = 0; v < s.nv; v++) {
        if (s.p_index[v] & 0x80000000u) point_from_words32(pts[v], P.const_pts + (size_t)(s.p_index[v] & 0x7fffffffu) * 32);
        else planar_load_point(pts[v], P.pts, P.n, s.p_index[v], item);
        load_scalar(a[v], P, s.vs[v], item);
    }
    for (int f = 0; f < s.nf; f++) {
        ft[f] = s.fbase[f] == 0 ? tab_g : (s.fbase[f] == 1 ? tab_k : tab_h);
        if (s.fbase[f] >= 3) { ft[f] = P.table_x + (size_t)(s.fbase[f] - 3) * EG_NARROW_ALLOC_WORDS; narrow[f] = true; }
        load_scalar(b[f], P, s.fs[f], item);
    }
    ge_ext acc;
    if (s.out_enc == 2) {       // all scalars halved: acc = Q with 2 Q = the commitment, encoded later with its siblings
        for (int v = 0; v < s.nv; v++) { sc h; sc_half(h, a[v]); a[v] = h; }
        for (int f = 0; f < s.nf; f++) { sc h; sc_half(h, b[f]); b[f] = h; }
        ge_msm_chain_rt<EG_MSM_MAXV>(acc, s.nv, pts, a, s.nf, ft, b, narrow);
        planar_store_point(P.term_pts, P.n, s.term, item, acc);
        return;
    }
    ge_msm_chain_rt<EG_MSM_MAXV>(acc, s.nv, pts, a, s.nf, ft, b, narrow);
    if (s.out_point) planar_store_point(P.pts_out, P.n, s.out_index, item, acc);
    if (s.out_enc) {
        uint32_t w[8];
        ge_encode(w, acc);
        planar_store_words(P.commit, P.n, s.out_index, 8, item, w);
    }
}

// ------------------------------------------------------------------ ring transcripts

// One slot = one ring in one hash stage: e_{j+1} = H(ring transcript, j, R_G(j), R_K(j))   (ring.rs:325-360)
struct ring_hash_slot {
    uint32_t ring_index;        // value appended as "i"
    uint32_t eq_index;          // value appended as "j"
    uint32_t enc_index;         // planar index of enc(R); enc(B) is enc_index + 1
    uint32_t commit_index;      // planar index of R_G; R_K is commit_index + 1
    uint32_t chal_index;        // planar index of the output challenge
};

struct ring_hash_params {
    size_t n;
    int n_slots;
    ring_hash_slot slots[EG_MAX_SLOTS];
    transcript prefix;          // state after RingProof::initialize_transcript (ring.rs:290-293)
    const uint32_t *enc;
    const uint32_t *commit;
    uint32_t *chal;
};

EG_HD void ring_hash_body(const ring_hash_params &P, size_t item, int slot) {
    const ring_hash_slot &s = P.slots[slot];
    transcript t = P.prefix;
    uint32_t w[16];
    merlin_append_message(t, EG_LBL("dom-sep"), (const uint8_t *)"ring_enc", 8);
    planar_load_words(w, P.enc, P.n, s.enc_index, 8, item);
    planar_load_words(w + 8, P.enc, P.n, s.enc_index + 1, 8, item);
    merlin_append_words(t, EG_LBL("enc"), w, 16);
    merlin_append_u64(t, EG_LBL("i"), s.ring_index);
    merlin_append_u64(t, EG_LBL("j"), s.eq_index);
    planar_load_words(w, P.commit, P.n, s.commit_index, 8, item);
    merlin_append_words(t, EG_LBL("R_G"), w, 8);
    planar_load_words(w, P.commit, P.n, s.commit_index + 1, 8, item);
    merlin_append_words(t, EG_LBL("R_K"), w, 8);
    sc c;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    planar_store_words(P.chal, P.n, s.chal_index, 8, item, c.v);
}

// ---- v2 ring engine: one thread = one ring of one item, all of its equations (ring.rs:322-366) --------------------
//
// R_G(j) = [s_j] G - [e_j] R ; R_K(j) = [s_j] K - [e_j] (B - [a_j] G) = [s_j] K - [e_j] B + [e_j a_j] G with a_j = j * step
// the admissible value of equation j (PreparedRange::new range.rs:341-355; [O, G] for bool / choice rings).  The window
// tables of R and B are built once per ring (ge_vtab_build) in a per-thread scratch region and serve every j; the two
// commitments of an equation are encoded together with one inversion (ge_double_compress2 on the half-scalar points).
struct ring_params {
    in_bufs in;
    size_t n;
    uint32_t n_rings;
    uint16_t sizes[EG_MAX_RINGS];           // equations per ring
    uint16_t starts[EG_MAX_RINGS];          // index of the ring's first response in the proof
    uint32_t ct_p_index[EG_MAX_RINGS];      // planar point index of R; B at +1
    uint32_t ct_enc_index[EG_MAX_RINGS];    // planar encoding index of R; B at +1
    uint64_t adm_step[EG_MAX_RINGS];
    uint8_t proof_buf;
    uint32_t proof_offset;                  // e0 | responses
    uint32_t commit_index0;                 // terminal commitments of ring r -> commit_index0 + 2r, +1
    transcript prefix;                      // after initialize_transcript (ring.rs:290-293)
    const uint32_t *pts;
    const uint32_t *enc;
    uint32_t *commit;
    uint32_t *scratch;                      // 2 * EG_VTAB_WORDS words per resident thread
    const uint32_t *table_g, *table_k;      // wide fixed-base tables
    uint32_t *term_pts;                     // when set: the half-scalar points of ring r's LAST equation go to planar
                                            // indexes 2r, 2r + 1 of this buffer and are encoded by k_terminal
};

// the ring's own transcript: prefix + start_proof("ring_enc") + "enc" + "i"   (ring.rs:325-331)
static EG_HD_NOINLINE void ring_transcript_start(transcript &rt, const transcript &prefix, const uint32_t enc_ct[16], uint32_t r) {
    rt = prefix;
    merlin_append_message(rt, EG_LBL("dom-sep"), (const uint8_t *)"ring_enc", 8);
    merlin_append_words(rt, EG_LBL("enc"), enc_ct, 16);
    merlin_append_u64(rt, EG_LBL("i"), r);
}

// e_{j+1} = H(ring transcript, j, R_G, R_K)   (ring.rs:354-360)
static EG_HD_NOINLINE void ring_next_challenge(sc &e, const transcript &rt, uint32_t j, const uint32_t cg[8], const uint32_t ck[8]) {
    transcript t = rt;
    merlin_append_u64(t, EG_LBL("j"), j);
    merlin_append_words(t, EG_LBL("R_G"), cg, 8);
    merlin_append_words(t, EG_LBL("R_K"), ck, 8);
    merlin_challenge_scalar(t, EG_LBL("c"), e);
}

template <int C>
EG_HD void ring_body(const ring_params &P, size_t item, uint32_t r, uint32_t *scratch, const uint32_t *tab_g, const uint32_t *tab_k) {
    uint32_t *tab_r = scratch, *tab_b = scratch + EG_VTAB_WORDS;
    {
        ge_ext pt;
        planar_load_point(pt, P.pts, P.n, P.ct_p_index[r], item);
        ge_vtab_build<C>(tab_r, pt);
        planar_load_point(pt, P.pts, P.n, P.ct_p_index[r] + 1, item);
        ge_vtab_build<C>(tab_b, pt);
    }
    const uint8_t *proof = in_ptr(P.in, P.proof_buf, item) + P.proof_offset;
    uint32_t w[16];
    sc e;
    load32_bytes(w, proof);
    bool ok = sc_from_words(e, w);
    if (!ok) e = sc_zero();                 // malformed items are flagged by k_scalars; keep the math defined
    planar_load_words(w, P.enc, P.n, P.ct_enc_index[r], 8, item);
    planar_load_words(w + 8, P.enc, P.n, P.ct_enc_index[r] + 1, 8, item);
    const uint32_t *enc_ct = w;
    const uint32_t size = P.sizes[r];
    transcript rt;                          // cloned per equation
    ring_transcript_start(rt, P.prefix, enc_ct, r);
    uint32_t cg[8], ck[8];
#pragma unroll 1
    for (uint32_t j = 0; j < size; j++) {
        sc s, ne, hs, hne, hea;
        load32_bytes(w, proof + 32 * (1 + P.starts[r] + j));
        if (!sc_from_words(s, w)) s = sc_zero();
        sc_neg(ne, e);
        sc_half(hs, s);
        sc_half(hne, ne);
        ge_ext qg, qk;
        ge_eval64<C>(qg, tab_r, hne, 1, tab_g, hs, tab_g, hs);
        const uint64_t a = P.adm_step[r] * (uint64_t)j;
        if (a != 0) {
            sc ea;
            sc_mul(ea, e, sc_from_u64(a));
            sc_half(hea, ea);
            ge_eval64<C>(qk, tab_b, hne, 2, tab_k, hs, tab_g, hea);
        } else {
            ge_eval64<C>(qk, tab_b, hne, 1, tab_k, hs, tab_k, hs);
        }
        if (j + 1 == size && P.term_pts) {
            planar_store_point(P.term_pts, P.n, 2 * r, item, qg);
            planar_store_point(P.term_pts, P.n, 2 * r + 1, item, qk);
            return;
        }
        ge_double_compress2(cg, ck, qg, qk);
        if (j + 1 < size) ring_next_challenge(e, rt, j, cg, ck);
    }
    planar_store_words(P.commit, P.n, P.commit_index0 + 2 * r, 8, item, cg);
    planar_store_words(P.commit, P.n, P.commit_index0 + 2 * r + 1, 8, item, ck);
}

// ---- pair engine: two adjacent lanes = one ring (small chunks) ------------------------------------------------------
//
// A chunk with fewer ring threads than the GPU has warp slots is latency-bound: what counts is the length of the longest
// per-thread chain, not the amount of work.  k_ring runs both sides of every equation in one thread (2 x 192 table
// doublings + 4 x 60), the per-equation pipeline pays 252 doublings per equation index.  Here lane 2p evaluates the G side
// (tables of R only), lane 2p + 1 the K side (tables of B): 192 + 60 per equation doublings on the critical path, each lane
// encodes its own commitment (one inversion) and the pair swaps the encodings by shuffle before both clone the
// transcript for the next challenge (ring.rs:342-360).  Same group elements, same bytes.

// Q = half-scalar point of side `side` of equation j: side 0: [s/2] G - [e/2] R, side 1: [s/2] K - [e/2] B + [e a_j / 2] G
template <int C>
EG_HD void ring_side_eval(ge_ext &q, const ring_params &P, uint32_t r, uint32_t j, int side, const uint32_t *tab, const sc &e,
                          const sc &s, const uint32_t *tab_g, const uint32_t *tab_k) {
    sc ne, hs, hne, hea;
    sc_neg(ne, e);
    sc_half(hs, s);
    sc_half(hne, ne);
    hea = hs;
    int nf = 1;
    const uint64_t a = side ? P.adm_step[r] * (uint64_t)j : 0;
    if (a != 0) {
        sc ea;
        sc_mul(ea, e, sc_from_u64(a));
        sc_half(hea, ea);
        nf = 2;
    }
    ge_eval64<C>(q, tab, hne, nf, side ? tab_k : tab_g, hs, tab_g, hea);
}

static EG_HD_NOINLINE void ge_double_compress1_call(uint32_t w[8], const ge_ext &Q) { ge_double_compress1(w, Q); }

#if defined(__CUDACC__) && !defined(EG_HOSTSIM)
// `tab`: EG_VTAB_WORDS words of scratch for this lane.  Both lanes of a pair share (item, r) and therefore every branch
// below; the shuffles name only the two lanes of the pair, so pairs of one warp may sit in different equations.
template <int C>
__device__ void ring_pair_body(const ring_params &P, size_t item, uint32_t r, int side, uint32_t *tab, const uint32_t *tab_g,
                               const uint32_t *tab_k) {
    {
        ge_ext pt;
        planar_load_point(pt, P.pts, P.n, P.ct_p_index[r] + (uint32_t)side, item);
        ge_vtab_build<C>(tab, pt);
    }
    const unsigned pair_mask = 3u << (threadIdx.x & 30u);
    const uint8_t *proof = in_ptr(P.in, P.proof_buf, item) + P.proof_offset;
    uint32_t w[16];
    sc e;
    load32_bytes(w, proof);
    if (!sc_from_words(e, w)) e = sc_zero();
    planar_load_words(w, P.enc, P.n, P.ct_enc_index[r], 8, item);
    planar_load_words(w + 8, P.enc, P.n, P.ct_enc_index[r] + 1, 8, item);
    const uint32_t size = P.sizes[r];
    transcript rt;
    ring_transcript_start(rt, P.prefix, w, r);
    uint32_t mine[8], other[8];
#pragma unroll 1
    for (uint32_t j = 0; j < size; j++) {
        sc s;
        load32_bytes(w, proof + 32 * (1 + P.starts[r] + j));
        if (!sc_from_words(s, w)) s = sc_zero();
        ge_ext q;
        ring_side_eval<C>(q, P, r, j, side, tab, e, s, tab_g, tab_k);
        if (j + 1 == size && P.term_pts) {
            planar_store_point(P.term_pts, P.n, 2 * r + (uint32_t)side, item, q);
            return;
        }
        ge_double_compress1_call(mine, q);
        if (j + 1 < size) {
            for (int k = 0; k < 8; k++) other[k] = __shfl_xor_sync(pair_mask, mine[k], 1);
            ring_next_challenge(e, rt, j, side ? other : mine, side ? mine : other);
        }
    }
    planar_store_words(P.commit, P.n, P.commit_index0 + 2 * r + (uint32_t)side, 8, item, mine);
}
#endif

// the same engine for the host harness: the two lanes of a pair one after the other (scratch: 2 * EG_VTAB_WORDS words)
template <int C>
EG_HD void ring_pair_host(const ring_params &P, size_t item, uint32_t r, uint32_t *scratch, const uint32_t *tab_g, const uint32_t *tab_k) {
    uint32_t *tab[2] = {scratch, scratch + EG_VTAB_WORDS};
    for (int side = 0; side < 2; side++) {
        ge_ext pt;
        planar_load_point(pt, P.pts, P.n, P.ct_p_index[r] + (uint32_t)side, item);
        ge_vtab_build<C>(tab[side], pt);
    }
    const uint8_t *proof = in_ptr(P.in, P.proof_buf, item) + P.proof_offset;
    uint32_t w[16];
    sc e;
    load32_bytes(w, proof);
    if (!sc_from_words(e, w)) e = sc_zero();
    planar_load_words(w, P.enc, P.n, P.ct_enc_index[r], 8, item);
    planar_load_words(w + 8, P.enc, P.n, P.ct_enc_index[r] + 1, 8, item);
    const uint32_t size = P.sizes[r];
    transcript rt;
    ring_transcript_start(rt, P.prefix, w, r);
    uint32_t c[2][8];
    for (uint32_t j = 0; j < size; j++) {
        sc s;
        load32_bytes(w, proof + 32 * (1 + P.starts[r] + j));
        if (!sc_from_words(s, w)) s = sc_zero();
        for (int side = 0; side < 2; side++) {
            ge_ext q;
            ring_side_eval<C>(q, P, r, j, side, tab[side], e, s, tab_g, tab_k);
            if (j + 1 == size && P.term_pts) planar_store_point(P.term_pts, P.n, 2 * r + (uint32_t)side, item, q);
            else ge_double_compress1_call(c[side], q);
        }
        if (j + 1 == size && P.term_pts) return;
        if (j + 1 < size) ring_next_challenge(e, rt, j, c[0], c[1]);
    }
    planar_store_words(P.commit, P.n, P.commit_index0 + 2 * r, 8, item, c[0]);
    planar_store_words(P.commit, P.n, P.commit_index0 + 2 * r + 1, 8, item, c[1]);
}

// ---- terminal commitments: encode(2 Q_k) for all deferred points of an item with ONE field inversion ---------------
//
// The commitments of a ring's last equation (and of an EncryptedChoice's sum proof) are only read by the outer
// transcripts, so their encodings are not needed inside the sequential chains: k_ring / k_commit store the half-scalar
// points and one thread per item encodes all of them here (Montgomery's trick over ge_dc_prepare's products): a 5-option
// ballot pays 12 x ~30 + 265 field operations instead of 5 x 304 + 2 x 280.
#define EG_TERM_MAX (2 * EG_MAX_RINGS + 2)

struct terminal_params {
    size_t n;
    uint32_t n_pts;
    uint16_t out_index[EG_TERM_MAX];        // planar index in `commit` of the encoding of point k
    const uint32_t *term_pts;
    uint32_t *commit;
};

EG_HD void terminal_body(const terminal_params &P, size_t item) {
    fe prefix[EG_TERM_MAX];
    fe run = fe_one();
#pragma unroll 1
    for (uint32_t k = 0; k < P.n_pts; k++) {
        ge_ext q;
        ge_dc_state st;
        fe t, u;
        planar_load_point(q, P.term_pts, P.n, k, item);
        ge_dc_prepare(st, t, q);
        fe_select(u, t, fe_one(), fe_iszero(t));
        if (k) fe_mul(run, run, u); else run = u;
        prefix[k] = run;
    }
    fe inv;
    fe_invert(inv, run);
#pragma unroll 1
    for (int k = (int)P.n_pts - 1; k >= 0; k--) {
        ge_ext q;
        ge_dc_state st;
        fe t, u, ik;
        planar_load_point(q, P.term_pts, P.n, (uint32_t)k, item);
        ge_dc_prepare(st, t, q);
        const bool z = fe_iszero(t);
        fe_select(u, t, fe_one(), z);
        if (k) { fe_mul(ik, inv, prefix[k - 1]); fe_mul(inv, inv, u); } else ik = inv;
        fe_select(ik, ik, fe_zero(), z);
        uint32_t w[8];
        ge_dc_finish(w, st, ik);
        planar_store_words(P.commit, P.n, P.out_index[k], 8, item, w);
    }
}

// ------------------------------------------------------------------ proving side: encrypt_bool / EncryptedChoice::new
//
// PublicKey::encrypt_bool (keys/impls.rs:77-89) and EncryptedChoice::new / ::single (choice.rs:288-349) for rings over
// the admissible pair [O, G].  Randomness is caller-supplied: item i consumes `draws` 64-byte blocks in the reference's
// draw order (SURVEY.md A.4), each reduced as in Ristretto::generate_scalar (ristretto.rs:28-32).  Ring k draws r_k, x_k
// and -- when its value is 0 -- the forged response s_1 while the rings are added (ring.rs:97-116); after the common
// challenge, rings whose value is 1 draw the forged s_0 in ring order (ring.rs:170-175); the sum proof nonce comes last.
// All fixed-base work goes through the wide tables (ge_eval_fixed); every encoding is produced by double-and-compress on the
// half-scalar point.
struct prove_params {
    size_t n;
    uint32_t options;
    uint32_t draws;              // 3 * options + single
    uint8_t single;
    const uint8_t *values;       // n * options, zero / non-zero
    const uint8_t *wide;         // n * draws * 64
    uint8_t *cts;                // n * options * 64
    uint8_t *ring;               // n * (1 + 2 * options) * 32 : e0 | responses
    uint8_t *sum;                // n * 64 : c | s
    transcript ring_prefix;      // Transcript::new(label) + initialize_transcript (ring.rs:290-293)
    transcript sum_prefix;       // Transcript::new("choice_encryption_sum") + start_proof("log_eq") + "K"
    uint32_t *pts;               // planar points: R_k at 2k, B_k at 2k+1
    uint32_t *enc;               // planar encodings of the same
    uint32_t *sec;               // planar scalars: r_k at 2k, x_k at 2k+1
    uint32_t *commit;            // planar encodings: terminal commitments of ring k at 2k, 2k+1
    uint32_t *chal;              // planar scalars: common challenge at 0
    const uint32_t *table_g, *table_k;
    rand_src rnd;                // caller-supplied blocks (`wide`) or in-kernel ChaCha20 (chacha.cuh); constant-time flag
};

EG_HD void prove_draw(sc &out, const prove_params &P, size_t item, uint32_t pos) {
    uint32_t w[16];
    if (P.rnd.seeded) {
        chacha20_block(w, P.rnd.key, rand_counter(P.rnd, item, pos));
    } else {
        const uint8_t *b = P.wide + (item * P.draws + pos) * 64;
        load32_bytes(w, b);
        load32_bytes(w + 8, b + 32);
    }
    sc_from_wide_words(out, w);
}

// out0 = encode([k] G), out1 = encode([k] K)
EG_HD void prove_commit_pair(uint32_t out0[8], uint32_t out1[8], const sc &k, const uint32_t *tab_g, const uint32_t *tab_k, bool ct) {
    sc h;
    sc_half(h, k);
    ge_ext q0, q1;
    ge_eval_fixed(q0, 1, tab_g, h, tab_g, h, ct);
    ge_eval_fixed(q1, 1, tab_k, h, tab_k, h, ct);
    ge_double_compress2(out0, out1, q0, q1);
}

// Forged equation with admissible value [a]G of a ring over the ciphertext (R, B) = ([r]G, [v]G + [r]K), challenge e and
// response s (ring.rs:104-116, 176-186): ([s]G - [e]R, [s]K - [e](B - [a]G)).  The prover knows r and v, so both
// commitments are fixed-base: [s - e r]G and [s - e r]K + [e (a - v)]G -- the same group elements, hence the same
// encodings, as the reference's vartime_double_mul_generator / vartime_multi_mul on R and B.
EG_HD void prove_forge_fixed(uint32_t cg[8], uint32_t ck[8], const sc &r, uint64_t v, const sc &e, const sc &s, uint64_t a,
                             const uint32_t *tab_g, const uint32_t *tab_k, bool ct) {
    sc er, t, d, u, ht, hu;
    sc_mul(er, e, r);
    sc_sub(t, s, er);
    if (a >= v) d = sc_from_u64(a - v);
    else { sc m = sc_from_u64(v - a); sc_neg(d, m); }
    sc_mul(u, e, d);
    sc_half(ht, t);
    sc_half(hu, u);
    ge_ext qg, qk;
    ge_eval_fixed(qg, 1, tab_g, ht, tab_g, ht, ct);
    ge_eval_fixed(qk, 2, tab_k, ht, tab_g, hu, ct);
    ge_double_compress2(cg, ck, qg, qk);
}

// phase 1, one thread per (item, ring k): ciphertext, nonce commitments, forged equation 1 when the value is 0
EG_HD void prove_ring1_body(const prove_params &P, size_t item, uint32_t k, uint32_t *scratch, const uint32_t *tab_g, const uint32_t *tab_k) {
    const uint8_t *vals = P.values + item * P.options;
    uint32_t pos = 0;
    for (uint32_t i = 0; i < k; i++) pos += 2 + (vals[i] ? 0 : 1);
    const bool v = vals[k] != 0;
    sc r, x, hr;
    prove_draw(r, P, item, pos);
    prove_draw(x, P, item, pos + 1);
    sc_half(hr, r);
    // ExtendedCiphertext::new (encryption.rs:310-327): R = [r]G, B = [v]G + [r]K
    ge_ext qr, qb;
    sc hone;
    sc_half(hone, sc_from_u64(1));
    const bool ct = P.rnd.ct != 0;
    if (ct && !v) hone = sc_zero();          // constant-time mode: always two terms, [0]G for a zero vote
    ge_eval_fixed(qr, 1, tab_g, hr, tab_g, hr, ct);
    ge_eval_fixed(qb, (v || ct) ? 2 : 1, tab_k, hr, tab_g, hone, ct);
    uint32_t enc_ct[16];
    ge_double_compress2(enc_ct, enc_ct + 8, qr, qb);
    uint8_t *ct_out = P.cts + (item * P.options + k) * 64;
    store32_bytes(ct_out, enc_ct);
    store32_bytes(ct_out + 32, enc_ct + 8);
    planar_store_words(P.enc, P.n, 2 * k, 8, item, enc_ct);
    planar_store_words(P.enc, P.n, 2 * k + 1, 8, item, enc_ct + 8);
    planar_store_words(P.sec, P.n, 2 * k, 8, item, r.v);
    planar_store_words(P.sec, P.n, 2 * k + 1, 8, item, x.v);
    // Ring::new (ring.rs:54-131): commitments of the real equation, then the forged ones above it
    uint32_t cg[8], ck[8];
    prove_commit_pair(cg, ck, x, tab_g, tab_k, ct);
    if (!v) {
        transcript rt;
        ring_transcript_start(rt, P.ring_prefix, enc_ct, k);
        sc e1, s1;
        ring_next_challenge(e1, rt, 0, cg, ck);
        prove_draw(s1, P, item, pos + 2);
        store32_bytes(P.ring + (item * (1 + 2 * (size_t)P.options) + 1 + 2 * k + 1) * 32, s1.v);
        prove_forge_fixed(cg, ck, r, 0, e1, s1, 1, tab_g, tab_k, ct);
    }
    planar_store_words(P.commit, P.n, 2 * k, 8, item, cg);
    planar_store_words(P.commit, P.n, 2 * k + 1, 8, item, ck);
}

// middle, one thread per item: common challenge (Ring::aggregate ring.rs:138-160) and the sum proof (choice.rs:58-75)
EG_HD void prove_common_body(const prove_params &P, size_t item, const uint32_t *tab_g, const uint32_t *tab_k) {
    transcript t = P.ring_prefix;
    uint32_t w[8], w2[8];
#pragma unroll 1
    for (uint32_t k = 0; k < P.options; k++) {
        planar_load_words(w, P.commit, P.n, 2 * k, 8, item);
        merlin_append_words(t, EG_LBL("R_G"), w, 8);
        planar_load_words(w, P.commit, P.n, 2 * k + 1, 8, item);
        merlin_append_words(t, EG_LBL("R_K"), w, 8);
    }
    sc e0;
    merlin_challenge_scalar(t, EG_LBL("c"), e0);
    planar_store_words(P.chal, P.n, 0, 8, item, e0.v);
    store32_bytes(P.ring + item * (1 + 2 * (size_t)P.options) * 32, e0.v);
    if (!P.single) return;
    // sum ciphertext = ([sum r]G, [sum v]G + [sum r]K); powers (sum R, sum B - G)
    const uint8_t *vals = P.values + item * P.options;
    sc sum_r = sc_zero(), r, vm1;
    uint64_t nv = 0;
#pragma unroll 1
    for (uint32_t k = 0; k < P.options; k++) {
        planar_load_words(r.v, P.sec, P.n, 2 * k, 8, item);
        sc_add(sum_r, sum_r, r);
        nv += vals[k] ? 1 : 0;
    }
    sc_sub(vm1, sc_from_u64(nv), sc_from_u64(1));
    sc hr, hv, x;
    sc_half(hr, sum_r);
    sc_half(hv, vm1);
    ge_ext q0, q1;
    const bool ct = P.rnd.ct != 0;
    ge_eval_fixed(q0, 1, tab_g, hr, tab_g, hr, ct);
    ge_eval_fixed(q1, 2, tab_k, hr, tab_g, hv, ct);
    ge_double_compress2(w, w2, q0, q1);
    transcript st = P.sum_prefix;
    merlin_append_words(st, EG_LBL("[r]G"), w, 8);
    merlin_append_words(st, EG_LBL("[r]K"), w2, 8);
    prove_draw(x, P, item, 3 * P.options);
    prove_commit_pair(w, w2, x, tab_g, tab_k, ct);
    merlin_append_words(st, EG_LBL("[x]G"), w, 8);
    merlin_append_words(st, EG_LBL("[x]K"), w2, 8);
    sc c, s;
    merlin_challenge_scalar(st, EG_LBL("c"), c);
    sc_muladd(s, c, sum_r, x);
    store32_bytes(P.sum + item * 64, c.v);
    store32_bytes(P.sum + item * 64 + 32, s.v);
}

// phase 2, one thread per (item, ring k): Ring::finalize (ring.rs:162-195)
EG_HD void prove_ring2_body(const prove_params &P, size_t item, uint32_t k, uint32_t *scratch, const uint32_t *tab_g, const uint32_t *tab_k) {
    const uint8_t *vals = P.values + item * P.options;
    const bool v = vals[k] != 0;
    sc e0, r, x, s;
    planar_load_words(e0.v, P.chal, P.n, 0, 8, item);
    planar_load_words(r.v, P.sec, P.n, 2 * k, 8, item);
    planar_load_words(x.v, P.sec, P.n, 2 * k + 1, 8, item);
    uint8_t *resp = P.ring + (item * (1 + 2 * (size_t)P.options) + 1 + 2 * k) * 32;
    if (!v) {
        sc_muladd(s, e0, r, x);
        store32_bytes(resp, s.v);
        return;
    }
    uint32_t pos = 0, before = 0;
    for (uint32_t i = 0; i < P.options; i++) { pos += 2 + (vals[i] ? 0 : 1); if (i < k && vals[i]) before++; }
    sc s0, e1;
    prove_draw(s0, P, item, pos + before);
    store32_bytes(resp, s0.v);
    uint32_t cg[8], ck[8], enc_ct[16];
    prove_forge_fixed(cg, ck, r, 1, e0, s0, 0, tab_g, tab_k, P.rnd.ct != 0);
    planar_load_words(enc_ct, P.enc, P.n, 2 * k, 8, item);
    planar_load_words(enc_ct + 8, P.enc, P.n, 2 * k + 1, 8, item);
    transcript rt;
    ring_transcript_start(rt, P.ring_prefix, enc_ct, k);
    ring_next_challenge(e1, rt, 0, cg, ck);
    sc_muladd(s, e1, r, x);
    store32_bytes(resp + 32, s.v);
}

// ------------------------------------------------------------------ proving side: RangeProof::new (general rings)
//
// PublicKey::encrypt_range (keys/impls.rs:121-141) = RangeProof::new (range.rs:462-473): encrypt the value, decompose it
// over the rings of the RangeDecomposition (range.rs decompose), encrypt every partial value but the last one
// (RingProofBuilder::add_value ring.rs:460-469), derive the last partial ciphertext from the others (range.rs:520-529),
// and close all rings with a common challenge.  Caller-supplied randomness, one 64-byte block per draw, in the
// reference's order:
//   block 0                      r of the main ciphertext (CiphertextWithValue::new)
//   then per ring k, in order:   [r_k unless k is the last ring]  x_k  s_{k,eq} for eq = vi_k+1 .. size_k-1   (Ring::new)
//   then per ring k, in order:   s_{k,eq} for eq = 0 .. vi_k-1                                               (Ring::finalize)
// n_rings + sum(size_k) blocks per item.  The last ring's ciphertext is ([r_last]G, [v_last]G + [r_last]K) with
// r_last = r - sum r_k: the same group elements as `ciphertext - sum partial` (ExtendedCiphertext arithmetic tracks the
// randomness, encryption.rs:329-357), computed without touching the other rings' points.
struct rprove_params {
    size_t n;
    uint32_t n_rings, total;                 // total = sum of ring sizes
    uint16_t sizes[EG_MAX_RINGS], starts[EG_MAX_RINGS];
    uint64_t steps[EG_MAX_RINGS];
    const uint64_t *values; size_t value_stride;     // value of item i = values[i * value_stride]
    // Items may be grouped into records (QuadraticVotingBallot: item = (ballot, option)): with group > 1 the address of
    // item i's data is base + (i / group) * stride + (i % group) * inner; group <= 1 is the flat base + i * stride.
    uint32_t group;
    size_t wide_inner, out_inner;
    const uint8_t *wide; size_t wide_stride;         // first randomness block of the item
    uint8_t *ct_out; size_t ct_stride;               // 64 B per item
    uint8_t *partial_out; size_t partial_stride;     // 64 (n_rings - 1) B per item
    uint8_t *ring_out; size_t ring_stride;           // 32 (1 + total) B per item: common challenge | responses
    transcript prefix;                               // Transcript::new(label) + "encryption_range_proof" + "range" + initialize_transcript
    uint32_t *pts, *enc, *sec, *commit, *chal;       // planar scratch; ring k: pts / enc / commit 2k, 2k+1; sec 2k = r_k, 2k+1 = x_k
    uint32_t *ct_sec;                                // optional planar scalar (index 0): r of the main ciphertext
    const uint32_t *table_g, *table_k;
    rand_src rnd;                                    // seeded: the item's stream is the RECORD's stream (group > 1: item / group),
                                                     // its blocks start at rnd.block0 + (item % group) * wide_inner / 64
    const uint8_t *ct_r;                             // RangeProof::from_ciphertext (range.rs:482-534): the main ciphertext exists
                                                     // already; its randomness (canonical scalar, 32 B per item) replaces draw 0
                                                     // and the remaining draws move up by one.  Flat batches only (group <= 1).
};

EG_HD size_t rprove_off(const rprove_params &P, size_t item, size_t stride, size_t inner) {
    return P.group > 1 ? (item / P.group) * stride + (item % P.group) * inner : item * stride;
}

EG_HD void rprove_draw(sc &out, const rprove_params &P, size_t item, uint32_t pos) {
    uint32_t w[16];
    if (P.ct_r) {
        if (pos == 0) {
            load32_bytes(w, P.ct_r + item * 32);
            if (!sc_from_words(out, w)) out = sc_zero();      // (validated on the host)
            return;
        }
        pos -= 1;
    }
    if (P.rnd.seeded) {
        const size_t record = P.group > 1 ? item / P.group : item;
        const uint32_t inner = P.group > 1 ? (uint32_t)((item % P.group) * (P.wide_inner / 64)) : 0u;
        chacha20_block(w, P.rnd.key, rand_counter(P.rnd, record, inner + pos));
    } else {
        const uint8_t *b = P.wide + rprove_off(P, item, P.wide_stride, P.wide_inner) + (size_t)pos * 64;
        load32_bytes(w, b);
        load32_bytes(w + 8, b + 32);
    }
    sc_from_wide_words(out, w);
}

// value index of ring k and the positions of its first phase-0 / phase-2 draws (RangeDecomposition::decompose)
struct rprove_pos { uint32_t vi, pos0, pos2; };

EG_HD rprove_pos rprove_layout(const rprove_params &P, uint64_t value, uint32_t k) {
    rprove_pos out = {0, 0, 0};
    uint32_t p0 = 1, fin_before = 0;
    for (uint32_t i = 0; i < P.n_rings; i++) {
        uint64_t idx = value / P.steps[i];
        if (idx > (uint64_t)P.sizes[i] - 1) idx = (uint64_t)P.sizes[i] - 1;
        value -= idx * P.steps[i];
        if (i == k) { out.vi = (uint32_t)idx; out.pos0 = p0; out.pos2 = fin_before; }
        p0 += (i + 1 < P.n_rings ? 1u : 0u) + 1u + (P.sizes[i] - 1u - (uint32_t)idx);
        if (i < k) fin_before += (uint32_t)idx;
    }
    out.pos2 += p0;         // finalize draws start after every ring's Ring::new draws
    return out;
}

// enc_ct = encodings of ([r]G, [v]G + [r]K)
EG_HD void rprove_encrypt(uint32_t enc_ct[16], const sc &r, uint64_t v, const uint32_t *tab_g, const uint32_t *tab_k, bool ct) {
    sc hr, hv;
    sc_half(hr, r);
    sc_half(hv, sc_from_u64(v));
    ge_ext qr, qb;
    ge_eval_fixed(qr, 1, tab_g, hr, tab_g, hr, ct);
    ge_eval_fixed(qb, (v || ct) ? 2 : 1, tab_k, hr, tab_g, hv, ct);
    ge_double_compress2(enc_ct, enc_ct + 8, qr, qb);
}

// phase 0, one thread per (item, slot): slot < n_rings = ring `slot` (ciphertext + Ring::new); slot == n_rings = main ciphertext
EG_HD void rprove_ring1_body(const rprove_params &P, size_t item, uint32_t slot, uint32_t *scratch, const uint32_t *tab_g, const uint32_t *tab_k) {
    const uint64_t value = P.values[item * P.value_stride];
    const uint32_t Rn = P.n_rings;
    uint32_t enc_ct[16];
    if (slot == Rn) {
        sc r;
        rprove_draw(r, P, item, 0);
        if (!P.ct_out && !P.ct_sec) return;           // from_ciphertext without the optional re-encryption
        rprove_encrypt(enc_ct, r, value, tab_g, tab_k, P.rnd.ct != 0);
        if (P.ct_out) {
            uint8_t *o = P.ct_out + rprove_off(P, item, P.ct_stride, P.out_inner);
            store32_bytes(o, enc_ct);
            store32_bytes(o + 32, enc_ct + 8);
        }
        if (P.ct_sec) planar_store_words(P.ct_sec, P.n, 0, 8, item, r.v);
        return;
    }
    const uint32_t k = slot, m = P.sizes[k];
    const rprove_pos L = rprove_layout(P, value, k);
    const bool last = (k + 1 == Rn);
    sc r, x;
    if (!last) {
        rprove_draw(r, P, item, L.pos0);
    } else {
        // r_last = r_ct - sum of the other rings' r (range.rs:520-521)
        rprove_draw(r, P, item, 0);
#pragma unroll 1
        for (uint32_t i = 0; i + 1 < Rn; i++) {
            sc ri;
            rprove_draw(ri, P, item, rprove_layout(P, value, i).pos0);
            sc_sub(r, r, ri);
        }
    }
    const bool ct = P.rnd.ct != 0;
    rprove_encrypt(enc_ct, r, (uint64_t)L.vi * P.steps[k], tab_g, tab_k, ct);
    if (!last) {
        uint8_t *o = P.partial_out + rprove_off(P, item, P.partial_stride, P.out_inner) + 64 * (size_t)k;
        store32_bytes(o, enc_ct);
        store32_bytes(o + 32, enc_ct + 8);
    }
    const uint32_t xpos = L.pos0 + (last ? 0u : 1u);
    rprove_draw(x, P, item, xpos);
    planar_store_words(P.enc, P.n, 2 * k, 8, item, enc_ct);
    planar_store_words(P.enc, P.n, 2 * k + 1, 8, item, enc_ct + 8);
    planar_store_words(P.sec, P.n, 2 * k, 8, item, r.v);
    planar_store_words(P.sec, P.n, 2 * k + 1, 8, item, x.v);
    // Ring::new (ring.rs:97-131): commitments of the real equation, then the forged equations above it
    uint32_t cg[8], ck[8];
    prove_commit_pair(cg, ck, x, tab_g, tab_k, ct);
    if (L.vi + 1 < m) {
        transcript rt;
        ring_transcript_start(rt, P.prefix, enc_ct, k);
        uint8_t *resp = P.ring_out + rprove_off(P, item, P.ring_stride, P.out_inner) + 32 * (1 + (size_t)P.starts[k]);
#pragma unroll 1
        for (uint32_t eq = L.vi + 1; eq < m; eq++) {
            sc e, s_;
            ring_next_challenge(e, rt, eq - 1, cg, ck);
            rprove_draw(s_, P, item, xpos + (eq - L.vi));
            store32_bytes(resp + 32 * (size_t)eq, s_.v);
            prove_forge_fixed(cg, ck, r, (uint64_t)L.vi * P.steps[k], e, s_, (uint64_t)eq * P.steps[k], tab_g, tab_k, ct);
        }
    }
    planar_store_words(P.commit, P.n, 2 * k, 8, item, cg);
    planar_store_words(P.commit, P.n, 2 * k + 1, 8, item, ck);
}

// phase 1, one thread per item: common challenge (Ring::aggregate ring.rs:138-160)
EG_HD void rprove_common_body(const rprove_params &P, size_t item) {
    transcript t = P.prefix;
    uint32_t w[8];
#pragma unroll 1
    for (uint32_t k = 0; k < P.n_rings; k++) {
        planar_load_words(w, P.commit, P.n, 2 * k, 8, item);
        merlin_append_words(t, EG_LBL("R_G"), w, 8);
        planar_load_words(w, P.commit, P.n, 2 * k + 1, 8, item);
        merlin_append_words(t, EG_LBL("R_K"), w, 8);
    }
    sc e0;
    merlin_challenge_scalar(t, EG_LBL("c"), e0);
    planar_store_words(P.chal, P.n, 0, 8, item, e0.v);
    store32_bytes(P.ring_out + rprove_off(P, item, P.ring_stride, P.out_inner), e0.v);
}

// phase 2, one thread per (item, ring k): Ring::finalize (ring.rs:162-195)
EG_HD void rprove_ring2_body(const rprove_params &P, size_t item, uint32_t k, uint32_t *scratch, const uint32_t *tab_g, const uint32_t *tab_k) {
    const uint64_t value = P.values[item * P.value_stride];
    const rprove_pos L = rprove_layout(P, value, k);
    sc e, r, x, s;
    planar_load_words(e.v, P.chal, P.n, 0, 8, item);
    planar_load_words(r.v, P.sec, P.n, 2 * k, 8, item);
    planar_load_words(x.v, P.sec, P.n, 2 * k + 1, 8, item);
    uint8_t *resp = P.ring_out + rprove_off(P, item, P.ring_stride, P.out_inner) + 32 * (1 + (size_t)P.starts[k]);
    if (L.vi > 0) {
        uint32_t enc_ct[16], cg[8], ck[8];
        planar_load_words(enc_ct, P.enc, P.n, 2 * k, 8, item);
        planar_load_words(enc_ct + 8, P.enc, P.n, 2 * k + 1, 8, item);
        transcript rt;
        ring_transcript_start(rt, P.prefix, enc_ct, k);
#pragma unroll 1
        for (uint32_t eq = 0; eq < L.vi; eq++) {
            sc s_;
            rprove_draw(s_, P, item, L.pos2 + eq);
            store32_bytes(resp + 32 * (size_t)eq, s_.v);
            prove_forge_fixed(cg, ck, r, (uint64_t)L.vi * P.steps[k], e, s_, (uint64_t)eq * P.steps[k], tab_g, tab_k, P.rnd.ct != 0);
            ring_next_challenge(e, rt, eq, cg, ck);
        }
    }
    sc_muladd(s, e, r, x);
    store32_bytes(resp + 32 * (size_t)L.vi, s.v);
}

// ------------------------------------------------------------------ PublicKey::encrypt / encrypt_zero (keys/impls.rs:16-53)
//
// encrypt: one draw r per item, (R, B) = ([r]G, [v]G + [r]K) (ExtendedCiphertext::new encryption.rs:310-327).
// encrypt_zero: r, then the LogEqualityProof::new nonce x (log_equality.rs:114-143); proof = c | c r + x.
struct encrypt_params {
    size_t n;
    uint8_t with_zero_proof;             // 0: encrypt(values[i]); 1: encrypt_zero + proof
    const uint64_t *values;              // mode 0
    const uint8_t *wide;                 // n * (1 + with_zero_proof) * 64
    uint8_t *cts;                        // n * 64
    uint8_t *proofs;                     // mode 1: n * 64
    transcript prefix;                   // mode 1: Transcript::new("zero_encryption") + start_proof("log_eq") + "K"
    const uint32_t *table_g, *table_k;
    rand_src rnd;
};

// block `k` of item `item`: from the caller's buffer at `b`, or generated
EG_HD void rand_block(uint32_t w[16], const rand_src &R, size_t item, uint32_t k, const uint8_t *b) {
    if (R.seeded) { chacha20_block(w, R.key, rand_counter(R, item, k)); return; }
    load32_bytes(w, b);
    load32_bytes(w + 8, b + 32);
}

EG_HD void encrypt_body(const encrypt_params &P, size_t item, const uint32_t *tab_g, const uint32_t *tab_k) {
    const uint32_t draws = 1 + P.with_zero_proof;
    uint32_t w[16], enc_ct[16];
    const uint8_t *b = P.wide + item * draws * 64;
    const bool ct = P.rnd.ct != 0;
    sc r;
    rand_block(w, P.rnd, item, 0, b);
    sc_from_wide_words(r, w);
    rprove_encrypt(enc_ct, r, P.with_zero_proof ? 0 : P.values[item], tab_g, tab_k, ct);
    store32_bytes(P.cts + item * 64, enc_ct);
    store32_bytes(P.cts + item * 64 + 32, enc_ct + 8);
    if (!P.with_zero_proof) return;
    sc x, c, s_;
    rand_block(w, P.rnd, item, 1, b + 64);
    sc_from_wide_words(x, w);
    uint32_t c0[8], c1[8];
    prove_commit_pair(c0, c1, x, tab_g, tab_k, ct);
    transcript t = P.prefix;
    merlin_append_words(t, EG_LBL("[r]G"), enc_ct, 8);
    merlin_append_words(t, EG_LBL("[r]K"), enc_ct + 8, 8);
    merlin_append_words(t, EG_LBL("[x]G"), c0, 8);
    merlin_append_words(t, EG_LBL("[x]K"), c1, 8);
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    sc_muladd(s_, c, r, x);
    store32_bytes(P.proofs + item * 64, c.v);
    store32_bytes(P.proofs + item * 64 + 32, s_.v);
}

// ------------------------------------------------------------------ proving side: SumOfSquaresProof::new (mul.rs:107-181)
//
// The prover knows the value x_i and randomness r_i of every ciphertext (R_i, X_i) = ([r_i]G, [x_i]G + [r_i]K), so each
// commitment is a fixed-base expression:
//   [e_r,i]G ; [e_x,i]G + [e_r,i]K ; sum [e_x,i]R_i + [e_z]G = [sum e_x,i r_i + e_z]G ;
//   sum [e_x,i]X_i + [e_z]K = [sum e_x,i x_i]G + [sum e_x,i r_i + e_z]K
// (the same group elements as the reference's multi_mul over R_i / X_i).  Draw order: e_z, then (e_r,i, e_x,i) per
// ciphertext.  One thread per ballot.  Used by QuadraticVotingBallot::new (quadratic_voting.rs:268-276).
struct sumsq_prove_params {
    size_t n;
    uint32_t m;                          // ciphertexts per item
    const uint64_t *values;              // n * m
    const uint8_t *wide; size_t wide_stride;   // first block of the proof's randomness
    const uint8_t *cts; size_t ct_stride, ct_inner;   // ciphertext i of item b at cts + b * ct_stride + i * ct_inner (64 B)
    const uint8_t *sum_ct;               // + b * ct_stride: the sum-of-squares ciphertext (64 B)
    uint8_t *proof; size_t proof_stride; // 32 (2m + 2) B: challenge | (r_resp, x_resp) * m | sum_resp
    const uint32_t *r_cts;               // planar scalars over n * m items (item b * m + i): r_i
    const uint32_t *r_sum;               // planar scalars over n items: randomness of the sum ciphertext
    transcript prefix;                   // Transcript::new(label) + start_proof("sum_of_squares") + "K"
    const uint32_t *table_g, *table_k;
    rand_src rnd;
};

EG_HD void sumsq_prove_body(const sumsq_prove_params &P, size_t item, const uint32_t *tab_g, const uint32_t *tab_k) {
    transcript t = P.prefix;
    uint32_t w[16], c0[8], c1[8];
    const uint8_t *wide = P.wide + item * P.wide_stride;
    const bool ct = P.rnd.ct != 0;
    sc e_z, e_r[EG_MSM_MAXV], e_x[EG_MSM_MAXV];
    rand_block(w, P.rnd, item, 0, wide);
    sc_from_wide_words(e_z, w);
    sc acc_r = e_z, acc_x = sc_zero();       // sum e_x,i r_i + e_z ; sum e_x,i x_i
    sc sum_random;                            // r_z - sum x_i r_i   (mul.rs:117,132-133)
    planar_load_words(sum_random.v, P.r_sum, P.n, 0, 8, item);
#pragma unroll 1
    for (uint32_t i = 0; i < P.m; i++) {
        const uint8_t *ct = P.cts + item * P.ct_stride + i * P.ct_inner;
        load32_bytes(w, ct);
        merlin_append_words(t, EG_LBL("R_x"), w, 8);
        load32_bytes(w, ct + 32);
        merlin_append_words(t, EG_LBL("X"), w, 8);
        const uint8_t *b = wide + 64 * (size_t)(1 + 2 * i);
        rand_block(w, P.rnd, item, 1 + 2 * i, b);
        sc_from_wide_words(e_r[i], w);
        rand_block(w, P.rnd, item, 2 + 2 * i, b + 64);
        sc_from_wide_words(e_x[i], w);
        sc her, hex_;
        sc_half(her, e_r[i]);
        sc_half(hex_, e_x[i]);
        ge_ext q0, q1;
        ge_eval_fixed(q0, 1, tab_g, her, tab_g, her, ct);
        ge_eval_fixed(q1, 2, tab_k, her, tab_g, hex_, ct);
        ge_double_compress2(c0, c1, q0, q1);
        merlin_append_words(t, EG_LBL("[e_r]G"), c0, 8);
        merlin_append_words(t, EG_LBL("[e_x]G + [e_r]K"), c1, 8);
        sc r_i, x_i = sc_from_u64(P.values[item * P.m + i]), tmp;
        planar_load_words(r_i.v, P.r_cts, P.n * P.m, 0, 8, item * P.m + i);
        sc_muladd(acc_r, e_x[i], r_i, acc_r);
        sc_muladd(acc_x, e_x[i], x_i, acc_x);
        sc_mul(tmp, x_i, r_i);
        sc_sub(sum_random, sum_random, tmp);
    }
    {
        sc ha, hx;
        sc_half(ha, acc_r);
        sc_half(hx, acc_x);
        ge_ext q0, q1;
        ge_eval_fixed(q0, 1, tab_g, ha, tab_g, ha, ct);
        ge_eval_fixed(q1, 2, tab_k, ha, tab_g, hx, ct);
        ge_double_compress2(c0, c1, q0, q1);
    }
    const uint8_t *zct = P.sum_ct + item * P.ct_stride;
    load32_bytes(w, zct);
    merlin_append_words(t, EG_LBL("R_z"), w, 8);
    load32_bytes(w, zct + 32);
    merlin_append_words(t, EG_LBL("Z"), w, 8);
    merlin_append_words(t, EG_LBL("[e_x]R_x + [e_z]G"), c0, 8);
    merlin_append_words(t, EG_LBL("[e_x]X + [e_z]K"), c1, 8);
    sc c, s;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    uint8_t *out = P.proof + item * P.proof_stride;
    store32_bytes(out, c.v);
#pragma unroll 1
    for (uint32_t i = 0; i < P.m; i++) {
        sc r_i, x_i = sc_from_u64(P.values[item * P.m + i]);
        planar_load_words(r_i.v, P.r_cts, P.n * P.m, 0, 8, item * P.m + i);
        sc_muladd(s, c, r_i, e_r[i]);
        store32_bytes(out + 32 * (size_t)(1 + 2 * i), s.v);
        sc_muladd(s, c, x_i, e_x[i]);
        store32_bytes(out + 32 * (size_t)(2 + 2 * i), s.v);
    }
    sc_muladd(s, c, sum_random, e_z);
    store32_bytes(out + 32 * (size_t)(1 + 2 * P.m), s.v);
}

// Outer transcript: absorb every ring's terminal commitments, compare with the common challenge (ring.rs:364-373)
struct ring_final_params {
    in_bufs in;
    size_t n;
    uint32_t n_rings;
    uint32_t commit_index0;     // ring r's terminal (R_G, R_K) at commit_index0 + 2r, +1
    uint8_t proof_buf;          // input buffer holding the ring proof; common challenge at offset `cc_offset`
    uint32_t cc_offset;
    transcript prefix;          // state after initialize_transcript
    const uint32_t *commit;
    uint32_t *result;           // per item: 1 = challenge matches
};

EG_HD void ring_final_body(const ring_final_params &P, size_t item) {
    transcript t = P.prefix;
    uint32_t w[8];
#pragma unroll 1
    for (uint32_t r = 0; r < P.n_rings; r++) {
        planar_load_words(w, P.commit, P.n, P.commit_index0 + 2 * r, 8, item);
        merlin_append_words(t, EG_LBL("R_G"), w, 8);
        planar_load_words(w, P.commit, P.n, P.commit_index0 + 2 * r + 1, 8, item);
        merlin_append_words(t, EG_LBL("R_K"), w, 8);
    }
    sc c, cc;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    load32_bytes(w, in_ptr(P.in, P.proof_buf, item) + P.cc_offset);
    bool ok = sc_from_words(cc, w);
    P.result[item] = (ok && sc_eq(c, cc)) ? 1u : 0u;
}

// LogEqualityProof transcript tail (log_equality.rs:169-179): prefix holds start_proof + "K"
struct logeq_final_params {
    in_bufs in;
    size_t n;
    uint32_t pow_enc_index;     // planar enc of the two powers ([r]G, [r]K) at pow_enc_index, +1
    uint32_t commit_index;      // planar commitments ([x]G, [x]K) at commit_index, +1
    uint8_t proof_buf;
    uint32_t c_offset;          // byte offset of the challenge in the proof item
    uint8_t prefix_per_item;    // 1: the transcript prefix is finished per item (share proofs: "K" = enc(R))
    uint32_t key_enc_index;     // planar enc index of the per-item log base (prefix_per_item = 1)
    transcript prefix;
    const uint32_t *enc;
    const uint32_t *commit;
    uint32_t *result;
};

EG_HD void logeq_final_body(const logeq_final_params &P, size_t item) {
    transcript t = P.prefix;
    uint32_t w[8];
    if (P.prefix_per_item) {
        merlin_append_message(t, EG_LBL("dom-sep"), (const uint8_t *)"log_eq", 6);
        planar_load_words(w, P.enc, P.n, P.key_enc_index, 8, item);
        merlin_append_words(t, EG_LBL("K"), w, 8);
    }
    planar_load_words(w, P.enc, P.n, P.pow_enc_index, 8, item);
    merlin_append_words(t, EG_LBL("[r]G"), w, 8);
    planar_load_words(w, P.enc, P.n, P.pow_enc_index + 1, 8, item);
    merlin_append_words(t, EG_LBL("[r]K"), w, 8);
    planar_load_words(w, P.commit, P.n, P.commit_index, 8, item);
    merlin_append_words(t, EG_LBL("[x]G"), w, 8);
    planar_load_words(w, P.commit, P.n, P.commit_index + 1, 8, item);
    merlin_append_words(t, EG_LBL("[x]K"), w, 8);
    sc c, cc;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    load32_bytes(w, in_ptr(P.in, P.proof_buf, item) + P.c_offset);
    bool ok = sc_from_words(cc, w);
    P.result[item] = (ok && sc_eq(c, cc)) ? 1u : 0u;
}

// ------------------------------------------------------------------ generic Fiat-Shamir tail of a sigma proof
//
// Appends a list of 32-byte messages (input encodings, recomputed commitments) to a prepared transcript prefix, squeezes
// the challenge and compares it with the proof's.  Used by CommitmentEquivalenceProof::verify (commitment.rs:198-248)
// and ProofOfPossession::verify (possession.rs:137-163); a message entry with count > 1 is a run of messages with the
// same label and consecutive indexes (the "K" / "R" runs of a multi-key proof of possession).
#define EG_SIGMA_MAX_MSGS 8

struct sigma_msg {
    uint8_t kind;               // 0: planar `enc`, 1: planar `commit`
    uint8_t label_len;
    char label[22];
    uint32_t index;             // first planar index
    uint32_t count;             // messages in the run
};

struct sigma_final_params {
    in_bufs in;
    size_t n;
    transcript prefix;
    int n_msgs;
    sigma_msg msgs[EG_SIGMA_MAX_MSGS];
    uint8_t proof_buf;
    uint32_t c_offset;          // byte offset of the proof's challenge in its item
    const uint32_t *enc;
    const uint32_t *commit;
    uint32_t *result;
};

EG_HD void sigma_final_body(const sigma_final_params &P, size_t item) {
    transcript t = P.prefix;
    uint32_t w[8];
#pragma unroll 1
    for (int m = 0; m < P.n_msgs; m++) {
        const sigma_msg &g = P.msgs[m];
        const uint32_t *base = g.kind ? P.commit : P.enc;
#pragma unroll 1
        for (uint32_t r = 0; r < g.count; r++) {
            planar_load_words(w, base, P.n, g.index + r, 8, item);
            merlin_append_words(t, g.label, g.label_len, w, 8);
        }
    }
    sc c, cc;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    load32_bytes(w, in_ptr(P.in, P.proof_buf, item) + P.c_offset);
    bool ok = sc_from_words(cc, w);
    P.result[item] = (ok && sc_eq(c, cc)) ? 1u : 0u;
}

// ------------------------------------------------------------------ derived ciphertexts

// EncryptedChoice: sum of the option ciphertexts (choice.rs:363) and the sum-proof powers (choice.rs:83-86):
// side 0: sum R ; side 1: sum B - G.  Stores the point and its encoding (both are hashed / multiplied later).
struct choice_sum_params {
    size_t n;
    uint32_t options;
    uint32_t out_p_index;       // points at out_p_index + side
    uint32_t out_enc_index;     // encodings at out_enc_index + side
    uint32_t *pts;
    uint32_t *enc;
};

EG_HD void choice_sum_body(const choice_sum_params &P, size_t item, int side) {
    ge_ext acc, q;
    planar_load_point(acc, P.pts, P.n, side, item);
#pragma unroll 1
    for (uint32_t k = 1; k < P.options; k++) {
        planar_load_point(q, P.pts, P.n, 2 * k + side, item);
        ge_add(acc, acc, q);
    }
    if (side == 1) ge_sub(acc, acc, ge_generator());
    planar_store_point(P.pts, P.n, P.out_p_index + side, item, acc);
    uint32_t w[8];
    ge_encode(w, acc);
    planar_store_words(P.enc, P.n, P.out_enc_index + side, 8, item, w);
}

// RangeProof: last ring's ciphertext = ct - sum(partial) (range.rs:564-572); point + encoding, per side
struct range_last_params {
    size_t n;
    uint32_t n_partial;         // n_rings - 1 partial ciphertexts at point indexes 2k + side (k < n_partial)
    uint32_t ct_p_index;        // main ciphertext at ct_p_index + side
    uint32_t out_p_index;       // last ring ciphertext at out_p_index + side
    uint32_t out_enc_index;
    uint32_t *pts;
    uint32_t *enc;
};

EG_HD void range_last_body(const range_last_params &P, size_t item, int side) {
    ge_ext acc, q;
    planar_load_point(acc, P.pts, P.n, P.ct_p_index + side, item);
#pragma unroll 1
    for (uint32_t k = 0; k < P.n_partial; k++) {
        planar_load_point(q, P.pts, P.n, 2 * k + side, item);
        ge_sub(acc, acc, q);
    }
    planar_store_point(P.pts, P.n, P.out_p_index + side, item, acc);
    uint32_t w[8];
    ge_encode(w, acc);
    planar_store_words(P.enc, P.n, P.out_enc_index + side, 8, item, w);
}

// ------------------------------------------------------------------ verdicts

// verdict precedence (SURVEY.md 3.1): malformed -> first failing check in the reference's order
struct verdict_params {
    size_t n;
    const uint32_t *flags;
    int n_checks;
    const uint32_t *check[8];   // per item 1 = passed
    size_t check_stride[8];     // item stride (1, or k when the check array holds k results per item)
    size_t check_offset[8];
    uint8_t code[8];            // verdict when check k is the first to fail
    uint8_t *verdicts;
};

EG_HD void verdict_body(const verdict_params &P, size_t item) {
    uint8_t v = 0;
    if (P.flags[item] & 1u) v = 1;
    else {
        for (int k = 0; k < P.n_checks; k++)
            if (!P.check[k][item * P.check_stride[k] + P.check_offset[k]]) { v = P.code[k]; break; }
    }
    P.verdicts[item] = v;
}

}  // namespace eg

// ------------------------------------------------------------------ setup bodies (once per context / receiver / range)

namespace eg {

// Wide fixed-base table of F (ge.cuh "fixed-base tables"), F given as an encoding; two stages.
// Stage 1 (one thread): status = 0 ok / 1 undecodable / 2 identity; bases[i] = 2^(W i) F, extended, 32 words each.
template <int BITS>
EG_HD void wide_bases_body(const uint32_t *enc_words, int use_generator, uint32_t *bases, uint32_t *status) {
    ge_ext F;
    bool ok = true;
    if (use_generator) F = ge_generator();
    else {
        uint32_t w[8];
        for (int k = 0; k < 8; k++) w[k] = enc_words[k];
        ok = ge_decode(F, w);                                  // the identity when rejected: the table stays well defined
    }
    *status = !ok ? 1u : (ge_is_identity(F) ? 2u : 0u);
#pragma unroll 1
    for (int i = 0; i < EG_BITS_WINDOWS(BITS); i++) {
        point_to_words32(bases + i * 32, F);
        if (i + 1 < EG_BITS_WINDOWS(BITS)) ge_hot_dbl(F, BITS);
    }
}

// Stage 2: thread tidx = (window i, block jb) writes entries m = jb * EG_WIDE_BLOCK + 1 .. + EG_WIDE_BLOCK of window i:
// table[(i * EG_WIDE_ENTRIES + m - 1) * 24 ..] = affine Niels form of m 2^(W i) F; one inversion per block.
template <int BITS>
EG_HD void wide_fill_body(size_t tidx, const uint32_t *bases, uint32_t *table) {
    const int blocks = EG_BITS_ENTRIES(BITS) / EG_WIDE_BLOCK;
    const int i = (int)(tidx / blocks), jb = (int)(tidx % blocks);
    ge_ext B, acc = ge_identity();
    point_from_words32(B, bases + i * 32);
    ge_cached cb;
    ge_to_cached(cb, B);
    const uint32_t first = (uint32_t)jb * EG_WIDE_BLOCK + 1;
    ge_p1p1 t;
#pragma unroll 1
    for (int bit = BITS - 1; bit >= 0; bit--) {
        ge_dbl(acc, acc);
        if ((first >> bit) & 1u) { ge_add_cached_p1p1(t, acc, cb, false); ge_p1p1_to_ext(acc, t); }
    }
    ge_ext pts[EG_WIDE_BLOCK];
    fe prod[EG_WIDE_BLOCK];
#pragma unroll 1
    for (int k = 0; k < EG_WIDE_BLOCK; k++) {
        if (k) { ge_add_cached_p1p1(t, acc, cb, false); ge_p1p1_to_ext(acc, t); }
        pts[k] = acc;
        if (k) fe_mul(prod[k], prod[k - 1], acc.Z); else prod[0] = acc.Z;
    }
    fe inv;
    fe_invert(inv, prod[EG_WIDE_BLOCK - 1]);
    uint32_t *out = table + ((size_t)i * EG_BITS_ENTRIES(BITS) + first - 1) * 24;
#pragma unroll 1
    for (int k = EG_WIDE_BLOCK - 1; k >= 0; k--) {
        fe zi, x, y, u;
        if (k) { fe_mul(zi, inv, prod[k - 1]); fe_mul(inv, inv, pts[k].Z); } else zi = inv;
        fe_mul(x, pts[k].X, zi); fe_mul(y, pts[k].Y, zi);
        fe_add(u, y, x); fe_towords(out + k * 24, u);
        fe_sub(u, y, x); fe_towords(out + k * 24 + 8, u);
        fe_mul(u, x, y); fe_mul(u, u, fe_const_2d()); fe_towords(out + k * 24 + 16, u);
    }
}

// adm[tid] = cached form of [values[tid]] G   (PreparedRange::new range.rs:341-355)
EG_HD void admissible_body(int tid, const uint64_t *values, uint32_t *adm) {
    uint64_t v = values[tid];
    ge_ext G = ge_generator(), acc = ge_identity();
#pragma unroll 1
    for (int bit = 63; bit >= 0; bit--) {
        ge_dbl(acc, acc);
        if ((v >> bit) & 1) ge_add(acc, acc, G);
    }
    ge_cached c;
    ge_to_cached(c, acc);
    uint32_t *o = adm + (size_t)tid * 32;
    for (int k = 0; k < 8; k++) { o[k] = c.YpX.v[k]; o[8 + k] = c.YmX.v[k]; o[16 + k] = c.Z.v[k]; o[24 + k] = c.T2d.v[k]; }
}


EG_HD void elements_validate_body(size_t i, const uint8_t *enc, uint8_t *ok) {
    uint32_t w[8];
    load32_bytes(w, enc + 32 * i);
    ge_ext p;
    ok[i] = ge_decode(p, w) ? 1 : 0;
}

EG_HD void scalars_validate_body(size_t i, const uint8_t *s, uint8_t *ok) {
    uint32_t w[8];
    load32_bytes(w, s + 32 * i);
    ok[i] = sc_is_canonical_words(w) ? 1 : 0;
}

// planar encoding 0 of every item -> 32-byte records; ok = 0 and the identity encoding for flagged (malformed) items
struct unpack_params { size_t n; uint32_t n_out; const uint32_t *commit; const uint32_t *flags; uint8_t *out; uint8_t *ok; };   // n_out encodings per item

EG_HD void unpack_body(const unpack_params &P, size_t item) {
    uint32_t w[8];
    const bool bad = (P.flags[item] & 1u) != 0;
    for (uint32_t q = 0; q < P.n_out; q++) {
        planar_load_words(w, P.commit, P.n, q, 8, item);
        if (bad) for (int k = 0; k < 8; k++) w[k] = 0;
        store32_bytes(P.out + 32 * (item * P.n_out + q), w);
    }
    P.ok[item] = bad ? 0 : 1;
}

// PublicKeySet::from_participants verdict (key_set.rs:128-140): interpolated key x (planar commit index 1 + (x - t)) must equal
// participant key x byte for byte (both are canonical encodings); planar commit 0 is the reconstructed shared key.
struct keyset_verdict_params {
    size_t n;
    uint32_t shares, threshold;
    const uint8_t *keys;            // n * shares * 32
    const uint32_t *commit;         // planar encodings
    const uint32_t *flags;
    uint8_t *shared_out;            // n * 32
    uint8_t *verdicts;
    uint8_t code_mismatch;
};

EG_HD void keyset_verdict_body(const keyset_verdict_params &P, size_t item) {
    uint32_t w[8], k[8];
    uint8_t v = 0;
    if (P.flags[item] & 1u) v = 1;
    else {
        for (uint32_t x = P.threshold; x < P.shares; x++) {
            planar_load_words(w, P.commit, P.n, 1 + (x - P.threshold), 8, item);
            load32_bytes(k, P.keys + (item * P.shares + x) * 32);
            bool same = true;
            for (int q = 0; q < 8; q++) same = same && (w[q] == k[q]);
            if (!same) { v = P.code_mismatch; break; }
        }
    }
    planar_load_words(w, P.commit, P.n, 0, 8, item);
    if (v) for (int q = 0; q < 8; q++) w[q] = 0;
    store32_bytes(P.shared_out + 32 * item, w);
    P.verdicts[item] = v;
}

// ------------------------------------------------------------------ wire format: Base64UrlUnpadded (serde.rs:19-80)
//
// Human-readable serde forms of every element / scalar / proof are unpadded base64url strings (serialize_bytes
// serde.rs:19-27, Base64Visitor :41-44).  Fields have fixed sizes, so a batch is n items of `chars` characters ->
// `bytes` bytes with chars = ceil(4 bytes / 3).  One thread = one 4-character group (3 bytes).  Decoding is strict like
// base64ct's: characters outside the URL-safe alphabet (including '=' padding) and non-zero trailing bits are rejected.
EG_HD int b64url_value(uint32_t c) {
    if (c - 'A' < 26u) return (int)(c - 'A');
    if (c - 'a' < 26u) return (int)(c - 'a') + 26;
    if (c - '0' < 10u) return (int)(c - '0') + 52;
    if (c == '-') return 62;
    if (c == '_') return 63;
    return -1;
}
EG_HD uint8_t b64url_char(uint32_t v) {
    return (uint8_t)(v < 26 ? 'A' + v : v < 52 ? 'a' + (v - 26) : v < 62 ? '0' + (v - 52) : v == 62 ? '-' : '_');
}

struct b64_params {
    size_t n;
    uint32_t bytes, chars, groups;      // per item; groups = ceil(chars / 4)
    uint8_t *text;
    uint8_t *raw;
    uint8_t *ok;                        // decode only: pre-set to 1, cleared by any failing group
    uint32_t ok_group;                  // strings per object (0 = 1): ok[item / ok_group] -- struct-level decoding, every
                                        // field of an object must decode
};

EG_HD void b64url_decode_body(const b64_params &P, size_t tid) {
    const size_t item = tid / P.groups;
    const uint32_t g = (uint32_t)(tid % P.groups);
    const uint8_t *src = P.text + item * P.chars + 4 * g;
    uint8_t *dst = P.raw + item * P.bytes + 3 * g;
    const uint32_t nc = (P.chars - 4 * g) < 4 ? (P.chars - 4 * g) : 4;      // 4, or 2 / 3 in the tail group
    int v[4] = {0, 0, 0, 0};
    bool good = nc != 1;
    for (uint32_t k = 0; k < nc; k++) { v[k] = b64url_value(src[k]); good = good && v[k] >= 0; }
    const uint32_t x = ((uint32_t)(v[0] & 63) << 18) | ((uint32_t)(v[1] & 63) << 12) | ((uint32_t)(v[2] & 63) << 6) | (uint32_t)(v[3] & 63);
    if (nc == 2) good = good && (x & 0xffffu) == 0;      // 4 unused bits of the second character
    if (nc == 3) good = good && (x & 0xffu) == 0;        // 2 unused bits of the third character
    const uint32_t nb = nc - 1;
    for (uint32_t k = 0; k < nb; k++) dst[k] = (uint8_t)(x >> (16 - 8 * k));
    if (!good) P.ok[P.ok_group > 1 ? item / P.ok_group : item] = 0;
}

EG_HD void b64url_encode_body(const b64_params &P, size_t tid) {
    const size_t item = tid / P.groups;
    const uint32_t g = (uint32_t)(tid % P.groups);
    const uint8_t *src = P.raw + item * P.bytes + 3 * g;
    uint8_t *dst = P.text + item * P.chars + 4 * g;
    const uint32_t nb = (P.bytes - 3 * g) < 3 ? (P.bytes - 3 * g) : 3;
    uint32_t x = 0;
    for (uint32_t k = 0; k < nb; k++) x |= (uint32_t)src[k] << (16 - 8 * k);
    for (uint32_t k = 0; k < nb + 1; k++) dst[k] = b64url_char((x >> (18 - 6 * k)) & 63);
}

EG_HD void scalars_from_wide_body(size_t i, const uint8_t *wide, uint8_t *out) {
    uint32_t w[16];
    load32_bytes(w, wide + 64 * i);
    load32_bytes(w + 8, wide + 64 * i + 32);
    sc r;
    sc_from_wide_words(r, w);
    store32_bytes(out + 32 * i, r.v);
}

// out = [a]A + [b]G (mode 0) or [b]G (mode 1): Group::vartime_double_mul_generator / mul_generator
EG_HD void double_mul_body(size_t i, const uint8_t *a, const uint8_t *A, const uint8_t *b, int mode, const uint32_t *tab_g,
                           uint8_t *out, uint8_t *okv) {
    uint32_t w[8];
    sc sa = sc_zero(), sb;
    ge_ext P = ge_identity();
    bool ok = true;
    if (mode == 0) {
        load32_bytes(w, a + 32 * i); ok = sc_from_words(sa, w) && ok;
        load32_bytes(w, A + 32 * i); ok = ge_decode(P, w) && ok;
    }
    load32_bytes(w, b + 32 * i); ok = sc_from_words(sb, w) && ok;
    ge_ext acc = ge_identity();
    if (ok) {
        const uint32_t *ft[1] = {tab_g};
        ge_msm_chain<1, 1>(acc, &P, &sa, ft, &sb);
    }
    ge_encode(w, acc);
    store32_bytes(out + 32 * i, w);
    if (okv) okv[i] = ok ? 1 : 0;
}

// out[c] = sum_p parts[p][c], ciphertext halves independently; tid over (c, half)
EG_HD void ciphertexts_sum_body(size_t tid, const uint8_t *parts, size_t n_parts, size_t n_cts, uint8_t *out, uint32_t *bad) {
    ge_ext acc = ge_identity(), q;
    uint32_t w[8];
    for (size_t p = 0; p < n_parts; p++) {
        load32_bytes(w, parts + (p * n_cts * 2 + tid) * 32);
        if (!ge_decode(q, w)) {
#if defined(__CUDA_ARCH__)
            atomicOr(bad, 1u);
#else
            *bad |= 1u;
#endif
        }
        ge_add(acc, acc, q);
    }
    ge_encode(w, acc);
    store32_bytes(out + 32 * tid, w);
}

}  // namespace eg

// ------------------------------------------------------------------ SumOfSquaresProof / share proofs / dlog table

namespace eg {

// SumOfSquaresProof::verify transcript (mul.rs:205-258).  prefix = Transcript::new(label) + start_proof("sum_of_squares")
// + "K".  Per item: n ciphertexts (input encodings), commitments (planar, from the msm kernel), the sum ciphertext.
struct sumsq_final_params {
    in_bufs in;
    size_t n;
    uint32_t n_cts;
    uint32_t ct_enc_index[EG_MSM_MAXV];   // planar enc of R_x; X at +1
    uint32_t sum_enc_index;               // planar enc of R_z; Z at +1
    uint32_t commit_index;                // [e_r]G_i at +2i, [e_x]G+[e_r]K_i at +2i+1, then the two sums at +2n, +2n+1
    uint8_t proof_buf;
    uint32_t c_offset;
    transcript prefix;
    const uint32_t *enc;
    const uint32_t *commit;
    uint32_t *result;
};

EG_HD void sumsq_final_body(const sumsq_final_params &P, size_t item) {
    transcript t = P.prefix;
    uint32_t w[8];
#pragma unroll 1
    for (uint32_t i = 0; i < P.n_cts; i++) {
        planar_load_words(w, P.enc, P.n, P.ct_enc_index[i], 8, item);
        merlin_append_words(t, EG_LBL("R_x"), w, 8);
        planar_load_words(w, P.enc, P.n, P.ct_enc_index[i] + 1, 8, item);
        merlin_append_words(t, EG_LBL("X"), w, 8);
        planar_load_words(w, P.commit, P.n, P.commit_index + 2 * i, 8, item);
        merlin_append_words(t, EG_LBL("[e_r]G"), w, 8);
        planar_load_words(w, P.commit, P.n, P.commit_index + 2 * i + 1, 8, item);
        merlin_append_words(t, EG_LBL("[e_x]G + [e_r]K"), w, 8);
    }
    planar_load_words(w, P.enc, P.n, P.sum_enc_index, 8, item);
    merlin_append_words(t, EG_LBL("R_z"), w, 8);
    planar_load_words(w, P.enc, P.n, P.sum_enc_index + 1, 8, item);
    merlin_append_words(t, EG_LBL("Z"), w, 8);
    planar_load_words(w, P.commit, P.n, P.commit_index + 2 * P.n_cts, 8, item);
    merlin_append_words(t, EG_LBL("[e_x]R_x + [e_z]G"), w, 8);
    planar_load_words(w, P.commit, P.n, P.commit_index + 2 * P.n_cts + 1, 8, item);
    merlin_append_words(t, EG_LBL("[e_x]X + [e_z]K"), w, 8);
    sc c, cc;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    load32_bytes(w, in_ptr(P.in, P.proof_buf, item) + P.c_offset);
    bool ok = sc_from_words(cc, w);
    P.result[item] = (ok && sc_eq(c, cc)) ? 1u : 0u;
}

// PublicKeySet::verify_share transcript tail (key_set.rs:216-226 -> log_equality.rs:167-173).
// prefix[j] = Transcript::new("elgamal_decryption_share") + commit(n, t, shared key) + "i" = indexes[j].
// The log base is the ciphertext's random element: "K" = enc(R) (PublicKey::from_element, keys/mod.rs:178-185).
struct share_final_params {
    in_bufs in;
    size_t n;                   // tallies
    uint32_t n_shares;
    uint32_t r_enc_index;       // planar enc(R)
    uint32_t share_enc_index0;  // planar enc of share j at +j
    uint32_t commit_index0;     // [x]G_j at +2j, [x]K_j at +2j+1
    uint8_t proof_buf;          // proofs: item stride n_shares*64, share j at 64j: c | s
    transcript prefix[8];
    uint32_t key_words[8][8];   // participant key encodings (constant per j)
    const uint32_t *enc;
    const uint32_t *commit;
    uint32_t *result;           // n * n_shares
};

EG_HD void share_final_body(const share_final_params &P, size_t item, int j) {
    transcript t = P.prefix[j];
    uint32_t w[8];
    merlin_append_message(t, EG_LBL("dom-sep"), (const uint8_t *)"log_eq", 6);
    planar_load_words(w, P.enc, P.n, P.r_enc_index, 8, item);
    merlin_append_words(t, EG_LBL("K"), w, 8);
    merlin_append_words(t, EG_LBL("[r]G"), P.key_words[j], 8);
    planar_load_words(w, P.enc, P.n, P.share_enc_index0 + j, 8, item);
    merlin_append_words(t, EG_LBL("[r]K"), w, 8);
    planar_load_words(w, P.commit, P.n, P.commit_index0 + 2 * j, 8, item);
    merlin_append_words(t, EG_LBL("[x]G"), w, 8);
    planar_load_words(w, P.commit, P.n, P.commit_index0 + 2 * j + 1, 8, item);
    merlin_append_words(t, EG_LBL("[x]K"), w, 8);
    sc c, cc;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    load32_bytes(w, in_ptr(P.in, P.proof_buf, item) + 64 * j);
    bool ok = sc_from_words(cc, w);
    P.result[item * P.n_shares + j] = (ok && sc_eq(c, cc)) ? 1u : 0u;
}

// DiscreteLogTable (encryption.rs:260-298) as an open-addressing table on the device: slot = 8 key words + value.
EG_HD uint64_t dlog_hash(const uint32_t w[8]) {
    uint64_t h = ((uint64_t)w[1] << 32) | w[0];
    h ^= h >> 29; h *= 0xbf58476d1ce4e5b9ULL; h ^= h >> 32;
    return h;
}

// thread t inserts the encodings of [lo + t*per .. lo + (t+1)*per) G: one variable-time [k]G, then additions of G
struct dlog_build_params {
    uint64_t lo, hi, per;
    size_t cap;                 // power of two
    uint32_t *keys;             // cap * 8
    unsigned long long *vals;   // cap, 0 = empty (value 0 is never stored, encryption.rs:270)
};

EG_HD void dlog_build_body(const dlog_build_params &P, size_t tid) {
    uint64_t v0 = P.lo + tid * P.per;
    if (v0 >= P.hi) return;
    uint64_t v1 = P.hi - v0 > P.per ? v0 + P.per : P.hi;      // v0 + per may wrap past 2^64 in the top slice
    ge_ext G = ge_generator(), acc = ge_identity();
    ge_cached cg;
    ge_to_cached(cg, G);
#pragma unroll 1
    for (int bit = 63; bit >= 0; bit--) {
        ge_dbl(acc, acc);
        if ((v0 >> bit) & 1) ge_add(acc, acc, G);
    }
#pragma unroll 1
    for (uint64_t v = v0; v < v1; v++) {
        if (v != 0) {
            uint32_t w[8];
            ge_encode(w, acc);
            size_t slot = (size_t)dlog_hash(w) & (P.cap - 1);
            for (;;) {
#if defined(__CUDA_ARCH__)
                unsigned long long prev = atomicCAS(&P.vals[slot], 0ULL, (unsigned long long)v);
#else
                unsigned long long prev = P.vals[slot];
                if (prev == 0) P.vals[slot] = v;
#endif
                if (prev == 0) { for (int k = 0; k < 8; k++) P.keys[slot * 8 + k] = w[k]; break; }
                slot = (slot + 1) & (P.cap - 1);
            }
        }
        ge_p1p1 t;
        ge_add_cached_p1p1(t, acc, cg, false);
        ge_p1p1_to_ext(acc, t);
    }
}

// lagrange_coefficients (sharing/mod.rs:139-170) of t <= EG_MSM_MAXV distinct participant indexes, each folded with the
// common scale prod_b (i_b + 1):  coeff[a] = scale / ((i_a + 1) prod_{b != a} (i_b - i_a)).  The t denominators share one
// inversion (Montgomery's trick: prefix products, one sc_invert, back-substitution), as the reference's invert_scalars.
// The host's batch constants (lagrange_scaled) and k_combine_select's per-tally coefficients both come from here.
EG_HD void lagrange_scaled_coeffs(uint32_t t, const uint32_t *indexes, sc *coeff) {
    sc scale = sc_from_u64(1), pre[EG_MSM_MAXV];
    for (uint32_t a = 0; a < t; a++) {
        sc e = sc_from_u64((uint64_t)indexes[a] + 1), mag = e;
        sc_mul(scale, scale, e);
        bool sign = false;
        for (uint32_t b = 0; b < t; b++) {
            if (b == a) continue;
            if (indexes[a] > indexes[b]) { sign = !sign; e = sc_from_u64(indexes[a] - indexes[b]); }
            else e = sc_from_u64(indexes[b] - indexes[a]);
            sc_mul(mag, mag, e);
        }
        if (sign) sc_neg(mag, mag);
        coeff[a] = mag;                                     // the denominator, until the back-substitution below
        if (a == 0) pre[0] = mag; else sc_mul(pre[a], pre[a - 1], mag);
    }
    sc inv;
    sc_invert(inv, pre[t - 1]);                             // 1 / (denominator 0 ... denominator a), a = t - 1 first
    for (uint32_t a = t; a-- > 0;) {
        sc d = coeff[a], c;
        if (a > 0) sc_mul(c, inv, pre[a - 1]); else c = inv;     // 1 / denominator a
        sc_mul(inv, inv, d);
        sc_mul(coeff[a], c, scale);     // (sum lambda_j S_j) * scale == sum (lambda_j * scale) S_j
    }
}

// Params::combine_shares (sharing/mod.rs:302-325) on the shares a tallier accepted: tally i has n_shares candidate shares
// (column j from participant indexes[j]) and combines the first t columns, in column order, whose verdict byte is EG_V_OK.
// Their encodings go to a compact row of t shares in `sel`, so that the decode reads no other column, and their Lagrange
// coefficients to the planar scalars `coeff` (k_msm reads them as scalar_src kind 1).  When the selection is columns
// 0 .. t-1 (every tally of a batch without rejected shares) the batch constants `first_coeff` are copied instead.  A tally
// with fewer than t accepted shares (combine_shares returns None) gets identity encodings, zero coefficients and flag bit
// 2u, which dlog_lookup_body turns into found 3.
struct combine_select_params {
    size_t n;
    uint32_t t, n_shares;
    const uint8_t *shares;          // n x n_shares x 32
    const uint8_t *verdicts;        // n x n_shares
    const uint32_t *indexes;        // n_shares distinct participant indexes
    const uint32_t *first_coeff;    // coefficients of columns 0 .. t-1, 8 words each
    uint8_t *sel;                   // n x t x 32
    uint32_t *coeff;                // planar scalars (8 words): t per item
    uint32_t *flags;                // per item; bit 2u = fewer than t accepted shares
};

EG_HD void combine_select_body(const combine_select_params &P, size_t item) {
    uint32_t col[EG_MSM_MAXV], idx[EG_MSM_MAXV], k = 0;
    bool first = true;
    const uint8_t *v = P.verdicts + item * P.n_shares;
    for (uint32_t j = 0; j < P.n_shares && k < P.t; j++)
        if (v[j] == 0) { first = first && j == k; col[k] = j; idx[k] = P.indexes[j]; k++; }
    uint8_t *out = P.sel + item * P.t * 32;
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (k < P.t) {
        for (uint32_t j = 0; j < P.t; j++) {
            store32_bytes(out + 32 * j, zero);
            planar_store_words(P.coeff, P.n, j, 8, item, zero);
        }
        P.flags[item] |= 2u;
        return;
    }
    const uint8_t *row = P.shares + item * P.n_shares * 32;
    uint32_t w[8];
    for (uint32_t j = 0; j < P.t; j++) {
        load32_bytes(w, row + 32 * col[j]);
        store32_bytes(out + 32 * j, w);
    }
    if (first) {
        for (uint32_t j = 0; j < P.t; j++) planar_store_words(P.coeff, P.n, j, 8, item, P.first_coeff + 8 * j);
        return;
    }
    sc c[EG_MSM_MAXV];
    lagrange_scaled_coeffs(P.t, idx, c);
    for (uint32_t j = 0; j < P.t; j++) planar_store_words(P.coeff, P.n, j, 8, item, c[j].v);
}

// decrypt_to_element (decryption.rs:129-131) + DiscreteLogTable::get (encryption.rs:287-297):
// M = B - D (D = recombined share, a planar point), identity -> Some(0), else table probe on the encoding
struct dlog_lookup_params {
    size_t n;
    uint32_t b_p_index, d_p_index;
    const uint32_t *pts;
    size_t cap;
    const uint32_t *keys;
    const unsigned long long *vals;
    const uint32_t *flags;      // 1u: malformed input; 2u: fewer accepted shares than the threshold (k_combine_select)
    unsigned long long *values;
    uint8_t *found;             // 1 found, 0 absent, 2 malformed input, 3 not combined
    uint8_t *enc;               // n * 32 or null: the encoding of M (read by the giant-step walk of a BSGS table)
};

// DiscreteLogTable::get (encryption.rs:287-297) on a non-identity element's encoding `w`: 1 and `value` when present, 0 absent
EG_HD uint8_t dlog_probe(const uint32_t w[8], size_t cap, const uint32_t *keys, const unsigned long long *vals, unsigned long long &value) {
    size_t slot = (size_t)dlog_hash(w) & (cap - 1);
    for (;;) {
        const unsigned long long v = vals[slot];
        if (v == 0) { value = 0; return 0; }
        bool eq = true;
        for (int k = 0; k < 8; k++) eq = eq && (keys[slot * 8 + k] == w[k]);
        if (eq) { value = v; return 1; }
        slot = (slot + 1) & (cap - 1);
    }
}

EG_HD void dlog_lookup_body(const dlog_lookup_params &P, size_t item) {
    // combine_shares returned None before anything was decrypted: 3 wins over 2, and found != 0 keeps the walk away
    if (P.flags[item] & 2u) { P.found[item] = 3; P.values[item] = 0; return; }
    if (P.flags[item] & 1u) { P.found[item] = 2; P.values[item] = 0; return; }
    ge_ext B, D, M;
    planar_load_point(B, P.pts, P.n, P.b_p_index, item);
    planar_load_point(D, P.pts, P.n, P.d_p_index, item);
    ge_sub(M, B, D);
    if (ge_is_identity(M)) { P.found[item] = 1; P.values[item] = 0; return; }
    uint32_t w[8];
    ge_encode(w, M);
    if (P.enc) store32_bytes(P.enc + item * 32, w);
    unsigned long long v = 0;
    P.found[item] = dlog_probe(w, P.cap, P.keys, P.vals, v);
    P.values[item] = v;
}

// DiscreteLogTable::get (encryption.rs:287-297) on caller-supplied element encodings: 2 when the encoding does not decode,
// 1 / 0 for the identity, else the table probe
struct dlog_get_params {
    size_t n;
    const uint8_t *enc;         // n * 32
    size_t cap;
    const uint32_t *keys;
    const unsigned long long *vals;
    unsigned long long *values;
    uint8_t *found;
};

EG_HD void dlog_get_body(const dlog_get_params &P, size_t item) {
    uint32_t w[8];
    load32_bytes(w, P.enc + item * 32);
    ge_ext M;
    unsigned long long v = 0;
    uint8_t f = 1;
    if (!ge_decode(M, w)) f = 2;
    else if (!ge_is_identity(M)) f = dlog_probe(w, P.cap, P.keys, P.vals, v);
    P.found[item] = f;
    P.values[item] = v;
}

// DiscreteLogTable::get over [lo, hi) by baby-step giant-step:the table holds the baby steps [lo, lo + m) and
// v = u + j m (u in [lo, lo + m), j < giants) is found by probing P_j = M - [j m]G.  Giant step 0 is the ordinary probe
// (dlog_lookup_body / decrypt_body); this walk takes the items it left at found 0 (decoded, absent) through j = 1 .. giants - 1.
// Thread (item, seg) walks j in [1 + seg * seg_steps, ...) on the half points Q_j = [1/2] P_j, so a block of
// EG_WALK_BLOCK steps is encoded with one inversion and no square root (ge_double_compress_n: encode(2 Q_j) = encode(P_j)).
// A hit sets found[item] = 1, which the item's other segments poll once per block to stop early.  Only one (u, j) can
// match (v < 2^64 < l), so any thread that finds it may write the result.
#define EG_WALK_BLOCK 8
struct dlog_walk_params {
    size_t n;
    const uint8_t *enc;         // n * 32: encodings of M (items at found != 0 are not read)
    uint8_t *found;             // n: 0 = unresolved so far; set to 1 on a hit
    unsigned long long *values; // n
    uint64_t lo, hi, m, giants; // giants = ceil((hi - lo) / m) >= 2
    uint64_t seg_steps;         // giant steps per thread (a multiple of EG_WALK_BLOCK)
    uint32_t segs;              // threads per item
    size_t cap;
    const uint32_t *keys;
    const unsigned long long *vals;
    const uint32_t *table_g;    // wide fixed-base table of G
    uint32_t step[24];          // -[m/2]G, affine Niels form
};

EG_HD uint8_t dlog_walk_poll(const uint8_t *found, size_t item) { return *(const volatile uint8_t *)(found + item); }

EG_HD void dlog_walk_body(const dlog_walk_params &P, size_t tid) {
    const size_t item = tid % P.n;
    const uint64_t seg = tid / P.n;
    const uint64_t j0 = 1 + seg * P.seg_steps;
    if (j0 >= P.giants || dlog_walk_poll(P.found, item) != 0) return;
    const uint64_t j1 = P.giants - j0 > P.seg_steps ? j0 + P.seg_steps : P.giants;
    uint32_t w[8];
    load32_bytes(w, P.enc + item * 32);
    ge_ext M, H, X, Q;
    ge_decode(M, w);                                            // decoded before (found 0, not 2)
    EG_ALIGN16 ge_cached tbl[8];
    ge_window_table(tbl, M);
    sc half;
    sc_half(half, sc_from_u64(1));
    ge_var_mul(H, tbl, half);                                   // [1/2] M
    sc c;
    sc_half(c, sc_from_u64(j0 * P.m));                          // j0 m < 2^32 * 2^28
    ge_eval_fixed(X, 1, P.table_g, c, P.table_g, c);
    ge_sub(Q, H, X);                                            // Q_j0 = [1/2] (M - [j0 m]G)
    ge_niels step;
    ge_niels_load(step, P.step, 0);
#pragma unroll 1
    for (uint64_t jb = j0; jb < j1; jb += EG_WALK_BLOCK) {
        if (jb != j0 && dlog_walk_poll(P.found, item) != 0) return;
        ge_ext q[EG_WALK_BLOCK];
        uint32_t e[EG_WALK_BLOCK][8];
#pragma unroll 1
        for (int k = 0; k < EG_WALK_BLOCK; k++) {
            q[k] = Q;
            ge_p1p1 t;
            ge_add_niels_p1p1(t, Q, step, false);
            ge_p1p1_to_ext(Q, t);
        }
        ge_double_compress_n<EG_WALK_BLOCK>(e, q);
#pragma unroll 1
        for (int k = 0; k < EG_WALK_BLOCK && jb + k < j1; k++) {
            const uint64_t jm = (jb + k) * P.m;
            bool zero = true;
            for (int i = 0; i < 8; i++) zero = zero && e[k][i] == 0;
            unsigned long long u = 0;
            bool hit;
            if (zero) hit = P.lo == 0;                              // P_j = [0]G: u = 0, never stored in the table
            else hit = dlog_probe(e[k], P.cap, P.keys, P.vals, u) != 0;
            const uint64_t v = (uint64_t)u + jm;
            if (hit && v >= jm && v < P.hi) {                       // v >= jm: u + j m did not pass 2^64
                P.values[item] = v;
#if defined(__CUDA_ARCH__)
                __threadfence();
#endif
                *(volatile uint8_t *)(P.found + item) = 1;
                return;
            }
        }
    }
}

// ------------------------------------------------------------------ decryption side: the talliers' operations
//
// One thread per ciphertext, with the holder's secret key s (a canonical scalar, the same in every lane):
//   EG_DEC_PLAIN  SecretKey::decrypt_to_element (keys/impls.rs:160-177): M = B - [s]R, encoded, then DiscreteLogTable::get
//                 (encryption.rs:287-297) when a table is given.
//   EG_DEC_PROOF  dh = [s]R with a LogEqualityProof over log base R (log_equality.rs:114-143): the share of
//                 ActiveParticipant::decrypt_share (participant.rs:163-185) or VerifiableDecryption::new with a custom key
//                 (decryption.rs:89-111) -- the two differ only in the transcript prefix and the public key, both host-made.
//                 Nonce x = one 64-byte block; [x]G from the wide table of G, [s/2]R and [x/2]R share one window table of R,
//                 the three encodings take one inversion (ge_double_compress_n on the half-scalar points); s = c s + x.
// CT = true (eg_ctx_set_prover_mode 1): the key and the nonce go through ge_var_mul_ct / ge_fixed_adds_ct.
#define EG_DEC_PLAIN 0
#define EG_DEC_PROOF 1

struct decrypt_params {
    size_t n;
    const uint8_t *cts;                  // n * 64
    const uint8_t *wide;                 // EG_DEC_PROOF, caller-supplied blocks: n * 64
    uint8_t *out;                        // n * 32: the element (plain, may be null) / dh (proof)
    uint8_t *proofs;                     // EG_DEC_PROOF: n * 64 = c | s
    unsigned long long *values;          // EG_DEC_PLAIN with a table: n
    uint8_t *flags;                      // n: plain: found (1 / 0 / 2 = does not decode); proof: ok
    uint32_t secret[8];                  // the key, by value (like rand_src's ChaCha seed)
    uint32_t key_words[8];               // EG_DEC_PROOF: encoding of [s]G, "[r]G" of the transcript
    transcript prefix;                   // EG_DEC_PROOF: up to and including start_proof("log_eq")
    size_t cap;                          // EG_DEC_PLAIN: dlog table (keys == null: no table)
    const uint32_t *keys;
    const unsigned long long *vals;
    const uint32_t *table_g;
    rand_src rnd;
};

template <int OP, bool CT>
EG_HD void decrypt_body(const decrypt_params &P, size_t item) {
    uint32_t w[8], w2[8];
    load32_bytes(w, P.cts + item * 64);
    ge_ext R, B;
    bool ok = ge_decode(R, w);
    if (OP == EG_DEC_PLAIN) {
        load32_bytes(w2, P.cts + item * 64 + 32);
        ok = ge_decode(B, w2) && ok;
    }
    if (!ok) {
        for (int k = 0; k < 8; k++) w[k] = 0;
        if (P.out) store32_bytes(P.out + item * 32, w);
        if (OP == EG_DEC_PLAIN) {
            P.flags[item] = 2;
            if (P.values) P.values[item] = 0;
        } else {
            store32_bytes(P.proofs + item * 64, w);
            store32_bytes(P.proofs + item * 64 + 32, w);
            P.flags[item] = 0;
        }
        return;
    }
    EG_ALIGN16 ge_cached tbl[8];
    ge_window_table(tbl, R);
    sc s;
    for (int k = 0; k < 8; k++) s.v[k] = P.secret[k];
    if (OP == EG_DEC_PLAIN) {
        ge_ext D, M;
        if (CT) ge_var_mul_ct(D, tbl, s); else ge_var_mul(D, tbl, s);
        ge_sub(M, B, D);
        ge_encode(w, M);
        if (P.out) store32_bytes(P.out + item * 32, w);
        uint8_t f = 1;
        if (P.keys) {
            unsigned long long v = 0;
            if (!ge_is_identity(M)) f = dlog_probe(w, P.cap, P.keys, P.vals, v);
            P.values[item] = v;
        }
        P.flags[item] = f;
        return;
    }
    uint32_t blk[16], enc[3][8];                             // dh | [x]G | [x]R
    sc x, hs, hx, c, resp;
    rand_block(blk, P.rnd, item, 0, P.wide + item * 64);
    sc_from_wide_words(x, blk);
    sc_half(hs, s);
    sc_half(hx, x);
    ge_ext q[3];
    if (CT) { ge_var_mul_ct(q[0], tbl, hs); ge_var_mul_ct(q[2], tbl, hx); }
    else { ge_var_mul(q[0], tbl, hs); ge_var_mul(q[2], tbl, hx); }
    ge_eval_fixed(q[1], 1, P.table_g, hx, P.table_g, hx, CT);
    ge_double_compress_n<3>(enc, q);
    transcript t = P.prefix;
    merlin_append_words(t, EG_LBL("K"), w, 8);                 // R's own bytes: canonical, as it decoded
    merlin_append_words(t, EG_LBL("[r]G"), P.key_words, 8);
    merlin_append_words(t, EG_LBL("[r]K"), enc[0], 8);
    merlin_append_words(t, EG_LBL("[x]G"), enc[1], 8);
    merlin_append_words(t, EG_LBL("[x]K"), enc[2], 8);
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    sc_muladd(resp, c, s, x);
    store32_bytes(P.out + item * 32, enc[0]);
    store32_bytes(P.proofs + item * 64, c.v);
    store32_bytes(P.proofs + item * 64 + 32, resp.v);
    P.flags[item] = 1;
}

// ------------------------------------------------------------------ proving side: CommitmentEquivalenceProof::new
//
// CommitmentEquivalenceProof::new (commitment.rs:126-196) for a ciphertext (R, B) = ([r]G, [v]G + [r]K) whose value v and
// randomness r the caller holds.  Draws: the commitment blinding b (SecretKey::generate), then the nonces e_r, e_v, e_c.
// Every point is fixed-base: R, B, C = [v]G + [b]H, [e_r]G, [e_v]G + [e_r]K, [e_v]G + [e_c]H; the six encodings share one
// inversion (ge_double_compress_n on the half-scalar points).  R and B are always computed because the transcript absorbs
// them; `cts` only decides whether they are written.  One thread per item.
struct ceq_prove_params {
    size_t n;
    const uint64_t *values;              // n
    const uint8_t *ct_r;                 // n * 32: canonical scalars (validated on the host)
    const uint8_t *wide;                 // caller-supplied blocks: n * 4 * 64
    uint8_t *cts;                        // n * 64 or null
    uint8_t *commitments;                // n * 32
    uint8_t *proofs;                     // n * 128 = c | s_r | s_v | s_c
    uint8_t *blindings;                  // n * 32 (secret)
    transcript prefix;                   // Transcript::new(label) + start_proof("commitment_equivalence") + "K"
    const uint32_t *table_g, *table_k, *table_h;
    rand_src rnd;
};

EG_HD void ceq_prove_body(const ceq_prove_params &P, size_t item) {
    const bool ct = P.rnd.ct != 0;
    uint32_t w[16];
    sc r, b, er, ev, ec, s;
    const sc v = sc_from_u64(P.values[item]);
    load32_bytes(w, P.ct_r + item * 32);
    if (!sc_from_words(r, w)) r = sc_zero();
    const uint8_t *blk = P.wide + item * 4 * 64;
    rand_block(w, P.rnd, item, 0, blk);
    sc_from_wide_words(b, w);
    rand_block(w, P.rnd, item, 1, blk + 64);
    sc_from_wide_words(er, w);
    rand_block(w, P.rnd, item, 2, blk + 128);
    sc_from_wide_words(ev, w);
    rand_block(w, P.rnd, item, 3, blk + 192);
    sc_from_wide_words(ec, w);
    ge_ext q[6];
    {
        sc hr, hv, hb;
        sc_half(hr, r);
        sc_half(hv, v);
        sc_half(hb, b);
        ge_eval_fixed(q[0], 1, P.table_g, hr, P.table_g, hr, ct);          // R = [r]G
        ge_eval_fixed(q[1], 2, P.table_k, hr, P.table_g, hv, ct);          // B = [r]K + [v]G
        ge_eval_fixed(q[2], 2, P.table_h, hb, P.table_g, hv, ct);          // C = [b]H + [v]G
    }
    {
        sc her, hev, hec;
        sc_half(her, er);
        sc_half(hev, ev);
        sc_half(hec, ec);
        ge_eval_fixed(q[3], 1, P.table_g, her, P.table_g, her, ct);        // [e_r]G
        ge_eval_fixed(q[4], 2, P.table_k, her, P.table_g, hev, ct);        // [e_v]G + [e_r]K
        ge_eval_fixed(q[5], 2, P.table_h, hec, P.table_g, hev, ct);        // [e_v]G + [e_c]H
    }
    uint32_t enc[6][8];
    ge_double_compress_n<6>(enc, q);
    transcript t = P.prefix;
    merlin_append_words(t, EG_LBL("R"), enc[0], 8);
    merlin_append_words(t, EG_LBL("B"), enc[1], 8);
    merlin_append_words(t, EG_LBL("C"), enc[2], 8);
    merlin_append_words(t, EG_LBL("[e_r]G"), enc[3], 8);
    merlin_append_words(t, EG_LBL("[e_v]G + [e_r]K"), enc[4], 8);
    merlin_append_words(t, EG_LBL("[e_v]G + [e_c]H"), enc[5], 8);
    sc c;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    uint8_t *out = P.proofs + item * 128;
    store32_bytes(out, c.v);
    sc_muladd(s, c, r, er);
    store32_bytes(out + 32, s.v);
    sc_muladd(s, c, v, ev);
    store32_bytes(out + 64, s.v);
    sc_muladd(s, c, b, ec);
    store32_bytes(out + 96, s.v);
    store32_bytes(P.commitments + item * 32, enc[2]);
    store32_bytes(P.blindings + item * 32, b.v);
    if (P.cts) {
        store32_bytes(P.cts + item * 64, enc[0]);
        store32_bytes(P.cts + item * 64 + 32, enc[1]);
    }
}

// ------------------------------------------------------------------ proving side: Keypair::from + ProofOfPossession::from_keys
//
// possession.rs:93-130 over k key pairs per proof, the public keys derived here ([s_j]G, so a key cannot mismatch its secret).
// One nonce draw x_j per key, in key order.  Phase 0, one thread per (item, key j): encode([s_j]G) into `keys`, encode([x_j]G)
// into planar scratch (index j over n items).  Phase 1, one thread per item: transcript start_proof("multi_pop"), "K" x k,
// "R" x k, challenge c; the responses c s_j + x_j re-draw x_j, so no nonce is ever stored.
struct pop_prove_params {
    size_t n;
    uint32_t k;                          // keys per proof, 1..64
    const uint8_t *secrets;              // n * k * 32: canonical scalars (validated on the host)
    const uint8_t *wide;                 // caller-supplied blocks: n * k * 64
    uint8_t *keys;                       // n * k * 32
    uint8_t *proofs;                     // n * (1 + k) * 32 = c | s_0 .. s_{k-1}
    uint32_t *enc;                       // planar encodings, index j over n items: [x_j]G
    transcript prefix;                   // Transcript::new(label) + start_proof("multi_pop")
    const uint32_t *table_g;
    rand_src rnd;
};

EG_HD void pop_nonce(sc &x, const pop_prove_params &P, size_t item, uint32_t j) {
    uint32_t w[16];
    rand_block(w, P.rnd, item, j, P.wide + (item * P.k + j) * 64);
    sc_from_wide_words(x, w);
}

EG_HD void pop_key_body(const pop_prove_params &P, size_t item, uint32_t j) {
    const bool ct = P.rnd.ct != 0;
    uint32_t w[8], enc[2][8];
    sc s, x, hs, hx;
    load32_bytes(w, P.secrets + (item * P.k + j) * 32);
    if (!sc_from_words(s, w)) s = sc_zero();
    pop_nonce(x, P, item, j);
    sc_half(hs, s);
    sc_half(hx, x);
    ge_ext q[2];
    ge_eval_fixed(q[0], 1, P.table_g, hs, P.table_g, hs, ct);
    ge_eval_fixed(q[1], 1, P.table_g, hx, P.table_g, hx, ct);
    ge_double_compress_n<2>(enc, q);
    store32_bytes(P.keys + (item * P.k + j) * 32, enc[0]);
    planar_store_words(P.enc, P.n, j, 8, item, enc[1]);
}

EG_HD void pop_final_body(const pop_prove_params &P, size_t item) {
    transcript t = P.prefix;
    uint32_t w[8];
#pragma unroll 1
    for (uint32_t j = 0; j < P.k; j++) {
        load32_bytes(w, P.keys + (item * P.k + j) * 32);
        merlin_append_words(t, EG_LBL("K"), w, 8);
    }
#pragma unroll 1
    for (uint32_t j = 0; j < P.k; j++) {
        planar_load_words(w, P.enc, P.n, j, 8, item);
        merlin_append_words(t, EG_LBL("R"), w, 8);
    }
    sc c;
    merlin_challenge_scalar(t, EG_LBL("c"), c);
    uint8_t *out = P.proofs + item * (1 + (size_t)P.k) * 32;
    store32_bytes(out, c.v);
#pragma unroll 1
    for (uint32_t j = 0; j < P.k; j++) {
        sc s, x, resp;
        load32_bytes(w, P.secrets + (item * P.k + j) * 32);
        if (!sc_from_words(s, w)) s = sc_zero();
        pop_nonce(x, P, item, j);
        sc_muladd(resp, c, s, x);
        store32_bytes(out + 32 * (1 + (size_t)j), resp.v);
    }
}

// ------------------------------------------------------------------ SumOfSquaresProof::new on its own: input staging
//
// k_sumsq_prove reads an item's ciphertexts and sum ciphertext from one record (ct_stride apart) and the randomness as
// planar scalars.  One thread per item packs the caller's flat arrays into that shape: records of (m + 1) * 64 B
// (m ciphertexts, then the sum ciphertext), r_i planar over n * m items, r_z planar over n items.
struct sumsq_stage_params {
    size_t n;
    uint32_t m;
    const uint8_t *cts;                  // n * m * 64
    const uint8_t *sum_cts;              // n * 64
    const uint8_t *r;                    // n * m * 32
    const uint8_t *r_sum;                // n * 32
    uint8_t *records;                    // n * (m + 1) * 64
    uint32_t *r_planar;                  // planar scalars over n * m items
    uint32_t *r_sum_planar;              // planar scalars over n items
};

EG_HD void sumsq_stage_body(const sumsq_stage_params &P, size_t item) {
    uint32_t w[8];
    uint8_t *rec = P.records + item * (P.m + 1) * 64;
#pragma unroll 1
    for (uint32_t i = 0; i < P.m; i++) {
        const size_t q = item * P.m + i;
        load32_bytes(w, P.cts + q * 64);
        store32_bytes(rec + 64 * (size_t)i, w);
        load32_bytes(w, P.cts + q * 64 + 32);
        store32_bytes(rec + 64 * (size_t)i + 32, w);
        load32_bytes(w, P.r + q * 32);
        planar_store_words(P.r_planar, P.n * P.m, 0, 8, q, w);
    }
    load32_bytes(w, P.sum_cts + item * 64);
    store32_bytes(rec + 64 * (size_t)P.m, w);
    load32_bytes(w, P.sum_cts + item * 64 + 32);
    store32_bytes(rec + 64 * (size_t)P.m + 32, w);
    load32_bytes(w, P.r_sum + item * 32);
    planar_store_words(P.r_sum_planar, P.n, 0, 8, item, w);
}


// QuadraticVotingBallot::verify precedence (quadratic_voting.rs:291-329): malformed anywhere, then the first failing
// vote range proof (Variant{i}), then the credit range proof, then the sum-of-squares proof.
struct qv_verdict_params {
    size_t n;
    uint32_t options;
    const uint32_t *flags_votes;    // n * options
    const uint32_t *flags_credit;   // n
    const uint32_t *flags_sumsq;    // n
    const uint32_t *res_votes;      // n * options
    const uint32_t *res_credit;     // n
    const uint32_t *res_sumsq;      // n
    uint8_t *verdicts;
};

EG_HD void qv_verdict_body(const qv_verdict_params &P, size_t item) {
    bool bad = (P.flags_credit[item] | P.flags_sumsq[item]) & 1u;
    for (uint32_t i = 0; i < P.options; i++) bad = bad || (P.flags_votes[item * P.options + i] & 1u);
    uint8_t v = 0;
    if (bad) v = 1;
    else {
        for (uint32_t i = 0; i < P.options && v == 0; i++)
            if (!P.res_votes[item * P.options + i]) v = (uint8_t)(16 + i);
        if (v == 0 && !P.res_credit[item]) v = 5;
        if (v == 0 && !P.res_sumsq[item]) v = 6;
    }
    P.verdicts[item] = v;
}

// per (tally, share): malformed ciphertext / share / proof scalars, else the log-equality check
struct share_verdict_params {
    size_t n;
    uint32_t n_shares;
    const uint32_t *flags;          // n * (n_shares + 1): [0] ciphertext, [1 + j] share j
    const uint32_t *result;         // n * n_shares
    uint8_t *verdicts;              // n * n_shares
};

EG_HD void share_verdict_body(const share_verdict_params &P, size_t tid) {
    size_t item = tid / P.n_shares, j = tid % P.n_shares;
    const uint32_t *f = P.flags + item * (P.n_shares + 1);
    uint8_t v = 0;
    if ((f[0] | f[1 + j]) & 1u) v = 1;
    else if (!P.result[tid]) v = 2;
    P.verdicts[tid] = v;
}

}  // namespace eg
