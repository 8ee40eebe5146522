// weighted_sum.cuh -- kernel bodies of the weighted tally fold (eg_ciphertexts_weighted_sum): a Pippenger bucket MSM over
// the 2 n_cts point columns of a batch of ciphertexts (R and B of each position), all columns sharing each item's scalar.
//
// Per chunk of items:
//   1. ws_scalars / ws_decode: canonical check and bit length of each included scalar; decode of each included element
//      into affine Niels form (Ristretto decoding yields Z = 1, so every bucket addition below is a mixed addition).
//   2. ws_recode: signed c-bit digits d in (-2^(c-1), 2^(c-1)] over the windows that the chunk's largest scalar needs,
//      and a histogram of (window, |d|).  Zero digits enter no bucket.
//   3. ws_hist_* / ws_scatter: counting sort of the (item, sign) pairs by key = window * 2^(c-1) + |d| - 1.  The sorted
//      list is shared by every column.
//   4. ws_accum: the list cut into equal runs, one thread per (column, run).  A bucket that lies wholly inside a run
//      (not its first or last piece) is stored; the first and last pieces go to a list of partial sums twice as long as
//      the number of runs, which the next level reduces the same way, until the list fits one run.  A bucket shared by
//      many runs (equal weights put every item into one bucket) is so added up by a tree, never by a serial chain.
//   5. ws_reduce / ws_window: sum_b b B_b per (column, window) by running sums over spans of EG_WS_SPAN buckets, then the
//      spans combined with the weights of their first bucket; ws_combine: c doublings per window (Horner), added to the
//      running total of the call; ws_emit: one RFC 9496 encoding per column.
// All arithmetic is variable-time in the scalars (weights are public).  The result is a group element with a canonical
// encoding, so the summation order (atomics in the histogram and the scatter) does not change a byte of it.
#pragma once

namespace eg {

// Window policy: c = floor(log2(chunk items)) - EG_WS_BITS_OFFSET, clamped to [EG_WS_BITS_MIN, EG_WS_BITS_MAX].  The test
// harness uses small constants so that batches of tens to hundreds of items reach every width and several levels of the
// run reduction.
#ifdef EG_HOSTSIM
#define EG_WS_BITS_MIN 2
#define EG_WS_BITS_MAX 5
#define EG_WS_BITS_OFFSET 3
#define EG_WS_RUN 4            // list entries per accumulation thread
#define EG_WS_SPAN 2           // buckets per bucket-reduction thread
#define EG_WS_SEG 4            // histogram entries per scan thread
#else
#define EG_WS_BITS_MIN 4
#define EG_WS_BITS_MAX 13
#define EG_WS_BITS_OFFSET 4
#define EG_WS_RUN 32
#define EG_WS_SPAN 32
#define EG_WS_SEG 256
#endif

struct ws_params {
    const uint8_t *cts;         // ciphertext j of item i: cts + i * item_stride + j * ct_stride
    size_t item_stride, ct_stride;
    const uint8_t *scalars;     // 32 bytes per item
    const uint8_t *verdicts;    // item i is included when verdicts[i] == 0 (EG_V_OK); NULL: every item
    size_t n;                   // items of the chunk
    uint32_t cols;              // 2 n_cts
    uint32_t c, B, wmax, span, S;   // window bits, buckets per window (2^(c-1)), windows of a 253-bit scalar, spans per window
                                    // (the group sum, group_sum.cuh: B = n_groups, wmax = 1)
    size_t lmax, cap;           // list capacity (wmax n), entries per column of each level buffer
    uint32_t *pts;              // planar Niels points: word w of column col of item i at (col * 24 + w) * n + i
    int32_t *digits;            // digit of window w of item i at w * n + i
    uint32_t *hist;             // wmax B + 1: counts, then exclusive offsets ([wmax B] = list length)
    uint32_t *cursor;           // wmax B scatter cursors
    uint32_t *segsum;           // per scan segment
    uint32_t *list_item;        // sorted list: item << 1 | negative
    uint32_t *list_key;
    uint32_t *lvl_key[2];       // partial sums of the run levels: entry e of column col at col * cap + e
    uint32_t *lvl_pts[2];       // 32 words per entry
    uint32_t *buckets;          // bucket key of column col at (col * wmax B + key) * 32
    uint32_t *rsum;             // per (column, window, span): 64 words (weighted sum, plain sum)
    uint32_t *wsum;             // per (column, window): 32 words
    uint32_t *running;          // per column: 32 words, the total over the chunks so far (group sum: per group and column)
    uint32_t *ctl;              // [0] largest bit length of the chunk's included scalars, [1] list length
    uint32_t *bad;              // a non-canonical scalar or an undecodable element in an included item (whole call);
                                // group sum: a group id out of range in an included item
};

EG_HD uint32_t ws_atomic_add(uint32_t *p, uint32_t v) {
#if defined(__CUDA_ARCH__)
    return atomicAdd(p, v);
#else
    const uint32_t o = *p;
    *p = o + v;
    return o;
#endif
}

EG_HD void ws_atomic_max(uint32_t *p, uint32_t v) {
#if defined(__CUDA_ARCH__)
    atomicMax(p, v);
#else
    if (v > *p) *p = v;
#endif
}

EG_HD void ws_set_bad(uint32_t *bad) {
#if defined(__CUDA_ARCH__)
    atomicOr(bad, 1u);
#else
    *bad |= 1u;
#endif
}

EG_HD bool ws_included(const ws_params &P, size_t i) { return !P.verdicts || P.verdicts[i] == 0; }

// windows of c-bit signed digits for scalars of at most `bits` bits: c W > bits, so the top digit takes the last carry
EG_HD uint32_t ws_windows(uint32_t bits, uint32_t c) { return bits == 0 ? 0 : bits / c + 1; }

// length of the list that run level `level` reduces (level 0: the sorted list of `len` entries); 0 once a level fits a run
EG_HD size_t ws_level_len(size_t len, int level) {
    for (int k = 0; k < level; k++) len = len <= EG_WS_RUN ? 0 : 2 * ((len + EG_WS_RUN - 1) / EG_WS_RUN);
    return len;
}

EG_HD void ws_store_point(uint32_t *o, const ge_ext &p) {
    for (int k = 0; k < 8; k++) { o[k] = p.X.v[k]; o[8 + k] = p.Y.v[k]; o[16 + k] = p.Z.v[k]; o[24 + k] = p.T.v[k]; }
}
EG_HD void ws_load_point(ge_ext &p, const uint32_t *o) {
    for (int k = 0; k < 8; k++) { p.X.v[k] = o[k]; p.Y.v[k] = o[8 + k]; p.Z.v[k] = o[16 + k]; p.T.v[k] = o[24 + k]; }
}

// ------------------------------------------------------------------ 1. scalars and elements

EG_HD void ws_scalars_body(const ws_params &P, size_t i) {
    if (!ws_included(P, i)) return;
    uint32_t w[8];
    load32_bytes(w, P.scalars + 32 * i);
    sc s;
    if (!sc_from_words(s, w)) { ws_set_bad(P.bad); return; }
    uint32_t bits = 0;
    for (int k = 7; k >= 0 && bits == 0; k--)
        if (w[k]) { uint32_t b = 0; while (b < 32 && (w[k] >> b)) b++; bits = 32 * (uint32_t)k + b; }
    if (bits) ws_atomic_max(P.ctl, bits);
}

// element col of item i into column col of P.pts; false (nothing stored) when it does not decode
EG_HD bool ws_decode_niels(const ws_params &P, size_t i, uint32_t col) {
    uint32_t w[8];
    load32_bytes(w, P.cts + i * P.item_stride + (size_t)(col >> 1) * P.ct_stride + 32 * (col & 1));
    ge_ext p;
    if (!ge_decode(p, w)) return false;
    fe t;                                           // Z = 1: (y + x, y - x, 2 d x y)
    uint32_t o[24];
    fe_add(t, p.Y, p.X); fe_towords(o, t);
    fe_sub(t, p.Y, p.X); fe_towords(o + 8, t);
    fe_mul(t, p.T, fe_const_2d()); fe_towords(o + 16, t);
    planar_store_words(P.pts, P.n, col, 24, i, o);
    return true;
}

EG_HD void ws_decode_body(const ws_params &P, size_t i, uint32_t col) {
    if (!ws_included(P, i)) return;
    if (!ws_decode_niels(P, i, col)) ws_set_bad(P.bad);
}

// ------------------------------------------------------------------ 2. signed digits and histogram

EG_HD void ws_recode_body(const ws_params &P, size_t i) {
    const uint32_t W = ws_windows(P.ctl[0], P.c);
    uint32_t s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (ws_included(P, i)) {
        load32_bytes(s, P.scalars + 32 * i);
        if (sc_geq_l(s)) for (int k = 0; k < 8; k++) s[k] = 0;
    }
    uint32_t carry = 0;
    for (uint32_t w = 0; w < W; w++) {
        const uint32_t bit = w * P.c, word = bit >> 5, sh = bit & 31;
        uint32_t v = s[word] >> sh;
        if (sh + P.c > 32 && word < 7) v |= s[word + 1] << (32 - sh);
        v = (v & ((1u << P.c) - 1)) + carry;
        int32_t d = (int32_t)v;
        carry = 0;
        if (v > P.B) { d -= (int32_t)(2 * P.B); carry = 1; }
        P.digits[(size_t)w * P.n + i] = d;
        if (d) ws_atomic_add(&P.hist[w * P.B + (uint32_t)(d < 0 ? -d : d) - 1], 1);
    }
}

// ------------------------------------------------------------------ 3. counting sort

EG_HD void ws_hist_sum_body(const ws_params &P, size_t seg) {
    const size_t E = (size_t)P.wmax * P.B, lo = seg * EG_WS_SEG, hi = lo + EG_WS_SEG < E ? lo + EG_WS_SEG : E;
    uint32_t s = 0;
    for (size_t k = lo; k < hi; k++) s += P.hist[k];
    P.segsum[seg] = s;
}

// one thread: exclusive scan of the segment sums; the list length goes to ctl[1] and hist[E]
EG_HD void ws_hist_scan_body(const ws_params &P) {
    const size_t E = (size_t)P.wmax * P.B, nseg = (E + EG_WS_SEG - 1) / EG_WS_SEG;
    uint32_t run = 0;
    for (size_t g = 0; g < nseg; g++) { const uint32_t v = P.segsum[g]; P.segsum[g] = run; run += v; }
    P.ctl[1] = run;
    P.hist[E] = run;
}

EG_HD void ws_hist_offsets_body(const ws_params &P, size_t seg) {
    const size_t E = (size_t)P.wmax * P.B, lo = seg * EG_WS_SEG, hi = lo + EG_WS_SEG < E ? lo + EG_WS_SEG : E;
    uint32_t run = P.segsum[seg];
    for (size_t k = lo; k < hi; k++) { const uint32_t v = P.hist[k]; P.hist[k] = run; P.cursor[k] = run; run += v; }
}

EG_HD void ws_scatter_body(const ws_params &P, uint32_t w, size_t i) {
    if (w >= ws_windows(P.ctl[0], P.c)) return;
    const int32_t d = P.digits[(size_t)w * P.n + i];
    if (d == 0) return;
    const uint32_t key = w * P.B + (uint32_t)(d < 0 ? -d : d) - 1;
    const uint32_t pos = ws_atomic_add(&P.cursor[key], 1);
    P.list_item[pos] = (uint32_t)(i << 1) | (d < 0 ? 1u : 0u);
    P.list_key[pos] = key;
}

// ------------------------------------------------------------------ 4. bucket accumulation in equal runs

// Run t of column col at level `level`: entries [t R, (t + 1) R) of that level's list.  Pieces of one key inside the run
// that are neither its first nor its last piece are whole buckets and are stored; the first and the last piece go to
// entries 2t and 2t + 1 of the next level (a run of one piece sends it with the identity as its last).  The level whose
// list fits one run stores every piece.
template <bool LEVEL0>
EG_HD void ws_accum_body(const ws_params &P, int level, uint32_t col, size_t t) {
    const size_t len = ws_level_len(P.ctl[1], level);
    const size_t a = t * EG_WS_RUN;
    if (a >= len) return;
    const size_t b = a + EG_WS_RUN < len ? a + EG_WS_RUN : len;
    const bool top = len <= EG_WS_RUN;
    const size_t E = (size_t)P.wmax * P.B;
    const uint32_t *in_key = LEVEL0 ? P.list_key : P.lvl_key[(level - 1) & 1] + (size_t)col * P.cap;
    const uint32_t *in_pts = LEVEL0 ? nullptr : P.lvl_pts[(level - 1) & 1] + (size_t)col * P.cap * 32;
    uint32_t *out_key = P.lvl_key[level & 1] + (size_t)col * P.cap;
    uint32_t *out_pts = P.lvl_pts[level & 1] + (size_t)col * P.cap * 32;
    auto flush = [&](uint32_t key, const ge_ext &acc, bool first, bool last) {
        if (top || (!first && !last)) { ws_store_point(P.buckets + ((size_t)col * E + key) * 32, acc); return; }
        if (first) { out_key[2 * t] = key; ws_store_point(out_pts + 2 * t * 32, acc); }
        if (last) {
            out_key[2 * t + 1] = key;
            if (first) ws_store_point(out_pts + (2 * t + 1) * 32, ge_identity());
            else ws_store_point(out_pts + (2 * t + 1) * 32, acc);
        }
    };
    ge_ext acc = ge_identity();
    uint32_t cur = in_key[a];
    bool first = true;
    for (size_t p = a; p < b; p++) {
        const uint32_t key = in_key[p];
        if (key != cur) { flush(cur, acc, first, false); acc = ge_identity(); cur = key; first = false; }
        ge_p1p1 r;
        if (LEVEL0) {
            const uint32_t e = P.list_item[p];
            uint32_t o[24];
            planar_load_words(o, P.pts, P.n, col, 24, e >> 1);
            ge_niels q;
            ge_niels_load(q, o, 0);
            ge_add_niels_p1p1(r, acc, q, (e & 1) != 0);
            ge_p1p1_to_ext(acc, r);
        } else {
            ge_ext q;
            ws_load_point(q, in_pts + p * 32);
            ge_add(acc, acc, q);
        }
    }
    flush(cur, acc, first, true);
}

// ------------------------------------------------------------------ 5. bucket reduction and window combination

// span r of window w of column col: (sum_j (j - lo + 1) B_j, sum_j B_j) over buckets j in [lo, lo + span), by running sums
// from the top
EG_HD void ws_reduce_body(const ws_params &P, uint32_t col, uint32_t w, uint32_t r) {
    if (w >= ws_windows(P.ctl[0], P.c)) return;
    const size_t E = (size_t)P.wmax * P.B;
    const uint32_t lo = r * P.span;
    ge_ext run = ge_identity(), acc = ge_identity(), q;
    bool started = false;
    for (uint32_t j = lo + P.span; j-- > lo;) {
        const uint32_t key = w * P.B + j;
        if (P.hist[key + 1] != P.hist[key]) {
            ws_load_point(q, P.buckets + ((size_t)col * E + key) * 32);
            ge_add(run, run, q);
            started = true;
        }
        if (started) ge_add(acc, acc, run);
    }
    uint32_t *o = P.rsum + (((size_t)col * P.wmax + w) * P.S + r) * 64;
    ws_store_point(o, acc);
    ws_store_point(o + 32, run);
}

// window w of column col: sum over spans of (weighted sum + [lo_r] plain sum), lo_r = r span; sum_r r X_r by running sums,
// then span (a power of two) by doublings
EG_HD void ws_window_body(const ws_params &P, uint32_t col, uint32_t w) {
    if (w >= ws_windows(P.ctl[0], P.c)) return;
    const uint32_t *in = P.rsum + ((size_t)col * P.wmax + w) * P.S * 64;
    ge_ext total = ge_identity(), u = ge_identity(), t = ge_identity(), q;
    for (uint32_t r = P.S; r-- > 0;) {
        ws_load_point(q, in + (size_t)r * 64);
        ge_add(total, total, q);
        if (r == 0) break;
        ws_load_point(q, in + (size_t)r * 64 + 32);
        ge_add(u, u, q);
        ge_add(t, t, u);
    }
    for (uint32_t s = P.span; s > 1; s >>= 1) ge_dbl(t, t);
    ge_add(total, total, t);
    ws_store_point(P.wsum + ((size_t)col * P.wmax + w) * 32, total);
}

// column col: sum_w 2^(c w) W_w (Horner from the top window), added to the running total (first chunk: replaces it)
EG_HD void ws_combine_body(const ws_params &P, uint32_t col, int first) {
    const uint32_t W = ws_windows(P.ctl[0], P.c);
    ge_ext acc = ge_identity(), q;
    for (uint32_t w = W; w-- > 0;) {
        if (w + 1 < W)
            for (uint32_t k = 0; k < P.c; k++) ge_dbl(acc, acc);
        ws_load_point(q, P.wsum + ((size_t)col * P.wmax + w) * 32);
        ge_add(acc, acc, q);
    }
    uint32_t *r = P.running + (size_t)col * 32;
    if (!first) { ws_load_point(q, r); ge_add(acc, acc, q); }
    ws_store_point(r, acc);
}

// column col of the result (Ciphertext::to_bytes: R then B); the identity when no chunk ran or the call is bad
EG_HD void ws_emit_body(const ws_params &P, uint32_t col, int empty, uint8_t *out, uint8_t *ok) {
    const bool bad = *P.bad != 0;
    ge_ext acc = ge_identity();
    if (!empty && !bad) ws_load_point(acc, P.running + (size_t)col * 32);
    uint32_t w[8];
    ge_encode(w, acc);
    store32_bytes(out + 64 * (size_t)(col >> 1) + 32 * (col & 1), w);
    if (col == 0) *ok = bad ? 0 : 1;
}

}  // namespace eg
