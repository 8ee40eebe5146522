// group_sum.cuh -- kernel bodies of the grouped tally fold (eg_ciphertexts_group_sum): out[g][j] = sum of cts[i][j] over the
// included items i with groups[i] == g.  It is the weighted sum's machinery (weighted_sum.cuh) with unit weights and the
// group as the bucket key: one window (wmax = 1) of B = n_groups buckets, so the key count E = wmax B of the counting sort
// and of the run accumulation is n_groups and their bodies run unchanged.
//
// Per chunk of items:
//   1. gs_decode: for each included item, the range check of its group id (the call-wide P.bad), its count in the group
//      histogram and the decode of its 2 n_cts elements into affine Niels form (ws_decode_niels).  An element that does
//      not decode flags its group (gbad[g]), not the call.
//   2. ws_hist_* / gs_scatter: counting sort of the included items by group; the list holds item indices, never negated.
//   3. ws_accum: the equal-run accumulation, so a group holding every item is added up by a tree.
//   4. gs_add: each non-empty bucket added to its (group, column) running total; the first chunk writes every total, the
//      identity for an empty bucket, so empty groups need no special case.
// After the last chunk gs_emit encodes every (group, column) total, or the identity for a flagged group, and writes ok.
// With unit weights each bucket is the answer: no recoding, bucket reduction or Horner step.  Time depends on the group
// ids and the mask, which are public.
#pragma once

namespace eg {

// gbad: one flag word per group (an included item of the group has an element that does not decode)
EG_HD void gs_decode_body(const ws_params &P, const uint32_t *groups, uint32_t *gbad, size_t i, uint32_t col) {
    if (!ws_included(P, i)) return;
    const uint32_t g = groups[i];
    if (g >= P.B) {
        if (col == 0) ws_set_bad(P.bad);
        return;
    }
    if (col == 0) ws_atomic_add(&P.hist[g], 1);
    if (!ws_decode_niels(P, i, col)) ws_set_bad(gbad + g);
}

EG_HD void gs_scatter_body(const ws_params &P, const uint32_t *groups, size_t i) {
    if (!ws_included(P, i)) return;
    const uint32_t g = groups[i];
    if (g >= P.B) return;
    const uint32_t pos = ws_atomic_add(&P.cursor[g], 1);
    P.list_item[pos] = (uint32_t)(i << 1);
    P.list_key[pos] = g;
}

// running total of (group g, column col): 32 words at (g * cols + col) * 32
EG_HD void gs_add_body(const ws_params &P, uint32_t g, uint32_t col, int first) {
    uint32_t *r = P.running + ((size_t)g * P.cols + col) * 32;
    if (P.hist[g + 1] == P.hist[g]) {
        if (first) ws_store_point(r, ge_identity());
        return;
    }
    ge_ext acc, q;
    ws_load_point(acc, P.buckets + ((size_t)col * P.B + g) * 32);
    if (!first) { ws_load_point(q, r); ge_add(acc, acc, q); }
    ws_store_point(r, acc);
}

// column col of group g (Ciphertext::to_bytes, n_cts ciphertexts per group); the identity when no chunk ran or the group
// is flagged, whose ok byte is then 0
EG_HD void gs_emit_body(const ws_params &P, const uint32_t *gbad, uint32_t g, uint32_t col, int empty, uint8_t *out, uint8_t *ok) {
    const bool bad = gbad[g] != 0;
    const size_t cell = (size_t)g * P.cols + col;
    ge_ext acc = ge_identity();
    if (!empty && !bad) ws_load_point(acc, P.running + cell * 32);
    uint32_t w[8];
    ge_encode(w, acc);
    store32_bytes(out + 32 * cell, w);
    if (col == 0) ok[g] = bad ? 0 : 1;
}

}  // namespace eg
