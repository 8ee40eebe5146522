/*
 * proofs.c -- zero-knowledge proofs of the hot path for the CPU oracle (test infrastructure, see
 * eg_oracle.h): RingProof (src/proofs/ring.rs), LogEqualityProof (src/proofs/log_equality.rs),
 * RangeDecomposition / RangeProof (src/proofs/range.rs), SumOfSquaresProof (src/proofs/mul.rs).
 * Prover sides are included because the reference's golden snapshots (tests/snapshots.rs) pin the
 * prover output byte-for-byte, and because they generate the seeded synthetic workloads.
 */
#include "eg_oracle.h"
#include "proofs_internal.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* ---------------------------------------------------------------- keys */

int eo_pk_from_bytes(eo_pk *pk, const uint8_t b[32]) {           /* keys/mod.rs:161-176 */
    if (!eo_pt_decode(&pk->element, b)) return 1;
    if (eo_pt_is_identity(&pk->element)) return 2;
    memcpy(pk->bytes, b, 32);
    return 0;
}

void eo_pk_from_element(eo_pk *pk, const eo_pt *p) {             /* keys/mod.rs:178-185 */
    pk->element = *p;
    eo_pt_encode(pk->bytes, p);
}

int eo_ct_decode(eo_ct *ct, const uint8_t b[64]) {
    return eo_pt_decode(&ct->R, b) && eo_pt_decode(&ct->B, b + 32);
}

void eo_ct_encode(uint8_t b[64], const eo_ct *ct) {             /* encryption.rs:155-160 */
    eo_pt_encode(b, &ct->R);
    eo_pt_encode(b + 32, &ct->B);
}

void eo_ct_add(eo_ct *r, const eo_ct *a, const eo_ct *b) {      /* encryption.rs:163-172 */
    eo_pt_add(&r->R, &a->R, &b->R);
    eo_pt_add(&r->B, &a->B, &b->B);
}

void eo_ct_sub(eo_ct *r, const eo_ct *a, const eo_ct *b) {      /* encryption.rs:180-189 */
    eo_pt_sub(&r->R, &a->R, &b->R);
    eo_pt_sub(&r->B, &a->B, &b->B);
}

void eo_ct_zero(eo_ct *r) { eo_pt_identity(&r->R); eo_pt_identity(&r->B); }   /* encryption.rs:123-128 */

/* ExtendedCiphertext::new encryption.rs:310-327 */
void eo_ext_ct_new(eo_ct *ct, eo_sc *r_out, const eo_pt *value, const eo_pk *pk, eo_rng *rng) {
    eo_pt dh;
    eo_rng_scalar(rng, r_out);
    eo_pt_mul_generator(&ct->R, r_out);
    eo_pt_mul(&dh, r_out, &pk->element);
    eo_pt_add(&ct->B, value, &dh);
}

/* ---------------------------------------------------------------- LogEqualityProof */

/* log_equality.rs:114-143 */
void eo_logeq_prove(const eo_pk *log_base, const eo_sc *secret, const eo_pt *pow_g, const eo_pt *pow_k,
                    eo_transcript *t, eo_rng *rng, eo_sc *challenge, eo_sc *response) {
    eo_sc x;
    eo_pt xg, xk;
    eo_transcript_start_proof(t, "log_eq");
    eo_transcript_append_message(t, "K", log_base->bytes, 32);
    eo_transcript_append_element(t, "[r]G", pow_g);
    eo_transcript_append_element(t, "[r]K", pow_k);
    eo_rng_scalar(rng, &x);
    eo_pt_mul_generator(&xg, &x);
    eo_pt_mul(&xk, &x, &log_base->element);
    eo_transcript_append_element(t, "[x]G", &xg);
    eo_transcript_append_element(t, "[x]K", &xk);
    eo_transcript_challenge_scalar(t, "c", challenge);
    eo_sc_mul(response, challenge, secret);
    eo_sc_add(response, response, &x);
}

/* log_equality.rs:153-180 */
int eo_logeq_verify(const eo_pk *log_base, const eo_pt *pow_g, const eo_pt *pow_k, eo_transcript *t,
                    const eo_sc *challenge, const eo_sc *response) {
    eo_sc neg_c, expected;
    eo_pt cg, ck;
    eo_sc_neg(&neg_c, challenge);
    eo_pt_double_mul_generator(&cg, &neg_c, pow_g, response);
    eo_sc scalars[2] = {neg_c, *response};
    eo_pt points[2] = {*pow_k, log_base->element};
    eo_pt_multi_mul(&ck, scalars, points, 2);
    eo_transcript_start_proof(t, "log_eq");
    eo_transcript_append_message(t, "K", log_base->bytes, 32);
    eo_transcript_append_element(t, "[r]G", pow_g);
    eo_transcript_append_element(t, "[r]K", pow_k);
    eo_transcript_append_element(t, "[x]G", &cg);
    eo_transcript_append_element(t, "[x]K", &ck);
    eo_transcript_challenge_scalar(t, "c", &expected);
    return eo_sc_eq(&expected, challenge) ? EO_OK : EO_CHALLENGE_MISMATCH;
}

/* ---------------------------------------------------------------- RingProof */

static void ring_transcript_init(eo_transcript *t, const eo_pk *pk) {       /* ring.rs:290-293 */
    eo_transcript_start_proof(t, "multi_ring_enc");
    eo_transcript_append_message(t, "K", pk->bytes, 32);
}

/* RingProofBuilder::new ring.rs:442-457 */
void eo_ring_builder_init(eo_ring_builder *b, const eo_pk *pk, eo_transcript *t, eo_rng *rng, eo_sc *responses) {
    ring_transcript_init(t, pk);
    b->pk = pk; b->transcript = t; b->rng = rng; b->responses = responses;
    b->n_rings = 0; b->used_responses = 0;
}

/* Ring::new ring.rs:54-131 via add_precomputed_value ring.rs:471-492 */
int eo_ring_builder_add_precomputed(eo_ring_builder *b, const eo_ct *ct, const eo_sc *ct_random,
                                    const eo_pt *admissible, size_t n_values, size_t value_index) {
    if (b->n_rings >= EO_MAX_RINGS || n_values == 0 || value_index >= n_values) return -1;
    eo_ring_state *ring = &b->rings[b->n_rings];
    ring->index = b->n_rings;
    ring->admissible = admissible;
    ring->n_values = n_values;
    ring->value_index = value_index;
    ring->ct = *ct;
    ring->discrete_log = *ct_random;
    ring->responses = b->responses + b->used_responses;
    b->used_responses += n_values;
    for (size_t i = 0; i < n_values; i++) eo_sc_from_u64(&ring->responses[i], 0);

    ring->transcript = *b->transcript;
    uint8_t enc[64];
    eo_ct_encode(enc, ct);
    eo_transcript_start_proof(&ring->transcript, "ring_enc");
    eo_transcript_append_message(&ring->transcript, "enc", enc, 64);
    eo_transcript_append_u64(&ring->transcript, "i", ring->index);

    eo_rng_scalar(b->rng, &ring->random_scalar);
    eo_pt c0, c1;
    eo_pt_mul_generator(&c0, &ring->random_scalar);
    eo_pt_mul(&c1, &ring->random_scalar, &b->pk->element);

    for (size_t eq = value_index + 1; eq < n_values; eq++) {
        eo_transcript et = ring->transcript;
        eo_sc challenge, neg_challenge, response;
        eo_transcript_append_u64(&et, "j", (uint64_t)eq - 1);
        eo_transcript_append_element(&et, "R_G", &c0);
        eo_transcript_append_element(&et, "R_K", &c1);
        eo_transcript_challenge_scalar(&et, "c", &challenge);
        eo_rng_scalar(b->rng, &response);
        ring->responses[eq] = response;
        eo_pt dh;
        eo_pt_sub(&dh, &ct->B, &admissible[eq]);
        eo_sc_neg(&neg_challenge, &challenge);
        /* G::mul_generator(&response) - random_element * &challenge */
        eo_pt_double_mul_generator(&c0, &neg_challenge, &ct->R, &response);
        eo_sc scalars[2] = {response, neg_challenge};
        eo_pt points[2] = {b->pk->element, dh};
        eo_pt_multi_mul(&c1, scalars, points, 2);
    }
    ring->terminal[0] = c0;
    ring->terminal[1] = c1;
    b->n_rings++;
    return 0;
}

/* RingProofBuilder::add_value ring.rs:460-469 */
int eo_ring_builder_add_value(eo_ring_builder *b, const eo_pt *admissible, size_t n_values, size_t value_index,
                              eo_ct *ct_out, eo_sc *random_out) {
    if (value_index >= n_values) return -1;
    eo_ext_ct_new(ct_out, random_out, &admissible[value_index], b->pk, b->rng);
    return eo_ring_builder_add_precomputed(b, ct_out, random_out, admissible, n_values, value_index);
}

/* Ring::finalize ring.rs:162-195 */
static void ring_finalize(eo_ring_builder *b, eo_ring_state *ring, const eo_sc *common_challenge) {
    eo_sc challenge = *common_challenge;
    for (size_t eq = 0; eq < ring->value_index; eq++) {
        eo_sc response, neg_challenge;
        eo_rng_scalar(b->rng, &response);
        ring->responses[eq] = response;
        eo_pt dh, c0, c1;
        eo_pt_sub(&dh, &ring->ct.B, &ring->admissible[eq]);
        eo_sc_neg(&neg_challenge, &challenge);
        eo_pt_double_mul_generator(&c0, &neg_challenge, &ring->ct.R, &response);
        eo_sc scalars[2] = {response, neg_challenge};
        eo_pt points[2] = {b->pk->element, dh};
        eo_pt_multi_mul(&c1, scalars, points, 2);
        eo_transcript et = ring->transcript;
        eo_transcript_append_u64(&et, "j", (uint64_t)eq);
        eo_transcript_append_element(&et, "R_G", &c0);
        eo_transcript_append_element(&et, "R_K", &c1);
        eo_transcript_challenge_scalar(&et, "c", &challenge);
    }
    eo_sc s;
    eo_sc_mul(&s, &challenge, &ring->discrete_log);
    eo_sc_add(&s, &s, &ring->random_scalar);
    ring->responses[ring->value_index] = s;
}

/* RingProofBuilder::build ring.rs:495-506 -> Ring::aggregate ring.rs:138-160 */
void eo_ring_builder_build(eo_ring_builder *b, eo_sc *common_challenge) {
    for (size_t i = 0; i < b->n_rings; i++) {
        eo_transcript_append_element(b->transcript, "R_G", &b->rings[i].terminal[0]);
        eo_transcript_append_element(b->transcript, "R_K", &b->rings[i].terminal[1]);
    }
    eo_transcript_challenge_scalar(b->transcript, "c", common_challenge);
    for (size_t i = 0; i < b->n_rings; i++) ring_finalize(b, &b->rings[i], common_challenge);
}

/* RingProof::verify ring.rs:302-374.  admissible[i] points at ring i's values; the length check
 * (ring.rs:310-315) is the caller's (fixed-stride layouts make it an API-level error). */
int eo_ring_verify(const eo_pk *pk, size_t n_rings, const eo_pt *const *admissible, const size_t *ring_sizes,
                   const eo_ct *cts, const eo_sc *common_challenge, const eo_sc *responses, eo_transcript *t) {
    ring_transcript_init(t, pk);
    eo_transcript initial = *t;
    size_t start = 0;
    for (size_t ri = 0; ri < n_rings; ri++) {
        eo_sc challenge = *common_challenge;
        eo_pt c0, c1;
        eo_pt_generator(&c0); eo_pt_generator(&c1);
        eo_transcript rt = initial;
        uint8_t enc[64];
        eo_ct_encode(enc, &cts[ri]);
        eo_transcript_start_proof(&rt, "ring_enc");
        eo_transcript_append_message(&rt, "enc", enc, 64);
        eo_transcript_append_u64(&rt, "i", (uint64_t)ri);
        for (size_t eq = 0; eq < ring_sizes[ri]; eq++) {
            const eo_sc *response = &responses[start + eq];
            eo_pt dh;
            eo_sc neg_challenge;
            eo_pt_sub(&dh, &cts[ri].B, &admissible[ri][eq]);
            eo_sc_neg(&neg_challenge, &challenge);
            eo_pt_double_mul_generator(&c0, &neg_challenge, &cts[ri].R, response);
            eo_sc scalars[2] = {*response, neg_challenge};
            eo_pt points[2] = {pk->element, dh};
            eo_pt_multi_mul(&c1, scalars, points, 2);
            if (eq + 1 < ring_sizes[ri]) {
                eo_transcript et = rt;
                eo_transcript_append_u64(&et, "j", (uint64_t)eq);
                eo_transcript_append_element(&et, "R_G", &c0);
                eo_transcript_append_element(&et, "R_K", &c1);
                eo_transcript_challenge_scalar(&et, "c", &challenge);
            }
        }
        start += ring_sizes[ri];
        eo_transcript_append_element(t, "R_G", &c0);
        eo_transcript_append_element(t, "R_K", &c1);
    }
    eo_sc expected;
    eo_transcript_challenge_scalar(t, "c", &expected);
    return eo_sc_eq(&expected, common_challenge) ? EO_OK : EO_CHALLENGE_MISMATCH;
}

int eo_scalars_decode(eo_sc *out, const uint8_t *bytes, size_t n) {    /* ring.rs:397-414 */
    for (size_t i = 0; i < n; i++)
        if (!eo_sc_from_canonical(&out[i], bytes + 32 * i)) return 0;
    return 1;
}

void eo_scalars_encode(uint8_t *bytes, const eo_sc *in, size_t n) {    /* ring.rs:383-393 */
    for (size_t i = 0; i < n; i++) eo_sc_tobytes(bytes + 32 * i, &in[i]);
}

/* ---------------------------------------------------------------- RangeDecomposition */

typedef struct opt_entry {
    uint64_t upper_bound, optimal_len;
    eo_range decomposition;
    struct opt_entry *next;
} opt_entry;

static uint64_t lower_len_estimate(uint64_t upper_bound) {            /* range.rs:302-305 (std) */
    return (uint64_t)ceil(log2((double)upper_bound) * 3.0);
}

static const opt_entry *optimize(uint64_t upper_bound, opt_entry **memo) {   /* range.rs:238-300 */
    for (opt_entry *e = *memo; e; e = e->next)
        if (e->upper_bound == upper_bound) return e;

    opt_entry *opt = (opt_entry *)calloc(1, sizeof *opt);
    opt->upper_bound = upper_bound;
    opt->optimal_len = upper_bound + 2;
    opt->decomposition.n_rings = 1;                       /* RangeDecomposition::just range.rs:155-161 */
    opt->decomposition.size[0] = upper_bound;
    opt->decomposition.step[0] = 1;

    for (uint64_t first = 2;; first++) {
        if (first + 2 > opt->optimal_len) break;
        uint64_t remaining = upper_bound - first;
        for (uint64_t mult = 2; mult <= first; mult++) {
            if (remaining % mult != 0) continue;
            uint64_t inner_ub = remaining / mult + 1;
            if (inner_ub < 2) break;
            uint64_t best_estimate = first + 2 + lower_len_estimate(inner_ub);
            if (best_estimate > opt->optimal_len) continue;
            const opt_entry *inner = optimize(inner_ub, memo);
            uint64_t cand_len = first + 2 + inner->optimal_len;
            uint32_t cand_rings = 1 + inner->decomposition.n_rings;
            if (cand_len < opt->optimal_len ||
                (cand_len == opt->optimal_len && cand_rings < opt->decomposition.n_rings)) {
                if (cand_rings > EO_MAX_RINGS) continue;
                opt->optimal_len = cand_len;
                /* combine_mul range.rs:163-171 */
                opt->decomposition = inner->decomposition;
                for (uint32_t i = 0; i < opt->decomposition.n_rings; i++) opt->decomposition.step[i] *= mult;
                opt->decomposition.size[opt->decomposition.n_rings] = first;
                opt->decomposition.step[opt->decomposition.n_rings] = 1;
                opt->decomposition.n_rings++;
            }
        }
    }
    opt->next = *memo;
    *memo = opt;
    return opt;
}

int eo_range_optimal(eo_range *out, uint64_t upper_bound) {           /* range.rs:148-153 */
    if (upper_bound < 2) return -1;
    opt_entry *memo = NULL;
    const opt_entry *opt = optimize(upper_bound, &memo);
    *out = opt->decomposition;
    while (memo) { opt_entry *n = memo->next; free(memo); memo = n; }
    return 0;
}

uint64_t eo_range_upper_bound(const eo_range *r) {                    /* range.rs:174-181 */
    uint64_t s = 0;
    for (uint32_t i = 0; i < r->n_rings; i++) s += (r->size[i] - 1) * r->step[i];
    return s + 1;
}

/* upper bound - 1, with the sum taken in 128 bits: from an upper bound of 2^64 on, every u64 value is in the range */
uint64_t eo_range_max_value(const eo_range *r) {
    unsigned __int128 s = 0;
    for (uint32_t i = 0; i < r->n_rings; i++) s += (unsigned __int128)(r->size[i] - 1) * r->step[i];
    return s > UINT64_MAX ? UINT64_MAX : (uint64_t)s;
}

uint64_t eo_range_rings_size(const eo_range *r) {                     /* range.rs:183-186 */
    uint64_t s = 0;
    for (uint32_t i = 0; i < r->n_rings; i++) s += r->size[i];
    return s;
}

size_t eo_range_display(const eo_range *r, char *buf, size_t cap) {   /* range.rs:110-124 */
    size_t off = 0;
    buf[0] = 0;
    for (uint32_t i = 0; i < r->n_rings; i++) {
        if (r->step[i] > 1) off += (size_t)snprintf(buf + off, cap - off, "%llu * ", (unsigned long long)r->step[i]);
        off += (size_t)snprintf(buf + off, cap - off, "0..%llu", (unsigned long long)r->size[i]);
        if (i + 1 < r->n_rings) off += (size_t)snprintf(buf + off, cap - off, " + ");
    }
    return off;
}

/* PreparedRange::new range.rs:341-355 */
int eo_prepared_range_init(eo_prepared_range *pr, const eo_range *range) {
    pr->range = *range;
    size_t total = (size_t)eo_range_rings_size(range);
    pr->values = (eo_pt *)malloc(total * sizeof(eo_pt));
    if (!pr->values) return -1;
    size_t off = 0;
    for (uint32_t i = 0; i < range->n_rings; i++) {
        pr->ring_values[i] = pr->values + off;
        pr->ring_sizes[i] = (size_t)range->size[i];
        for (uint64_t j = 0; j < range->size[i]; j++) {
            eo_sc k;
            eo_sc_from_u64(&k, j * range->step[i]);
            eo_pt_mul_generator(&pr->values[off + j], &k);
        }
        off += (size_t)range->size[i];
    }
    return 0;
}

void eo_prepared_range_free(eo_prepared_range *pr) { free(pr->values); pr->values = NULL; }

/* RangeDecomposition::decompose range.rs:199-210 */
static void range_decompose(const eo_range *r, size_t *indexes, uint64_t value) {
    for (uint32_t i = 0; i < r->n_rings; i++) {
        uint64_t idx = value / r->step[i];
        if (idx > r->size[i] - 1) idx = r->size[i] - 1;
        indexes[i] = (size_t)idx;
        value -= idx * r->step[i];
    }
}

/* RangeProof::from_ciphertext range.rs:482-534 (ciphertext already drawn by RangeProof::new :469) */
int eo_range_prove_prepared(const eo_pk *pk, const eo_prepared_range *pr, uint64_t value, const eo_ct *ct,
                            const eo_sc *ct_random, eo_transcript *t, eo_rng *rng,
                            eo_ct *partial /* n_rings-1 */, eo_sc *common_challenge, eo_sc *responses) {
    const eo_range *range = &pr->range;
    if (value > eo_range_max_value(range)) return -1;
    size_t indexes[EO_MAX_RINGS];
    char display[EO_MAX_RINGS * 48];
    range_decompose(range, indexes, value);
    size_t dlen = eo_range_display(range, display, sizeof display);
    eo_transcript_start_proof(t, "encryption_range_proof");
    eo_transcript_append_message(t, "range", (const uint8_t *)display, dlen);

    eo_ring_builder *b = (eo_ring_builder *)malloc(sizeof *b);
    if (!b) return -1;
    eo_ring_builder_init(b, pk, t, rng, responses);
    eo_ct cumulative;
    eo_sc cumulative_r;
    eo_ct_zero(&cumulative);
    eo_sc_from_u64(&cumulative_r, 0);
    for (uint32_t i = 0; i + 1 < range->n_rings; i++) {
        eo_sc r;
        eo_ring_builder_add_value(b, pr->ring_values[i], pr->ring_sizes[i], indexes[i], &partial[i], &r);
        eo_ct_add(&cumulative, &cumulative, &partial[i]);
        eo_sc_add(&cumulative_r, &cumulative_r, &r);
    }
    eo_ct last;
    eo_sc last_r;
    eo_ct_sub(&last, ct, &cumulative);
    eo_sc_sub(&last_r, ct_random, &cumulative_r);
    uint32_t li = range->n_rings - 1;
    eo_ring_builder_add_precomputed(b, &last, &last_r, pr->ring_values[li], pr->ring_sizes[li], indexes[li]);
    eo_ring_builder_build(b, common_challenge);
    free(b);
    return 0;
}

/* RangeProof::verify range.rs:547-577 */
int eo_range_verify_prepared(const eo_pk *pk, const eo_prepared_range *pr, const eo_ct *ct, const eo_ct *partial,
                             const eo_sc *common_challenge, const eo_sc *responses, eo_transcript *t) {
    const eo_range *range = &pr->range;
    char display[EO_MAX_RINGS * 48];
    size_t dlen = eo_range_display(range, display, sizeof display);
    eo_transcript_start_proof(t, "encryption_range_proof");
    eo_transcript_append_message(t, "range", (const uint8_t *)display, dlen);
    eo_ct cts[EO_MAX_RINGS], sum;
    eo_ct_zero(&sum);
    for (uint32_t i = 0; i + 1 < range->n_rings; i++) {
        eo_ct_add(&sum, &sum, &partial[i]);
        cts[i] = partial[i];
    }
    eo_ct_sub(&cts[range->n_rings - 1], ct, &sum);
    return eo_ring_verify(pk, range->n_rings, (const eo_pt *const *)pr->ring_values, pr->ring_sizes, cts,
                          common_challenge, responses, t);
}

/* byte-level wrappers: RangeProof::new range.rs:462-473 */
int eo_range_prove(const uint8_t pkb[32], const eo_range *range, const char *label, uint64_t value, eo_rng *rng,
                   uint8_t ctb[64], uint8_t sk_r_out[32], uint8_t *partialb, uint8_t *ringb) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    eo_prepared_range pr;
    if (eo_prepared_range_init(&pr, range)) return -1;
    size_t total = (size_t)eo_range_rings_size(range);
    eo_sc *responses = (eo_sc *)malloc(total * sizeof(eo_sc));
    eo_ct partial[EO_MAX_RINGS];
    eo_transcript t;
    eo_transcript_new(&t, label);
    /* CiphertextWithValue::new encryption.rs:403-407 */
    eo_sc v, r, cc;
    eo_pt vg;
    eo_ct ct;
    eo_sc_from_u64(&v, value);
    eo_pt_mul_generator(&vg, &v);
    eo_ext_ct_new(&ct, &r, &vg, &pk, rng);
    int rc = eo_range_prove_prepared(&pk, &pr, value, &ct, &r, &t, rng, partial, &cc, responses);
    if (rc == 0) {
        eo_ct_encode(ctb, &ct);
        if (sk_r_out) eo_sc_tobytes(sk_r_out, &r);
        for (uint32_t i = 0; i + 1 < range->n_rings; i++) eo_ct_encode(partialb + 64 * i, &partial[i]);
        eo_sc_tobytes(ringb, &cc);
        eo_scalars_encode(ringb + 32, responses, total);
    }
    free(responses);
    eo_prepared_range_free(&pr);
    return rc;
}

int eo_range_verify_bytes_prepared(const eo_pk *pk, const eo_prepared_range *pr, const char *label,
                                   const uint8_t ctb[64], const uint8_t *partialb, const uint8_t *ringb) {
    const eo_range *range = &pr->range;
    size_t total = (size_t)eo_range_rings_size(range);
    eo_ct ct, partial[EO_MAX_RINGS];
    eo_sc cc, responses_stack[64], *responses = responses_stack;
    int rc;
    if (total > 64) responses = (eo_sc *)malloc(total * sizeof(eo_sc));
    if (!eo_ct_decode(&ct, ctb)) { rc = EO_MALFORMED; goto done; }
    for (uint32_t i = 0; i + 1 < range->n_rings; i++)
        if (!eo_ct_decode(&partial[i], partialb + 64 * i)) { rc = EO_MALFORMED; goto done; }
    if (!eo_sc_from_canonical(&cc, ringb) || !eo_scalars_decode(responses, ringb + 32, total)) { rc = EO_MALFORMED; goto done; }
    eo_transcript t;
    eo_transcript_new(&t, label);
    rc = eo_range_verify_prepared(pk, pr, &ct, partial, &cc, responses, &t);
done:
    if (responses != responses_stack) free(responses);
    return rc;
}

int eo_range_verify(const uint8_t pkb[32], const eo_range *range, const char *label, const uint8_t ctb[64],
                    const uint8_t *partialb, const uint8_t *ringb) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    eo_prepared_range pr;
    if (eo_prepared_range_init(&pr, range)) return -1;
    int rc = eo_range_verify_bytes_prepared(&pk, &pr, label, ctb, partialb, ringb);
    eo_prepared_range_free(&pr);
    return rc;
}

/* ---------------------------------------------------------------- SumOfSquaresProof */

/* mul.rs:107-181 */
void eo_sumsq_prove_internal(const eo_pk *pk, size_t n, const eo_ct *cts, const eo_sc *values, const eo_sc *randomness,
                             const eo_ct *sum_ct, const eo_sc *sum_randomness, eo_transcript *t, eo_rng *rng,
                             eo_sc *challenge, eo_sc *ct_responses /* 2n */, eo_sc *sum_response) {
    eo_transcript_start_proof(t, "sum_of_squares");
    eo_transcript_append_message(t, "K", pk->bytes, 32);
    eo_sc sum_scalar, sum_random = *sum_randomness;
    eo_rng_scalar(rng, &sum_scalar);
    eo_sc e_r[EO_MAX_TERMS_SUMSQ], e_x[EO_MAX_TERMS_SUMSQ + 1];
    for (size_t i = 0; i < n; i++) {
        eo_transcript_append_element(t, "R_x", &cts[i].R);
        eo_transcript_append_element(t, "X", &cts[i].B);
        eo_rng_scalar(rng, &e_r[i]);
        eo_pt rc, vc, tmp;
        eo_pt_mul_generator(&rc, &e_r[i]);
        eo_transcript_append_element(t, "[e_r]G", &rc);
        eo_rng_scalar(rng, &e_x[i]);
        eo_pt_mul_generator(&vc, &e_x[i]);
        eo_pt_mul(&tmp, &e_r[i], &pk->element);
        eo_pt_add(&vc, &vc, &tmp);
        eo_transcript_append_element(t, "[e_x]G + [e_r]K", &vc);
        eo_sc neg_v, prod;
        eo_sc_neg(&neg_v, &values[i]);
        eo_sc_mul(&prod, &randomness[i], &neg_v);
        eo_sc_add(&sum_random, &sum_random, &prod);
    }
    e_x[n] = sum_scalar;
    eo_pt elems[EO_MAX_TERMS_SUMSQ + 1], rsum, vsum;
    for (size_t i = 0; i < n; i++) elems[i] = cts[i].R;
    eo_pt_generator(&elems[n]);
    eo_pt_multi_mul(&rsum, e_x, elems, n + 1);
    for (size_t i = 0; i < n; i++) elems[i] = cts[i].B;
    elems[n] = pk->element;
    eo_pt_multi_mul(&vsum, e_x, elems, n + 1);
    eo_transcript_append_element(t, "R_z", &sum_ct->R);
    eo_transcript_append_element(t, "Z", &sum_ct->B);
    eo_transcript_append_element(t, "[e_x]R_x + [e_z]G", &rsum);
    eo_transcript_append_element(t, "[e_x]X + [e_z]K", &vsum);
    eo_transcript_challenge_scalar(t, "c", challenge);
    for (size_t i = 0; i < n; i++) {
        eo_sc_mul(&ct_responses[2 * i], challenge, &randomness[i]);
        eo_sc_add(&ct_responses[2 * i], &ct_responses[2 * i], &e_r[i]);
        eo_sc_mul(&ct_responses[2 * i + 1], challenge, &values[i]);
        eo_sc_add(&ct_responses[2 * i + 1], &ct_responses[2 * i + 1], &e_x[i]);
    }
    eo_sc_mul(sum_response, challenge, &sum_random);
    eo_sc_add(sum_response, sum_response, &sum_scalar);
}

/* mul.rs:190-260 */
int eo_sumsq_verify_internal(const eo_pk *pk, size_t n, const eo_ct *cts, const eo_ct *sum_ct, eo_transcript *t,
                             const eo_sc *challenge, const eo_sc *ct_responses, const eo_sc *sum_response) {
    eo_transcript_start_proof(t, "sum_of_squares");
    eo_transcript_append_message(t, "K", pk->bytes, 32);
    eo_sc neg_c;
    eo_sc_neg(&neg_c, challenge);
    eo_pt G;
    eo_pt_generator(&G);
    for (size_t i = 0; i < n; i++) {
        eo_transcript_append_element(t, "R_x", &cts[i].R);
        eo_transcript_append_element(t, "X", &cts[i].B);
        const eo_sc *r_resp = &ct_responses[2 * i], *v_resp = &ct_responses[2 * i + 1];
        eo_pt rc, vc;
        eo_pt_double_mul_generator(&rc, &neg_c, &cts[i].R, r_resp);
        eo_transcript_append_element(t, "[e_r]G", &rc);
        eo_sc scalars[3] = {*v_resp, *r_resp, neg_c};
        eo_pt points[3] = {G, pk->element, cts[i].B};
        eo_pt_multi_mul(&vc, scalars, points, 3);
        eo_transcript_append_element(t, "[e_x]G + [e_r]K", &vc);
    }
    eo_sc scalars[EO_MAX_TERMS_SUMSQ + 2];
    eo_pt elems[EO_MAX_TERMS_SUMSQ + 2], rsum, vsum;
    for (size_t i = 0; i < n; i++) scalars[i] = ct_responses[2 * i + 1];   /* OddItems mul.rs:266 */
    scalars[n] = *sum_response;
    scalars[n + 1] = neg_c;
    for (size_t i = 0; i < n; i++) elems[i] = cts[i].R;
    elems[n] = G; elems[n + 1] = sum_ct->R;
    eo_pt_multi_mul(&rsum, scalars, elems, n + 2);
    for (size_t i = 0; i < n; i++) elems[i] = cts[i].B;
    elems[n] = pk->element; elems[n + 1] = sum_ct->B;
    eo_pt_multi_mul(&vsum, scalars, elems, n + 2);
    eo_transcript_append_element(t, "R_z", &sum_ct->R);
    eo_transcript_append_element(t, "Z", &sum_ct->B);
    eo_transcript_append_element(t, "[e_x]R_x + [e_z]G", &rsum);
    eo_transcript_append_element(t, "[e_x]X + [e_z]K", &vsum);
    eo_sc expected;
    eo_transcript_challenge_scalar(t, "c", &expected);
    return eo_sc_eq(&expected, challenge) ? EO_OK : EO_CHALLENGE_MISMATCH;
}

int eo_sumsq_prove(const uint8_t pkb[32], uint32_t n, const uint8_t *ctsb, const uint8_t *valuesb,
                   const uint8_t *randb, const uint8_t sum_ctb[64], const uint8_t sum_randb[32],
                   const char *label, eo_rng *rng, uint8_t *proof) {
    if (n > EO_MAX_TERMS_SUMSQ) return -1;
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    eo_ct cts[EO_MAX_TERMS_SUMSQ], sum_ct;
    eo_sc values[EO_MAX_TERMS_SUMSQ], rands[EO_MAX_TERMS_SUMSQ], sum_rand;
    for (uint32_t i = 0; i < n; i++) {
        if (!eo_ct_decode(&cts[i], ctsb + 64 * i)) return -1;
        if (!eo_sc_from_canonical(&values[i], valuesb + 32 * i)) return -1;
        if (!eo_sc_from_canonical(&rands[i], randb + 32 * i)) return -1;
    }
    if (!eo_ct_decode(&sum_ct, sum_ctb) || !eo_sc_from_canonical(&sum_rand, sum_randb)) return -1;
    eo_transcript t;
    eo_transcript_new(&t, label);
    eo_sc c, resp[2 * EO_MAX_TERMS_SUMSQ], sr;
    eo_sumsq_prove_internal(&pk, n, cts, values, rands, &sum_ct, &sum_rand, &t, rng, &c, resp, &sr);
    eo_sc_tobytes(proof, &c);
    eo_scalars_encode(proof + 32, resp, 2 * n);
    eo_sc_tobytes(proof + 32 + 64 * n, &sr);
    return 0;
}

int eo_sumsq_verify_bytes(const eo_pk *pk, uint32_t n, const uint8_t *ctsb, const uint8_t sum_ctb[64],
                          const char *label, const uint8_t *proof) {
    if (n > EO_MAX_TERMS_SUMSQ) return -1;
    eo_ct cts[EO_MAX_TERMS_SUMSQ], sum_ct;
    eo_sc c, resp[2 * EO_MAX_TERMS_SUMSQ], sr;
    for (uint32_t i = 0; i < n; i++)
        if (!eo_ct_decode(&cts[i], ctsb + 64 * i)) return EO_MALFORMED;
    if (!eo_ct_decode(&sum_ct, sum_ctb)) return EO_MALFORMED;
    if (!eo_sc_from_canonical(&c, proof) || !eo_scalars_decode(resp, proof + 32, 2 * n) ||
        !eo_sc_from_canonical(&sr, proof + 32 + 64 * n))
        return EO_MALFORMED;
    eo_transcript t;
    eo_transcript_new(&t, label);
    return eo_sumsq_verify_internal(pk, n, cts, &sum_ct, &t, &c, resp, &sr);
}

int eo_sumsq_verify(const uint8_t pkb[32], uint32_t n, const uint8_t *ctsb, const uint8_t sum_ctb[64],
                    const char *label, const uint8_t *proof) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    return eo_sumsq_verify_bytes(&pk, n, ctsb, sum_ctb, label, proof);
}
