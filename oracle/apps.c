/*
 * apps.c -- protocol objects and applications of the hot path for the CPU oracle (test infrastructure,
 * see eg_oracle.h): key/encryption helpers (src/keys/impls.rs, src/encryption.rs), EncryptedChoice
 * (src/app/choice.rs), QuadraticVotingBallot (src/app/quadratic_voting.rs), threshold decryption
 * (src/sharing/ and src/decryption.rs), DiscreteLogTable (src/encryption.rs:260-298), and the threaded
 * batch loops that stand in for the reference's per-ballot `for` loop (examples/voting.rs:189-204).
 */
#include "eg_oracle.h"
#include "proofs_internal.h"
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

void eo_oracle_init(void) {
    eo_pt g;
    eo_sc one;
    eo_sc_from_u64(&one, 1);
    eo_pt_mul_generator(&g, &one);     /* forces constants + basepoint table */
}

/* ---------------------------------------------------------------- keys / plain encryption */

void eo_keypair_generate(eo_rng *rng, uint8_t sk[32], uint8_t pk[32]) {     /* keys/mod.rs:285-291 */
    eo_sc s;
    eo_pt p;
    eo_rng_scalar(rng, &s);
    eo_pt_mul_generator(&p, &s);
    eo_sc_tobytes(sk, &s);
    eo_pt_encode(pk, &p);
}

int eo_encrypt(const uint8_t pkb[32], uint64_t value, eo_rng *rng, uint8_t ctb[64]) {   /* keys/impls.rs:16-23 */
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    eo_sc v, r;
    eo_pt vg;
    eo_ct ct;
    eo_sc_from_u64(&v, value);
    eo_pt_mul_generator(&vg, &v);
    eo_ext_ct_new(&ct, &r, &vg, &pk, rng);
    eo_ct_encode(ctb, &ct);
    return 0;
}

int eo_decrypt_to_element(const uint8_t skb[32], const uint8_t ctb[64], uint8_t out[32]) {  /* keys/impls.rs:160-163 */
    eo_sc sk;
    eo_ct ct;
    if (!eo_sc_from_canonical(&sk, skb) || !eo_ct_decode(&ct, ctb)) return -1;
    eo_pt dh, m;
    eo_pt_mul(&dh, &sk, &ct.R);
    eo_pt_sub(&m, &ct.B, &dh);
    eo_pt_encode(out, &m);
    return 0;
}

/* ---------------------------------------------------------------- zero encryption */

int eo_encrypt_zero(const uint8_t pkb[32], eo_rng *rng, uint8_t ctb[64], uint8_t proof[64]) {   /* keys/impls.rs:31-52 */
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    eo_sc r, c, s;
    eo_ct ct;
    eo_rng_scalar(rng, &r);
    eo_pt_mul_generator(&ct.R, &r);
    eo_pt_mul(&ct.B, &r, &pk.element);
    eo_transcript t;
    eo_transcript_new(&t, "zero_encryption");
    eo_logeq_prove(&pk, &r, &ct.R, &ct.B, &t, rng, &c, &s);
    eo_ct_encode(ctb, &ct);
    eo_sc_tobytes(proof, &c);
    eo_sc_tobytes(proof + 32, &s);
    return 0;
}

static int verify_zero_pk(const eo_pk *pk, const uint8_t ctb[64], const uint8_t proof[64]) {    /* keys/impls.rs:59-69 */
    eo_ct ct;
    eo_sc c, s;
    if (!eo_ct_decode(&ct, ctb)) return EO_MALFORMED;
    if (!eo_sc_from_canonical(&c, proof) || !eo_sc_from_canonical(&s, proof + 32)) return EO_MALFORMED;
    eo_transcript t;
    eo_transcript_new(&t, "zero_encryption");
    return eo_logeq_verify(pk, &ct.R, &ct.B, &t, &c, &s);
}

int eo_verify_zero(const uint8_t pkb[32], const uint8_t ctb[64], const uint8_t proof[64]) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    return verify_zero_pk(&pk, ctb, proof);
}

/* ---------------------------------------------------------------- bool encryption */

static void bool_values(eo_pt v[2]) { eo_pt_identity(&v[0]); eo_pt_generator(&v[1]); }

static int encrypt_bool_pk(const eo_pk *pk, int value, eo_rng *rng, uint8_t ctb[64], uint8_t proof[96]) {  /* keys/impls.rs:77-89 */
    eo_pt admissible[2];
    bool_values(admissible);
    eo_sc responses[2], cc, r;
    eo_ct ct;
    eo_transcript t;
    eo_transcript_new(&t, "bool_encryption");
    eo_ring_builder *b = (eo_ring_builder *)malloc(sizeof *b);
    if (!b) return -1;
    eo_ring_builder_init(b, pk, &t, rng, responses);
    eo_ring_builder_add_value(b, admissible, 2, value ? 1 : 0, &ct, &r);
    eo_ring_builder_build(b, &cc);
    free(b);
    eo_ct_encode(ctb, &ct);
    eo_sc_tobytes(proof, &cc);
    eo_scalars_encode(proof + 32, responses, 2);
    return 0;
}

int eo_encrypt_bool(const uint8_t pkb[32], int value, eo_rng *rng, uint8_t ctb[64], uint8_t proof[96]) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    return encrypt_bool_pk(&pk, value, rng, ctb, proof);
}

static int verify_bool_pk(const eo_pk *pk, const uint8_t ctb[64], const uint8_t proof[96]) {   /* keys/impls.rs:101-113 */
    eo_ct ct;
    eo_sc cc, responses[2];
    if (!eo_ct_decode(&ct, ctb)) return EO_MALFORMED;
    if (!eo_sc_from_canonical(&cc, proof) || !eo_scalars_decode(responses, proof + 32, 2)) return EO_MALFORMED;
    eo_pt admissible[2];
    bool_values(admissible);
    const eo_pt *adm[1] = {admissible};
    size_t sizes[1] = {2};
    eo_transcript t;
    eo_transcript_new(&t, "bool_encryption");
    return eo_ring_verify(pk, 1, adm, sizes, &ct, &cc, responses, &t);
}

int eo_verify_bool(const uint8_t pkb[32], const uint8_t ctb[64], const uint8_t proof[96]) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    return verify_bool_pk(&pk, ctb, proof);
}

/* ---------------------------------------------------------------- EncryptedChoice */

#define EO_MAX_OPTIONS EO_MAX_RINGS

static int choice_new_pk(const eo_pk *pk, uint32_t n, const uint8_t *choices, int single, eo_rng *rng,
                         uint8_t *ctsb, uint8_t *ringb, uint8_t *sumb) {        /* choice.rs:313-349 */
    if (n == 0 || n > EO_MAX_OPTIONS) return -1;
    eo_pt admissible[2];
    bool_values(admissible);
    eo_sc responses[2 * EO_MAX_OPTIONS], cc, rs[EO_MAX_OPTIONS];
    eo_ct cts[EO_MAX_OPTIONS];
    eo_transcript t;
    eo_transcript_new(&t, "encrypted_choice_ranges");
    eo_ring_builder *b = (eo_ring_builder *)malloc(sizeof *b);
    if (!b) return -1;
    eo_ring_builder_init(b, pk, &t, rng, responses);
    for (uint32_t i = 0; i < n; i++)
        eo_ring_builder_add_value(b, admissible, 2, choices[i] ? 1 : 0, &cts[i], &rs[i]);
    eo_ring_builder_build(b, &cc);
    free(b);
    for (uint32_t i = 0; i < n; i++) eo_ct_encode(ctsb + 64 * i, &cts[i]);
    eo_sc_tobytes(ringb, &cc);
    eo_scalars_encode(ringb + 32, responses, 2 * n);
    if (single) {
        /* SingleChoice::prove choice.rs:58-75 */
        eo_ct sum = cts[0];
        eo_sc sum_r = rs[0];
        for (uint32_t i = 1; i < n; i++) { eo_ct_add(&sum, &sum, &cts[i]); eo_sc_add(&sum_r, &sum_r, &rs[i]); }
        eo_pt g, bmg;
        eo_pt_generator(&g);
        eo_pt_sub(&bmg, &sum.B, &g);
        eo_transcript st;
        eo_transcript_new(&st, "choice_encryption_sum");
        eo_sc c, s;
        eo_logeq_prove(pk, &sum_r, &sum.R, &bmg, &st, rng, &c, &s);
        eo_sc_tobytes(sumb, &c);
        eo_sc_tobytes(sumb + 32, &s);
    }
    return 0;
}

int eo_choice_new(const uint8_t pkb[32], uint32_t n, const uint8_t *choices, int single, eo_rng *rng,
                  uint8_t *ctsb, uint8_t *ringb, uint8_t *sumb) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    return choice_new_pk(&pk, n, choices, single, rng, ctsb, ringb, sumb);
}

/* choice.rs:358-380; decoded ciphertexts are returned through cts_out for the tally */
static int choice_verify_pk(const eo_pk *pk, uint32_t n, int single, const uint8_t *ctsb, const uint8_t *ringb,
                            const uint8_t *sumb, eo_ct *cts_out) {
    if (n == 0 || n > EO_MAX_OPTIONS) return -1;
    eo_ct cts_local[EO_MAX_OPTIONS], *cts = cts_out ? cts_out : cts_local;
    eo_sc cc, responses[2 * EO_MAX_OPTIONS], sc, ss;
    for (uint32_t i = 0; i < n; i++)
        if (!eo_ct_decode(&cts[i], ctsb + 64 * i)) return EO_MALFORMED;
    if (!eo_sc_from_canonical(&cc, ringb) || !eo_scalars_decode(responses, ringb + 32, 2 * n)) return EO_MALFORMED;
    if (single && (!eo_sc_from_canonical(&sc, sumb) || !eo_sc_from_canonical(&ss, sumb + 32))) return EO_MALFORMED;

    eo_ct sum = cts[0];
    for (uint32_t i = 1; i < n; i++) eo_ct_add(&sum, &sum, &cts[i]);
    if (single) {
        /* SingleChoice::verify choice.rs:77-95 */
        eo_pt g, bmg;
        eo_pt_generator(&g);
        eo_pt_sub(&bmg, &sum.B, &g);
        eo_transcript st;
        eo_transcript_new(&st, "choice_encryption_sum");
        if (eo_logeq_verify(pk, &sum.R, &bmg, &st, &sc, &ss) != EO_OK) return EO_CHOICE_SUM;
    }
    eo_pt admissible[2];
    bool_values(admissible);
    const eo_pt *adm[EO_MAX_OPTIONS];
    size_t sizes[EO_MAX_OPTIONS];
    for (uint32_t i = 0; i < n; i++) { adm[i] = admissible; sizes[i] = 2; }
    eo_transcript t;
    eo_transcript_new(&t, "encrypted_choice_ranges");
    if (eo_ring_verify(pk, n, adm, sizes, cts, &cc, responses, &t) != EO_OK) return EO_CHOICE_RANGE;
    return EO_OK;
}

int eo_choice_verify(const uint8_t pkb[32], uint32_t n, int single, const uint8_t *ctsb, const uint8_t *ringb,
                     const uint8_t *sumb) {
    eo_pk pk;
    if (eo_pk_from_bytes(&pk, pkb)) return -1;
    return choice_verify_pk(&pk, n, single, ctsb, ringb, sumb, NULL);
}

/* ---------------------------------------------------------------- Quadratic voting */

uint64_t eo_isqrt(uint64_t x) {                                   /* quadratic_voting.rs:127-143 */
    uint64_t root = 0, power_of_4 = 1ULL << 62;
    while (power_of_4 > x) power_of_4 /= 4;
    while (power_of_4 > 0) {
        if (x >= root + power_of_4) { x -= root + power_of_4; root = root / 2 + power_of_4; }
        else root /= 2;
        power_of_4 /= 4;
    }
    return root;
}

int eo_qv_params_new(eo_qv_params *p, uint32_t options, uint64_t credits) {   /* quadratic_voting.rs:63-76 */
    if (options == 0 || credits == 0 || options > EO_MAX_TERMS_SUMSQ) return -1;
    p->options = options;
    p->credits = credits;
    uint64_t max_votes = eo_isqrt(credits);
    if (eo_range_optimal(&p->vote_range, max_votes + 1)) return -1;
    if (eo_range_optimal(&p->credit_range, credits + 1)) return -1;
    return 0;
}

static size_t range_item_size(const eo_range *r) {   /* ct | partial | ring proof */
    return 64 + 64 * (size_t)(r->n_rings - 1) + 32 * (1 + (size_t)eo_range_rings_size(r));
}

size_t eo_qv_ballot_size(const eo_qv_params *p) {
    return p->options * range_item_size(&p->vote_range) + range_item_size(&p->credit_range) +
           32 * (2 * (size_t)p->options + 2);
}

typedef struct {
    eo_pk pk;
    eo_qv_params params;
    eo_prepared_range vote, credit;
} qv_ctx;

static int qv_ctx_init(qv_ctx *c, const uint8_t pkb[32], const eo_qv_params *p) {
    if (eo_pk_from_bytes(&c->pk, pkb)) return -1;
    c->params = *p;
    if (eo_prepared_range_init(&c->vote, &p->vote_range)) return -1;
    if (eo_prepared_range_init(&c->credit, &p->credit_range)) { eo_prepared_range_free(&c->vote); return -1; }
    return 0;
}

static void qv_ctx_free(qv_ctx *c) { eo_prepared_range_free(&c->vote); eo_prepared_range_free(&c->credit); }

/* one `RangeProof::new` (range.rs:462-473) serialised at `out`; returns ciphertext + randomness */
static int qv_range_new(const qv_ctx *c, const eo_prepared_range *pr, const char *label, uint64_t value, eo_rng *rng,
                        uint8_t *out, eo_ct *ct, eo_sc *r) {
    size_t total = (size_t)eo_range_rings_size(&pr->range);
    eo_sc *responses = (eo_sc *)malloc(total * sizeof(eo_sc));
    eo_ct partial[EO_MAX_RINGS];
    eo_sc v, cc;
    eo_pt vg;
    eo_transcript t;
    eo_transcript_new(&t, label);
    eo_sc_from_u64(&v, value);
    eo_pt_mul_generator(&vg, &v);
    eo_ext_ct_new(ct, r, &vg, &c->pk, rng);
    int rc = eo_range_prove_prepared(&c->pk, pr, value, ct, r, &t, rng, partial, &cc, responses);
    if (rc == 0) {
        eo_ct_encode(out, ct);
        uint32_t np = pr->range.n_rings - 1;
        for (uint32_t i = 0; i < np; i++) eo_ct_encode(out + 64 + 64 * i, &partial[i]);
        eo_sc_tobytes(out + 64 + 64 * np, &cc);
        eo_scalars_encode(out + 64 + 64 * np + 32, responses, total);
    }
    free(responses);
    return rc;
}

static int qv_new_ctx(const qv_ctx *c, const uint64_t *votes, eo_rng *rng, uint8_t *ballot) {   /* quadratic_voting.rs:234-284 */
    const uint32_t n = c->params.options;
    eo_ct cts[EO_MAX_TERMS_SUMSQ], credit_ct;
    eo_sc rs[EO_MAX_TERMS_SUMSQ], vals[EO_MAX_TERMS_SUMSQ], credit_r;
    uint64_t credit = 0;
    size_t vsz = range_item_size(&c->params.vote_range), csz = range_item_size(&c->params.credit_range);
    for (uint32_t i = 0; i < n; i++) credit += votes[i] * votes[i];
    for (uint32_t i = 0; i < n; i++) {
        if (qv_range_new(c, &c->vote, "quadratic_voting_variant", votes[i], rng, ballot + vsz * i, &cts[i], &rs[i])) return -1;
        eo_sc_from_u64(&vals[i], votes[i]);
    }
    if (qv_range_new(c, &c->credit, "quadratic_voting_credit_range", credit, rng, ballot + vsz * n, &credit_ct, &credit_r)) return -1;
    eo_transcript t;
    eo_transcript_new(&t, "quadratic_voting_credit_equiv");
    eo_sc ch, resp[2 * EO_MAX_TERMS_SUMSQ], sr;
    eo_sumsq_prove_internal(&c->pk, n, cts, vals, rs, &credit_ct, &credit_r, &t, rng, &ch, resp, &sr);
    uint8_t *p = ballot + vsz * n + csz;
    eo_sc_tobytes(p, &ch);
    eo_scalars_encode(p + 32, resp, 2 * n);
    eo_sc_tobytes(p + 32 + 64 * n, &sr);
    return 0;
}

int eo_qv_new(const uint8_t pkb[32], const eo_qv_params *p, const uint64_t *votes, eo_rng *rng, uint8_t *ballot) {
    qv_ctx c;
    if (qv_ctx_init(&c, pkb, p)) return -1;
    int rc = qv_new_ctx(&c, votes, rng, ballot);
    qv_ctx_free(&c);
    return rc;
}

/* quadratic_voting.rs:291-329.  Every element/scalar of the ballot is deserialised before `verify` can
 * be called in the reference, so MALFORMED anywhere takes precedence over verification errors. */
static int qv_verify_ctx(const qv_ctx *c, const uint8_t *ballot, eo_ct *votes_out) {
    const uint32_t n = c->params.options;
    size_t vsz = range_item_size(&c->params.vote_range), csz = range_item_size(&c->params.credit_range);
    size_t total = eo_qv_ballot_size(&c->params);
    /* deserialisation pass */
    {
        eo_pt tmp;
        eo_sc s;
        for (uint32_t i = 0; i <= n; i++) {
            const eo_range *r = i < n ? &c->params.vote_range : &c->params.credit_range;
            const uint8_t *p = ballot + vsz * i;
            size_t n_pts = 2 * (size_t)r->n_rings, n_sc = 1 + (size_t)eo_range_rings_size(r);
            for (size_t k = 0; k < n_pts; k++) if (!eo_pt_decode(&tmp, p + 32 * k)) return EO_MALFORMED;
            for (size_t k = 0; k < n_sc; k++) if (!eo_sc_from_canonical(&s, p + 32 * (n_pts + k))) return EO_MALFORMED;
        }
        for (const uint8_t *p = ballot + vsz * n + csz; p < ballot + total; p += 32)
            if (!eo_sc_from_canonical(&s, p)) return EO_MALFORMED;
    }
    for (uint32_t i = 0; i < n; i++) {
        const uint8_t *p = ballot + vsz * i;
        int rc = eo_range_verify_bytes_prepared(&c->pk, &c->vote, "quadratic_voting_variant", p, p + 64,
                                                p + 64 + 64 * (c->params.vote_range.n_rings - 1));
        if (rc != EO_OK) return EO_QV_VARIANT_BASE + (int)i;
    }
    {
        const uint8_t *p = ballot + vsz * n;
        int rc = eo_range_verify_bytes_prepared(&c->pk, &c->credit, "quadratic_voting_credit_range", p, p + 64,
                                                p + 64 + 64 * (c->params.credit_range.n_rings - 1));
        if (rc != EO_OK) return EO_QV_CREDIT_RANGE;
    }
    uint8_t ctsb[64 * EO_MAX_TERMS_SUMSQ];
    for (uint32_t i = 0; i < n; i++) memcpy(ctsb + 64 * i, ballot + vsz * i, 64);
    int rc = eo_sumsq_verify_bytes(&c->pk, n, ctsb, ballot + vsz * n, "quadratic_voting_credit_equiv",
                                   ballot + vsz * n + csz);
    if (rc != EO_OK) return EO_QV_CREDIT_EQUIV;
    if (votes_out)
        for (uint32_t i = 0; i < n; i++) eo_ct_decode(&votes_out[i], ballot + vsz * i);
    return EO_OK;
}

int eo_qv_verify(const uint8_t pkb[32], const eo_qv_params *p, const uint8_t *ballot) {
    qv_ctx c;
    if (qv_ctx_init(&c, pkb, p)) return -1;
    int rc = qv_verify_ctx(&c, ballot, NULL);
    qv_ctx_free(&c);
    return rc;
}

/* ---------------------------------------------------------------- threshold decryption */

int eo_dealer_new(uint32_t shares, uint32_t threshold, eo_rng *rng, eo_keyset *ks, uint8_t *secret_shares) {
    /* Dealer::new participant.rs:35-52 (the proof of possession is not on the hot path and not drawn here);
     * secret_share_for_participant participant.rs:69-82; PublicKeySet::new key_set.rs:60-79 */
    if (shares == 0 || shares > 64 || threshold == 0 || threshold > shares) return -1;
    eo_sc poly[64];
    for (uint32_t i = 0; i < threshold; i++) eo_rng_scalar(rng, &poly[i]);
    ks->shares = shares;
    ks->threshold = threshold;
    eo_pt p;
    eo_pt_mul_generator(&p, &poly[0]);
    eo_pt_encode(ks->shared_key, &p);
    for (uint32_t idx = 0; idx < shares; idx++) {
        eo_sc power, val;
        eo_sc_from_u64(&power, idx + 1);
        eo_sc_from_u64(&val, 0);
        for (int k = (int)threshold - 1; k >= 0; k--) {
            eo_sc_mul(&val, &val, &power);
            eo_sc_add(&val, &val, &poly[k]);
        }
        eo_sc_tobytes(secret_shares + 32 * idx, &val);
        eo_pt_mul_generator(&p, &val);
        eo_pt_encode(ks->participant_keys[idx], &p);
    }
    return 0;
}

static void keyset_commit(const eo_keyset *ks, eo_transcript *t) {            /* key_set.rs:167-171 */
    eo_transcript_append_u64(t, "n", ks->shares);
    eo_transcript_append_u64(t, "t", ks->threshold);
    eo_transcript_append_message(t, "K", ks->shared_key, 32);
}

int eo_decrypt_share(const eo_keyset *ks, uint32_t index, const uint8_t secret_share[32], const uint8_t ctb[64],
                     eo_rng *rng, uint8_t share[32], uint8_t proof[64]) {      /* participant.rs:163-185 */
    eo_ct ct;
    eo_sc sk, c, s;
    eo_pt dh, our_key;
    if (index >= ks->shares || !eo_ct_decode(&ct, ctb) || !eo_sc_from_canonical(&sk, secret_share)) return -1;
    if (!eo_pt_decode(&our_key, ks->participant_keys[index])) return -1;
    eo_pt_mul(&dh, &sk, &ct.R);
    eo_transcript t;
    eo_transcript_new(&t, "elgamal_decryption_share");
    keyset_commit(ks, &t);
    eo_transcript_append_u64(&t, "i", index);
    eo_pk base;
    eo_pk_from_element(&base, &ct.R);
    eo_logeq_prove(&base, &sk, &our_key, &dh, &t, rng, &c, &s);
    eo_pt_encode(share, &dh);
    eo_sc_tobytes(proof, &c);
    eo_sc_tobytes(proof + 32, &s);
    return 0;
}

int eo_verify_share(const eo_keyset *ks, uint32_t index, const uint8_t ctb[64], const uint8_t share[32],
                    const uint8_t proof[64]) {                                 /* key_set.rs:209-228 */
    eo_ct ct;
    eo_pt key_share, dh;
    eo_sc c, s;
    if (index >= ks->shares) return -1;
    if (!eo_ct_decode(&ct, ctb) || !eo_pt_decode(&dh, share)) return EO_MALFORMED;   /* decryption.rs:168-177 */
    if (!eo_sc_from_canonical(&c, proof) || !eo_sc_from_canonical(&s, proof + 32)) return EO_MALFORMED;
    if (!eo_pt_decode(&key_share, ks->participant_keys[index])) return -1;
    eo_transcript t;
    eo_transcript_new(&t, "elgamal_decryption_share");
    keyset_commit(ks, &t);
    eo_transcript_append_u64(&t, "i", index);
    eo_pk base;
    eo_pk_from_element(&base, &ct.R);
    return eo_logeq_verify(&base, &key_share, &dh, &t, &c, &s);
}

/* VerifiableDecryption::new with a custom key, decryption.rs:89-111: dh = [sk]R, LogEqualityProof over log base R after
 * start_proof("decryption_with_custom_key") on Transcript::new(label). */
int eo_decryption_prove(const uint8_t secret[32], const char *transcript_label, const uint8_t ctb[64], eo_rng *rng,
                        uint8_t dh_out[32], uint8_t proof[64]) {
    eo_ct ct;
    eo_sc sk, c, s;
    eo_pt dh, key;
    if (!eo_ct_decode(&ct, ctb) || !eo_sc_from_canonical(&sk, secret)) return -1;
    eo_pt_mul_generator(&key, &sk);
    eo_pt_mul(&dh, &sk, &ct.R);
    eo_transcript t;
    eo_transcript_new(&t, transcript_label);
    eo_transcript_start_proof(&t, "decryption_with_custom_key");
    eo_pk base;
    eo_pk_from_element(&base, &ct.R);
    eo_logeq_prove(&base, &sk, &key, &dh, &t, rng, &c, &s);
    eo_pt_encode(dh_out, &dh);
    eo_sc_tobytes(proof, &c);
    eo_sc_tobytes(proof + 32, &s);
    return 0;
}

/* CandidateDecryption::from_bytes + ::verify, decryption.rs:168-205 */
int eo_decryption_verify(const uint8_t key[32], const char *transcript_label, const uint8_t ctb[64], const uint8_t dh_in[32],
                         const uint8_t proof[64]) {
    eo_ct ct;
    eo_pt k, dh;
    eo_sc c, s;
    if (!eo_pt_decode(&k, key)) return -1;
    if (!eo_ct_decode(&ct, ctb) || !eo_pt_decode(&dh, dh_in)) return EO_MALFORMED;
    if (!eo_sc_from_canonical(&c, proof) || !eo_sc_from_canonical(&s, proof + 32)) return EO_MALFORMED;
    eo_transcript t;
    eo_transcript_new(&t, transcript_label);
    eo_transcript_start_proof(&t, "decryption_with_custom_key");
    eo_pk base;
    eo_pk_from_element(&base, &ct.R);
    return eo_logeq_verify(&base, &k, &dh, &t, &c, &s);
}

static void lagrange(const uint32_t *indexes, uint32_t t, eo_sc *coeffs, eo_sc *scale) {   /* sharing/mod.rs:139-170 */
    for (uint32_t a = 0; a < t; a++) {
        int sign = 0;
        eo_sc mag, e;
        eo_sc_from_u64(&mag, 1);
        for (uint32_t b = 0; b < t; b++) {
            if (indexes[a] > indexes[b]) { sign ^= 1; eo_sc_from_u64(&e, indexes[a] - indexes[b]); }
            else if (indexes[a] < indexes[b]) eo_sc_from_u64(&e, indexes[b] - indexes[a]);
            else eo_sc_from_u64(&e, (uint64_t)indexes[a] + 1);
            eo_sc_mul(&mag, &mag, &e);
        }
        if (sign) eo_sc_neg(&mag, &mag);
        eo_sc_invert(&coeffs[a], &mag);
    }
    eo_sc_from_u64(scale, 1);
    for (uint32_t a = 0; a < t; a++) {
        eo_sc e;
        eo_sc_from_u64(&e, (uint64_t)indexes[a] + 1);
        eo_sc_mul(scale, scale, &e);
    }
}

void eo_lagrange_coefficients(const uint32_t *indexes, uint32_t t, uint8_t *coeffs, uint8_t scaleb[32]) {
    eo_sc c[64], scale;
    lagrange(indexes, t, c, &scale);
    eo_scalars_encode(coeffs, c, t);
    eo_sc_tobytes(scaleb, &scale);
}

int eo_combine_decrypt(uint32_t t, const uint32_t *indexes, const uint8_t *sharesb, const uint8_t ctb[64],
                       uint8_t out_element[32]) {
    /* Params::combine_shares sharing/mod.rs:302-325, then decrypt_to_element decryption.rs:129-131 */
    if (t == 0 || t > 16) return -1;
    eo_sc coeffs[16], scale;
    eo_pt shares[16], restored, dh, m;
    eo_ct ct;
    if (!eo_ct_decode(&ct, ctb)) return 1;
    for (uint32_t i = 0; i < t; i++)
        if (!eo_pt_decode(&shares[i], sharesb + 32 * i)) return 1;
    lagrange(indexes, t, coeffs, &scale);
    eo_pt_multi_mul(&restored, coeffs, shares, t);
    eo_pt_mul(&dh, &scale, &restored);
    eo_pt_sub(&m, &ct.B, &dh);
    eo_pt_encode(out_element, &m);
    return 0;
}

/* ---------------------------------------------------------------- DiscreteLogTable */

struct eo_dlog_table {
    size_t cap;            /* power of two */
    uint8_t *keys;         /* cap * 32 */
    uint64_t *vals;        /* cap; 0 = empty (value 0 is never stored, encryption.rs:270) */
};

static uint64_t key_hash(const uint8_t k[32]) {
    uint64_t h = 0;
    for (int i = 0; i < 8; i++) h |= (uint64_t)k[i] << (8 * i);
    h ^= h >> 29; h *= 0xbf58476d1ce4e5b9ULL; h ^= h >> 32;
    return h;
}

eo_dlog_table *eo_dlog_table_new(uint64_t lo, uint64_t hi) {     /* encryption.rs:267-284 */
    if (hi < lo) return NULL;
    eo_dlog_table *t = (eo_dlog_table *)calloc(1, sizeof *t);
    size_t n = (size_t)(hi - lo), cap = 16;
    while (cap < 2 * n + 2) cap <<= 1;
    t->cap = cap;
    t->keys = (uint8_t *)calloc(cap, 32);
    t->vals = (uint64_t *)calloc(cap, 8);
    eo_pt cur, g;
    eo_sc s;
    eo_pt_generator(&g);
    eo_sc_from_u64(&s, lo);
    eo_pt_mul_generator(&cur, &s);
    for (uint64_t v = lo; v < hi; v++) {
        if (v != 0) {
            uint8_t key[32];
            eo_pt_encode(key, &cur);
            size_t slot = (size_t)key_hash(key) & (cap - 1);
            while (t->vals[slot]) slot = (slot + 1) & (cap - 1);
            memcpy(t->keys + 32 * slot, key, 32);
            t->vals[slot] = v;
        }
        eo_pt_add(&cur, &cur, &g);
    }
    return t;
}

void eo_dlog_table_free(eo_dlog_table *t) {
    if (!t) return;
    free(t->keys); free(t->vals); free(t);
}

int eo_dlog_table_get(const eo_dlog_table *t, const uint8_t element[32], uint64_t *value) {   /* encryption.rs:287-297 */
    eo_pt p;
    if (!eo_pt_decode(&p, element)) return -1;
    if (eo_pt_is_identity(&p)) { *value = 0; return 1; }
    size_t slot = (size_t)key_hash(element) & (t->cap - 1);
    while (t->vals[slot]) {
        if (memcmp(t->keys + 32 * slot, element, 32) == 0) { *value = t->vals[slot]; return 1; }
        slot = (slot + 1) & (t->cap - 1);
    }
    return 0;
}

/* ---------------------------------------------------------------- threaded batch loops */

int eo_hw_threads(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}

typedef void (*item_fn)(void *ctx, size_t i);

typedef struct { item_fn fn; void *ctx; size_t lo, hi; } worker_arg;

static void *worker(void *p) {
    worker_arg *a = (worker_arg *)p;
    for (size_t i = a->lo; i < a->hi; i++) a->fn(a->ctx, i);
    return NULL;
}

static void parallel_for(item_fn fn, void *ctx, size_t n, int threads) {
    eo_oracle_init();
    if (threads <= 0) threads = eo_hw_threads();
    if ((size_t)threads > n) threads = n ? (int)n : 1;
    if (threads == 1) { for (size_t i = 0; i < n; i++) fn(ctx, i); return; }
    pthread_t *tid = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    worker_arg *args = (worker_arg *)malloc(sizeof(worker_arg) * (size_t)threads);
    for (int t = 0; t < threads; t++) {
        args[t].fn = fn; args[t].ctx = ctx;
        args[t].lo = n * (size_t)t / (size_t)threads;
        args[t].hi = n * (size_t)(t + 1) / (size_t)threads;
        pthread_create(&tid[t], NULL, worker, &args[t]);
    }
    for (int t = 0; t < threads; t++) pthread_join(tid[t], NULL);
    free(tid); free(args);
}

static void item_rng(eo_rng *rng, const uint8_t seed[32], size_t index) {
    eo_rng_from_seed(rng, seed, (uint64_t)index << 20);
}

/* --- bool */
typedef struct { eo_pk pk; const uint8_t *seed; size_t first; uint8_t *cts, *proofs; const uint8_t *ccts, *cproofs; uint8_t *verdicts; } bool_ctx;

static void gen_bool_item(void *p, size_t i) {
    bool_ctx *c = (bool_ctx *)p;
    eo_rng rng;
    item_rng(&rng, c->seed, c->first + i);
    encrypt_bool_pk(&c->pk, (int)((c->first + i) & 1), &rng, c->cts + 64 * i, c->proofs + 96 * i);
}

int eo_gen_bool_batch(const uint8_t pkb[32], const uint8_t seed[32], size_t first, size_t n, uint8_t *cts,
                      uint8_t *proofs, int threads) {
    bool_ctx c;
    if (eo_pk_from_bytes(&c.pk, pkb)) return -1;
    c.seed = seed; c.first = first; c.cts = cts; c.proofs = proofs;
    parallel_for(gen_bool_item, &c, n, threads);
    return 0;
}

static void verify_bool_item(void *p, size_t i) {
    bool_ctx *c = (bool_ctx *)p;
    c->verdicts[i] = (uint8_t)verify_bool_pk(&c->pk, c->ccts + 64 * i, c->cproofs + 96 * i);
}

int eo_verify_bool_batch(const uint8_t pkb[32], size_t n, const uint8_t *cts, const uint8_t *proofs,
                         uint8_t *verdicts, int threads) {
    bool_ctx c;
    if (eo_pk_from_bytes(&c.pk, pkb)) return -1;
    c.ccts = cts; c.cproofs = proofs; c.verdicts = verdicts;
    parallel_for(verify_bool_item, &c, n, threads);
    return 0;
}

/* --- choice */
typedef struct {
    eo_pk pk; uint32_t options; int single; const uint8_t *seed; size_t first;
    uint8_t *cts, *rings, *sums; const uint8_t *ccts, *crings, *csums; uint8_t *verdicts;
    size_t n; int threads; eo_ct *partial_tallies; uint8_t *partial_valid;
} choice_ctx;

static void gen_choice_item(void *p, size_t i) {
    choice_ctx *c = (choice_ctx *)p;
    eo_rng rng;
    uint8_t flags[EO_MAX_OPTIONS];
    item_rng(&rng, c->seed, c->first + i);
    for (uint32_t k = 0; k < c->options; k++) flags[k] = ((c->first + i) % c->options) == k;
    choice_new_pk(&c->pk, c->options, flags, 1, &rng, c->cts + 64 * c->options * i,
                  c->rings + 32 * (1 + 2 * c->options) * i, c->sums + 64 * i);
}

int eo_gen_choice_batch(const uint8_t pkb[32], uint32_t options, const uint8_t seed[32], size_t first, size_t n,
                        uint8_t *cts, uint8_t *rings, uint8_t *sums, int threads) {
    choice_ctx c;
    if (options == 0 || options > EO_MAX_OPTIONS) return -1;
    if (eo_pk_from_bytes(&c.pk, pkb)) return -1;
    c.options = options; c.seed = seed; c.first = first; c.cts = cts; c.rings = rings; c.sums = sums;
    parallel_for(gen_choice_item, &c, n, threads);
    return 0;
}

/* chunk worker: verify + fold the verified ciphertexts into a per-chunk tally (examples/voting.rs:200-203) */
static void verify_choice_chunk(void *p, size_t chunk) {
    choice_ctx *c = (choice_ctx *)p;
    size_t lo = c->n * chunk / (size_t)c->threads, hi = c->n * (chunk + 1) / (size_t)c->threads;
    eo_ct *tally = c->partial_tallies + chunk * c->options;
    for (uint32_t k = 0; k < c->options; k++) eo_ct_zero(&tally[k]);
    for (size_t i = lo; i < hi; i++) {
        eo_ct cts[EO_MAX_OPTIONS];
        int v = choice_verify_pk(&c->pk, c->options, c->single, c->ccts + 64 * c->options * i,
                                 c->crings + 32 * (1 + 2 * c->options) * i, c->csums ? c->csums + 64 * i : NULL, cts);
        c->verdicts[i] = (uint8_t)v;
        if (v == EO_OK && c->partial_tallies)
            for (uint32_t k = 0; k < c->options; k++) eo_ct_add(&tally[k], &tally[k], &cts[k]);
    }
}

int eo_verify_choice_batch(const uint8_t pkb[32], uint32_t options, int single, size_t n, const uint8_t *cts,
                           const uint8_t *rings, const uint8_t *sums, uint8_t *verdicts, uint8_t *tallyb, int threads) {
    choice_ctx c;
    if (options == 0 || options > EO_MAX_OPTIONS) return -1;
    if (eo_pk_from_bytes(&c.pk, pkb)) return -1;
    if (threads <= 0) threads = eo_hw_threads();
    if ((size_t)threads > n) threads = n ? (int)n : 1;
    c.options = options; c.single = single; c.ccts = cts; c.crings = rings; c.csums = sums; c.verdicts = verdicts;
    c.n = n; c.threads = threads;
    c.partial_tallies = (eo_ct *)malloc(sizeof(eo_ct) * options * (size_t)threads);
    parallel_for(verify_choice_chunk, &c, (size_t)threads, threads);
    if (tallyb) {
        for (uint32_t k = 0; k < options; k++) {
            eo_ct acc;
            eo_ct_zero(&acc);
            for (int t = 0; t < threads; t++) eo_ct_add(&acc, &acc, &c.partial_tallies[(size_t)t * options + k]);
            eo_ct_encode(tallyb + 64 * k, &acc);
        }
    }
    free(c.partial_tallies);
    return 0;
}

/* --- range */
typedef struct {
    eo_pk pk; eo_prepared_range pr; const char *label; const uint8_t *seed; size_t first; const uint64_t *values;
    uint8_t *cts, *partials, *rings; const uint8_t *ccts, *cpartials, *crings; uint8_t *verdicts;
} range_ctx;

static void gen_range_item(void *p, size_t i) {
    range_ctx *c = (range_ctx *)p;
    const eo_range *r = &c->pr.range;
    size_t total = (size_t)eo_range_rings_size(r), np = r->n_rings - 1;
    eo_rng rng;
    item_rng(&rng, c->seed, c->first + i);
    eo_sc *responses = (eo_sc *)malloc(total * sizeof(eo_sc));
    eo_ct partial[EO_MAX_RINGS], ct;
    eo_sc v, rr, cc;
    eo_pt vg;
    eo_transcript t;
    eo_transcript_new(&t, c->label);
    eo_sc_from_u64(&v, c->values[i]);
    eo_pt_mul_generator(&vg, &v);
    eo_ext_ct_new(&ct, &rr, &vg, &c->pk, &rng);
    eo_range_prove_prepared(&c->pk, &c->pr, c->values[i], &ct, &rr, &t, &rng, partial, &cc, responses);
    eo_ct_encode(c->cts + 64 * i, &ct);
    for (size_t k = 0; k < np; k++) eo_ct_encode(c->partials + 64 * (np * i + k), &partial[k]);
    uint8_t *ring = c->rings + 32 * (1 + total) * i;
    eo_sc_tobytes(ring, &cc);
    eo_scalars_encode(ring + 32, responses, total);
    free(responses);
}

int eo_gen_range_batch(const uint8_t pkb[32], const eo_range *range, const char *label, const uint8_t seed[32],
                       size_t first, size_t n, const uint64_t *values, uint8_t *cts, uint8_t *partials,
                       uint8_t *rings, int threads) {
    range_ctx c;
    if (eo_pk_from_bytes(&c.pk, pkb)) return -1;
    uint64_t max_value = eo_range_max_value(range);
    for (size_t i = 0; i < n; i++) if (values[i] > max_value) return -1;
    if (eo_prepared_range_init(&c.pr, range)) return -1;
    c.label = label; c.seed = seed; c.first = first; c.values = values; c.cts = cts; c.partials = partials; c.rings = rings;
    parallel_for(gen_range_item, &c, n, threads);
    eo_prepared_range_free(&c.pr);
    return 0;
}

static void verify_range_item(void *p, size_t i) {
    range_ctx *c = (range_ctx *)p;
    const eo_range *r = &c->pr.range;
    size_t total = (size_t)eo_range_rings_size(r), np = r->n_rings - 1;
    c->verdicts[i] = (uint8_t)eo_range_verify_bytes_prepared(&c->pk, &c->pr, c->label, c->ccts + 64 * i,
                                                            c->cpartials + 64 * np * i, c->crings + 32 * (1 + total) * i);
}

int eo_verify_range_batch(const uint8_t pkb[32], const eo_range *range, const char *label, size_t n,
                          const uint8_t *cts, const uint8_t *partials, const uint8_t *rings, uint8_t *verdicts, int threads) {
    range_ctx c;
    if (eo_pk_from_bytes(&c.pk, pkb)) return -1;
    if (eo_prepared_range_init(&c.pr, range)) return -1;
    c.label = label; c.ccts = cts; c.cpartials = partials; c.crings = rings; c.verdicts = verdicts;
    parallel_for(verify_range_item, &c, n, threads);
    eo_prepared_range_free(&c.pr);
    return 0;
}

/* --- quadratic voting */
typedef struct {
    qv_ctx q; const uint8_t *seed; size_t first; const uint64_t *votes; uint8_t *ballots; const uint8_t *cballots;
    uint8_t *verdicts; size_t n; int threads; eo_ct *partial_tallies; size_t bsz;
} qvb_ctx;

static void gen_qv_item(void *p, size_t i) {
    qvb_ctx *c = (qvb_ctx *)p;
    eo_rng rng;
    item_rng(&rng, c->seed, c->first + i);
    qv_new_ctx(&c->q, c->votes + (size_t)c->q.params.options * i, &rng, c->ballots + c->bsz * i);
}

int eo_gen_qv_batch(const uint8_t pkb[32], const eo_qv_params *p, const uint8_t seed[32], size_t first, size_t n,
                    const uint64_t *votes, uint8_t *ballots, int threads) {
    qvb_ctx c;
    if (qv_ctx_init(&c.q, pkb, p)) return -1;
    c.seed = seed; c.first = first; c.votes = votes; c.ballots = ballots; c.bsz = eo_qv_ballot_size(p);
    parallel_for(gen_qv_item, &c, n, threads);
    qv_ctx_free(&c.q);
    return 0;
}

static void verify_qv_chunk(void *p, size_t chunk) {
    qvb_ctx *c = (qvb_ctx *)p;
    const uint32_t options = c->q.params.options;
    size_t lo = c->n * chunk / (size_t)c->threads, hi = c->n * (chunk + 1) / (size_t)c->threads;
    eo_ct *tally = c->partial_tallies + chunk * options;
    for (uint32_t k = 0; k < options; k++) eo_ct_zero(&tally[k]);
    for (size_t i = lo; i < hi; i++) {
        eo_ct votes[EO_MAX_TERMS_SUMSQ];
        int v = qv_verify_ctx(&c->q, c->cballots + c->bsz * i, votes);
        c->verdicts[i] = (uint8_t)v;
        if (v == EO_OK)
            for (uint32_t k = 0; k < options; k++) eo_ct_add(&tally[k], &tally[k], &votes[k]);
    }
}

int eo_verify_qv_batch(const uint8_t pkb[32], const eo_qv_params *p, size_t n, const uint8_t *ballots,
                       uint8_t *verdicts, uint8_t *tallyb, int threads) {
    qvb_ctx c;
    if (qv_ctx_init(&c.q, pkb, p)) return -1;
    if (threads <= 0) threads = eo_hw_threads();
    if ((size_t)threads > n) threads = n ? (int)n : 1;
    c.cballots = ballots; c.verdicts = verdicts; c.n = n; c.threads = threads; c.bsz = eo_qv_ballot_size(p);
    c.partial_tallies = (eo_ct *)malloc(sizeof(eo_ct) * p->options * (size_t)threads);
    parallel_for(verify_qv_chunk, &c, (size_t)threads, threads);
    if (tallyb) {
        for (uint32_t k = 0; k < p->options; k++) {
            eo_ct acc;
            eo_ct_zero(&acc);
            for (int t = 0; t < threads; t++) eo_ct_add(&acc, &acc, &c.partial_tallies[(size_t)t * p->options + k]);
            eo_ct_encode(tallyb + 64 * k, &acc);
        }
    }
    free(c.partial_tallies);
    qv_ctx_free(&c.q);
    return 0;
}

/* ================================================================== CommitmentEquivalenceProof (proofs/commitment.rs)
 * Proof bytes (the reference has serde only; field order of the struct, commitment.rs:126-135):
 *   challenge | randomness_response | value_response | commitment_response  = 128 B.                           */

/* commitment.rs:146-193.  Draw order: e_r, e_v, e_c. */
static void ceq_prove_pk(const eo_pk *pk, const eo_ct *ct, const eo_sc *value, const eo_sc *randomness, const eo_sc *blinding,
                         const eo_pt *h, eo_transcript *t, eo_rng *rng, uint8_t commitment[32], uint8_t proof[128]) {
    eo_pt c, vg, bh, er_g, ev_g, er_k, ec_h, eb, ec;
    eo_pt_mul_generator(&vg, value);
    eo_pt_mul(&bh, blinding, h);
    eo_pt_add(&c, &vg, &bh);
    eo_transcript_start_proof(t, "commitment_equivalence");
    eo_transcript_append_message(t, "K", pk->bytes, 32);
    eo_transcript_append_element(t, "R", &ct->R);
    eo_transcript_append_element(t, "B", &ct->B);
    eo_transcript_append_element(t, "C", &c);
    eo_sc e_r, e_v, e_c, ch, s;
    eo_rng_scalar(rng, &e_r);
    eo_rng_scalar(rng, &e_v);
    eo_rng_scalar(rng, &e_c);
    eo_pt_mul_generator(&er_g, &e_r);
    eo_transcript_append_element(t, "[e_r]G", &er_g);
    eo_pt_mul_generator(&ev_g, &e_v);
    eo_pt_mul(&er_k, &e_r, &pk->element);
    eo_pt_add(&eb, &ev_g, &er_k);
    eo_transcript_append_element(t, "[e_v]G + [e_r]K", &eb);
    eo_pt_mul(&ec_h, &e_c, h);
    eo_pt_add(&ec, &ev_g, &ec_h);
    eo_transcript_append_element(t, "[e_v]G + [e_c]H", &ec);
    eo_transcript_challenge_scalar(t, "c", &ch);
    eo_sc_tobytes(proof, &ch);
    eo_sc_mul(&s, &ch, randomness); eo_sc_add(&s, &s, &e_r); eo_sc_tobytes(proof + 32, &s);
    eo_sc_mul(&s, &ch, value);      eo_sc_add(&s, &s, &e_v); eo_sc_tobytes(proof + 64, &s);
    eo_sc_mul(&s, &ch, blinding);   eo_sc_add(&s, &s, &e_c); eo_sc_tobytes(proof + 96, &s);
    eo_pt_encode(commitment, &c);
}

/* commitment.rs:198-248 */
static int ceq_verify_pk(const eo_pk *pk, const eo_pt *h, const char *label, const uint8_t ctb[64], const uint8_t commitment[32],
                         const uint8_t proof[128]) {
    eo_ct ct;
    eo_pt c;
    eo_sc s[4];
    if (!eo_ct_decode(&ct, ctb) || !eo_pt_decode(&c, commitment)) return EO_MALFORMED;
    if (!eo_scalars_decode(s, proof, 4)) return EO_MALFORMED;
    eo_transcript t;
    eo_transcript_new(&t, label);
    eo_transcript_start_proof(&t, "commitment_equivalence");
    eo_transcript_append_message(&t, "K", pk->bytes, 32);
    eo_transcript_append_element(&t, "R", &ct.R);
    eo_transcript_append_element(&t, "B", &ct.B);
    eo_transcript_append_element(&t, "C", &c);
    eo_sc neg_c, expected;
    eo_sc_neg(&neg_c, &s[0]);
    eo_pt e;
    eo_pt_double_mul_generator(&e, &neg_c, &ct.R, &s[1]);
    eo_transcript_append_element(&t, "[e_r]G", &e);
    eo_pt g;
    eo_sc one;
    eo_sc_from_u64(&one, 1);
    eo_pt_mul_generator(&g, &one);
    eo_sc sc3[3] = {s[2], s[1], neg_c};
    eo_pt pt3[3] = {g, pk->element, ct.B};
    eo_pt_multi_mul(&e, sc3, pt3, 3);
    eo_transcript_append_element(&t, "[e_v]G + [e_r]K", &e);
    eo_sc sc3b[3] = {s[2], s[3], neg_c};
    eo_pt pt3b[3] = {g, *h, c};
    eo_pt_multi_mul(&e, sc3b, pt3b, 3);
    eo_transcript_append_element(&t, "[e_v]G + [e_c]H", &e);
    eo_transcript_challenge_scalar(&t, "c", &expected);
    return eo_sc_eq(&expected, &s[0]) ? EO_OK : EO_CHALLENGE_MISMATCH;
}

/* tests/snapshots.rs:163-189 order: CiphertextWithValue::new(value) (draws r), SecretKey::generate (blinding), proof */
int eo_commitment_equiv_prove(const uint8_t pkb[32], uint64_t value, const uint8_t hb[32], const char *label, eo_rng *rng,
                              uint8_t ctb[64], uint8_t commitment[32], uint8_t proof[128], uint8_t blinding_out[32]) {
    eo_pk pk;
    eo_pt h, vg;
    if (eo_pk_from_bytes(&pk, pkb) || !eo_pt_decode(&h, hb)) return -1;
    eo_sc v, r, blinding;
    eo_ct ct;
    eo_sc_from_u64(&v, value);
    eo_pt_mul_generator(&vg, &v);
    eo_ext_ct_new(&ct, &r, &vg, &pk, rng);
    eo_rng_scalar(rng, &blinding);
    eo_transcript t;
    eo_transcript_new(&t, label);
    ceq_prove_pk(&pk, &ct, &v, &r, &blinding, &h, &t, rng, commitment, proof);
    eo_ct_encode(ctb, &ct);
    if (blinding_out) eo_sc_tobytes(blinding_out, &blinding);
    return 0;
}

int eo_commitment_equiv_verify(const uint8_t pkb[32], const uint8_t hb[32], const char *label, const uint8_t ctb[64],
                               const uint8_t commitment[32], const uint8_t proof[128]) {
    eo_pk pk;
    eo_pt h;
    if (eo_pk_from_bytes(&pk, pkb) || !eo_pt_decode(&h, hb)) return -1;
    return ceq_verify_pk(&pk, &h, label, ctb, commitment, proof);
}

typedef struct {
    eo_pk pk; eo_pt h; const uint8_t *hb; const char *label; const uint8_t *seed; size_t first; const uint64_t *values;
    uint8_t *cts, *commitments, *proofs; const uint8_t *ccts, *ccommitments, *cproofs; uint8_t *verdicts;
} ceq_ctx;

static void gen_ceq_item(void *p, size_t i) {
    ceq_ctx *c = (ceq_ctx *)p;
    eo_rng rng;
    item_rng(&rng, c->seed, c->first + i);
    eo_commitment_equiv_prove(c->pk.bytes, c->values[i], c->hb, c->label, &rng, c->cts + 64 * i, c->commitments + 32 * i,
                              c->proofs + 128 * i, NULL);
}

int eo_gen_ceq_batch(const uint8_t pkb[32], const uint8_t hb[32], const char *label, const uint8_t seed[32], size_t first,
                     size_t n, const uint64_t *values, uint8_t *cts, uint8_t *commitments, uint8_t *proofs, int threads) {
    ceq_ctx c;
    if (eo_pk_from_bytes(&c.pk, pkb) || !eo_pt_decode(&c.h, hb)) return -1;
    c.hb = hb; c.label = label; c.seed = seed; c.first = first; c.values = values;
    c.cts = cts; c.commitments = commitments; c.proofs = proofs;
    parallel_for(gen_ceq_item, &c, n, threads);
    return 0;
}

static void verify_ceq_item(void *p, size_t i) {
    ceq_ctx *c = (ceq_ctx *)p;
    c->verdicts[i] = (uint8_t)ceq_verify_pk(&c->pk, &c->h, c->label, c->ccts + 64 * i, c->ccommitments + 32 * i, c->cproofs + 128 * i);
}

int eo_verify_ceq_batch(const uint8_t pkb[32], const uint8_t hb[32], const char *label, size_t n, const uint8_t *cts,
                        const uint8_t *commitments, const uint8_t *proofs, uint8_t *verdicts, int threads) {
    ceq_ctx c;
    if (eo_pk_from_bytes(&c.pk, pkb) || !eo_pt_decode(&c.h, hb)) return -1;
    c.label = label; c.ccts = cts; c.ccommitments = commitments; c.cproofs = proofs; c.verdicts = verdicts;
    parallel_for(verify_ceq_item, &c, n, threads);
    return 0;
}

/* ================================================================== ProofOfPossession (proofs/possession.rs)
 * Proof bytes: challenge | responses[k]  = 32 (1 + k) B (struct field order, possession.rs:71-76).             */

/* possession.rs:94-130: secrets / public keys of k keypairs; one nonce draw per key, in key order */
int eo_pop_prove(uint32_t k, const uint8_t *secrets /* k*32 */, const uint8_t *keys /* k*32 */, const char *label, eo_rng *rng,
                 uint8_t *proof /* 32 (1+k) */) {
    if (k == 0 || k > EO_MAX_RINGS) return -1;
    eo_transcript t;
    eo_transcript_new(&t, label);
    eo_transcript_start_proof(&t, "multi_pop");
    for (uint32_t i = 0; i < k; i++) eo_transcript_append_message(&t, "K", keys + 32 * i, 32);
    eo_sc nonce[EO_MAX_RINGS], ch;
    for (uint32_t i = 0; i < k; i++) {
        eo_pt r;
        eo_rng_scalar(rng, &nonce[i]);
        eo_pt_mul_generator(&r, &nonce[i]);
        eo_transcript_append_element(&t, "R", &r);
    }
    eo_transcript_challenge_scalar(&t, "c", &ch);
    eo_sc_tobytes(proof, &ch);
    for (uint32_t i = 0; i < k; i++) {
        eo_sc x, s;
        if (!eo_sc_from_canonical(&x, secrets + 32 * i)) return -1;
        eo_sc_mul(&s, &x, &ch);
        eo_sc_add(&s, &s, &nonce[i]);
        eo_sc_tobytes(proof + 32 * (1 + i), &s);
    }
    return 0;
}

/* possession.rs:137-163.  Keys are PublicKey values: an undecodable or identity key is rejected when the key is
 * parsed (keys/mod.rs:161-176) -> EO_MALFORMED here. */
int eo_pop_verify(uint32_t k, const uint8_t *keys, const char *label, const uint8_t *proof) {
    if (k == 0 || k > EO_MAX_RINGS) return -1;
    eo_pk pk[EO_MAX_RINGS];
    eo_sc ch, s[EO_MAX_RINGS], neg_c, expected;
    for (uint32_t i = 0; i < k; i++)
        if (eo_pk_from_bytes(&pk[i], keys + 32 * i)) return EO_MALFORMED;
    if (!eo_sc_from_canonical(&ch, proof) || !eo_scalars_decode(s, proof + 32, k)) return EO_MALFORMED;
    eo_transcript t;
    eo_transcript_new(&t, label);
    eo_transcript_start_proof(&t, "multi_pop");
    for (uint32_t i = 0; i < k; i++) eo_transcript_append_message(&t, "K", keys + 32 * i, 32);
    eo_sc_neg(&neg_c, &ch);
    for (uint32_t i = 0; i < k; i++) {
        eo_pt r;
        eo_pt_double_mul_generator(&r, &neg_c, &pk[i].element, &s[i]);
        eo_transcript_append_element(&t, "R", &r);
    }
    eo_transcript_challenge_scalar(&t, "c", &expected);
    return eo_sc_eq(&expected, &ch) ? EO_OK : EO_CHALLENGE_MISMATCH;
}

typedef struct { uint32_t k; const char *label; const uint8_t *seed; size_t first; uint8_t *keys, *proofs; const uint8_t *ckeys, *cproofs; uint8_t *verdicts; } pop_ctx;

static void gen_pop_item(void *p, size_t i) {
    pop_ctx *c = (pop_ctx *)p;
    eo_rng rng;
    uint8_t secrets[32 * EO_MAX_RINGS];
    item_rng(&rng, c->seed, c->first + i);
    for (uint32_t j = 0; j < c->k; j++) eo_keypair_generate(&rng, secrets + 32 * j, c->keys + 32 * ((size_t)c->k * i + j));
    eo_pop_prove(c->k, secrets, c->keys + 32 * (size_t)c->k * i, c->label, &rng, c->proofs + 32 * (size_t)(1 + c->k) * i);
}

/* item i: k fresh keypairs (k draws) then the proof (k draws) */
int eo_gen_pop_batch(uint32_t k, const char *label, const uint8_t seed[32], size_t first, size_t n, uint8_t *keys,
                     uint8_t *proofs, int threads) {
    if (k == 0 || k > EO_MAX_RINGS) return -1;
    pop_ctx c;
    c.k = k; c.label = label; c.seed = seed; c.first = first; c.keys = keys; c.proofs = proofs;
    parallel_for(gen_pop_item, &c, n, threads);
    return 0;
}

static void verify_pop_item(void *p, size_t i) {
    pop_ctx *c = (pop_ctx *)p;
    c->verdicts[i] = (uint8_t)eo_pop_verify(c->k, c->ckeys + 32 * (size_t)c->k * i, c->label, c->cproofs + 32 * (size_t)(1 + c->k) * i);
}

int eo_verify_pop_batch(uint32_t k, const char *label, size_t n, const uint8_t *keys, const uint8_t *proofs, uint8_t *verdicts,
                        int threads) {
    if (k == 0 || k > EO_MAX_RINGS) return -1;
    pop_ctx c;
    c.k = k; c.label = label; c.ckeys = keys; c.cproofs = proofs; c.verdicts = verdicts;
    parallel_for(verify_pop_item, &c, n, threads);
    return 0;
}

/* ================================================================== PublicKeySet::from_participants (sharing/key_set.rs:87-144)
 * Returns 0 and the shared key when the participant keys are consistent, EO_MALFORMED when a key is not a valid
 * PublicKey (keys/mod.rs:161-176), EO_MALFORMED_PARTICIPANT_KEYS (Error::MalformedParticipantKeys) otherwise;
 * -1 for invalid parameters (ParticipantCountMismatch is the caller's framing: the batch has a fixed stride). */
int eo_keyset_from_participants(uint32_t shares, uint32_t threshold, const uint8_t *keys, uint8_t shared_key[32]) {
    if (shares == 0 || shares > 64 || threshold == 0 || threshold > shares) return -1;
    eo_pk pk[64];
    for (uint32_t i = 0; i < shares; i++)
        if (eo_pk_from_bytes(&pk[i], keys + 32 * i)) return EO_MALFORMED;
    uint32_t indexes[64];
    for (uint32_t i = 0; i < threshold; i++) indexes[i] = i;
    eo_sc denominators[64], scale;
    lagrange(indexes, threshold, denominators, &scale);
    eo_pt starting[64], acc, shared;
    for (uint32_t i = 0; i < threshold; i++) starting[i] = pk[i].element;
    eo_pt_multi_mul(&acc, denominators, starting, threshold);
    eo_pt_mul(&shared, &scale, &acc);
    eo_sc inverses[64];
    for (uint32_t i = 0; i < shares; i++) {        /* invert_scalars on 1..=n (key_set.rs:106-110) */
        eo_sc v;
        eo_sc_from_u64(&v, (uint64_t)i + 1);
        eo_sc_invert(&inverses[i], &v);
    }
    for (uint32_t x = threshold; x < shares; x++) {
        eo_sc key_scale, kd[64], e;
        eo_sc_from_u64(&key_scale, 1);
        for (uint32_t idx = 0; idx < threshold; idx++) {
            eo_sc_from_u64(&e, (uint64_t)(x - idx));
            eo_sc_mul(&key_scale, &key_scale, &e);
        }
        for (uint32_t idx = 0; idx < threshold; idx++) {
            eo_sc_from_u64(&e, (uint64_t)idx + 1);
            eo_sc_mul(&kd[idx], &denominators[idx], &e);
            eo_sc_mul(&kd[idx], &kd[idx], &inverses[x - idx - 1]);
        }
        if (threshold % 2 == 0) eo_sc_neg(&key_scale, &key_scale);
        eo_pt interpolated, scaled;
        eo_pt_multi_mul(&interpolated, kd, starting, threshold);
        eo_pt_mul(&scaled, &key_scale, &interpolated);
        if (!eo_pt_eq(&scaled, &pk[x].element)) return EO_MALFORMED_PARTICIPANT_KEYS;
    }
    eo_pt_encode(shared_key, &shared);
    return 0;
}
