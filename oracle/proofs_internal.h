/* proofs_internal.h -- oracle-internal types shared by proofs.c and apps.c (test infrastructure). */
#ifndef EG_ORACLE_PROOFS_INTERNAL_H
#define EG_ORACLE_PROOFS_INTERNAL_H

#include "eg_oracle.h"

#define EO_MAX_TERMS_SUMSQ 15      /* SumOfSquaresProof / QuadraticVotingBallot: the engine's 1..15 */

typedef struct { eo_pt R, B; } eo_ct;     /* Ciphertext encryption.rs:96-101: (random_element, blinded_element) */

int  eo_ct_decode(eo_ct *ct, const uint8_t b[64]);
void eo_ct_encode(uint8_t b[64], const eo_ct *ct);
void eo_ct_add(eo_ct *r, const eo_ct *a, const eo_ct *b);
void eo_ct_sub(eo_ct *r, const eo_ct *a, const eo_ct *b);
void eo_ct_zero(eo_ct *r);
void eo_ext_ct_new(eo_ct *ct, eo_sc *r_out, const eo_pt *value, const eo_pk *pk, eo_rng *rng);

void eo_logeq_prove(const eo_pk *log_base, const eo_sc *secret, const eo_pt *pow_g, const eo_pt *pow_k,
                    eo_transcript *t, eo_rng *rng, eo_sc *challenge, eo_sc *response);
int  eo_logeq_verify(const eo_pk *log_base, const eo_pt *pow_g, const eo_pt *pow_k, eo_transcript *t,
                     const eo_sc *challenge, const eo_sc *response);

typedef struct {                          /* Ring ring.rs:22-37 */
    size_t index;
    const eo_pt *admissible;
    size_t n_values, value_index;
    eo_ct ct;
    eo_transcript transcript;
    eo_sc *responses;
    eo_pt terminal[2];
    eo_sc discrete_log, random_scalar;
} eo_ring_state;

typedef struct {                          /* RingProofBuilder ring.rs:421-427 */
    const eo_pk *pk;
    eo_transcript *transcript;
    eo_rng *rng;
    eo_sc *responses;
    size_t used_responses;
    size_t n_rings;
    eo_ring_state rings[EO_MAX_RINGS];
} eo_ring_builder;

void eo_ring_builder_init(eo_ring_builder *b, const eo_pk *pk, eo_transcript *t, eo_rng *rng, eo_sc *responses);
int  eo_ring_builder_add_precomputed(eo_ring_builder *b, const eo_ct *ct, const eo_sc *ct_random,
                                     const eo_pt *admissible, size_t n_values, size_t value_index);
int  eo_ring_builder_add_value(eo_ring_builder *b, const eo_pt *admissible, size_t n_values, size_t value_index,
                               eo_ct *ct_out, eo_sc *random_out);
void eo_ring_builder_build(eo_ring_builder *b, eo_sc *common_challenge);
int  eo_ring_verify(const eo_pk *pk, size_t n_rings, const eo_pt *const *admissible, const size_t *ring_sizes,
                    const eo_ct *cts, const eo_sc *common_challenge, const eo_sc *responses, eo_transcript *t);

int  eo_scalars_decode(eo_sc *out, const uint8_t *bytes, size_t n);
void eo_scalars_encode(uint8_t *bytes, const eo_sc *in, size_t n);

typedef struct {                          /* PreparedRange range.rs:329-333 */
    eo_range range;
    eo_pt *values;
    eo_pt *ring_values[EO_MAX_RINGS];
    size_t ring_sizes[EO_MAX_RINGS];
} eo_prepared_range;

int  eo_prepared_range_init(eo_prepared_range *pr, const eo_range *range);
void eo_prepared_range_free(eo_prepared_range *pr);
int  eo_range_prove_prepared(const eo_pk *pk, const eo_prepared_range *pr, uint64_t value, const eo_ct *ct,
                             const eo_sc *ct_random, eo_transcript *t, eo_rng *rng,
                             eo_ct *partial, eo_sc *common_challenge, eo_sc *responses);
int  eo_range_verify_prepared(const eo_pk *pk, const eo_prepared_range *pr, const eo_ct *ct, const eo_ct *partial,
                              const eo_sc *common_challenge, const eo_sc *responses, eo_transcript *t);
int  eo_range_verify_bytes_prepared(const eo_pk *pk, const eo_prepared_range *pr, const char *label,
                                    const uint8_t ctb[64], const uint8_t *partialb, const uint8_t *ringb);

void eo_sumsq_prove_internal(const eo_pk *pk, size_t n, const eo_ct *cts, const eo_sc *values, const eo_sc *randomness,
                             const eo_ct *sum_ct, const eo_sc *sum_randomness, eo_transcript *t, eo_rng *rng,
                             eo_sc *challenge, eo_sc *ct_responses, eo_sc *sum_response);
int  eo_sumsq_verify_internal(const eo_pk *pk, size_t n, const eo_ct *cts, const eo_ct *sum_ct, eo_transcript *t,
                              const eo_sc *challenge, const eo_sc *ct_responses, const eo_sc *sum_response);
int  eo_sumsq_verify_bytes(const eo_pk *pk, uint32_t n, const uint8_t *ctsb, const uint8_t sum_ctb[64],
                           const char *label, const uint8_t *proof);

void eo_oracle_init(void);    /* forces lazy constant/table init before threads start */

#endif
