/*
 * eg_oracle.h -- CPU ORACLE for the elastic-elgamal hot path (TEST INFRASTRUCTURE ONLY).
 *
 * This is a plain-C restatement of the reference's algorithm for the batch-verification path
 * (slowli/elastic-elgamal v0.3.1).  It exists only as a checker: `tests/`, `__graft_entry__.smoke()`
 * and `bench.py`'s cpu_baseline / `--impl reference` legs may load it; the product library
 * (elastic_elgamal_b200/csrc -> libeg_b200.so) never links, loads or calls it.
 *
 * Parity is PINNED: tests/test_oracle_golden.py reproduces the reference's 12 seeded Ristretto
 * snapshot vectors byte-for-byte (tests/snapshots.rs:31-189 + tests/snapshots/ *-ristretto.snap,
 * committed as tests/golden/ristretto_snapshots.json) and the KATs listed in SURVEY.md 8(c).
 *
 * The arithmetic lives in third-party crates that are NOT vendored under /root/reference
 * (curve25519-dalek =5.0.0-rc.0, merlin 3.0.0 + keccak 0.1.6, rand_chacha 0.10.0); it is restated
 * from the public specifications: RFC 9496 (ristretto255), RFC 8032 (edwards25519), STROBE v1.0.2 /
 * Merlin v1.0 framing, RFC 8439 (ChaCha20 block function), PCG32 (rand_core seed_from_u64).
 * Protocol logic follows the reference file:line cited at each function.
 */
#ifndef EG_ORACLE_H
#define EG_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ field GF(2^255-19) */
typedef struct { uint64_t v[5]; } eo_fe;   /* radix 2^51 */

void eo_fe_frombytes(eo_fe *h, const uint8_t s[32]);      /* ignores bit 255 */
void eo_fe_tobytes(uint8_t s[32], const eo_fe *h);        /* canonical */
void eo_fe_mul(eo_fe *h, const eo_fe *f, const eo_fe *g);
void eo_fe_sq(eo_fe *h, const eo_fe *f);
void eo_fe_add(eo_fe *h, const eo_fe *f, const eo_fe *g);
void eo_fe_sub(eo_fe *h, const eo_fe *f, const eo_fe *g);
void eo_fe_neg(eo_fe *h, const eo_fe *f);
void eo_fe_invert(eo_fe *h, const eo_fe *f);
int  eo_fe_sqrt_ratio_i(eo_fe *r, const eo_fe *u, const eo_fe *v); /* RFC 9496 4.2 */

/* ------------------------------------------------------------------ scalars mod l */
typedef struct { uint64_t v[4]; } eo_sc;   /* canonical value < l, little-endian limbs */

int  eo_sc_from_canonical(eo_sc *s, const uint8_t b[32]);  /* 0 if b >= l (ristretto.rs:59-62) */
void eo_sc_from_wide(eo_sc *s, const uint8_t b[64]);       /* ristretto.rs:28-38 */
void eo_sc_from_u64(eo_sc *s, uint64_t x);
void eo_sc_tobytes(uint8_t b[32], const eo_sc *s);
void eo_sc_add(eo_sc *r, const eo_sc *a, const eo_sc *b);
void eo_sc_sub(eo_sc *r, const eo_sc *a, const eo_sc *b);
void eo_sc_neg(eo_sc *r, const eo_sc *a);
void eo_sc_mul(eo_sc *r, const eo_sc *a, const eo_sc *b);
void eo_sc_invert(eo_sc *r, const eo_sc *a);
int  eo_sc_eq(const eo_sc *a, const eo_sc *b);

/* ------------------------------------------------------------------ group (ristretto255) */
typedef struct { eo_fe X, Y, Z, T; } eo_pt;   /* extended twisted Edwards, a = -1 */

void eo_pt_identity(eo_pt *p);
void eo_pt_generator(eo_pt *p);
void eo_pt_add(eo_pt *r, const eo_pt *p, const eo_pt *q);
void eo_pt_sub(eo_pt *r, const eo_pt *p, const eo_pt *q);
void eo_pt_neg(eo_pt *r, const eo_pt *p);
void eo_pt_double(eo_pt *r, const eo_pt *p);
int  eo_pt_decode(eo_pt *p, const uint8_t s[32]);          /* RFC 9496 4.3.1; ristretto.rs:93 */
void eo_pt_encode(uint8_t s[32], const eo_pt *p);          /* RFC 9496 4.3.2; ristretto.rs:88 */
int  eo_pt_is_identity(const eo_pt *p);
int  eo_pt_eq(const eo_pt *p, const eo_pt *q);
/* r = sum scalars[i] * points[i]; variable time (ristretto.rs:139-146). n <= 16 */
void eo_pt_multi_mul(eo_pt *r, const eo_sc *scalars, const eo_pt *points, size_t n);
/* r = a*A + b*G (ristretto.rs:131-137) */
void eo_pt_double_mul_generator(eo_pt *r, const eo_sc *a, const eo_pt *A, const eo_sc *b);
void eo_pt_mul_generator(eo_pt *r, const eo_sc *k);        /* ristretto.rs:105-121 */
void eo_pt_mul(eo_pt *r, const eo_sc *k, const eo_pt *p);

/* byte-level helpers for the python test layer */
int  eo_point_decode_check(const uint8_t s[32]);
int  eo_point_mul_bytes(uint8_t out[32], const uint8_t scalar[32], const uint8_t point[32]);
void eo_point_mul_generator_bytes(uint8_t out[32], const uint8_t scalar[32]);
int  eo_point_add_bytes(uint8_t out[32], const uint8_t a[32], const uint8_t b[32]);
int  eo_point_sub_bytes(uint8_t out[32], const uint8_t a[32], const uint8_t b[32]);
void eo_scalar_reduce_wide_bytes(uint8_t out[32], const uint8_t in[64]);
int  eo_scalar_is_canonical(const uint8_t in[32]);
void eo_scalar_muladd_bytes(uint8_t out[32], const uint8_t a[32], const uint8_t b[32], const uint8_t c[32]);
void eo_scalar_invert_bytes(uint8_t out[32], const uint8_t a[32]);
void eo_fe_mul_bytes(uint8_t out[32], const uint8_t a[32], const uint8_t b[32]);
void eo_fe_invert_bytes(uint8_t out[32], const uint8_t a[32]);

/* ------------------------------------------------------------------ Merlin transcript */
typedef struct {
    uint8_t state[200];
    uint8_t pos, pos_begin, cur_flags;
} eo_transcript;

void eo_keccak_f1600(uint8_t state[200]);
void eo_transcript_new(eo_transcript *t, const char *label);                 /* merlin Transcript::new */
void eo_transcript_append_message(eo_transcript *t, const char *label, const uint8_t *msg, size_t len);
void eo_transcript_append_u64(eo_transcript *t, const char *label, uint64_t x);
void eo_transcript_challenge_bytes(eo_transcript *t, const char *label, uint8_t *out, size_t len);
/* TranscriptForGroup, proofs/mod.rs:29-57 */
void eo_transcript_start_proof(eo_transcript *t, const char *label);
void eo_transcript_append_element(eo_transcript *t, const char *label, const eo_pt *p);
void eo_transcript_challenge_scalar(eo_transcript *t, const char *label, eo_sc *out);

/* ------------------------------------------------------------------ ChaCha20 RNG (rand_chacha)
 * or a replay of caller-supplied blocks.  A replaying rng hands out blocks[0], blocks[1], ... in order (`block` counts the
 * draws) so that a prover runs on exactly the blocks the library's `wide_rand` form takes.  Its state lives in the 32 key
 * bytes, marked by EO_RNG_REPLAY_TAG, so eo_rng keeps its 40-byte layout: every caller that allocates the struct itself
 * (the ctypes mirror in tests/oracle.py, checked against eo_rng_size()) stays valid.  A draw past the last block yields a
 * 0xff block and leaves the rng overrun for good (eo_rng_overrun); tests/oracle.py raises on it, so a wrong draw count can
 * neither wrap around nor pass as zeros. */
#define EO_RNG_REPLAY_TAG "eo_rng replay v1"               /* 16 bytes, no terminator stored */
typedef struct {
    union {
        uint8_t key[32];                                    /* ChaCha20 key */
        struct {
            uint8_t tag[16];                                /* EO_RNG_REPLAY_TAG */
            const uint8_t *blocks;                          /* n_blocks * 64 caller-owned bytes */
            uint64_t n_blocks;
        } replay;
    };
    uint64_t block;                                         /* ChaCha20: next block counter; replay: draws so far */
} eo_rng;

size_t eo_rng_size(void);                                   /* sizeof(eo_rng) = 40, for the ctypes mirror */
void eo_rng_from_seed(eo_rng *r, const uint8_t seed[32], uint64_t first_block);
void eo_rng_seed_from_u64(eo_rng *r, uint64_t seed);        /* rand_core SeedableRng::seed_from_u64 */
void eo_rng_from_blocks(eo_rng *r, const uint8_t *blocks, uint64_t n_blocks);   /* replay; `blocks` must outlive r */
int  eo_rng_overrun(const eo_rng *r);                       /* 1: a replay was asked for more blocks than it holds */
uint64_t eo_rng_blocks_left(const eo_rng *r);            /* blocks a replay has not handed out yet (0 for ChaCha20) */
void eo_rng_block(eo_rng *r, uint8_t out[64]);              /* next 64-byte keystream (or replayed) block */
void eo_rng_scalar(eo_rng *r, eo_sc *out);                  /* Ristretto::generate_scalar, ristretto.rs:28-32 */

/* ------------------------------------------------------------------ verdict codes
 * Shared with include/eg_b200.h (same numeric values; the tests assert equality). */
enum {
    EO_OK = 0,
    EO_MALFORMED = 1,           /* undecodable element / non-canonical scalar: rejected by from_bytes/serde */
    EO_CHALLENGE_MISMATCH = 2,  /* VerificationError::ChallengeMismatch (proofs/mod.rs:63-69) */
    EO_CHOICE_SUM = 3,          /* ChoiceVerificationError::Sum (choice.rs:93) */
    EO_CHOICE_RANGE = 4,        /* ChoiceVerificationError::Range (choice.rs:379) */
    EO_QV_CREDIT_RANGE = 5,     /* QuadraticVotingError::CreditRange (quadratic_voting.rs:315-316) */
    EO_QV_CREDIT_EQUIV = 6,     /* QuadraticVotingError::CreditEquivalence (quadratic_voting.rs:325-326) */
    EO_MALFORMED_PARTICIPANT_KEYS = 7,  /* sharing::Error::MalformedParticipantKeys (sharing/key_set.rs:137-139) */
    EO_QV_VARIANT_BASE = 16     /* + option index: QuadraticVotingError::Variant (quadratic_voting.rs:305) */
};

/* ------------------------------------------------------------------ keys / encryption */
typedef struct { uint8_t bytes[32]; eo_pt element; } eo_pk;   /* keys/mod.rs:122-125 */

/* PublicKey::from_bytes keys/mod.rs:161-176: 0 ok, 1 invalid element, 2 identity */
int  eo_pk_from_bytes(eo_pk *pk, const uint8_t b[32]);
void eo_pk_from_element(eo_pk *pk, const eo_pt *p);                        /* keys/mod.rs:178-185 */
void eo_keypair_generate(eo_rng *rng, uint8_t sk[32], uint8_t pk[32]);     /* keys/mod.rs:285-291 */
int  eo_encrypt(const uint8_t pk[32], uint64_t value, eo_rng *rng, uint8_t ct[64]);   /* keys/impls.rs:16-23 */
int  eo_decrypt_to_element(const uint8_t sk[32], const uint8_t ct[64], uint8_t out[32]); /* keys/impls.rs:160-163 */

/* LogEqualityProof over (zero encryption), keys/impls.rs:31-69 */
int  eo_encrypt_zero(const uint8_t pk[32], eo_rng *rng, uint8_t ct[64], uint8_t proof[64]);
int  eo_verify_zero(const uint8_t pk[32], const uint8_t ct[64], const uint8_t proof[64]);

/* encrypt_bool / verify_bool, keys/impls.rs:77-113 */
int  eo_encrypt_bool(const uint8_t pk[32], int value, eo_rng *rng, uint8_t ct[64], uint8_t proof[96]);
int  eo_verify_bool(const uint8_t pk[32], const uint8_t ct[64], const uint8_t proof[96]);

/* EncryptedChoice, app/choice.rs:288-380.  choices: n flags; cts: n*64; ring: (1+2n)*32; sum: 64 (single only) */
int  eo_choice_new(const uint8_t pk[32], uint32_t n, const uint8_t *choices, int single, eo_rng *rng,
                   uint8_t *cts, uint8_t *ring, uint8_t *sum);
int  eo_choice_verify(const uint8_t pk[32], uint32_t n, int single,
                      const uint8_t *cts, const uint8_t *ring, const uint8_t *sum);

/* RangeDecomposition, proofs/range.rs:106-324 */
#define EO_MAX_RINGS 64
typedef struct {
    uint32_t n_rings;
    uint64_t size[EO_MAX_RINGS];
    uint64_t step[EO_MAX_RINGS];
} eo_range;

int      eo_range_optimal(eo_range *out, uint64_t upper_bound);            /* range.rs:148-153 */
uint64_t eo_range_upper_bound(const eo_range *r);                          /* range.rs:174-181 (wraps from 2^64 on) */
uint64_t eo_range_max_value(const eo_range *r);                            /* upper bound - 1, saturated at 2^64 - 1 */
uint64_t eo_range_rings_size(const eo_range *r);                           /* range.rs:183-186 */
size_t   eo_range_display(const eo_range *r, char *buf, size_t cap);       /* range.rs:110-124 */

/* RangeProof, range.rs:462-577.  partial: (n_rings-1)*64; ring: (1+rings_size)*32 */
int  eo_range_prove(const uint8_t pk[32], const eo_range *range, const char *transcript_label,
                    uint64_t value, eo_rng *rng, uint8_t ct[64], uint8_t sk_r_out[32],
                    uint8_t *partial, uint8_t *ring);
int  eo_range_verify(const uint8_t pk[32], const eo_range *range, const char *transcript_label,
                     const uint8_t ct[64], const uint8_t *partial, const uint8_t *ring);

/* SumOfSquaresProof, proofs/mul.rs:107-260.  proof: (2n+2)*32 = challenge | responses | sum_response.
 * values/randomness are canonical scalars (32 B each), cts are 64 B each. */
int  eo_sumsq_prove(const uint8_t pk[32], uint32_t n, const uint8_t *cts, const uint8_t *values,
                    const uint8_t *randomness, const uint8_t sum_ct[64], const uint8_t sum_randomness[32],
                    const char *transcript_label, eo_rng *rng, uint8_t *proof);
int  eo_sumsq_verify(const uint8_t pk[32], uint32_t n, const uint8_t *cts, const uint8_t sum_ct[64],
                     const char *transcript_label, const uint8_t *proof);

/* QuadraticVotingBallot, app/quadratic_voting.rs:63-329 */
typedef struct {
    uint32_t options;
    uint64_t credits;
    eo_range vote_range;
    eo_range credit_range;
} eo_qv_params;

uint64_t eo_isqrt(uint64_t x);                                             /* quadratic_voting.rs:127-143 */
int      eo_qv_params_new(eo_qv_params *p, uint32_t options, uint64_t credits); /* quadratic_voting.rs:63-76 */
size_t   eo_qv_ballot_size(const eo_qv_params *p);
/* ballot layout (bytes): for each option: ct(64) | partial | ring ; credit: ct | partial | ring ; sumsq proof */
int  eo_qv_new(const uint8_t pk[32], const eo_qv_params *p, const uint64_t *votes, eo_rng *rng, uint8_t *ballot);
int  eo_qv_verify(const uint8_t pk[32], const eo_qv_params *p, const uint8_t *ballot);

/* Threshold decryption, sharing/ *.rs, decryption.rs */
typedef struct {
    uint32_t shares, threshold;
    uint8_t shared_key[32];
    uint8_t participant_keys[64][32];
} eo_keyset;

/* Dealer::new + secret_share_for_participant (participant.rs:35-83) without the proof of possession:
 * draws `threshold` secrets; participant secret i = poly(i+1). */
int  eo_dealer_new(uint32_t shares, uint32_t threshold, eo_rng *rng, eo_keyset *ks, uint8_t *secret_shares /* shares*32 */);
/* ActiveParticipant::decrypt_share participant.rs:163-185 */
int  eo_decrypt_share(const eo_keyset *ks, uint32_t index, const uint8_t secret_share[32], const uint8_t ct[64],
                      eo_rng *rng, uint8_t share[32], uint8_t proof[64]);
/* PublicKeySet::verify_share key_set.rs:209-228 */
int  eo_verify_share(const eo_keyset *ks, uint32_t index, const uint8_t ct[64], const uint8_t share[32],
                     const uint8_t proof[64]);

/* VerifiableDecryption::new / CandidateDecryption::verify with a custom key, decryption.rs:89-111,189-205 */
int  eo_decryption_prove(const uint8_t secret[32], const char *transcript_label, const uint8_t ct[64], eo_rng *rng,
                         uint8_t dh_out[32], uint8_t proof[64]);
int  eo_decryption_verify(const uint8_t key[32], const char *transcript_label, const uint8_t ct[64], const uint8_t dh[32],
                          const uint8_t proof[64]);
/* lagrange_coefficients sharing/mod.rs:139-170: out coeffs t*32, scale 32 */
void eo_lagrange_coefficients(const uint32_t *indexes, uint32_t t, uint8_t *coeffs, uint8_t scale[32]);
/* Params::combine_shares sharing/mod.rs:302-325 + VerifiableDecryption::decrypt_to_element decryption.rs:129-131:
 * out = B - combined. returns 0 ok, 1 malformed */
int  eo_combine_decrypt(uint32_t t, const uint32_t *indexes, const uint8_t *shares /* t*32 */,
                        const uint8_t ct[64], uint8_t out_element[32]);

/* DiscreteLogTable encryption.rs:260-298 */
typedef struct eo_dlog_table eo_dlog_table;
eo_dlog_table *eo_dlog_table_new(uint64_t lo, uint64_t hi);  /* values lo..hi (exclusive) */
void eo_dlog_table_free(eo_dlog_table *t);
/* returns 1 and sets *value if found (identity -> 0 always), 0 if absent, -1 if element undecodable */
int  eo_dlog_table_get(const eo_dlog_table *t, const uint8_t element[32], uint64_t *value);

/* ------------------------------------------------------------------ batch helpers (threads)
 * Deterministic synthetic workload generation + CPU baseline loops.  Item i draws from an
 * independent ChaCha20 stream: key = seed, first block = i << 20 (SURVEY.md 8(d)). */
int  eo_gen_bool_batch(const uint8_t pk[32], const uint8_t seed[32], size_t first, size_t n,
                       uint8_t *cts, uint8_t *proofs, int threads);
int  eo_verify_bool_batch(const uint8_t pk[32], size_t n, const uint8_t *cts, const uint8_t *proofs,
                          uint8_t *verdicts, int threads);
int  eo_gen_choice_batch(const uint8_t pk[32], uint32_t options, const uint8_t seed[32], size_t first, size_t n,
                         uint8_t *cts, uint8_t *rings, uint8_t *sums, int threads);
/* verdicts + tally (options*64; sum over OK ballots, choice.rs:358 + examples/voting.rs:200-203) */
int  eo_verify_choice_batch(const uint8_t pk[32], uint32_t options, int single, size_t n,
                            const uint8_t *cts, const uint8_t *rings, const uint8_t *sums,
                            uint8_t *verdicts, uint8_t *tally, int threads);
int  eo_gen_range_batch(const uint8_t pk[32], const eo_range *range, const char *label, const uint8_t seed[32],
                        size_t first, size_t n, const uint64_t *values,
                        uint8_t *cts, uint8_t *partials, uint8_t *rings, int threads);
int  eo_verify_range_batch(const uint8_t pk[32], const eo_range *range, const char *label, size_t n,
                           const uint8_t *cts, const uint8_t *partials, const uint8_t *rings,
                           uint8_t *verdicts, int threads);
int  eo_gen_qv_batch(const uint8_t pk[32], const eo_qv_params *p, const uint8_t seed[32], size_t first, size_t n,
                     const uint64_t *votes /* n*options */, uint8_t *ballots, int threads);
int  eo_verify_qv_batch(const uint8_t pk[32], const eo_qv_params *p, size_t n, const uint8_t *ballots,
                        uint8_t *verdicts, uint8_t *tally, int threads);
/* CommitmentEquivalenceProof proofs/commitment.rs:126-248.  proof = challenge | s_r | s_v | s_c (128 B; struct field
 * order, the reference has serde only).  prove follows tests/snapshots.rs:163-189: encrypt(value) draws r, then the
 * commitment blinding, then e_r, e_v, e_c.  verify returns a verdict (EO_OK / EO_MALFORMED / EO_CHALLENGE_MISMATCH),
 * -1 when the receiver key or the blinding base is invalid. */
int  eo_commitment_equiv_prove(const uint8_t pk[32], uint64_t value, const uint8_t blinding_base[32], const char *label,
                               eo_rng *rng, uint8_t ct[64], uint8_t commitment[32], uint8_t proof[128],
                               uint8_t blinding_out[32] /* may be NULL */);
int  eo_commitment_equiv_verify(const uint8_t pk[32], const uint8_t blinding_base[32], const char *label,
                                const uint8_t ct[64], const uint8_t commitment[32], const uint8_t proof[128]);
int  eo_gen_ceq_batch(const uint8_t pk[32], const uint8_t blinding_base[32], const char *label, const uint8_t seed[32],
                      size_t first, size_t n, const uint64_t *values, uint8_t *cts, uint8_t *commitments, uint8_t *proofs,
                      int threads);
int  eo_verify_ceq_batch(const uint8_t pk[32], const uint8_t blinding_base[32], const char *label, size_t n,
                         const uint8_t *cts, const uint8_t *commitments, const uint8_t *proofs, uint8_t *verdicts, int threads);

/* ProofOfPossession proofs/possession.rs:71-163.  proof = challenge | responses[k] (32 (1 + k) B). */
int  eo_pop_prove(uint32_t k, const uint8_t *secrets, const uint8_t *keys, const char *label, eo_rng *rng, uint8_t *proof);
int  eo_pop_verify(uint32_t k, const uint8_t *keys, const char *label, const uint8_t *proof);
int  eo_gen_pop_batch(uint32_t k, const char *label, const uint8_t seed[32], size_t first, size_t n, uint8_t *keys,
                      uint8_t *proofs, int threads);
int  eo_verify_pop_batch(uint32_t k, const char *label, size_t n, const uint8_t *keys, const uint8_t *proofs,
                         uint8_t *verdicts, int threads);
/* PublicKeySet::from_participants sharing/key_set.rs:87-144: verdict (EO_OK / EO_MALFORMED /
 * EO_MALFORMED_PARTICIPANT_KEYS) and, when OK, the reconstructed shared key; -1 for invalid (shares, threshold). */
int  eo_keyset_from_participants(uint32_t shares, uint32_t threshold, const uint8_t *keys /* shares*32 */,
                                 uint8_t shared_key[32]);
int  eo_hw_threads(void);

#ifdef __cplusplus
}
#endif
#endif /* EG_ORACLE_H */
