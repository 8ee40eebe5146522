/*
 * eg_b200.h -- C ABI of the B200 batch engine for elastic-elgamal's verification hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8(b)): a batch entry point that is semantically
 *     items.iter().map(|x| x.verify(&params))          (+ the homomorphic tally fold)
 * for the reference's per-item calls.  Every function cites the reference interface it replaces.
 * A Rust `-sys` crate binds these symbols 1:1 (see INTEGRATION.md and rust/); nothing here depends on
 * torch, NCCL or C++ types: plain pointers and sizes only.
 *
 * Conventions
 *   - All byte layouts follow the reference's `to_bytes` forms: Ciphertext = R || B (64 B,
 *     src/encryption.rs:155-160); RingProof = e0 || s_0 || ... (src/proofs/ring.rs:383-393);
 *     LogEqualityProof = c || s (src/proofs/log_equality.rs:184-189); VerifiableDecryption = 32 B element
 *     (src/decryption.rs:118-122).  Batches are contiguous arrays of such items.
 *   - Host entry points (`eg_*_batch`) take HOST pointers and copy to/from the device themselves.
 *     `_dev` variants take DEVICE pointers on the context's device and run on the context's stream
 *     (results are complete when the call returns).
 *   - The return value reports API / CUDA failures only.  Per-item outcomes are verdict bytes that
 *     enumerate the reference's error variants in the reference's precedence order.
 *   - Never unwinds across the boundary.  A context is used from one host thread at a time (!Sync);
 *     different contexts are independent.  There is no CPU fallback: without a CUDA device
 *     eg_ctx_create fails with EG_ERR_NO_DEVICE.
 */
#ifndef EG_B200_H
#define EG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct eg_ctx eg_ctx;
typedef struct eg_dlog_table eg_dlog_table;
typedef int32_t eg_status;

enum {
    EG_SUCCESS = 0,
    EG_ERR_INVALID_ARG = 1,       /* null pointer, zero options, inconsistent sizes (reference: assert!/panic! on the caller side) */
    EG_ERR_INVALID_ELEMENT = 2,   /* PublicKeyConversionError::InvalidGroupElement, src/keys/mod.rs:166-167 */
    EG_ERR_IDENTITY_KEY = 3,      /* PublicKeyConversionError::IdentityKey, src/keys/mod.rs:168-169 */
    EG_ERR_NO_RECEIVER = 4,       /* a verification entry point was called before eg_ctx_set_receiver */
    EG_ERR_NO_DEVICE = 5,         /* no usable CUDA device (there is no CPU fallback) */
    EG_ERR_CUDA = 6,              /* CUDA runtime failure; see eg_last_error */
    EG_ERR_OUT_OF_MEMORY = 7,
    EG_ERR_LEN_MISMATCH = 8,      /* VerificationError::LenMismatch / OptionsLenMismatch (src/proofs/mod.rs:70-78,
                                     src/app/choice.rs:149-158): in a fixed-stride batch this is an API-level error */
    EG_ERR_NCCL = 9               /* NCCL could not be loaded / a collective failed; see eg_last_error */
};

/* Per-item verdicts (uint8_t).  0 = Ok(..); the rest mirror the reference's error enums. */
enum {
    EG_V_OK = 0,
    EG_V_MALFORMED = 1,           /* an element does not decode or a scalar is not canonical: the reference rejects
                                     these before `verify`, in from_bytes / serde (src/proofs/ring.rs:397-414,
                                     src/serde.rs:195-198,258-261, src/decryption.rs:168-177) */
    EG_V_CHALLENGE_MISMATCH = 2,  /* VerificationError::ChallengeMismatch, src/proofs/mod.rs:63-69 */
    EG_V_CHOICE_SUM = 3,          /* ChoiceVerificationError::Sum, src/app/choice.rs:93 */
    EG_V_CHOICE_RANGE = 4,        /* ChoiceVerificationError::Range, src/app/choice.rs:379 */
    EG_V_QV_CREDIT_RANGE = 5,     /* QuadraticVotingError::CreditRange, src/app/quadratic_voting.rs:315-316 */
    EG_V_QV_CREDIT_EQUIV = 6,     /* QuadraticVotingError::CreditEquivalence, src/app/quadratic_voting.rs:325-326 */
    EG_V_MALFORMED_PARTICIPANT_KEYS = 7,  /* sharing::Error::MalformedParticipantKeys, src/sharing/key_set.rs:137-139 */
    EG_V_QV_VARIANT_BASE = 16     /* + option index: QuadraticVotingError::Variant{index}, src/app/quadratic_voting.rs:305 */
};

/* ---- context ------------------------------------------------------------------------------------ */

/* Creates a context on CUDA device `device_id` (one context per GPU / per process rank).
 * Owns a stream, the fixed-base tables for G and for the receiver key (8.25 GiB of device memory each: 24-bit windows,
 * DESIGN.md "Data layout"), transcript prefixes, scratch. */
eg_status eg_ctx_create(int device_id, eg_ctx **out);
void      eg_ctx_destroy(eg_ctx *ctx);
/* Human-readable description of the last failure on this context ("" if none). Never NULL. */
const char *eg_last_error(const eg_ctx *ctx);
/* Library build identification: "eg_b200 <version> sm_100a". */
const char *eg_version(void);

/* ---- multi-GPU (SURVEY.md 8(e)) ------------------------------------------------------------------
 * The loop being replaced (examples/voting.rs:188-204) is a map over independent ballots with a commutative fold, so a
 * batch shards across the GPUs of one box; the only exchange is the per-GPU partial tally (options x 64 B), which the
 * library combines itself: ONE ncclAllGather over NVLink followed by a point-addition kernel (NCCL has no
 * elliptic-curve reduction operator).  NCCL is bound at run time (libnccl.so.2), only when one of these is called.
 *
 * (1) One process, several devices.  The context owns one child context per device (own streams, tables, scratch) and a
 *     communicator from ncclCommInitAll.  Every host-pointer batch entry point then shards the batch contiguously
 *     across the devices (one host thread each); verdicts come back in input order; `tally` outputs are the totals over
 *     all devices.  `_dev` entry points need a single-device context (EG_ERR_INVALID_ARG); helper entry points (group
 *     helpers, wire codec, key-set validation, proofs of possession, commitment equivalence) run on the first device. */
eg_status eg_ctx_create_multi(const int *device_ids, int n_dev, eg_ctx **out);
/* (2) One process per GPU (torchrun / MPI style).  Rank 0 obtains a unique id, the host distributes its 128 bytes over
 *     any channel it already has, every rank attaches it to its single-device context (ncclCommInitRank; collective).
 *     From then on the `tally` output of eg_verify_choice_batch[_dev] and eg_verify_qv_batch is the total over all ranks
 *     (identical bytes on every rank) and those calls are collective: every rank calls them, with its own slice of the
 *     batch (n may differ, 0 included) and the same options / `tally != NULL`.  Verdicts stay local to the rank. */
#define EG_COMM_ID_BYTES 128
eg_status eg_comm_unique_id(uint8_t id[EG_COMM_ID_BYTES]);
eg_status eg_ctx_attach_comm(eg_ctx *ctx, const uint8_t id[EG_COMM_ID_BYTES], int rank, int world);
/* rank / world of the attached communicator (0 / 1 without one); devices = children of a multi-device context (else 1) */
eg_status eg_ctx_comm_info(const eg_ctx *ctx, int *rank, int *world, int *devices);

/* PublicKey::<Ristretto>::from_bytes (src/keys/mod.rs:161-176): validates K (decodable, not the identity),
 * keeps its bytes for the transcripts (PublicKey::as_bytes :188-190) and builds K's fixed-base table. */
eg_status eg_ctx_set_receiver(eg_ctx *ctx, const uint8_t key[32]);

/* The Pedersen blinding base H of CommitmentEquivalenceProof (`commitment_blinding_base`, src/proofs/commitment.rs:140-145),
 * e.g. the Bulletproofs base of tests/snapshots.rs:253-257.  Validated like a public key (decodable, not the identity);
 * gets the same fixed-base table as G and K. */
eg_status eg_ctx_set_blinding_base(eg_ctx *ctx, const uint8_t base[32]);

/* ---- group-level helpers (Group / ElementOps / ScalarOps for Ristretto, src/group/ristretto.rs) -- */

/* ElementOps::deserialize_element :93-95 over a batch: ok[i] = 1 if encodings[i] decodes */
eg_status eg_elements_validate(eg_ctx *ctx, size_t n, const uint8_t *encodings /* n*32 */, uint8_t *ok /* n */);
/* ScalarOps::deserialize_scalar :59-62 over a batch: ok[i] = 1 if canonical (< l) */
eg_status eg_scalars_validate(eg_ctx *ctx, size_t n, const uint8_t *scalars /* n*32 */, uint8_t *ok /* n */);
/* ScalarOps::scalar_from_random_bytes :34-38: 64 bytes -> canonical scalar */
eg_status eg_scalars_from_wide(eg_ctx *ctx, size_t n, const uint8_t *wide /* n*64 */, uint8_t *scalars /* n*32 */);
/* Group::vartime_double_mul_generator :131-137 over a batch: out[i] = [a_i]A_i + [b_i]G.
 * ok[i] = 0 (and out[i] = identity encoding) if A_i does not decode or a scalar is not canonical. */
eg_status eg_double_mul_generator_batch(eg_ctx *ctx, size_t n, const uint8_t *a /* n*32 */, const uint8_t *A /* n*32 */,
                                        const uint8_t *b /* n*32 */, uint8_t *out /* n*32 */, uint8_t *ok /* n */);
/* Group::mul_generator :105-107 over a batch: out[i] = [k_i]G */
eg_status eg_mul_generator_batch(eg_ctx *ctx, size_t n, const uint8_t *k /* n*32 */, uint8_t *out /* n*32 */, uint8_t *ok);
/* Group::vartime_multi_mul :139-146 over a batch: out[i] = sum_j [scalars[i][j]] points[i][j], 1 <= terms <= 16.
 * ok[i] = 0 (and out[i] = identity encoding) if a point does not decode or a scalar is not canonical. */
eg_status eg_multi_mul_batch(eg_ctx *ctx, size_t n, uint32_t terms, const uint8_t *scalars /* n*terms*32 */,
                             const uint8_t *points /* n*terms*32 */, uint8_t *out /* n*32 */, uint8_t *ok /* n */);
/* The Ciphertext operators of src/encryption.rs:163-226 (Add :163, Sub :180, Mul<&Scalar> :197, Mul<u64> :208, Neg :217)
 * over a batch, as one linear combination per item: out[i] = sum_j [scalars[i][j]] cts[i][j] on the R and the B parts, 1 <= terms <= 16.
 * a + b = scalars (1, 1); a - b = (1, l - 1); -a = (l - 1); a * k = (k).  ok[i] = 0 (and out[i] = two identity encodings)
 * if an element does not decode or a scalar is not canonical. */
eg_status eg_ciphertexts_lincomb_batch(eg_ctx *ctx, size_t n, uint32_t terms, const uint8_t *scalars /* n*terms*32 */,
                                       const uint8_t *cts /* n*terms*64 */, uint8_t *out /* n*64 */, uint8_t *ok /* n */);
/* Ciphertext + Ciphertext folded over a batch (src/encryption.rs:163-172): out = sum of the n_parts rows,
 * each row = n_cts ciphertexts.  Used to combine per-GPU partial tallies. ok = 0 if any element is malformed. */
eg_status eg_ciphertexts_sum(eg_ctx *ctx, size_t n_parts, size_t n_cts, const uint8_t *parts /* n_parts*n_cts*64 */,
                             uint8_t *out /* n_cts*64 */, uint8_t *ok /* 1 */);

/* ---- wire format (src/serde.rs:19-80) ----------------------------------------------------------- */

/* The human-readable serde form of every element, scalar and proof is an unpadded base64url string
 * (serialize_bytes :19-27 / Base64Visitor :41-44, base64ct::Base64UrlUnpadded).  Fields have fixed sizes, so a batch is
 * n strings of eg_base64url_chars(bytes_per_item) = ceil(4 * bytes / 3) characters, back to back, no terminators.
 * Decoding is strict like base64ct's: ok[i] = 0 for characters outside the URL-safe alphabet ('=' padding included)
 * or non-zero trailing bits; raw[i] is then unspecified.  (A wrong string length is the caller's framing error.) */
size_t    eg_base64url_chars(size_t bytes_per_item);
eg_status eg_base64url_decode_batch(eg_ctx *ctx, size_t n, size_t bytes_per_item, const char *text, uint8_t *raw /* n*bytes */,
                                    uint8_t *ok /* n */);
eg_status eg_base64url_encode_batch(eg_ctx *ctx, size_t n, size_t bytes_per_item, const uint8_t *raw, char *text);
eg_status eg_base64url_decode_batch_dev(eg_ctx *ctx, size_t n, size_t bytes_per_item, const char *d_text, uint8_t *d_raw,
                                        uint8_t *d_ok);
eg_status eg_base64url_encode_batch_dev(eg_ctx *ctx, size_t n, size_t bytes_per_item, const uint8_t *d_raw, char *d_text);

/* Struct-level form of the same wire format.  An object is F fields = F strings of 43 characters (every field is a 32-byte
 * element or scalar), concatenated in struct-field order -- which is also the order of the flat binary layouts this header
 * uses, so the decoded bytes feed the batch entry points directly.  eg_wire_fields gives F for the objects whose vectors
 * carry a minimum length in the reference (`VecHelper<_, MIN>`, src/serde.rs:303-355) and returns 0 when `count` violates
 * it -- the reference fails deserialisation there with `invalid_length`; composite objects (RangeProof = (n_rings - 1)
 * ciphertexts + a ring proof, EncryptedChoice, QuadraticVotingBallot) are sums of these.  ok[i] = 1 iff all F strings of
 * object i are valid base64url; fields_per_object == 0 is EG_ERR_LEN_MISMATCH. */
enum {
    EG_WIRE_CIPHERTEXT = 0,             /* 2 fields */
    EG_WIRE_DECRYPTION = 1,             /* VerifiableDecryption: 1 field */
    EG_WIRE_LOG_EQUALITY_PROOF = 2,     /* 2 fields */
    EG_WIRE_COMMITMENT_EQUIV_PROOF = 3, /* 4 fields */
    EG_WIRE_RING_PROOF = 4,             /* 1 + count responses, count >= 2 (src/proofs/ring.rs:285) */
    EG_WIRE_POSSESSION_PROOF = 5,       /* 1 + count responses, count >= 1 (src/proofs/possession.rs:74) */
    EG_WIRE_SUMSQ_PROOF = 6             /* 1 + count ciphertext responses + 1, count >= 2 (src/proofs/mul.rs:89) */
};
size_t    eg_wire_fields(int kind, uint32_t count);
eg_status eg_wire_decode_batch(eg_ctx *ctx, size_t fields_per_object, size_t n, const char *text /* n*F*43 */,
                               uint8_t *raw /* n*F*32 */, uint8_t *ok /* n */);
eg_status eg_wire_encode_batch(eg_ctx *ctx, size_t fields_per_object, size_t n, const uint8_t *raw /* n*F*32 */,
                               char *text /* n*F*43 */);

/* ---- proofs and applications ------------------------------------------------------------------- */

/* PublicKey::verify_zero (src/keys/impls.rs:59-69) -> LogEqualityProof::verify (src/proofs/log_equality.rs:153-180) */
eg_status eg_verify_zero_batch(eg_ctx *ctx, size_t n, const uint8_t *cts /* n*64 */, const uint8_t *proofs /* n*64 */,
                               uint8_t *verdicts /* n */);
/* PublicKey::verify_bool (src/keys/impls.rs:101-113) -> RingProof::verify (src/proofs/ring.rs:302-374) */
eg_status eg_verify_bool_batch(eg_ctx *ctx, size_t n, const uint8_t *cts /* n*64 */, const uint8_t *proofs /* n*96 */,
                               uint8_t *verdicts /* n */);
/* EncryptedChoice::verify (src/app/choice.rs:358-380) for n ballots with `options` options each, followed by the
 * tally fold of examples/voting.rs:200-203 over the ballots whose verdict is EG_V_OK.
 *   single != 0: SingleChoice (sum proofs checked first, src/app/choice.rs:77-95); 0: MultiChoice (sums may be NULL).
 *   tally (options*64, may be NULL): sum of the verified ballots' ciphertexts, Ciphertext::to_bytes form. */
eg_status eg_verify_choice_batch(eg_ctx *ctx, size_t n, uint32_t options, int single,
                                 const uint8_t *choices /* n*options*64 */, const uint8_t *ring_proofs /* n*(1+2*options)*32 */,
                                 const uint8_t *sum_proofs /* n*64 or NULL */, uint8_t *verdicts /* n */,
                                 uint8_t *tally /* options*64 or NULL */);

/* RangeDecomposition (src/proofs/range.rs:106-108): rings listed as in `Display` (:110-124), most significant
 * first; ring i admits the values step[i] * {0, .., size[i]-1}. */
typedef struct {
    uint32_t n_rings;
    uint32_t reserved;
    uint64_t size[64];
    uint64_t step[64];
} eg_range;

/* RangeDecomposition::optimal (src/proofs/range.rs:148-153) */
eg_status eg_range_optimal(uint64_t upper_bound, eg_range *out);
/* Display for RangeDecomposition (src/proofs/range.rs:110-124); returns the length written (no NUL counted) */
size_t    eg_range_display(const eg_range *range, char *buf, size_t cap);

/* PublicKey::verify_range (src/keys/impls.rs:143-151) -> RangeProof::verify (src/proofs/range.rs:547-577);
 * `transcript_label` is the Transcript::new label ("ciphertext_range" for verify_range). */
eg_status eg_verify_range_batch(eg_ctx *ctx, const eg_range *range, const char *transcript_label, size_t n,
                                const uint8_t *cts /* n*64 */, const uint8_t *partial_cts /* n*(n_rings-1)*64 */,
                                const uint8_t *ring_proofs /* n*(1+sum(size))*32 */, uint8_t *verdicts /* n */);

/* QuadraticVotingParams::new (src/app/quadratic_voting.rs:63-76) */
typedef struct {
    uint32_t options;
    uint32_t reserved;
    uint64_t credits;
    eg_range vote_range;     /* optimal(isqrt(credits) + 1) */
    eg_range credit_range;   /* optimal(credits + 1) */
} eg_qv_params;
eg_status eg_qv_params_new(uint32_t options, uint64_t credits, eg_qv_params *out);
size_t    eg_qv_ballot_size(const eg_qv_params *params);
/* QuadraticVotingBallot::verify (src/app/quadratic_voting.rs:291-329) + tally of the vote ciphertexts.
 * Ballot bytes: for each option ct | partial cts | ring proof; then credit ct | partial cts | ring proof;
 * then SumOfSquaresProof = challenge | 2*options responses | sum response (src/proofs/mul.rs:86-93). */
eg_status eg_verify_qv_batch(eg_ctx *ctx, const eg_qv_params *params, size_t n, const uint8_t *ballots,
                             uint8_t *verdicts /* n */, uint8_t *tally /* options*64 or NULL */);

/* SumOfSquaresProof::verify (src/proofs/mul.rs:190-260; benched alone at benches/basics.rs:176) over a batch: item i proves
 * that sum_cts[i] encrypts the sum of squares of the values in its `count` ciphertexts (1..15), with `Transcript::new(label)`.
 * Proof layout = struct field order (:86-93): challenge | (r_resp, v_resp) x count | sum_resp = 32 (2 count + 2) bytes.
 * verdicts: EG_V_OK / EG_V_MALFORMED / EG_V_CHALLENGE_MISMATCH.  (A responses / ciphertexts count mismatch,
 * VerificationError::LenMismatch, cannot occur in a fixed-stride batch.) */
eg_status eg_verify_sumsq_batch(eg_ctx *ctx, const char *transcript_label, uint32_t count, size_t n, const uint8_t *cts /* n*count*64 */,
                                const uint8_t *sum_cts /* n*64 */, const uint8_t *proofs /* n*(2 count+2)*32 */, uint8_t *verdicts /* n */);

/* CandidateDecryption::verify (src/decryption.rs:189-205): item i claims that dh_elements[i] = [x]R_i for the secret key x
 * of the public `key` (custom key, not a key-set participant), proved by a LogEqualityProof with
 * `Transcript::new(label)` + start_proof("decryption_with_custom_key").  `key` is validated like PublicKey::from_bytes
 * (EG_ERR_INVALID_ELEMENT).  verdicts: EG_V_OK / EG_V_MALFORMED (CandidateDecryption::from_bytes :168-177, or a
 * non-canonical scalar) / EG_V_CHALLENGE_MISMATCH.  Needs no receiver key. */
eg_status eg_verify_decryption_batch(eg_ctx *ctx, const char *transcript_label, const uint8_t key[32], size_t n,
                                     const uint8_t *cts /* n*64 */, const uint8_t *dh_elements /* n*32 */,
                                     const uint8_t *proofs /* n*64 */, uint8_t *verdicts /* n */);

/* PublicKeySet (src/sharing/key_set.rs:19-26) */
typedef struct {
    uint32_t shares, threshold;
    uint8_t shared_key[32];
    uint8_t participant_keys[64][32];
} eg_keyset;

/* PublicKeySet::verify_share (src/sharing/key_set.rs:209-228) for n_tallies ciphertexts x n_shares candidate shares
 * each; share j of every tally comes from participant `indexes[j]`.  At most 8 shares per call (EG_ERR_INVALID_ARG
 * beyond; call again with the next group of participants).  Participant keys are validated like PublicKey::from_bytes
 * (src/keys/mod.rs:161-176): undecodable or identity -> EG_ERR_INVALID_ELEMENT. */
eg_status eg_verify_shares_batch(eg_ctx *ctx, const eg_keyset *keyset, size_t n_tallies, uint32_t n_shares,
                                 const uint32_t *indexes /* n_shares */, const uint8_t *cts /* n_tallies*64 */,
                                 const uint8_t *shares /* n_tallies*n_shares*32 */,
                                 const uint8_t *proofs /* n_tallies*n_shares*64 */,
                                 uint8_t *verdicts /* n_tallies*n_shares */);

/* CommitmentEquivalenceProof::verify (src/proofs/commitment.rs:198-248) over a batch, against the receiver key and the
 * blinding base of the context, with `Transcript::new(label)`.  The reference gives this proof a serde form only; the
 * 128-byte layout is the struct's field order (:126-135): challenge | randomness_response | value_response |
 * commitment_response.  verdicts: EG_V_OK / EG_V_MALFORMED / EG_V_CHALLENGE_MISMATCH. */
eg_status eg_verify_commitment_equiv_batch(eg_ctx *ctx, const char *transcript_label, size_t n, const uint8_t *cts /* n*64 */,
                                           const uint8_t *commitments /* n*32 */, const uint8_t *proofs /* n*128 */,
                                           uint8_t *verdicts /* n */);

/* ProofOfPossession::verify (src/proofs/possession.rs:137-163) over a batch of proofs for `keys_per_proof` public keys
 * each (1..64), with `Transcript::new(label)`.  Proof layout = struct field order (:71-76): challenge | responses.
 * A key that does not decode or is the identity is EG_V_MALFORMED (PublicKey::from_bytes, src/keys/mod.rs:161-176); a
 * responses / keys count mismatch cannot occur in a fixed-stride batch.  Needs no receiver key. */
eg_status eg_verify_possession_batch(eg_ctx *ctx, const char *transcript_label, uint32_t keys_per_proof, size_t n,
                                     const uint8_t *keys /* n*keys_per_proof*32 */,
                                     const uint8_t *proofs /* n*(1+keys_per_proof)*32 */, uint8_t *verdicts /* n */);

/* PublicKeySet::from_participants (src/sharing/key_set.rs:87-144) over n_sets key sets with the same (shares, threshold),
 * threshold <= 16: reconstructs each shared key from the first `threshold` participant keys and checks that the other
 * participant keys lie on the same polynomial.  verdicts: EG_V_OK (shared_keys[i] set), EG_V_MALFORMED (a key does not
 * decode or is the identity), EG_V_MALFORMED_PARTICIPANT_KEYS.  `ParticipantCountMismatch` cannot occur in a fixed-stride
 * batch.  Needs no receiver key. */
eg_status eg_keysets_validate_batch(eg_ctx *ctx, uint32_t shares, uint32_t threshold, size_t n_sets,
                                    const uint8_t *keys /* n_sets*shares*32 */, uint8_t *shared_keys /* n_sets*32 */,
                                    uint8_t *verdicts /* n_sets */);

/* DiscreteLogTable::new (src/encryption.rs:267-284) for the values lo..hi (exclusive); lives on the device */
eg_status eg_dlog_table_create(eg_ctx *ctx, uint64_t lo, uint64_t hi, eg_dlog_table **out);
void      eg_dlog_table_destroy(eg_dlog_table *table);

/* Params::combine_shares (src/sharing/mod.rs:302-325) on the first `threshold` shares of every tally, then
 * VerifiableDecryption::decrypt (src/decryption.rs:138-144) through DiscreteLogTable::get (src/encryption.rs:287-297).
 * found[i] = 1 and values[i] set when the decrypted element is in the table (identity -> 0), found[i] = 0 when it
 * is not (Option::None), found[i] = 2 when an input element does not decode. */
eg_status eg_combine_decrypt_batch(eg_ctx *ctx, uint32_t threshold, const uint32_t *indexes /* threshold */,
                                   size_t n_tallies, uint32_t share_stride /* shares per tally in `shares` */,
                                   const uint8_t *cts /* n_tallies*64 */, const uint8_t *shares,
                                   const eg_dlog_table *table, uint64_t *values /* n */, uint8_t *found /* n */);

/* ---- encryption side (encrypt_* drop-ins with caller-supplied randomness) ----------------------- */

/* PublicKey::encrypt (src/keys/impls.rs:16-23 -> ExtendedCiphertext::new src/encryption.rs:310-327): one block per item
 * (the randomness r); cts[i] = ([r]G, [values[i]]G + [r]K). */
eg_status eg_encrypt_batch(eg_ctx *ctx, size_t n, const uint64_t *values /* n */, const uint8_t *wide_rand /* n*64 */,
                           uint8_t *cts /* n*64 */);
/* PublicKey::encrypt_zero (src/keys/impls.rs:30-53): two blocks per item (r, then the LogEqualityProof::new nonce,
 * src/proofs/log_equality.rs:114-143); proofs[i] = challenge | response as LogEqualityProof::to_bytes. */
eg_status eg_encrypt_zero_batch(eg_ctx *ctx, size_t n, const uint8_t *wide_rand /* n*2*64 */, uint8_t *cts /* n*64 */,
                                uint8_t *proofs /* n*64 */);
/* PublicKey::encrypt_bool (src/keys/impls.rs:77-89).  The reference draws from a CryptoRng; here the caller supplies the
 * randomness: item i consumes three 64-byte blocks in the reference's draw order (SURVEY.md A.4: r, x, forged
 * response), each reduced mod l as Ristretto::generate_scalar does (src/group/ristretto.rs:28-32).  With blocks taken
 * from the same ChaCha20 stream the outputs are byte-identical to the reference's.  values[i] != 0 encrypts `true`. */
eg_status eg_encrypt_bool_batch(eg_ctx *ctx, size_t n, const uint8_t *values /* n */, const uint8_t *wide_rand /* n*3*64 */,
                                uint8_t *cts /* n*64 */, uint8_t *proofs /* n*96 */);
/* EncryptedChoice::new / ::single (src/app/choice.rs:288-349): values[i*options + k] != 0 marks option k of ballot i
 * (exactly one for `single`); item i consumes 3*options (+1 for the sum proof when `single`) blocks: r, x and -- for a
 * zero option -- the forged response per option in option order, then the forged responses of the chosen options,
 * then the sum-proof nonce.  sum_proofs may be NULL when single == 0.  With single != 0 a row that does not mark exactly
 * one option is EG_ERR_INVALID_ARG (EncryptedChoice::single cannot produce such a ballot, src/app/choice.rs:288-306). */
eg_status eg_encrypt_choice_batch(eg_ctx *ctx, size_t n, uint32_t options, int single, const uint8_t *values /* n*options */,
                                  const uint8_t *wide_rand /* n*(3*options+single)*64 */, uint8_t *choices /* n*options*64 */,
                                  uint8_t *ring_proofs /* n*(1+2*options)*32 */, uint8_t *sum_proofs /* n*64 */);

/* PublicKey::encrypt_range (src/keys/impls.rs:121-141) = RangeProof::new (src/proofs/range.rs:462-534) with
 * `Transcript::new(label)`.  Item i consumes eg_range_prover_draws(range) = n_rings + sum(ring sizes) blocks in the
 * reference's draw order: r of the ciphertext; per ring, in order: r of the partial ciphertext (not for the last ring,
 * which is derived, range.rs:520-529), the ring's nonce, the forged responses above the value's index (ring.rs:97-131);
 * then per ring, in order, the forged responses below it (Ring::finalize ring.rs:162-195).  values[i] must be below the
 * range's upper bound (the reference panics, range.rs:365-369): EG_ERR_INVALID_ARG otherwise.
 * Outputs use the layouts eg_verify_range_batch reads. */
size_t    eg_range_prover_draws(const eg_range *range);
eg_status eg_encrypt_range_batch(eg_ctx *ctx, const eg_range *range, const char *transcript_label, size_t n,
                                 const uint64_t *values /* n */, const uint8_t *wide_rand /* n*draws*64 */,
                                 uint8_t *cts /* n*64 */, uint8_t *partials /* n*(n_rings-1)*64 */,
                                 uint8_t *ring_proofs /* n*(1+sum sizes)*32 */);

/* RangeProof::from_ciphertext (src/proofs/range.rs:482-534): proofs for ciphertexts that exist already (made with
 * CiphertextWithValue::new / eg_encrypt_batch), whose values and randomness the caller holds.  ct_randomness = one canonical
 * scalar per item (EG_ERR_INVALID_ARG otherwise); item i consumes eg_range_prover_draws(range) - 1 blocks, in the order
 * above without its first block.  cts (optional, may be NULL) receives the re-encryption ([r]G, [v]G + [r]K) for checking. */
eg_status eg_prove_range_batch(eg_ctx *ctx, const eg_range *range, const char *transcript_label, size_t n, const uint64_t *values /* n */,
                               const uint8_t *ct_randomness /* n*32 */, const uint8_t *wide_rand /* n*(draws-1)*64 */,
                               uint8_t *cts /* n*64 or NULL */, uint8_t *partials, uint8_t *ring_proofs);

/* QuadraticVotingBallot::new (src/app/quadratic_voting.rs:234-284).  votes[i*options + k] = votes of ballot i for
 * option k.  Item i consumes eg_qv_prover_draws(params) blocks: one RangeProof::new per option over the vote range, one for
 * credit = sum votes^2 over the credit range, then SumOfSquaresProof::new (src/proofs/mul.rs:107-181: e_z, then e_r, e_x per
 * option).  A vote or credit outside its range (a panic in the reference) is EG_ERR_INVALID_ARG.
 * Ballots use the layout eg_verify_qv_batch reads. */
size_t    eg_qv_prover_draws(const eg_qv_params *params);
eg_status eg_encrypt_qv_batch(eg_ctx *ctx, const eg_qv_params *params, size_t n, const uint64_t *votes /* n*options */,
                              const uint8_t *wide_rand /* n*draws*64 */, uint8_t *ballots /* n*eg_qv_ballot_size */);

/* ---- encryption side with in-kernel randomness ---------------------------------------------------
 * The same provers, but every 64-byte block is produced inside the kernel by ChaCha20 (RFC 8439 block function, 64-bit
 * block counter, stream id 0 -- rand_chacha's ChaCha20Rng, the generator of tests/snapshots.rs:31-34 and
 * benches/basics.rs:17) instead of crossing PCIe (64 B per draw: 2560 B per range proof, 3392 B per quadratic-voting
 * ballot).  `seed` is the 32-byte ChaCha20 key; item i of the batch draws from its own stream: draw number k (in the draw
 * order documented above for the caller-supplied form) is the block with counter  counter_base + (i << 20) + k.  Hence
 *   - the outputs equal those of the caller-supplied form fed with these blocks, byte for byte;
 *   - counter_base = 1, n = 1 and the key of `ChaChaRng::seed_from_u64(12345)` reproduces the reference snapshots (block 0
 *     of that stream is the receiver's secret key, tests/snapshots.rs:32-34);
 *   - the seed is a SECRET of the same weight as the randomness it replaces: one seed per batch from the host's CSPRNG. */
eg_status eg_encrypt_batch_seeded(eg_ctx *ctx, size_t n, const uint64_t *values, const uint8_t seed[32], uint64_t counter_base,
                                  uint8_t *cts);
eg_status eg_encrypt_zero_batch_seeded(eg_ctx *ctx, size_t n, const uint8_t seed[32], uint64_t counter_base, uint8_t *cts,
                                       uint8_t *proofs);
eg_status eg_encrypt_bool_batch_seeded(eg_ctx *ctx, size_t n, const uint8_t *values, const uint8_t seed[32], uint64_t counter_base,
                                       uint8_t *cts, uint8_t *proofs);
eg_status eg_encrypt_choice_batch_seeded(eg_ctx *ctx, size_t n, uint32_t options, int single, const uint8_t *values,
                                         const uint8_t seed[32], uint64_t counter_base, uint8_t *choices, uint8_t *ring_proofs,
                                         uint8_t *sum_proofs);
eg_status eg_encrypt_range_batch_seeded(eg_ctx *ctx, const eg_range *range, const char *transcript_label, size_t n,
                                        const uint64_t *values, const uint8_t seed[32], uint64_t counter_base, uint8_t *cts,
                                        uint8_t *partials, uint8_t *ring_proofs);
eg_status eg_prove_range_batch_seeded(eg_ctx *ctx, const eg_range *range, const char *transcript_label, size_t n, const uint64_t *values,
                                      const uint8_t *ct_randomness /* n*32 */, const uint8_t seed[32], uint64_t counter_base,
                                      uint8_t *cts /* or NULL */, uint8_t *partials, uint8_t *ring_proofs);
eg_status eg_encrypt_qv_batch_seeded(eg_ctx *ctx, const eg_qv_params *params, size_t n, const uint64_t *votes, const uint8_t seed[32],
                                     uint64_t counter_base, uint8_t *ballots);

/* Side-channel posture of the encryption side (the reference: constant-time G::mul_generator / multi_mul and zeroizing
 * secret wrappers, src/proofs/ring.rs:97-116, src/group/mod.rs:79).
 *   constant_time = 0 (default): secret scalars (randomness r, nonces x) walk the wide-window (24-bit) fixed-base tables with
 *     secret-dependent addresses and skip zero digits -- fastest; appropriate when the GPU is not shared with an adversary.
 *   constant_time = 1: every fixed-base multiplication by a secret scalar uses 64 signed 4-bit windows, reads all eight
 *     candidate entries of a window and selects with masks, always adds; no branch or address depends on a secret scalar
 *     (64 instead of 11 additions per base).  Scalar arithmetic mod l is branch-free in both modes.  As in the reference, the
 *     *shape* of a ring proof's computation (which equation is the real one) follows the encrypted value.
 * In both modes the device scratch that held randomness, nonces, plaintext values and staged randomness blocks is zeroed
 * before a prover call returns.  Verification entry points only handle public data and stay variable-time. */
eg_status eg_ctx_set_prover_mode(eg_ctx *ctx, int constant_time);

/* ---- decryption side (the talliers' operations; they hold a secret) ------------------------------
 * None of these needs a receiver key.  A secret that is not a canonical scalar is EG_ERR_INVALID_ARG.  The secret's digits
 * follow eg_ctx_set_prover_mode like the nonces' (s = c secret + x: a leaked nonce reveals the key), the key travels by
 * value in the kernel launch parameters, and the staging buffers are zeroed before a host-pointer call returns.  On a
 * multi-device context the host forms shard the batch; item i keeps its own randomness either way. */

/* SecretKey::decrypt_to_element / decrypt (src/keys/impls.rs:160-177) -> DiscreteLogTable::get (src/encryption.rs:287-297).
 * elements (n*32, may be NULL): encode(B - [secret]R).  table may be NULL (then values may be NULL).
 * found[i]: as eg_combine_decrypt_batch (1 found / identity -> 0, 0 absent, 2 ciphertext does not decode);
 * without a table 1 = decoded, 2 = does not decode. */
eg_status eg_decrypt_batch(eg_ctx *ctx, const uint8_t secret[32], size_t n, const uint8_t *cts /* n*64 */,
                           const eg_dlog_table *table, uint8_t *elements, uint64_t *values, uint8_t *found /* n */);

/* ActiveParticipant::decrypt_share (src/sharing/participant.rs:163-185): participant `index` of `keyset` with its secret
 * share; one 64-byte block per item (the LogEqualityProof::new nonce, src/proofs/log_equality.rs:114-143).
 * shares[i] / proofs[i] in the layouts eg_verify_shares_batch reads (one column of its n_tallies x n_shares arrays).
 * ok[i] = 0 (outputs zeroed) when cts[i] does not decode.  index >= keyset->shares is EG_ERR_INVALID_ARG; the participant
 * key is validated like PublicKey::from_bytes (EG_ERR_INVALID_ELEMENT); [secret_share]G != participant_keys[index] is
 * EG_ERR_INVALID_ARG (the reference cannot build such an ActiveParticipant). */
eg_status eg_decrypt_share_batch(eg_ctx *ctx, const eg_keyset *keyset, uint32_t index, const uint8_t secret_share[32], size_t n,
                                 const uint8_t *cts /* n*64 */, const uint8_t *wide_rand /* n*64 */, uint8_t *shares /* n*32 */,
                                 uint8_t *proofs /* n*64 */, uint8_t *ok /* n */);
eg_status eg_decrypt_share_batch_seeded(eg_ctx *ctx, const eg_keyset *keyset, uint32_t index, const uint8_t secret_share[32], size_t n,
                                        const uint8_t *cts, const uint8_t seed[32], uint64_t counter_base, uint8_t *shares,
                                        uint8_t *proofs, uint8_t *ok);
/* device pointers on a single-device context; seed == NULL -> one block per item at d_wide_rand (as eg_encrypt_*_batch_dev) */
eg_status eg_decrypt_share_batch_dev(eg_ctx *ctx, const eg_keyset *keyset, uint32_t index, const uint8_t secret_share[32], size_t n,
                                     const uint8_t *d_cts, const uint8_t *d_wide_rand, const uint8_t seed[32], uint64_t counter_base,
                                     uint8_t *d_shares, uint8_t *d_proofs, uint8_t *d_ok);

/* VerifiableDecryption::new with the key pair (secret, [secret]G) (src/decryption.rs:89-111), Transcript::new(label).
 * One block per item (the proof nonce).  Outputs are what eg_verify_decryption_batch(label, [secret]G, ...) accepts;
 * ok[i] = 0 (outputs zeroed) when cts[i] does not decode. */
eg_status eg_prove_decryption_batch(eg_ctx *ctx, const char *transcript_label, const uint8_t secret[32], size_t n,
                                    const uint8_t *cts /* n*64 */, const uint8_t *wide_rand /* n*64 */, uint8_t *dh_elements /* n*32 */,
                                    uint8_t *proofs /* n*64 */, uint8_t *ok /* n */);
eg_status eg_prove_decryption_batch_seeded(eg_ctx *ctx, const char *transcript_label, const uint8_t secret[32], size_t n,
                                           const uint8_t *cts, const uint8_t seed[32], uint64_t counter_base, uint8_t *dh_elements,
                                           uint8_t *proofs, uint8_t *ok);

/* ---- device-pointer variants (inputs already resident in HBM; same semantics) ------------------- */
eg_status eg_verify_bool_batch_dev(eg_ctx *ctx, size_t n, const uint8_t *d_cts, const uint8_t *d_proofs, uint8_t *d_verdicts);
eg_status eg_verify_choice_batch_dev(eg_ctx *ctx, size_t n, uint32_t options, int single, const uint8_t *d_choices,
                                     const uint8_t *d_ring_proofs, const uint8_t *d_sum_proofs, uint8_t *d_verdicts,
                                     uint8_t *d_tally);
eg_status eg_verify_range_batch_dev(eg_ctx *ctx, const eg_range *range, const char *transcript_label, size_t n,
                                    const uint8_t *d_cts, const uint8_t *d_partial_cts, const uint8_t *d_ring_proofs,
                                    uint8_t *d_verdicts);
/* QuadraticVotingBallot::verify, PublicKeySet::verify_share and combine_shares + decrypt on device buffers */
eg_status eg_verify_qv_batch_dev(eg_ctx *ctx, const eg_qv_params *params, size_t n, const uint8_t *d_ballots, uint8_t *d_verdicts,
                                 uint8_t *d_tally);
eg_status eg_verify_shares_batch_dev(eg_ctx *ctx, const eg_keyset *keyset, size_t n_tallies, uint32_t n_shares, const uint32_t *indexes,
                                     const uint8_t *d_cts, const uint8_t *d_shares, const uint8_t *d_proofs, uint8_t *d_verdicts);
eg_status eg_combine_decrypt_batch_dev(eg_ctx *ctx, uint32_t threshold, const uint32_t *indexes, size_t n_tallies, uint32_t share_stride,
                                       const uint8_t *d_cts, const uint8_t *d_shares, const eg_dlog_table *table, uint64_t *d_values,
                                       uint8_t *d_found);
/* Provers on device buffers: values in, objects out, all in HBM of the context's device.  Randomness: `seed` (32 bytes, HOST
 * pointer) + counter_base as in the _seeded forms, or -- with seed == NULL -- blocks already resident at d_wide_rand in the
 * layout of the host forms.  The domain checks the host forms make on the values (exactly one option for `single`, value
 * below the range's bound) are the caller's here: a violating item yields an object that fails verification. */
eg_status eg_encrypt_bool_batch_dev(eg_ctx *ctx, size_t n, const uint8_t *d_values, const uint8_t *d_wide_rand, const uint8_t seed[32],
                                    uint64_t counter_base, uint8_t *d_cts, uint8_t *d_proofs);
eg_status eg_encrypt_choice_batch_dev(eg_ctx *ctx, size_t n, uint32_t options, int single, const uint8_t *d_values,
                                      const uint8_t *d_wide_rand, const uint8_t seed[32], uint64_t counter_base, uint8_t *d_choices,
                                      uint8_t *d_ring_proofs, uint8_t *d_sum_proofs);
eg_status eg_encrypt_range_batch_dev(eg_ctx *ctx, const eg_range *range, const char *transcript_label, size_t n, const uint64_t *d_values,
                                     const uint8_t *d_wide_rand, const uint8_t seed[32], uint64_t counter_base, uint8_t *d_cts,
                                     uint8_t *d_partials, uint8_t *d_ring_proofs);
/* eg_ciphertexts_sum on device buffers, asynchronous on the context's stream: the local combine after the all_gather
 * of per-GPU partial tallies.  *d_bad_flag (optional, device) becomes non-zero when a part does not decode. */
eg_status eg_ciphertexts_sum_dev(eg_ctx *ctx, size_t n_parts, size_t n_cts, const uint8_t *d_parts, uint8_t *d_out,
                                 uint32_t *d_bad_flag);

/* ---- instrumentation --------------------------------------------------------------------------- */
/* Number of kernels this context has launched since creation (bench.py's `gpu_launches`). */
uint64_t  eg_kernel_launch_count(const eg_ctx *ctx);
/* Device time in ms of the last batch call (CUDA events on the context's stream), split by stage:
 * [0] decode + derived ciphertexts, [1] commitments + transcripts + verdicts, [2] the k_commit launches alone
 * (one event pair per launch), [3] tally, [4] total of [0]+[1]+[3]. */
eg_status eg_last_timings(const eg_ctx *ctx, float out_ms[5]);
/* The equation-evaluation kernels (k_ring + k_commit) in the last batch call: number of launches, number of
 * verification-equation sides evaluated, summed device time of those launches (one CUDA event pair per launch). */
eg_status eg_last_commit_stats(const eg_ctx *ctx, uint64_t *launches, uint64_t *tasks, float *ms);
/* The same split by kernel: kind 0 = k_commit (single-use equation sides), kind 1 = k_ring (one thread per ring),
 * kind 2 = k_msm (general multi-scalar sums: share proofs, sum-of-squares, Lagrange recombination; tasks = sums),
 * kind 3 = k_ring_pair (two lanes per ring, small chunks; tasks = equation sides). */
eg_status eg_last_kernel_stats(const eg_ctx *ctx, int kind, uint64_t *launches, uint64_t *tasks, float *ms);
/* On-device self-test of the tuned GF(2^255-19) multiply / square / add / sub against the portable formulation on
 * n pseudo-random and edge-case operands; *mismatches must come back 0. */
eg_status eg_selftest_field(eg_ctx *ctx, size_t n, uint64_t seed, uint64_t *mismatches);
/* Tuning knob: items processed per internal chunk (0 = default 262144).  Results do not depend on it. */
eg_status eg_ctx_set_chunk_items(eg_ctx *ctx, size_t items);
/* Tuning / A-B knob for RingProof verification: 2 = one thread per ring with per-point chunked window tables (k_ring,
 * 64 doublings per equation; the engine for large batches); 1 = one launch per equation index with one thread per
 * equation side (k_commit + k_ring_hash, 252 doublings); 3 = two lanes per ring, one per equation side, each with the
 * chunked tables of its own point (k_ring_pair: the shortest per-thread chain, for chunks smaller than the GPU);
 * 0 (default) = chosen per chunk from the measured crossovers: 3 for small chunks that are rings only (bool, range, QV),
 * 1 for small chunks with extra single-use equations (the sum proof of an EncryptedChoice), 2 otherwise.  Results do
 * not depend on it. */
eg_status eg_ctx_set_ring_mode(eg_ctx *ctx, int mode);
/* Tuning knob for PublicKeySet::verify_share / CandidateDecryption::verify: from `min_tallies` per call on, the keys the
 * shares are checked against (batch constants) get 48 MiB fixed-base tables of their own (built on the device in ~1 ms each,
 * kept while the same keys are used), which removes the 252-doubling chain on the key from every share.  Default 32768
 * (a table costs about what it saves on 12 000 tallies); 0 = always, SIZE_MAX = never.  Results do not depend on it. */
eg_status eg_ctx_set_key_table_min(eg_ctx *ctx, size_t min_tallies);
/* Raw CUDA stream handle (cudaStream_t) so callers can order their own work / time with events on it. */
void     *eg_ctx_stream(const eg_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* EG_B200_H */
