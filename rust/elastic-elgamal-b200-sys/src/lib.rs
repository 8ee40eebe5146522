//! Raw `extern "C"` declarations for `include/eg_b200.h` (1:1, no logic).
//!
//! NOTE: this crate is *source only* in the build image (no rustc there); it is the binding a maintainer of
//! `slowli/elastic-elgamal` would compile against `libeg_b200.so`.  See INTEGRATION.md.
#![allow(non_camel_case_types)]

use core::ffi::{c_char, c_int, c_void};

#[repr(C)]
pub struct eg_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct eg_dlog_table {
    _private: [u8; 0],
}
pub type eg_status = i32;

pub const EG_SUCCESS: eg_status = 0;
pub const EG_ERR_INVALID_ARG: eg_status = 1;
pub const EG_ERR_INVALID_ELEMENT: eg_status = 2;
pub const EG_ERR_IDENTITY_KEY: eg_status = 3;
pub const EG_ERR_NO_RECEIVER: eg_status = 4;
pub const EG_ERR_NO_DEVICE: eg_status = 5;
pub const EG_ERR_CUDA: eg_status = 6;
pub const EG_ERR_OUT_OF_MEMORY: eg_status = 7;
pub const EG_ERR_LEN_MISMATCH: eg_status = 8;
pub const EG_ERR_NCCL: eg_status = 9;

/// Size of the NCCL unique id exchanged by `eg_comm_unique_id` / `eg_ctx_attach_comm`.
pub const EG_COMM_ID_BYTES: usize = 128;

pub const EG_WIRE_CIPHERTEXT: c_int = 0;
pub const EG_WIRE_DECRYPTION: c_int = 1;
pub const EG_WIRE_LOG_EQUALITY_PROOF: c_int = 2;
pub const EG_WIRE_COMMITMENT_EQUIV_PROOF: c_int = 3;
pub const EG_WIRE_RING_PROOF: c_int = 4;
pub const EG_WIRE_POSSESSION_PROOF: c_int = 5;
pub const EG_WIRE_SUMSQ_PROOF: c_int = 6;

pub const EG_V_OK: u8 = 0;
pub const EG_V_MALFORMED: u8 = 1;
pub const EG_V_CHALLENGE_MISMATCH: u8 = 2;
pub const EG_V_CHOICE_SUM: u8 = 3;
pub const EG_V_CHOICE_RANGE: u8 = 4;
pub const EG_V_QV_CREDIT_RANGE: u8 = 5;
pub const EG_V_QV_CREDIT_EQUIV: u8 = 6;
pub const EG_V_MALFORMED_PARTICIPANT_KEYS: u8 = 7;
pub const EG_V_QV_VARIANT_BASE: u8 = 16;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct eg_range {
    pub n_rings: u32,
    pub reserved: u32,
    pub size: [u64; 64],
    pub step: [u64; 64],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct eg_qv_params {
    pub options: u32,
    pub reserved: u32,
    pub credits: u64,
    pub vote_range: eg_range,
    pub credit_range: eg_range,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct eg_keyset {
    pub shares: u32,
    pub threshold: u32,
    pub shared_key: [u8; 32],
    pub participant_keys: [[u8; 32]; 64],
}

extern "C" {
    pub fn eg_ctx_create_multi(device_ids: *const c_int, n_dev: c_int, out: *mut *mut eg_ctx) -> eg_status;
    pub fn eg_comm_unique_id(id: *mut u8) -> eg_status;
    pub fn eg_ctx_attach_comm(ctx: *mut eg_ctx, id: *const u8, rank: c_int, world: c_int) -> eg_status;
    pub fn eg_ctx_comm_info(ctx: *const eg_ctx, rank: *mut c_int, world: *mut c_int, devices: *mut c_int) -> eg_status;
    pub fn eg_ctx_create(device_id: c_int, out: *mut *mut eg_ctx) -> eg_status;
    pub fn eg_ctx_destroy(ctx: *mut eg_ctx);
    pub fn eg_last_error(ctx: *const eg_ctx) -> *const c_char;
    pub fn eg_version() -> *const c_char;
    pub fn eg_ctx_set_receiver(ctx: *mut eg_ctx, key: *const u8) -> eg_status;

    pub fn eg_wire_fields(kind: c_int, count: u32) -> usize;
    pub fn eg_wire_decode_batch(ctx: *mut eg_ctx, fields_per_object: usize, n: usize, text: *const c_char, raw: *mut u8, ok: *mut u8) -> eg_status;
    pub fn eg_wire_encode_batch(ctx: *mut eg_ctx, fields_per_object: usize, n: usize, raw: *const u8, text: *mut c_char) -> eg_status;
    pub fn eg_elements_validate(ctx: *mut eg_ctx, n: usize, encodings: *const u8, ok: *mut u8) -> eg_status;
    pub fn eg_scalars_validate(ctx: *mut eg_ctx, n: usize, scalars: *const u8, ok: *mut u8) -> eg_status;
    pub fn eg_scalars_from_wide(ctx: *mut eg_ctx, n: usize, wide: *const u8, scalars: *mut u8) -> eg_status;
    pub fn eg_double_mul_generator_batch(ctx: *mut eg_ctx, n: usize, a: *const u8, big_a: *const u8, b: *const u8,
                                         out: *mut u8, ok: *mut u8) -> eg_status;
    pub fn eg_mul_generator_batch(ctx: *mut eg_ctx, n: usize, k: *const u8, out: *mut u8, ok: *mut u8) -> eg_status;
    pub fn eg_ciphertexts_sum(ctx: *mut eg_ctx, n_parts: usize, n_cts: usize, parts: *const u8, out: *mut u8,
                              ok: *mut u8) -> eg_status;

    pub fn eg_verify_zero_batch(ctx: *mut eg_ctx, n: usize, cts: *const u8, proofs: *const u8, verdicts: *mut u8) -> eg_status;
    pub fn eg_verify_bool_batch(ctx: *mut eg_ctx, n: usize, cts: *const u8, proofs: *const u8, verdicts: *mut u8) -> eg_status;
    pub fn eg_verify_choice_batch(ctx: *mut eg_ctx, n: usize, options: u32, single: c_int, choices: *const u8,
                                  ring_proofs: *const u8, sum_proofs: *const u8, verdicts: *mut u8, tally: *mut u8) -> eg_status;
    pub fn eg_range_optimal(upper_bound: u64, out: *mut eg_range) -> eg_status;
    pub fn eg_range_display(range: *const eg_range, buf: *mut c_char, cap: usize) -> usize;
    pub fn eg_verify_range_batch(ctx: *mut eg_ctx, range: *const eg_range, transcript_label: *const c_char, n: usize,
                                 cts: *const u8, partial_cts: *const u8, ring_proofs: *const u8, verdicts: *mut u8) -> eg_status;
    pub fn eg_qv_params_new(options: u32, credits: u64, out: *mut eg_qv_params) -> eg_status;
    pub fn eg_qv_ballot_size(params: *const eg_qv_params) -> usize;
    pub fn eg_verify_qv_batch(ctx: *mut eg_ctx, params: *const eg_qv_params, n: usize, ballots: *const u8,
                              verdicts: *mut u8, tally: *mut u8) -> eg_status;
    pub fn eg_verify_sumsq_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, count: u32, n: usize, cts: *const u8, sum_cts: *const u8, proofs: *const u8, verdicts: *mut u8) -> eg_status;
    pub fn eg_verify_decryption_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, key: *const u8, n: usize, cts: *const u8, dh_elements: *const u8, proofs: *const u8, verdicts: *mut u8) -> eg_status;
    pub fn eg_verify_shares_batch(ctx: *mut eg_ctx, keyset: *const eg_keyset, n_tallies: usize, n_shares: u32,
                                  indexes: *const u32, cts: *const u8, shares: *const u8, proofs: *const u8,
                                  verdicts: *mut u8) -> eg_status;
    pub fn eg_keysets_validate_batch(ctx: *mut eg_ctx, shares: u32, threshold: u32, n_sets: usize, keys: *const u8,
                                     shared_keys: *mut u8, verdicts: *mut u8) -> eg_status;
    pub fn eg_dlog_table_create(ctx: *mut eg_ctx, lo: u64, hi: u64, out: *mut *mut eg_dlog_table) -> eg_status;
    pub fn eg_dlog_table_destroy(table: *mut eg_dlog_table);
    pub fn eg_dlog_table_create_bsgs(ctx: *mut eg_ctx, lo: u64, hi: u64, baby_steps: u64, out: *mut *mut eg_dlog_table) -> eg_status;
    pub fn eg_dlog_lookup_batch(ctx: *mut eg_ctx, table: *const eg_dlog_table, n: usize, elements: *const u8, values: *mut u64,
                                found: *mut u8) -> eg_status;
    pub fn eg_combine_decrypt_batch(ctx: *mut eg_ctx, threshold: u32, indexes: *const u32, n_tallies: usize,
                                    share_stride: u32, cts: *const u8, shares: *const u8, table: *const eg_dlog_table,
                                    values: *mut u64, found: *mut u8) -> eg_status;
    pub fn eg_combine_decrypt_accepted_batch(ctx: *mut eg_ctx, threshold: u32, n_shares: u32, indexes: *const u32, n_tallies: usize,
                                             cts: *const u8, shares: *const u8, verdicts: *const u8, table: *const eg_dlog_table,
                                             values: *mut u64, found: *mut u8) -> eg_status;

    pub fn eg_verify_bool_batch_dev(ctx: *mut eg_ctx, n: usize, d_cts: *const u8, d_proofs: *const u8, d_verdicts: *mut u8) -> eg_status;
    pub fn eg_verify_choice_batch_dev(ctx: *mut eg_ctx, n: usize, options: u32, single: c_int, d_choices: *const u8,
                                      d_ring_proofs: *const u8, d_sum_proofs: *const u8, d_verdicts: *mut u8,
                                      d_tally: *mut u8) -> eg_status;
    pub fn eg_verify_range_batch_dev(ctx: *mut eg_ctx, range: *const eg_range, transcript_label: *const c_char, n: usize,
                                     d_cts: *const u8, d_partial_cts: *const u8, d_ring_proofs: *const u8,
                                     d_verdicts: *mut u8) -> eg_status;

    pub fn eg_ctx_set_blinding_base(ctx: *mut eg_ctx, base: *const u8) -> eg_status;
    pub fn eg_ctx_set_ring_mode(ctx: *mut eg_ctx, mode: c_int) -> eg_status;
    pub fn eg_ctx_set_key_table_min(ctx: *mut eg_ctx, min_tallies: usize) -> eg_status;

    pub fn eg_multi_mul_batch(ctx: *mut eg_ctx, n: usize, terms: u32, scalars: *const u8, points: *const u8, out: *mut u8,
                              ok: *mut u8) -> eg_status;
    pub fn eg_ciphertexts_lincomb_batch(ctx: *mut eg_ctx, n: usize, terms: u32, scalars: *const u8, cts: *const u8, out: *mut u8,
                                        ok: *mut u8) -> eg_status;
    pub fn eg_verify_qv_batch_dev(ctx: *mut eg_ctx, params: *const eg_qv_params, n: usize, d_ballots: *const u8, d_verdicts: *mut u8, d_tally: *mut u8) -> eg_status;
    pub fn eg_verify_shares_batch_dev(ctx: *mut eg_ctx, keyset: *const eg_keyset, n_tallies: usize, n_shares: u32, indexes: *const u32, d_cts: *const u8, d_shares: *const u8, d_proofs: *const u8, d_verdicts: *mut u8) -> eg_status;
    pub fn eg_combine_decrypt_batch_dev(ctx: *mut eg_ctx, threshold: u32, indexes: *const u32, n_tallies: usize, share_stride: u32, d_cts: *const u8, d_shares: *const u8, table: *const eg_dlog_table, d_values: *mut u64, d_found: *mut u8) -> eg_status;
    pub fn eg_combine_decrypt_accepted_batch_dev(ctx: *mut eg_ctx, threshold: u32, n_shares: u32, indexes: *const u32, n_tallies: usize, d_cts: *const u8, d_shares: *const u8, d_verdicts: *const u8, table: *const eg_dlog_table, d_values: *mut u64, d_found: *mut u8) -> eg_status;
    pub fn eg_encrypt_bool_batch_dev(ctx: *mut eg_ctx, n: usize, d_values: *const u8, d_wide_rand: *const u8, seed: *const u8, counter_base: u64, d_cts: *mut u8, d_proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_choice_batch_dev(ctx: *mut eg_ctx, n: usize, options: u32, single: c_int, d_values: *const u8, d_wide_rand: *const u8, seed: *const u8, counter_base: u64, d_choices: *mut u8, d_ring_proofs: *mut u8, d_sum_proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_range_batch_dev(ctx: *mut eg_ctx, range: *const eg_range, transcript_label: *const c_char, n: usize, d_values: *const u64, d_wide_rand: *const u8, seed: *const u8, counter_base: u64, d_cts: *mut u8, d_partials: *mut u8, d_ring_proofs: *mut u8) -> eg_status;
    pub fn eg_ciphertexts_sum_dev(ctx: *mut eg_ctx, n_parts: usize, n_cts: usize, d_parts: *const u8, d_out: *mut u8,
                                  d_bad: *mut u32) -> eg_status;
    pub fn eg_ciphertexts_weighted_sum(ctx: *mut eg_ctx, n: usize, n_cts: u32, item_stride: usize, ct_stride: usize, cts: *const u8,
                                       scalars: *const u8, verdicts: *const u8, out: *mut u8, ok: *mut u8) -> eg_status;
    pub fn eg_ciphertexts_weighted_sum_dev(ctx: *mut eg_ctx, n: usize, n_cts: u32, item_stride: usize, ct_stride: usize, d_cts: *const u8,
                                           d_scalars: *const u8, d_verdicts: *const u8, d_out: *mut u8, d_ok: *mut u8) -> eg_status;
    pub fn eg_ciphertexts_group_sum(ctx: *mut eg_ctx, n: usize, n_cts: u32, item_stride: usize, ct_stride: usize, cts: *const u8,
                                    groups: *const u32, n_groups: u32, verdicts: *const u8, out: *mut u8, ok: *mut u8) -> eg_status;
    pub fn eg_ciphertexts_group_sum_dev(ctx: *mut eg_ctx, n: usize, n_cts: u32, item_stride: usize, ct_stride: usize, d_cts: *const u8,
                                        d_groups: *const u32, n_groups: u32, d_verdicts: *const u8, d_out: *mut u8, d_ok: *mut u8) -> eg_status;

    pub fn eg_base64url_chars(bytes_per_item: usize) -> usize;
    pub fn eg_base64url_decode_batch(ctx: *mut eg_ctx, n: usize, bytes_per_item: usize, text: *const c_char, raw: *mut u8,
                                     ok: *mut u8) -> eg_status;
    pub fn eg_base64url_encode_batch(ctx: *mut eg_ctx, n: usize, bytes_per_item: usize, raw: *const u8, text: *mut c_char) -> eg_status;
    pub fn eg_base64url_decode_batch_dev(ctx: *mut eg_ctx, n: usize, bytes_per_item: usize, d_text: *const c_char,
                                         d_raw: *mut u8, d_ok: *mut u8) -> eg_status;
    pub fn eg_base64url_encode_batch_dev(ctx: *mut eg_ctx, n: usize, bytes_per_item: usize, d_raw: *const u8,
                                         d_text: *mut c_char) -> eg_status;

    pub fn eg_verify_commitment_equiv_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, n: usize, cts: *const u8,
                                            commitments: *const u8, proofs: *const u8, verdicts: *mut u8) -> eg_status;
    pub fn eg_verify_possession_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, keys_per_proof: u32, n: usize,
                                      keys: *const u8, proofs: *const u8, verdicts: *mut u8) -> eg_status;

    pub fn eg_encrypt_batch(ctx: *mut eg_ctx, n: usize, values: *const u64, wide_rand: *const u8, cts: *mut u8) -> eg_status;
    pub fn eg_encrypt_zero_batch(ctx: *mut eg_ctx, n: usize, wide_rand: *const u8, cts: *mut u8, proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_bool_batch(ctx: *mut eg_ctx, n: usize, values: *const u8, wide_rand: *const u8, cts: *mut u8,
                                 proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_choice_batch(ctx: *mut eg_ctx, n: usize, options: u32, single: c_int, values: *const u8,
                                   wide_rand: *const u8, choices: *mut u8, ring_proofs: *mut u8, sum_proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_batch_seeded(ctx: *mut eg_ctx, n: usize, values: *const u64, seed: *const u8, counter_base: u64, cts: *mut u8) -> eg_status;
    pub fn eg_encrypt_zero_batch_seeded(ctx: *mut eg_ctx, n: usize, seed: *const u8, counter_base: u64, cts: *mut u8, proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_bool_batch_seeded(ctx: *mut eg_ctx, n: usize, values: *const u8, seed: *const u8, counter_base: u64, cts: *mut u8, proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_choice_batch_seeded(ctx: *mut eg_ctx, n: usize, options: u32, single: c_int, values: *const u8, seed: *const u8, counter_base: u64, choices: *mut u8, ring_proofs: *mut u8, sum_proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_range_batch_seeded(ctx: *mut eg_ctx, range: *const eg_range, transcript_label: *const c_char, n: usize, values: *const u64, seed: *const u8, counter_base: u64, cts: *mut u8, partials: *mut u8, ring_proofs: *mut u8) -> eg_status;
    pub fn eg_encrypt_qv_batch_seeded(ctx: *mut eg_ctx, params: *const eg_qv_params, n: usize, votes: *const u64, seed: *const u8, counter_base: u64, ballots: *mut u8) -> eg_status;
    pub fn eg_ctx_set_prover_mode(ctx: *mut eg_ctx, constant_time: c_int) -> eg_status;
    pub fn eg_range_prover_draws(range: *const eg_range) -> usize;
    pub fn eg_encrypt_range_batch(ctx: *mut eg_ctx, range: *const eg_range, transcript_label: *const c_char, n: usize,
                                  values: *const u64, wide_rand: *const u8, cts: *mut u8, partials: *mut u8,
                                  ring_proofs: *mut u8) -> eg_status;
    pub fn eg_prove_range_batch(ctx: *mut eg_ctx, range: *const eg_range, transcript_label: *const c_char, n: usize, values: *const u64, ct_randomness: *const u8, wide_rand: *const u8, cts: *mut u8, partials: *mut u8, ring_proofs: *mut u8) -> eg_status;
    pub fn eg_prove_range_batch_seeded(ctx: *mut eg_ctx, range: *const eg_range, transcript_label: *const c_char, n: usize, values: *const u64, ct_randomness: *const u8, seed: *const u8, counter_base: u64, cts: *mut u8, partials: *mut u8, ring_proofs: *mut u8) -> eg_status;
    pub fn eg_qv_prover_draws(params: *const eg_qv_params) -> usize;
    pub fn eg_encrypt_qv_batch(ctx: *mut eg_ctx, params: *const eg_qv_params, n: usize, votes: *const u64,
                               wide_rand: *const u8, ballots: *mut u8) -> eg_status;

    // decryption side (SecretKey::decrypt, ActiveParticipant::decrypt_share, VerifiableDecryption::new)
    pub fn eg_decrypt_batch(ctx: *mut eg_ctx, secret: *const u8, n: usize, cts: *const u8, table: *const eg_dlog_table,
                            elements: *mut u8, values: *mut u64, found: *mut u8) -> eg_status;
    pub fn eg_decrypt_share_batch(ctx: *mut eg_ctx, keyset: *const eg_keyset, index: u32, secret_share: *const u8, n: usize,
                                  cts: *const u8, wide_rand: *const u8, shares: *mut u8, proofs: *mut u8, ok: *mut u8) -> eg_status;
    pub fn eg_decrypt_share_batch_seeded(ctx: *mut eg_ctx, keyset: *const eg_keyset, index: u32, secret_share: *const u8, n: usize,
                                         cts: *const u8, seed: *const u8, counter_base: u64, shares: *mut u8, proofs: *mut u8,
                                         ok: *mut u8) -> eg_status;
    pub fn eg_decrypt_share_batch_dev(ctx: *mut eg_ctx, keyset: *const eg_keyset, index: u32, secret_share: *const u8, n: usize,
                                      d_cts: *const u8, d_wide_rand: *const u8, seed: *const u8, counter_base: u64, d_shares: *mut u8,
                                      d_proofs: *mut u8, d_ok: *mut u8) -> eg_status;
    pub fn eg_prove_decryption_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, secret: *const u8, n: usize, cts: *const u8,
                                     wide_rand: *const u8, dh_elements: *mut u8, proofs: *mut u8, ok: *mut u8) -> eg_status;
    pub fn eg_prove_decryption_batch_seeded(ctx: *mut eg_ctx, transcript_label: *const c_char, secret: *const u8, n: usize,
                                            cts: *const u8, seed: *const u8, counter_base: u64, dh_elements: *mut u8, proofs: *mut u8,
                                            ok: *mut u8) -> eg_status;
    pub fn eg_prove_commitment_equiv_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, n: usize, values: *const u64,
                                           ct_randomness: *const u8, wide_rand: *const u8, cts: *mut u8, commitments: *mut u8,
                                           proofs: *mut u8, blindings: *mut u8) -> eg_status;
    pub fn eg_prove_commitment_equiv_batch_seeded(ctx: *mut eg_ctx, transcript_label: *const c_char, n: usize, values: *const u64,
                                                  ct_randomness: *const u8, seed: *const u8, counter_base: u64, cts: *mut u8,
                                                  commitments: *mut u8, proofs: *mut u8, blindings: *mut u8) -> eg_status;
    pub fn eg_prove_sumsq_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, count: u32, n: usize, cts: *const u8, values: *const u64,
                                randomness: *const u8, sum_cts: *const u8, sum_randomness: *const u8, wide_rand: *const u8,
                                proofs: *mut u8) -> eg_status;
    pub fn eg_prove_sumsq_batch_seeded(ctx: *mut eg_ctx, transcript_label: *const c_char, count: u32, n: usize, cts: *const u8,
                                       values: *const u64, randomness: *const u8, sum_cts: *const u8, sum_randomness: *const u8,
                                       seed: *const u8, counter_base: u64, proofs: *mut u8) -> eg_status;
    pub fn eg_prove_possession_batch(ctx: *mut eg_ctx, transcript_label: *const c_char, keys_per_proof: u32, n: usize, secrets: *const u8,
                                     wide_rand: *const u8, keys: *mut u8, proofs: *mut u8) -> eg_status;
    pub fn eg_prove_possession_batch_seeded(ctx: *mut eg_ctx, transcript_label: *const c_char, keys_per_proof: u32, n: usize,
                                            secrets: *const u8, seed: *const u8, counter_base: u64, keys: *mut u8, proofs: *mut u8)
                                            -> eg_status;

    pub fn eg_last_kernel_stats(ctx: *const eg_ctx, kind: c_int, launches: *mut u64, tasks: *mut u64, ms: *mut f32) -> eg_status;
    pub fn eg_kernel_launch_count(ctx: *const eg_ctx) -> u64;
    pub fn eg_last_timings(ctx: *const eg_ctx, out_ms: *mut f32) -> eg_status;
    pub fn eg_last_commit_stats(ctx: *const eg_ctx, launches: *mut u64, tasks: *mut u64, ms: *mut f32) -> eg_status;
    pub fn eg_selftest_field(ctx: *mut eg_ctx, n: usize, seed: u64, mismatches: *mut u64) -> eg_status;
    pub fn eg_ctx_set_chunk_items(ctx: *mut eg_ctx, items: usize) -> eg_status;
    pub fn eg_ctx_stream(ctx: *const eg_ctx) -> *mut c_void;
}
