// elastic_elgamal_b200.hpp -- header-only C++17 mirror of the reference's API surface for the batch path, over the
// C ABI of eg_b200.h.  Names follow slowli/elastic-elgamal: PublicKey (src/keys/mod.rs:122), Ciphertext
// (src/encryption.rs:96), RingProof (src/proofs/ring.rs:282), LogEqualityProof (src/proofs/log_equality.rs:96),
// EncryptedChoice / ChoiceParams (src/app/choice.rs:276,132).  Objects are the reference's `to_bytes` forms.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "eg_b200.h"

namespace elastic_elgamal_b200 {

struct Error : std::runtime_error {
    eg_status status;
    Error(eg_status s, const std::string &m) : std::runtime_error(m), status(s) {}
};

// per-item outcome, mirroring VerificationError / ChoiceVerificationError / QuadraticVotingError
enum class Verdict : uint8_t {
    Ok = EG_V_OK, Malformed = EG_V_MALFORMED, ChallengeMismatch = EG_V_CHALLENGE_MISMATCH, ChoiceSum = EG_V_CHOICE_SUM,
    ChoiceRange = EG_V_CHOICE_RANGE, QvCreditRange = EG_V_QV_CREDIT_RANGE, QvCreditEquivalence = EG_V_QV_CREDIT_EQUIV,
    QvVariantBase = EG_V_QV_VARIANT_BASE
};

using Element = std::array<uint8_t, 32>;
using Scalar = std::array<uint8_t, 32>;
struct Ciphertext { Element random_element, blinded_element; };                       // to_bytes: R || B
struct LogEqualityProof { Scalar challenge, response; };                              // to_bytes: c || s
struct RingProof { Scalar common_challenge; std::vector<Scalar> ring_responses; };    // to_bytes: e0 || s...
struct PublicKey { Element bytes; };
// src/proofs/commitment.rs:126-135 (serde only in the reference; bytes = struct field order)
struct CommitmentEquivalenceProof { Scalar challenge, randomness_response, value_response, commitment_response; };
// src/proofs/possession.rs:71-76
struct ProofOfPossession { Scalar challenge; std::vector<Scalar> responses; };
// src/proofs/range.rs:446-450 + the ciphertext it speaks about
struct RangeProof { std::vector<Ciphertext> partial_ciphertexts; RingProof inner; };

struct ChoiceParams { PublicKey receiver; uint32_t options_count; bool single; };     // ChoiceParams::{single, multi}
struct EncryptedChoice { std::vector<Ciphertext> choices; RingProof range_proof; LogEqualityProof sum_proof; };

struct ChoiceBatchResult { std::vector<Verdict> verdicts; std::vector<Ciphertext> tally; };
// src/proofs/mul.rs:86-93
struct SumOfSquaresProof { Scalar challenge; std::vector<Scalar> ciphertext_responses; Scalar sum_response; };
// src/app/quadratic_voting.rs:205-217 (CiphertextWithRangeProof = ciphertext + range proof)
struct CiphertextWithRangeProof { Ciphertext ciphertext; RangeProof range_proof; };
struct QuadraticVotingBallot { std::vector<CiphertextWithRangeProof> votes; CiphertextWithRangeProof credit; SumOfSquaresProof credit_equivalence_proof; };
// src/sharing/key_set.rs:19-26
struct PublicKeySet { uint32_t shares, threshold; PublicKey shared_key; std::vector<PublicKey> participant_keys; };
// 32-byte ChaCha20 key + block counter base for the provers that generate their randomness in the kernel (eg_*_batch_seeded)
struct Seed { std::array<uint8_t, 32> key; uint64_t counter_base = 0; };
struct DecryptedValue { bool found; uint64_t value; };       // Option<u64> of DiscreteLogTable::get

class Engine {
  public:
    explicit Engine(int device = 0) {
        eg_status st = eg_ctx_create(device, &ctx_);
        if (st != EG_SUCCESS) throw Error(st, "eg_ctx_create failed: no CUDA device (the engine has no CPU fallback)");
    }
    // one process, several GPUs: batches shard across them and tallies are combined inside the library (eg_ctx_create_multi)
    explicit Engine(const std::vector<int> &devices) {
        eg_status st = eg_ctx_create_multi(devices.data(), (int)devices.size(), &ctx_);
        if (st != EG_SUCCESS) throw Error(st, "eg_ctx_create_multi failed (devices / libnccl.so.2?)");
    }
    ~Engine() {
        for (eg_dlog_table *t : tables_) eg_dlog_table_destroy(t);
        eg_ctx_destroy(ctx_);
    }
    // one process per GPU: rank 0 makes the id, the host distributes it, every rank attaches (collective)
    static std::array<uint8_t, EG_COMM_ID_BYTES> comm_unique_id() {
        std::array<uint8_t, EG_COMM_ID_BYTES> id{};
        eg_status st = eg_comm_unique_id(id.data());
        if (st != EG_SUCCESS) throw Error(st, "eg_comm_unique_id failed (libnccl.so.2?)");
        return id;
    }
    void attach_comm(const std::array<uint8_t, EG_COMM_ID_BYTES> &id, int rank, int world) { check(eg_ctx_attach_comm(ctx_, id.data(), rank, world)); }
    void set_constant_time_provers(bool on) { check(eg_ctx_set_prover_mode(ctx_, on ? 1 : 0)); }
    // tuning knobs (results never depend on them): ring-proof engine 0..3, tallies per call from which share verification
    // builds fixed-base tables for the keys
    void set_ring_engine(int mode) { check(eg_ctx_set_ring_mode(ctx_, mode)); }
    void set_key_table_min(size_t min_tallies) { check(eg_ctx_set_key_table_min(ctx_, min_tallies)); }
    Engine(const Engine &) = delete;
    Engine &operator=(const Engine &) = delete;

    // PublicKey::from_bytes
    void set_receiver(const PublicKey &key) { check(eg_ctx_set_receiver(ctx_, key.bytes.data())); }

    // keys.iter().map(|(ct, proof)| receiver.verify_bool(ct, proof))
    std::vector<Verdict> verify_bool_batch(const std::vector<Ciphertext> &cts, const std::vector<RingProof> &proofs) {
        if (cts.size() != proofs.size()) throw Error(EG_ERR_LEN_MISMATCH, "ciphertexts / proofs size mismatch");
        std::vector<uint8_t> c, p, v(cts.size());
        for (size_t i = 0; i < cts.size(); i++) {
            if (proofs[i].ring_responses.size() != 2) throw Error(EG_ERR_LEN_MISMATCH, "items in all rings");   // ring.rs:310-315
            append(c, cts[i]);
            append(p, proofs[i]);
        }
        check(eg_verify_bool_batch(ctx_, cts.size(), c.data(), p.data(), v.data()));
        return to_verdicts(v);
    }

    // ballots.iter().map(|b| b.verify(&params)) + the tally fold (examples/voting.rs:189-204)
    ChoiceBatchResult verify_batch(const ChoiceParams &params, const std::vector<EncryptedChoice> &ballots) {
        const uint32_t m = params.options_count;
        std::vector<uint8_t> c, r, s, v(ballots.size()), t(64 * (size_t)m);
        for (const auto &b : ballots) {
            if (b.choices.size() != m) throw Error(EG_ERR_LEN_MISMATCH, "number of options in the ballot");        // choice.rs:149-158
            if (b.range_proof.ring_responses.size() != 2 * (size_t)m) throw Error(EG_ERR_LEN_MISMATCH, "items in all rings");
            for (const auto &ct : b.choices) append(c, ct);
            append(r, b.range_proof);
            if (params.single) { s.insert(s.end(), b.sum_proof.challenge.begin(), b.sum_proof.challenge.end());
                                 s.insert(s.end(), b.sum_proof.response.begin(), b.sum_proof.response.end()); }
        }
        check(eg_verify_choice_batch(ctx_, ballots.size(), m, params.single ? 1 : 0, c.data(), r.data(),
                                     params.single ? s.data() : nullptr, v.data(), t.data()));
        ChoiceBatchResult out;
        out.verdicts = to_verdicts(v);
        out.tally.resize(m);
        for (uint32_t k = 0; k < m; k++) {
            std::copy(t.begin() + 64 * k, t.begin() + 64 * k + 32, out.tally[k].random_element.begin());
            std::copy(t.begin() + 64 * k + 32, t.begin() + 64 * k + 64, out.tally[k].blinded_element.begin());
        }
        return out;
    }

    // proofs.iter().map(|(ct, proof)| receiver.verify_range(&range, ct, proof))   (keys/impls.rs:143-151)
    std::vector<Verdict> verify_range_batch(const eg_range &range, const std::vector<Ciphertext> &cts, const std::vector<RangeProof> &proofs,
                                            const std::string &label = "ciphertext_range") {
        if (cts.size() != proofs.size()) throw Error(EG_ERR_LEN_MISMATCH, "ciphertexts / proofs size mismatch");
        size_t total = 0;
        for (uint32_t r = 0; r < range.n_rings; r++) total += range.size[r];
        std::vector<uint8_t> c, pc, r, v(cts.size());
        for (size_t i = 0; i < cts.size(); i++) {
            if (proofs[i].partial_ciphertexts.size() + 1 != range.n_rings) throw Error(EG_ERR_LEN_MISMATCH, "number of rings");  // range.rs:555-559
            if (proofs[i].inner.ring_responses.size() != total) throw Error(EG_ERR_LEN_MISMATCH, "items in all rings");
            append(c, cts[i]);
            for (const auto &ct : proofs[i].partial_ciphertexts) append(pc, ct);
            append(r, proofs[i].inner);
        }
        check(eg_verify_range_batch(ctx_, &range, label.c_str(), cts.size(), c.data(), range.n_rings > 1 ? pc.data() : nullptr, r.data(), v.data()));
        return to_verdicts(v);
    }

    // CommitmentEquivalenceProof::verify over a batch (commitment.rs:198-248); `blinding_base` = H
    void set_blinding_base(const Element &base) { check(eg_ctx_set_blinding_base(ctx_, base.data())); }
    std::vector<Verdict> verify_commitment_equivalence_batch(const std::vector<Ciphertext> &cts, const std::vector<Element> &commitments,
                                                             const std::vector<CommitmentEquivalenceProof> &proofs, const std::string &label) {
        if (cts.size() != proofs.size() || cts.size() != commitments.size()) throw Error(EG_ERR_LEN_MISMATCH, "batch size mismatch");
        std::vector<uint8_t> c, k, p, v(cts.size());
        for (size_t i = 0; i < cts.size(); i++) {
            append(c, cts[i]);
            k.insert(k.end(), commitments[i].begin(), commitments[i].end());
            for (const Scalar *s : {&proofs[i].challenge, &proofs[i].randomness_response, &proofs[i].value_response, &proofs[i].commitment_response})
                p.insert(p.end(), s->begin(), s->end());
        }
        check(eg_verify_commitment_equiv_batch(ctx_, label.c_str(), cts.size(), c.data(), k.data(), p.data(), v.data()));
        return to_verdicts(v);
    }

    // ProofOfPossession::verify over a batch of proofs for `keys_per_proof` keys each (possession.rs:137-163)
    std::vector<Verdict> verify_possession_batch(const std::vector<std::vector<PublicKey>> &keys, const std::vector<ProofOfPossession> &proofs,
                                                 const std::string &label) {
        if (keys.size() != proofs.size()) throw Error(EG_ERR_LEN_MISMATCH, "batch size mismatch");
        if (keys.empty()) return {};
        const size_t kpp = keys[0].size();
        std::vector<uint8_t> k, p, v(keys.size());
        for (size_t i = 0; i < keys.size(); i++) {
            if (keys[i].size() != kpp || proofs[i].responses.size() != kpp) throw Error(EG_ERR_LEN_MISMATCH, "public keys");   // possession.rs:147
            for (const auto &key : keys[i]) k.insert(k.end(), key.bytes.begin(), key.bytes.end());
            p.insert(p.end(), proofs[i].challenge.begin(), proofs[i].challenge.end());
            for (const auto &s : proofs[i].responses) p.insert(p.end(), s.begin(), s.end());
        }
        check(eg_verify_possession_batch(ctx_, label.c_str(), (uint32_t)kpp, keys.size(), k.data(), p.data(), v.data()));
        return to_verdicts(v);
    }

    // ballots.iter().map(|b| b.verify(&params)) + the tally fold (quadratic_voting.rs:291-329)
    // The Ciphertext operators (src/encryption.rs:160-226) over a batch: out[i] = sum_j rows[i][j].first * rows[i][j].second.
    // a + b = {(1, a), (1, b)}; a - b = {(1, a), (l - 1, b)}; -a = {(l - 1, a)}; a * k = {(k, a)}.
    std::vector<Ciphertext> combine_ciphertexts(const std::vector<std::vector<std::pair<Scalar, Ciphertext>>> &rows) {
        const size_t n = rows.size(), terms = n ? rows[0].size() : 1;
        std::vector<uint8_t> s, c, out(n * 64), ok(n);
        for (const auto &row : rows) {
            if (row.size() != terms) throw Error(EG_ERR_INVALID_ARG, "rows must have the same number of terms");
            for (const auto &t : row) s.insert(s.end(), t.first.begin(), t.first.end());
            for (const auto &t : row) append(c, t.second);
        }
        check(eg_ciphertexts_lincomb_batch(ctx_, n, (uint32_t)terms, s.data(), c.data(), out.data(), ok.data()));
        for (size_t i = 0; i < n; i++)
            if (!ok[i]) throw Error(EG_ERR_INVALID_ARG, "malformed element or scalar in a ciphertext combination");
        return to_ciphertexts(out);
    }

    // The weighted tally fold total[j] += items[i][j] * scalars[i] (src/encryption.rs:163,197) over the items whose verdict
    // is 0 (every item when `verdicts` is empty), e.g. the verdicts of verify_choice_batch.  Variable-time in the scalars.
    std::vector<Ciphertext> weighted_sum(const std::vector<std::vector<Ciphertext>> &items, const std::vector<Scalar> &scalars,
                                         const std::vector<uint8_t> &verdicts = {}) {
        const size_t n = items.size(), n_cts = n ? items[0].size() : 1;
        if (scalars.size() != n || (!verdicts.empty() && verdicts.size() != n))
            throw Error(EG_ERR_INVALID_ARG, "one scalar and verdict per item");
        std::vector<uint8_t> s, c, out(n_cts * 64);
        uint8_t ok = 0;
        for (size_t i = 0; i < n; i++) {
            if (items[i].size() != n_cts) throw Error(EG_ERR_INVALID_ARG, "items must have the same number of ciphertexts");
            s.insert(s.end(), scalars[i].begin(), scalars[i].end());
            for (const auto &ct : items[i]) append(c, ct);
        }
        check(eg_ciphertexts_weighted_sum(ctx_, n, (uint32_t)n_cts, 64 * n_cts, 64, c.data(), s.data(),
                                          verdicts.empty() ? nullptr : verdicts.data(), out.data(), &ok));
        if (!ok) throw Error(EG_ERR_INVALID_ARG, "malformed element or scalar in a weighted sum");
        return to_ciphertexts(out);
    }

    ChoiceBatchResult verify_qv_batch(uint32_t options, uint64_t credits, const std::vector<QuadraticVotingBallot> &ballots) {
        eg_qv_params qp;
        check(eg_qv_params_new(options, credits, &qp));
        const size_t size = eg_qv_ballot_size(&qp);
        std::vector<uint8_t> b, v(ballots.size()), t(64 * (size_t)options);
        for (const auto &ballot : ballots) {
            const size_t before = b.size();
            for (const auto &vote : ballot.votes) append(b, vote);
            append(b, ballot.credit);
            append(b, ballot.credit_equivalence_proof);
            if (b.size() - before != size) throw Error(EG_ERR_LEN_MISMATCH, "number of options in the ballot");      // quadratic_voting.rs:292-298
        }
        check(eg_verify_qv_batch(ctx_, &qp, ballots.size(), b.data(), v.data(), t.data()));
        ChoiceBatchResult out;
        out.verdicts = to_verdicts(v);
        out.tally = to_ciphertexts(t);
        return out;
    }

    // proof.verify(cts.iter(), sum_ct, receiver, transcript) over a batch (mul.rs:190-260)
    std::vector<Verdict> verify_sum_of_squares_batch(uint32_t count, const std::vector<Ciphertext> &cts, const std::vector<Ciphertext> &sum_cts,
                                                     const std::vector<SumOfSquaresProof> &proofs, const std::string &label) {
        if (cts.size() != proofs.size() * count || sum_cts.size() != proofs.size()) throw Error(EG_ERR_LEN_MISMATCH, "batch size mismatch");
        std::vector<uint8_t> c, s, p, v(proofs.size());
        for (const auto &ct : cts) append(c, ct);
        for (const auto &ct : sum_cts) append(s, ct);
        for (const auto &proof : proofs) {
            if (proof.ciphertext_responses.size() != 2 * (size_t)count) throw Error(EG_ERR_LEN_MISMATCH, "ciphertext responses");   // mul.rs:198-203
            append(p, proof);
        }
        check(eg_verify_sumsq_batch(ctx_, label.c_str(), count, proofs.size(), c.data(), s.data(), p.data(), v.data()));
        return to_verdicts(v);
    }

    // key_set.verify_share(share, ct, index, proof) for every tally x listed participant (key_set.rs:209-228)
    std::vector<Verdict> verify_shares_batch(const PublicKeySet &ks, const std::vector<uint32_t> &indexes, const std::vector<Ciphertext> &cts,
                                             const std::vector<Element> &shares, const std::vector<LogEqualityProof> &proofs) {
        const size_t n = cts.size(), s = indexes.size();
        if (shares.size() != n * s || proofs.size() != n * s || ks.participant_keys.size() != ks.shares || ks.shares > 64)
            throw Error(EG_ERR_LEN_MISMATCH, "batch size mismatch");
        eg_keyset k{};
        k.shares = ks.shares; k.threshold = ks.threshold;
        std::copy(ks.shared_key.bytes.begin(), ks.shared_key.bytes.end(), k.shared_key);
        for (uint32_t i = 0; i < ks.shares; i++) std::copy(ks.participant_keys[i].bytes.begin(), ks.participant_keys[i].bytes.end(), k.participant_keys[i]);
        std::vector<uint8_t> c, sh, p, v(n * s);
        for (const auto &ct : cts) append(c, ct);
        for (const auto &e : shares) sh.insert(sh.end(), e.begin(), e.end());
        for (const auto &proof : proofs) append(p, proof);
        check(eg_verify_shares_batch(ctx_, &k, n, (uint32_t)s, indexes.data(), c.data(), sh.data(), p.data(), v.data()));
        return to_verdicts(v);
    }

    // candidate.verify(ct, key, proof, transcript) over a batch, one custom key (decryption.rs:189-205)
    std::vector<Verdict> verify_decryption_batch(const PublicKey &key, const std::vector<Ciphertext> &cts, const std::vector<Element> &dh_elements,
                                                 const std::vector<LogEqualityProof> &proofs, const std::string &label) {
        if (dh_elements.size() != cts.size() || proofs.size() != cts.size()) throw Error(EG_ERR_LEN_MISMATCH, "batch size mismatch");
        std::vector<uint8_t> c, d, p, v(cts.size());
        for (const auto &ct : cts) append(c, ct);
        for (const auto &e : dh_elements) d.insert(d.end(), e.begin(), e.end());
        for (const auto &proof : proofs) append(p, proof);
        check(eg_verify_decryption_batch(ctx_, label.c_str(), key.bytes.data(), cts.size(), c.data(), d.data(), p.data(), v.data()));
        return to_verdicts(v);
    }

    // DiscreteLogTable::new(lo..hi) on the device(s); owned by the engine
    eg_dlog_table *dlog_table(uint64_t lo, uint64_t hi) {
        eg_dlog_table *t = nullptr;
        check(eg_dlog_table_create(ctx_, lo, hi, &t));
        tables_.push_back(t);
        return t;
    }

    // DiscreteLogTable::new(lo..hi) by baby-step giant-step (baby_steps values on the device, up to 2^32 giant steps per
    // lookup); owned by the engine
    eg_dlog_table *dlog_table_bsgs(uint64_t lo, uint64_t hi, uint64_t baby_steps) {
        eg_dlog_table *t = nullptr;
        check(eg_dlog_table_create_bsgs(ctx_, lo, hi, baby_steps, &t));
        tables_.push_back(t);
        return t;
    }

    // DiscreteLogTable::get over a batch of elements (encryption.rs:287-297); the identity is found with value 0
    std::vector<DecryptedValue> dlog_lookup_batch(const eg_dlog_table *table, const std::vector<Element> &elements) {
        const size_t n = elements.size();
        std::vector<uint8_t> el, found(n);
        std::vector<uint64_t> values(n);
        for (const auto &e : elements) el.insert(el.end(), e.begin(), e.end());
        check(eg_dlog_lookup_batch(ctx_, table, n, el.data(), values.data(), found.data()));
        std::vector<DecryptedValue> out(n);
        for (size_t i = 0; i < n; i++) out[i] = DecryptedValue{found[i] == 1, values[i]};
        return out;
    }

    // params.combine_shares(..) + decrypt(ct, &table) per tally (sharing/mod.rs:302-325, decryption.rs:138-144)
    std::vector<DecryptedValue> combine_decrypt_batch(const std::vector<uint32_t> &indexes, const std::vector<Ciphertext> &cts,
                                                      const std::vector<Element> &shares, const eg_dlog_table *table) {
        const size_t n = cts.size(), t = indexes.size();
        if (shares.size() != n * t) throw Error(EG_ERR_LEN_MISMATCH, "batch size mismatch");
        std::vector<uint8_t> c, sh, found(n);
        std::vector<uint64_t> values(n);
        for (const auto &ct : cts) append(c, ct);
        for (const auto &e : shares) sh.insert(sh.end(), e.begin(), e.end());
        check(eg_combine_decrypt_batch(ctx_, (uint32_t)t, indexes.data(), n, (uint32_t)t, c.data(), sh.data(), table, values.data(), found.data()));
        std::vector<DecryptedValue> out(n);
        for (size_t i = 0; i < n; i++) out[i] = DecryptedValue{found[i] == 1, values[i]};
        return out;
    }

    // secret.decrypt(ct, &table) over a batch (keys/impls.rs:160-177); table == nullptr: decrypt_to_element only (found = decoded)
    std::vector<DecryptedValue> decrypt_batch(const Scalar &secret, const std::vector<Ciphertext> &cts, const eg_dlog_table *table,
                                              std::vector<Element> *elements = nullptr) {
        const size_t n = cts.size();
        std::vector<uint8_t> c, el(32 * n), found(n);
        std::vector<uint64_t> values(n);
        for (const auto &ct : cts) append(c, ct);
        check(eg_decrypt_batch(ctx_, secret.data(), n, c.data(), table, el.data(), table ? values.data() : nullptr, found.data()));
        if (elements) {
            elements->assign(n, Element{});
            for (size_t i = 0; i < n; i++) std::copy(el.begin() + 32 * i, el.begin() + 32 * (i + 1), (*elements)[i].begin());
        }
        std::vector<DecryptedValue> out(n);
        for (size_t i = 0; i < n; i++) out[i] = DecryptedValue{found[i] == 1, values[i]};
        return out;
    }

    // participant.decrypt_share(ct, rng) over a batch with in-kernel randomness (participant.rs:163-185): shares + proofs
    std::pair<std::vector<Element>, std::vector<LogEqualityProof>> decrypt_share_batch(const PublicKeySet &ks, uint32_t index, const Scalar &secret_share,
                                                                                       const std::vector<Ciphertext> &cts, const Seed &seed) {
        if (ks.participant_keys.size() != ks.shares || ks.shares > 64) throw Error(EG_ERR_LEN_MISMATCH, "key set size mismatch");
        eg_keyset k{};
        k.shares = ks.shares; k.threshold = ks.threshold;
        std::copy(ks.shared_key.bytes.begin(), ks.shared_key.bytes.end(), k.shared_key);
        for (uint32_t i = 0; i < ks.shares; i++) std::copy(ks.participant_keys[i].bytes.begin(), ks.participant_keys[i].bytes.end(), k.participant_keys[i]);
        const size_t n = cts.size();
        std::vector<uint8_t> c, d(32 * n), p(64 * n), ok(n);
        for (const auto &ct : cts) append(c, ct);
        check(eg_decrypt_share_batch_seeded(ctx_, &k, index, secret_share.data(), n, c.data(), seed.key.data(), seed.counter_base, d.data(), p.data(), ok.data()));
        return split_log_eq(d, p);
    }

    // VerifiableDecryption::new(ct, &(secret, [secret]G), &mut Transcript::new(label), rng) over a batch (decryption.rs:89-111)
    std::pair<std::vector<Element>, std::vector<LogEqualityProof>> prove_decryption_batch(const Scalar &secret, const std::vector<Ciphertext> &cts,
                                                                                          const std::string &label, const Seed &seed) {
        const size_t n = cts.size();
        std::vector<uint8_t> c, d(32 * n), p(64 * n), ok(n);
        for (const auto &ct : cts) append(c, ct);
        check(eg_prove_decryption_batch_seeded(ctx_, label.c_str(), secret.data(), n, c.data(), seed.key.data(), seed.counter_base, d.data(), p.data(), ok.data()));
        return split_log_eq(d, p);
    }

    // CommitmentEquivalenceProof::new over a batch of existing ciphertexts of values[i] with randomness ct_randomness[i]
    // (commitment.rs:126-196), in-kernel randomness.  Needs the receiver key and the blinding base; blindings are secret.
    struct CommitmentEquivalence { Ciphertext ciphertext; CommitmentEquivalenceProof proof; Element commitment; Scalar blinding; };
    std::vector<CommitmentEquivalence> prove_commitment_equiv_batch(const std::vector<uint64_t> &values, const std::vector<Scalar> &ct_randomness,
                                                                    const std::string &label, const Seed &seed) {
        const size_t n = values.size();
        if (ct_randomness.size() != n) throw Error(EG_ERR_LEN_MISMATCH, "one randomness per value");
        std::vector<uint8_t> r, c(64 * n), m(32 * n), p(128 * n), b(32 * n);
        for (const auto &s : ct_randomness) r.insert(r.end(), s.begin(), s.end());
        check(eg_prove_commitment_equiv_batch_seeded(ctx_, label.c_str(), n, values.data(), r.data(), seed.key.data(), seed.counter_base, c.data(),
                                                     m.data(), p.data(), b.data()));
        std::vector<CommitmentEquivalence> out(n);
        for (size_t i = 0; i < n; i++) {
            std::copy_n(&c[64 * i], 32, out[i].ciphertext.random_element.begin());
            std::copy_n(&c[64 * i + 32], 32, out[i].ciphertext.blinded_element.begin());
            Scalar *f[4] = {&out[i].proof.challenge, &out[i].proof.randomness_response, &out[i].proof.value_response, &out[i].proof.commitment_response};
            for (int k = 0; k < 4; k++) std::copy_n(&p[128 * i + 32 * k], 32, f[k]->begin());
            std::copy_n(&m[32 * i], 32, out[i].commitment.begin());
            std::copy_n(&b[32 * i], 32, out[i].blinding.begin());
        }
        std::fill(b.begin(), b.end(), 0);
        return out;
    }

    // SumOfSquaresProof::new over a batch (mul.rs:107-181): item i has `count` ciphertexts cts[i*count..] of values with
    // randomness, and the sum ciphertext sum_cts[i] with sum_randomness[i]; in-kernel randomness.
    std::vector<SumOfSquaresProof> prove_sumsq_batch(uint32_t count, const std::vector<Ciphertext> &cts, const std::vector<uint64_t> &values,
                                                     const std::vector<Scalar> &randomness, const std::vector<Ciphertext> &sum_cts,
                                                     const std::vector<Scalar> &sum_randomness, const std::string &label, const Seed &seed) {
        const size_t n = sum_cts.size();
        if (cts.size() != n * count || values.size() != n * count || randomness.size() != n * count || sum_randomness.size() != n)
            throw Error(EG_ERR_LEN_MISMATCH, "count ciphertexts, values and randomness per sum ciphertext");
        std::vector<uint8_t> c, s, r, sr, p(32 * (2 * (size_t)count + 2) * n);
        for (const auto &ct : cts) append(c, ct);
        for (const auto &ct : sum_cts) append(s, ct);
        for (const auto &x : randomness) r.insert(r.end(), x.begin(), x.end());
        for (const auto &x : sum_randomness) sr.insert(sr.end(), x.begin(), x.end());
        check(eg_prove_sumsq_batch_seeded(ctx_, label.c_str(), count, n, c.data(), values.data(), r.data(), s.data(), sr.data(), seed.key.data(),
                                          seed.counter_base, p.data()));
        std::vector<SumOfSquaresProof> out(n);
        const uint8_t *q = p.data();
        for (auto &proof : out) {
            std::copy_n(q, 32, proof.challenge.begin()); q += 32;
            proof.ciphertext_responses.resize(2 * (size_t)count);
            for (auto &x : proof.ciphertext_responses) { std::copy_n(q, 32, x.begin()); q += 32; }
            std::copy_n(q, 32, proof.sum_response.begin()); q += 32;
        }
        return out;
    }

    // Keypair::from(secret) for keys_per_proof secrets per item, then ProofOfPossession::from_keys (possession.rs:93-130);
    // in-kernel randomness.  Returns the public keys (item-major) and the proofs.
    std::pair<std::vector<PublicKey>, std::vector<ProofOfPossession>> prove_possession_batch(uint32_t keys_per_proof, const std::vector<Scalar> &secrets,
                                                                                          const std::string &label, const Seed &seed) {
        const size_t k = keys_per_proof;
        if (k == 0 || secrets.size() % k) throw Error(EG_ERR_LEN_MISMATCH, "keys_per_proof secrets per proof");
        const size_t n = secrets.size() / k;
        std::vector<uint8_t> s, keys(32 * k * n), p(32 * (1 + k) * n);
        for (const auto &x : secrets) s.insert(s.end(), x.begin(), x.end());
        check(eg_prove_possession_batch_seeded(ctx_, label.c_str(), keys_per_proof, n, s.data(), seed.key.data(), seed.counter_base, keys.data(), p.data()));
        std::fill(s.begin(), s.end(), 0);
        std::vector<PublicKey> pks(k * n);
        for (size_t j = 0; j < k * n; j++) std::copy_n(&keys[32 * j], 32, pks[j].bytes.begin());
        std::vector<ProofOfPossession> proofs(n);
        for (size_t i = 0; i < n; i++) {
            const uint8_t *q = &p[32 * (1 + k) * i];
            std::copy_n(q, 32, proofs[i].challenge.begin());
            proofs[i].responses.resize(k);
            for (size_t j = 0; j < k; j++) std::copy_n(q + 32 * (1 + j), 32, proofs[i].responses[j].begin());
        }
        return {pks, proofs};
    }

    // key.encrypt_bool(value, rng) over a batch with in-kernel randomness (keys/impls.rs:77-89)
    std::pair<std::vector<Ciphertext>, std::vector<RingProof>> encrypt_bool_batch(const std::vector<uint8_t> &values, const Seed &seed) {
        const size_t n = values.size();
        std::vector<uint8_t> c(64 * n), p(96 * n);
        check(eg_encrypt_bool_batch_seeded(ctx_, n, values.data(), seed.key.data(), seed.counter_base, c.data(), p.data()));
        std::vector<RingProof> proofs(n);
        for (size_t i = 0; i < n; i++) proofs[i] = ring_proof(p.data() + 96 * i, 2);
        return {to_ciphertexts(c), proofs};
    }

    // EncryptedChoice::single(params, choice, rng) over a batch with in-kernel randomness (choice.rs:288-306)
    std::vector<EncryptedChoice> encrypt_single_choice_batch(uint32_t options, const std::vector<uint32_t> &choices, const Seed &seed) {
        const size_t n = choices.size(), ring = 32 * (1 + 2 * (size_t)options);
        std::vector<uint8_t> values(n * options, 0), c(64 * n * options), r(ring * n), s(64 * n);
        for (size_t i = 0; i < n; i++) {
            if (choices[i] >= options) throw Error(EG_ERR_INVALID_ARG, "invalid choice");       // choice.rs:293-297
            values[i * options + choices[i]] = 1;
        }
        check(eg_encrypt_choice_batch_seeded(ctx_, n, options, 1, values.data(), seed.key.data(), seed.counter_base, c.data(), r.data(), s.data()));
        std::vector<EncryptedChoice> out(n);
        for (size_t i = 0; i < n; i++) {
            std::vector<uint8_t> row(c.begin() + 64 * options * i, c.begin() + 64 * options * (i + 1));
            out[i].choices = to_ciphertexts(row);
            out[i].range_proof = ring_proof(r.data() + ring * i, 2 * options);
            std::copy(s.begin() + 64 * i, s.begin() + 64 * i + 32, out[i].sum_proof.challenge.begin());
            std::copy(s.begin() + 64 * i + 32, s.begin() + 64 * i + 64, out[i].sum_proof.response.begin());
        }
        return out;
    }

    eg_ctx *raw() { return ctx_; }

  private:
    eg_ctx *ctx_ = nullptr;
    std::vector<eg_dlog_table *> tables_;
    static void append(std::vector<uint8_t> &o, const LogEqualityProof &p) {
        o.insert(o.end(), p.challenge.begin(), p.challenge.end());
        o.insert(o.end(), p.response.begin(), p.response.end());
    }
    static void append(std::vector<uint8_t> &o, const CiphertextWithRangeProof &x) {
        append(o, x.ciphertext);
        for (const auto &ct : x.range_proof.partial_ciphertexts) append(o, ct);
        append(o, x.range_proof.inner);
    }
    static void append(std::vector<uint8_t> &o, const SumOfSquaresProof &p) {
        o.insert(o.end(), p.challenge.begin(), p.challenge.end());
        for (const auto &s : p.ciphertext_responses) o.insert(o.end(), s.begin(), s.end());
        o.insert(o.end(), p.sum_response.begin(), p.sum_response.end());
    }
    static std::vector<Ciphertext> to_ciphertexts(const std::vector<uint8_t> &t) {
        std::vector<Ciphertext> out(t.size() / 64);
        for (size_t k = 0; k < out.size(); k++) {
            std::copy(t.begin() + 64 * k, t.begin() + 64 * k + 32, out[k].random_element.begin());
            std::copy(t.begin() + 64 * k + 32, t.begin() + 64 * k + 64, out[k].blinded_element.begin());
        }
        return out;
    }
    static std::pair<std::vector<Element>, std::vector<LogEqualityProof>> split_log_eq(const std::vector<uint8_t> &d, const std::vector<uint8_t> &p) {
        const size_t n = d.size() / 32;
        std::vector<Element> el(n);
        std::vector<LogEqualityProof> pr(n);
        for (size_t i = 0; i < n; i++) {
            std::copy(d.begin() + 32 * i, d.begin() + 32 * (i + 1), el[i].begin());
            std::copy(p.begin() + 64 * i, p.begin() + 64 * i + 32, pr[i].challenge.begin());
            std::copy(p.begin() + 64 * i + 32, p.begin() + 64 * (i + 1), pr[i].response.begin());
        }
        return {el, pr};
    }
    static RingProof ring_proof(const uint8_t *p, size_t responses) {
        RingProof out;
        std::copy(p, p + 32, out.common_challenge.begin());
        out.ring_responses.resize(responses);
        for (size_t k = 0; k < responses; k++) std::copy(p + 32 * (1 + k), p + 32 * (2 + k), out.ring_responses[k].begin());
        return out;
    }
    void check(eg_status st) { if (st != EG_SUCCESS) throw Error(st, eg_last_error(ctx_)); }
    static void append(std::vector<uint8_t> &o, const Ciphertext &ct) {
        o.insert(o.end(), ct.random_element.begin(), ct.random_element.end());
        o.insert(o.end(), ct.blinded_element.begin(), ct.blinded_element.end());
    }
    static void append(std::vector<uint8_t> &o, const RingProof &p) {
        o.insert(o.end(), p.common_challenge.begin(), p.common_challenge.end());
        for (const auto &s : p.ring_responses) o.insert(o.end(), s.begin(), s.end());
    }
    static std::vector<Verdict> to_verdicts(const std::vector<uint8_t> &v) {
        std::vector<Verdict> out(v.size());
        for (size_t i = 0; i < v.size(); i++) out[i] = static_cast<Verdict>(v[i]);
        return out;
    }
};

}  // namespace elastic_elgamal_b200
